"""Render sample levels of levels_400.txt as game screenshots for tests/test_levels.py:
    python tests/golden/make_level_images.py
The reference's own 400 screenshots are not part of this repository.  These stand in for them:
1080x2340 images in the layout tiler_slider_b200/levels.py reads (dataloader.py:8-133 of the
reference): the board in rows 665:1710 on the background colour, cells in the empty-cell colour
separated by background lines, a tile as a coloured ring, a target as a coloured dot, a blocked
cell filled, and in multi-colour levels tile k and target k in the same colour.  Output:
tests/golden/level_images/<name>.png (lossless, a few KB each), except puzzle_multi_001 as a
JPEG (lossy, like the game's screenshots; `load_level` looks levels up by <name>.jpg).
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tiler_slider_b200.levels import BACKGROUND_RGB, EMPTY_CELL_RGB  # noqa: E402
from tiler_slider_b200.puzzle import load_puzzle_file  # noqa: E402

SAMPLE = ["puzzle_multi_001", "puzzle_single_001", "puzzle_single_051", "puzzle_multi_061",
          "puzzle_single_151", "puzzle_multi_111"]
JPEG_LEVEL = "puzzle_multi_001"
WIDTH, HEIGHT = 1080, 2340
BOARD_TOP, BOARD_SIDE = 700, 960           # inside the parser's crop (rows 665:1710, cols 15:-15)
GAP = 12                                   # background line between cells, pixels
BLOCKED_RGB = (70, 70, 90)
SINGLE_RGB = (250, 150, 40)
MULTI_RGB = [(230, 60, 60), (240, 210, 40), (140, 80, 210)]


def names():
    return [ln[2:].strip() for ln in open(os.path.join(HERE, "levels_400.txt")) if ln.startswith("# puzzle")]


def render(p) -> np.ndarray:
    img = np.empty((HEIGHT, WIDTH, 3), np.uint8)
    img[:] = BACKGROUND_RGB
    S = p.size
    cell = (BOARD_SIDE - (S + 1) * GAP) // S
    x0 = (WIDTH - (S * cell + (S + 1) * GAP)) // 2

    def box(r, c):
        y, x = BOARD_TOP + GAP + r * (cell + GAP), x0 + GAP + c * (cell + GAP)
        return img[y:y + cell, x:x + cell]

    for r in range(S):
        for c in range(S):
            box(r, c)[:] = EMPTY_CELL_RGB
    for r, c in p.blocked_locations:
        box(r, c)[:] = BLOCKED_RGB
    half = cell // 2
    for k, ((tr, tc), (gr, gc)) in enumerate(zip(p.initial_locations, p.target_locations)):
        rgb = MULTI_RGB[k] if p.multiple_colors else SINGLE_RGB
        t = box(tr, tc)
        t[:] = rgb                                                  # ring: coloured cell, empty centre
        cv2.circle(t, (half, half), int(0.25 * cell), tuple(int(v) for v in EMPTY_CELL_RGB), -1)
        cv2.circle(box(gr, gc), (half, half), int(0.2 * cell), rgb, -1)   # dot
    return img


def main():
    levels = dict(zip(names(), load_puzzle_file(os.path.join(HERE, "levels_400.txt"))))
    out = os.path.join(HERE, "level_images")
    os.makedirs(out, exist_ok=True)
    for name in SAMPLE:
        bgr = cv2.cvtColor(render(levels[name]), cv2.COLOR_RGB2BGR)
        if name == JPEG_LEVEL:
            cv2.imwrite(os.path.join(out, f"{name}.jpg"), bgr, [cv2.IMWRITE_JPEG_QUALITY, 75])
        else:
            cv2.imwrite(os.path.join(out, f"{name}.png"), bgr, [cv2.IMWRITE_PNG_COMPRESSION, 9])
    print(len(SAMPLE), "images in", out)


if __name__ == "__main__":
    main()
