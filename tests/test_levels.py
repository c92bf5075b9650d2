"""Level ingest (tiler_slider_b200/levels.py) against the reference's own image parser.

tests/golden/levels_400.txt holds the 400 levels as decoded by the UNMODIFIED reference
(ImageLoader.parse_puzzle_image, dataloader.py:44-133; tests/golden/make_levels.py).  The
screenshots themselves (99 MB of JPEGs) live only in the reference checkout, which is not part of
this repository.  tests/golden/level_images holds six of those levels rendered in the screenshot
layout (tests/golden/make_level_images.py), checked against the same decodings everywhere; the
full 400-screenshot comparison runs where $TS_REFERENCE names the reference checkout."""
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
DATA = os.path.join(os.environ.get("TS_REFERENCE", ""), "data")
GOLD = os.path.join(HERE, "golden", "levels_400.txt")
SAMPLES = os.path.join(HERE, "golden", "level_images")


def _same(got, w, name):
    assert (got.size, got.multiple_colors) == (w.size, w.multiple_colors), name
    assert got.blocked_locations == w.blocked_locations, name
    assert got.initial_locations == w.initial_locations, name
    assert got.target_locations == w.target_locations, name


def test_sample_levels_match_the_reference_decoding():
    from tiler_slider_b200.levels import export_levels, load_level, load_level_image
    from tiler_slider_b200.puzzle import load_puzzle_file, parse_puzzle_file_text
    names = [ln[2:].strip() for ln in open(GOLD) if ln.startswith("# puzzle")]
    want = dict(zip(names, load_puzzle_file(GOLD)))
    files = sorted(os.listdir(SAMPLES))
    assert len(files) == 6
    for f in files:
        _same(load_level_image(os.path.join(SAMPLES, f)), want[os.path.splitext(f)[0]], f)
    p = load_level("puzzle_multi_001", SAMPLES)
    assert p.initial_locations == [(0, 3), (3, 2)] and p.target_locations == [(0, 0), (3, 0)]
    again = parse_puzzle_file_text(export_levels(os.path.join(SAMPLES, f) for f in files))
    for f, a in zip(files, again):
        _same(a, want[os.path.splitext(f)[0]], f)


@pytest.mark.skipif(not os.environ.get("TS_REFERENCE") or not os.path.isdir(DATA),
                    reason="needs $TS_REFERENCE: a checkout of the reference with its data/*.jpg")
def test_every_level_matches_the_reference_parser():
    from tiler_slider_b200.levels import export_levels, load_level, load_level_image
    from tiler_slider_b200.puzzle import load_puzzle_file, parse_puzzle_file_text
    want = load_puzzle_file(GOLD)
    names = sorted(f for f in os.listdir(DATA) if f.endswith(".jpg"))
    assert len(names) == len(want) == 400
    for name, w in zip(names, want):
        _same(load_level_image(os.path.join(DATA, name)), w, name)
    p = load_level("puzzle_multi_001", DATA)
    assert p.initial_locations == [(0, 3), (3, 2)] and p.target_locations == [(0, 0), (3, 0)]
    text = export_levels(os.path.join(DATA, n) for n in names[:5])
    again = parse_puzzle_file_text(text)
    assert [a.initial_locations for a in again] == [w.initial_locations for w in want[:5]]
