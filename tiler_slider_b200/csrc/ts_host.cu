// ts_host.cu -- ts_step_host: the step through HOST buffers, as a host-side driver of the
// reference's env.step() loop (explainrl/environment/environment.py:100-143) would call it.
//
// The env range is cut into chunks; chunk c runs on stream c % n_streams as
//   H2D actions  ->  ts_step on that sub-range  ->  D2H reward, done
// so the PCIe uploads, the kernel and the downloads of neighbouring chunks overlap
// (H2D and D2H use separate copy engines).  The call returns after all streams drained.
#include <cstdio>
#include <vector>
#include "ts_common.cuh"
#include "../../include/tiler_slider.h"

struct ts_host_ctx {
    std::vector<cudaStream_t> streams;
};

extern "C" {

int ts_host_ctx_create(ts_host_ctx** out, int n_streams) {
    if (!out || n_streams < 1 || n_streams > 16) return TS_E_BAD_ARGUMENT;
    ts_host_ctx* c = new ts_host_ctx();
    for (int i = 0; i < n_streams; ++i) {
        cudaStream_t s;
        cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            for (cudaStream_t t : c->streams) cudaStreamDestroy(t);
            delete c;
            return (int)e;
        }
        c->streams.push_back(s);
    }
    *out = c;
    return 0;
}

int ts_host_ctx_destroy(ts_host_ctx* ctx) {
    if (!ctx) return 0;
    for (cudaStream_t s : ctx->streams) cudaStreamDestroy(s);
    delete ctx;
    return 0;
}

int ts_step_host(ts_host_ctx* ctx, const ts_step_args* a, const uint8_t* h_actions, float* h_reward,
                 uint8_t* h_done, uint8_t* h_flags, int64_t chunk_envs) {
    if (!ctx || !a || !h_actions) return TS_E_NULL_POINTER;
    if (!h_flags && (!h_reward || !h_done)) return TS_E_NULL_POINTER;   // need reward+done, or the flag byte
    if (!a->d_actions || !a->d_reward || !a->d_done) return TS_E_NULL_POINTER;
    if (h_flags && !a->d_flags) return TS_E_NULL_POINTER;
    if (chunk_envs <= 0 || chunk_envs % ts::CAP_ALIGN != 0) return TS_E_BAD_ARGUMENT;
    const int ns = (int)ctx->streams.size();
    int rc = 0;
    int c = 0;
    for (int64_t off = 0; off < a->n_envs && rc == 0; off += chunk_envs, ++c) {
        const int64_t n = (a->n_envs - off < chunk_envs) ? a->n_envs - off : chunk_envs;
        const int64_t e0 = a->first_env + off;
        cudaStream_t s = ctx->streams[c % ns];
        cudaError_t e = cudaMemcpyAsync(const_cast<uint8_t*>(a->d_actions) + e0, h_actions + off, (size_t)n,
                                        cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) { rc = (int)e; break; }
        ts_step_args sub = *a;
        sub.first_env = e0;
        sub.n_envs = n;
        rc = ts_step(&sub, s);
        if (rc) break;
        e = cudaSuccess;
        if (h_reward) e = cudaMemcpyAsync(h_reward + off, a->d_reward + e0, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && h_done)
            e = cudaMemcpyAsync(h_done + off, a->d_done + e0, (size_t)n, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && h_flags)
            e = cudaMemcpyAsync(h_flags + off, a->d_flags + e0, (size_t)n, cudaMemcpyDeviceToHost, s);
        if (e != cudaSuccess) rc = (int)e;
    }
    for (cudaStream_t s : ctx->streams) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess && rc == 0) rc = (int)e;
    }
    return rc;
}

}  // extern "C"
