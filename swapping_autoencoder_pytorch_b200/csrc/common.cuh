// Shared helpers for the sm_100a kernels behind include/sae_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/sae_b200.h"

namespace sae {

extern thread_local char g_err[512];
extern std::atomic<int64_t> g_launches;

inline int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(SAE_E_CUDA, "%s: launch failed: %s", what, cudaGetErrorString(e));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SAE_OK;
}

#define SAE_CUDA_TRY(expr)                                                                   \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess)                                                               \
            return ::sae::fail(SAE_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,      \
                               cudaGetErrorString(_e));                                      \
    } while (0)

// Device properties are queried once per process (device 0's SM count is representative: one
// process drives one GPU in this design).
int sm_count();

// Deterministic cross-block reductions.  Float atomics add in whatever order the blocks happen to finish, so the last bits
// of a reduced gradient — and, through the optimiser, every later training step — would change from run to run.  Instead,
// every block writes its partial sums to its own slice of a workspace with plain stores, and det_reduce adds the slices
// in index order.
//
// det_workspace: a device buffer of at least nfloats floats, library-owned and grow-only.  A buffer is never freed once
// handed out, because captured CUDA graphs keep its address; all users run in stream order, one after the other.
// Returns nullptr (and sets the error text) when the allocation fails.
float* det_workspace(size_t nfloats);
// out[c] += sum over b = 0 .. parts-1 (in that order) of ws[b * n + c], for c < n; columns c < n_a go to a[c] (skipped if
// a is null), the rest to b[c - n_a] (skipped if b is null).  ws must come from det_workspace(det_reduce_floats(n, parts)):
// the reduction uses the space behind the parts * n partials.
size_t det_reduce_floats(int64_t n, int parts);
int det_reduce(float* a, int64_t n_a, float* b, const float* ws, int64_t n, int parts, cudaStream_t st);
inline int det_reduce(float* out, const float* ws, int64_t n, int parts, cudaStream_t st) {
    return det_reduce(out, n, nullptr, ws, n, parts, st);
}

__device__ __forceinline__ float rna_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// Epilogue shared by the conv kernels (see sae_conv_epilogue in the header).
struct EpiParams {
    const float* bias;
    const float* noise;
    const float* residual;
    float nw;          // resolved on device from noise_weight pointer
    const float* noise_weight;
    float alpha, gain, res_scale;
    int act, round_tf32;
    uint32_t* act_mask;   // optional: sign bits of the activation output, 1 bit per element (see sae_conv_epilogue)
};

inline EpiParams make_epi(const sae_conv_epilogue* e) {
    EpiParams p;
    p.bias = nullptr; p.noise = nullptr; p.residual = nullptr; p.noise_weight = nullptr;
    p.nw = 0.f; p.alpha = 0.2f; p.gain = 1.f; p.res_scale = 1.f; p.act = 1; p.round_tf32 = 0; p.act_mask = nullptr;
    if (e) {
        p.bias = e->bias; p.noise = e->noise; p.noise_weight = e->noise_weight;
        p.residual = e->residual; p.alpha = e->alpha; p.gain = e->gain;
        p.res_scale = e->res_scale; p.act = e->act; p.round_tf32 = e->round_tf32; p.act_mask = e->act_mask;
    }
    return p;
}

__device__ __forceinline__ float apply_epi(const EpiParams& e, float v, int64_t pixel, int col, int64_t ldc) {
    if (e.bias) v += __ldg(e.bias + col);
    if (e.noise) v += __ldg(e.noise_weight) * __ldg(e.noise + pixel);
    if (e.act == 3) v = (v > 0.f ? v : v * e.alpha);
    v *= e.gain;
    if (e.residual) v = (v + __ldg(e.residual + pixel * ldc + col)) * e.res_scale;
    if (e.round_tf32) v = rna_tf32(v);
    return v;
}

}  // namespace sae
