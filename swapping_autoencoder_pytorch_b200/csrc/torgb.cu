// ToRGB: the 1x1 style-modulated convolution without demodulation that ends the generator
// (models/networks/stylegan2_layers.py:408-427 -> ModulatedConv2d(in, 3, 1, demodulate=False), :266-325).
//
//   y[n, p, o] = bias[o] + sum_c x[n, p, c] * (s[n, c] * w[o, c]),     o < 3 (stored as 4 channels, the 4th zero)
//
// With 3 output channels this is a bandwidth problem, not a GEMM: 2 * 3 FLOP per 4 input bytes.  The reference multiplies
// the whole activation by the style (one read + one write of the largest tensor of the generator), runs a grouped conv and adds
// the bias (two more passes); the generic implicit-GEMM path of this library needed the modulate pass plus a K = C GEMM with
// N = 4.  Here x is read ONCE: a warp owns a strip of pixels of one sample, lane l holds the 3 x 4 combined weights
// s[n, c] * w[o, c] of its four channels c = 4l + 128j in registers, reads its float4 of every pixel and the three partial
// sums are reduced with shuffles.  Backward, also one pass over x: dx = sum_o dy[o] * s * w (written) and the per-sample
// weight gradient G[n, o, c] = sum_p dy[n, p, o] x[n, p, c] (registers -> one row of partial sums per strip, added in strip order), from which the caller
// forms ds = sum_o G * w and dw = sum_n G * s on [N, 3, C] values.
#include "common.cuh"

namespace sae {

constexpr int TORGB_MAXJ = 8;            // C <= 128 * 8 = 1024 input channels

template <int NJ>
__global__ void __launch_bounds__(256)
torgb_fwd_kernel(const float* __restrict__ x, const float* __restrict__ s, const float* __restrict__ w,
                 const float* __restrict__ bias, float* __restrict__ y, int N, int64_t HW, int C, int strips_per_sample,
                 float wscale, int round_tf32) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t warps_total = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t strip_len = (HW + strips_per_sample - 1) / strips_per_sample;
    const float b0 = bias ? __ldg(bias) : 0.f, b1 = bias ? __ldg(bias + 1) : 0.f, b2 = bias ? __ldg(bias + 2) : 0.f;
    for (int64_t item = warp_global; item < (int64_t)N * strips_per_sample; item += warps_total) {
        const int n = (int)(item / strips_per_sample);
        const int64_t p_begin = (item % strips_per_sample) * strip_len;
        const int64_t p_end = min(p_begin + strip_len, HW);
        float wc[NJ][3][4];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int c = 4 * lane + 128 * j;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float sv = (c + u < C) ? __ldg(s + (int64_t)n * C + c + u) * wscale : 0.f;
#pragma unroll
                for (int o = 0; o < 3; ++o) wc[j][o][u] = (c + u < C) ? sv * __ldg(w + (int64_t)o * C + c + u) : 0.f;
            }
        }
        const float* xn = x + (int64_t)n * HW * C;
        float* yn = y + (int64_t)n * HW * 4;
        // four pixels per trip: their loads are issued back to back before any of them is consumed
        constexpr int UP = 4;
        for (int64_t p0 = p_begin; p0 < p_end; p0 += UP) {
            float4 v[UP][NJ];
#pragma unroll
            for (int u = 0; u < UP; ++u)
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int c = 4 * lane + 128 * j;
                    v[u][j] = (c < C && p0 + u < p_end) ? __ldg(reinterpret_cast<const float4*>(xn + (p0 + u) * C + c))
                                                         : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            float a[UP][3];
#pragma unroll
            for (int u = 0; u < UP; ++u) {
                a[u][0] = a[u][1] = a[u][2] = 0.f;
#pragma unroll
                for (int j = 0; j < NJ; ++j)
#pragma unroll
                    for (int o = 0; o < 3; ++o)
                        a[u][o] += v[u][j].x * wc[j][o][0] + v[u][j].y * wc[j][o][1] + v[u][j].z * wc[j][o][2] + v[u][j].w * wc[j][o][3];
            }
#pragma unroll
            for (int u = 0; u < UP; ++u)
#pragma unroll
                for (int o = 0; o < 3; ++o) a[u][o] = warp_sum(a[u][o]);
            // lane u stores pixel p0 + u
#pragma unroll
            for (int u = 0; u < UP; ++u) {
                if (lane == u && p0 + u < p_end) {
                    float r0 = a[u][0] + b0, r1 = a[u][1] + b1, r2 = a[u][2] + b2;
                    if (round_tf32) { r0 = rna_tf32(r0); r1 = rna_tf32(r1); r2 = rna_tf32(r2); }
                    *reinterpret_cast<float4*>(yn + (p0 + u) * 4) = make_float4(r0, r1, r2, 0.f);
                }
            }
        }
    }
}

template <int NJ>
__global__ void __launch_bounds__(256)
torgb_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ s, const float* __restrict__ w,
                 float* __restrict__ dx, float* __restrict__ gw, int N, int64_t HW, int W_img, int C, int strips_per_sample,
                 float wscale, int64_t ds_n, int64_t ds_c, int64_t ds_h, int64_t ds_w, int round_tf32) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t warps_total = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t strip_len = (HW + strips_per_sample - 1) / strips_per_sample;
    for (int64_t item = warp_global; item < (int64_t)N * strips_per_sample; item += warps_total) {
        const int n = (int)(item / strips_per_sample);
        const int64_t p_begin = (item % strips_per_sample) * strip_len;
        const int64_t p_end = min(p_begin + strip_len, HW);
        float wc[NJ][3][4], g[NJ][3][4];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int c = 4 * lane + 128 * j;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float sv = (c + u < C) ? __ldg(s + (int64_t)n * C + c + u) * wscale : 0.f;
#pragma unroll
                for (int o = 0; o < 3; ++o) {
                    wc[j][o][u] = (c + u < C) ? sv * __ldg(w + (int64_t)o * C + c + u) : 0.f;
                    g[j][o][u] = 0.f;
                }
            }
        }
        const float* xn = x + (int64_t)n * HW * C;
        float* dxn = dx ? dx + (int64_t)n * HW * C : nullptr;
        const float* dyn = dy + (int64_t)n * ds_n;
        for (int64_t p = p_begin; p < p_end; ++p) {
            const int64_t ph = p / W_img, pw = p - ph * W_img;
            const float* d = dyn + ph * ds_h + pw * ds_w;
            const float d0 = __ldg(d), d1 = __ldg(d + ds_c), d2 = __ldg(d + 2 * ds_c);
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int c = 4 * lane + 128 * j;
                if (c < C) {
                    if (gw) {
                        const float4 v = ldg_stream(reinterpret_cast<const float4*>(xn + p * C + c));
                        g[j][0][0] += d0 * v.x; g[j][0][1] += d0 * v.y; g[j][0][2] += d0 * v.z; g[j][0][3] += d0 * v.w;
                        g[j][1][0] += d1 * v.x; g[j][1][1] += d1 * v.y; g[j][1][2] += d1 * v.z; g[j][1][3] += d1 * v.w;
                        g[j][2][0] += d2 * v.x; g[j][2][1] += d2 * v.y; g[j][2][2] += d2 * v.z; g[j][2][3] += d2 * v.w;
                    }
                    if (dxn) {
                        float4 o;
                        o.x = d0 * wc[j][0][0] + d1 * wc[j][1][0] + d2 * wc[j][2][0];
                        o.y = d0 * wc[j][0][1] + d1 * wc[j][1][1] + d2 * wc[j][2][1];
                        o.z = d0 * wc[j][0][2] + d1 * wc[j][1][2] + d2 * wc[j][2][2];
                        o.w = d0 * wc[j][0][3] + d1 * wc[j][1][3] + d2 * wc[j][2][3];
                        if (round_tf32) { o.x = rna_tf32(o.x); o.y = rna_tf32(o.y); o.z = rna_tf32(o.z); o.w = rna_tf32(o.w); }
                        *reinterpret_cast<float4*>(dxn + p * C + c) = o;
                    }
                }
            }
        }
        if (gw) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int c = 4 * lane + 128 * j;
#pragma unroll
                for (int o = 0; o < 3; ++o)
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (c + u < C) gw[(((item % strips_per_sample) * N + n) * 3 + o) * C + c + u] = g[j][o][u];
            }
        }
    }
}

static int torgb_strips(int N, int64_t HW) {
    // enough warps to fill the machine (8 warps x 8 blocks per SM), strips of at least 64 pixels
    int64_t want = ((int64_t)sm_count() * 64 + N - 1) / (N > 0 ? N : 1);
    int64_t cap = HW / 64 > 0 ? HW / 64 : 1;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return (int)want;
}

}  // namespace sae

using namespace sae;

extern "C" int sae_torgb_forward(const float* x, const float* s, const float* w, const float* bias, float* y,
                                 int N, int H, int W, int C, float wscale, int round_tf32, void* stream) {
    if (N == 0) return SAE_OK;
    if (!x || !s || !w || !y || N < 0 || H <= 0 || W <= 0) return fail(SAE_E_INVALID, "torgb_forward: bad arguments");
    if (C <= 0 || C % 4 != 0 || C > 128 * TORGB_MAXJ) return fail(SAE_E_UNSUPPORTED, "torgb_forward: C must be a multiple of 4, <= %d", 128 * TORGB_MAXJ);
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) return fail(SAE_E_INVALID, "torgb_forward: unaligned pointer");
    const int64_t HW = (int64_t)H * W;
    const int strips = torgb_strips(N, HW);
    const int64_t warps = (int64_t)N * strips;
    int64_t blocks = (warps + 7) / 8;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    const int nj = (C + 127) / 128;
    cudaStream_t st = (cudaStream_t)stream;
#define SAE_TORGB_FWD(NJ) torgb_fwd_kernel<NJ><<<(unsigned)blocks, 256, 0, st>>>(x, s, w, bias, y, N, HW, C, strips, wscale, round_tf32)
    switch (nj) {
        case 1: SAE_TORGB_FWD(1); break;
        case 2: SAE_TORGB_FWD(2); break;
        case 3: case 4: SAE_TORGB_FWD(4); break;
        default: SAE_TORGB_FWD(8); break;
    }
#undef SAE_TORGB_FWD
    return check_launch("torgb_forward");
}

extern "C" int sae_torgb_backward(const float* dy, const float* x, const float* s, const float* w, float* dx, float* gw,
                                  int N, int H, int W, int C, float wscale,
                                  int64_t ds_n, int64_t ds_c, int64_t ds_h, int64_t ds_w, int round_tf32, void* stream) {
    if (N == 0) return SAE_OK;
    if (!dy || !x || !s || !w || (!dx && !gw) || N < 0 || H <= 0 || W <= 0) return fail(SAE_E_INVALID, "torgb_backward: bad arguments");
    if (C <= 0 || C % 4 != 0 || C > 128 * TORGB_MAXJ) return fail(SAE_E_UNSUPPORTED, "torgb_backward: C must be a multiple of 4, <= %d", 128 * TORGB_MAXJ);
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx)) & 15) return fail(SAE_E_INVALID, "torgb_backward: unaligned pointer");
    const int64_t HW = (int64_t)H * W;
    const int strips = torgb_strips(N, HW);
    const int64_t warps = (int64_t)N * strips;
    int64_t blocks = (warps + 7) / 8;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    const int nj = (C + 127) / 128;
    cudaStream_t st = (cudaStream_t)stream;
    // gw: one row of partial sums per strip, [strip][N][3][C], added in strip order after the kernel
    float* part = nullptr;
    if (gw) {
        part = det_workspace(det_reduce_floats((int64_t)N * 3 * C, strips));
        if (!part) return SAE_E_CUDA;
    }
#define SAE_TORGB_BWD(NJ) torgb_bwd_kernel<NJ><<<(unsigned)blocks, 256, 0, st>>>(dy, x, s, w, dx, part, N, HW, W, C, strips, wscale, ds_n, ds_c, ds_h, ds_w, round_tf32)
    switch (nj) {
        case 1: SAE_TORGB_BWD(1); break;
        case 2: SAE_TORGB_BWD(2); break;
        case 3: case 4: SAE_TORGB_BWD(4); break;
        default: SAE_TORGB_BWD(8); break;
    }
#undef SAE_TORGB_BWD
    int rc = check_launch("torgb_backward");
    if (rc || !gw) return rc;
    return det_reduce(gw, part, (int64_t)N * 3 * C, strips, st);
}
