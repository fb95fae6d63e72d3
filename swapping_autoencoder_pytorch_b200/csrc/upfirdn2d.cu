// upfirdn2d on NHWC fp32 — replaces models/networks/stylegan2_op/upfirdn2d_kernel.cu:52-137 of the
// reference.  HBM-bound: algorithmic traffic 4*(N_in + N_out) bytes (SURVEY.md §8(d)).
//
// Design (B200): channels are the innermost (minor) dimension, so one warp reads 32 consecutive
// float4 = 512 contiguous bytes per tap and writes 512 contiguous bytes per output pixel; the
// (up to kh*kw) tap re-reads of a neighbourhood are served by L1/L2 (a 4x4 FIR touches each input
// line 16 times within a few hundred cycles from neighbouring warps of the same CTA).  Taps live in
// shared memory, already flipped, so the inner loop is a plain correlation.  A column-strip variant
// keeps a rolling kh x kw register window so each input element is loaded kw (not kh*kw) times.
#include "common.cuh"
#include "tc_common.cuh"

namespace sae {

struct FirParams {
    int64_t major;
    int in_h, in_w, minor;
    int kh, kw;
    int up_x, up_y, down_x, down_y;
    int pad_x0, pad_y0;
    int out_h, out_w;
    int round_tf32;
};

constexpr int kMaxTaps = 32 * 32;

__device__ __forceinline__ int floordiv(int a, int b) {
    int q = a / b;
    return (q * b > a) ? q - 1 : q;
}

// Generic kernel: one thread per VEC output channels of one output pixel.
template <int VEC>
__global__ void __launch_bounds__(256)
fir_generic_kernel(const float* __restrict__ x, const float* __restrict__ k, float* __restrict__ out, FirParams p) {
    __shared__ float sk[kMaxTaps];
    const int ntaps = p.kh * p.kw;
    for (int i = threadIdx.x; i < ntaps; i += blockDim.x) {
        int ky = i / p.kw, kx = i - ky * p.kw;
        sk[i] = k[(p.kh - 1 - ky) * p.kw + (p.kw - 1 - kx)];   // flipped: true convolution
    }
    __syncthreads();

    const int cv = p.minor / VEC;
    const int64_t total = p.major * (int64_t)p.out_h * p.out_w * cv;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int c = (int)(idx % cv);
        int64_t pix = idx / cv;
        int ox = (int)(pix % p.out_w);
        int64_t t = pix / p.out_w;
        int oy = (int)(t % p.out_h);
        int64_t n = t / p.out_h;

        // position of tap (0,0) in zero-upsampled, unpadded coordinates
        const int uy0 = oy * p.down_y - p.pad_y0;
        const int ux0 = ox * p.down_x - p.pad_x0;
        float acc[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[v] = 0.f;

        const float* xn = x + n * (int64_t)p.in_h * p.in_w * p.minor + (int64_t)c * VEC;
        for (int ky = 0; ky < p.kh; ++ky) {
            int uy = uy0 + ky;
            if (uy < 0) continue;
            int iy = uy / p.up_y;
            if (iy * p.up_y != uy || iy >= p.in_h) continue;
            for (int kx = 0; kx < p.kw; ++kx) {
                int ux = ux0 + kx;
                if (ux < 0) continue;
                int ix = ux / p.up_x;
                if (ix * p.up_x != ux || ix >= p.in_w) continue;
                float w = sk[ky * p.kw + kx];
                const float* src = xn + ((int64_t)iy * p.in_w + ix) * p.minor;
                if (VEC == 4) {
                    float4 v = __ldg(reinterpret_cast<const float4*>(src));
                    acc[0] = fmaf(v.x, w, acc[0]);
                    acc[1 % VEC] = fmaf(v.y, w, acc[1 % VEC]);
                    acc[2 % VEC] = fmaf(v.z, w, acc[2 % VEC]);
                    acc[3 % VEC] = fmaf(v.w, w, acc[3 % VEC]);
                } else {
                    acc[0] = fmaf(__ldg(src), w, acc[0]);
                }
            }
        }
        float* dst = out + pix * p.minor + (int64_t)c * VEC;
        if (p.round_tf32) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) acc[v] = rna_tf32(acc[v]);
        }
        if (VEC == 4) {
            *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1 % VEC], acc[2 % VEC], acc[3 % VEC]);
        } else {
            dst[0] = acc[0];
        }
    }
}

// Column-strip kernel for the training hot path (up = down = 1, kh,kw <= 4, minor % 4 == 0):
// a thread owns (n, ox, c4) and walks ROWS output rows downwards keeping the last KH input rows x KW
// columns in registers, so every input float4 is loaded KW times instead of KH*KW times.
template <int KH, int KW, int ROWS>
__global__ void __launch_bounds__(256)
fir_strip_kernel(const float* __restrict__ x, const float* __restrict__ k, float* __restrict__ out, FirParams p) {
    __shared__ float sk[KH * KW];
    if (threadIdx.x < KH * KW) {
        int ky = threadIdx.x / KW, kx = threadIdx.x - ky * KW;
        sk[threadIdx.x] = k[(KH - 1 - ky) * KW + (KW - 1 - kx)];
    }
    __syncthreads();
    float w[KH][KW];
#pragma unroll
    for (int a = 0; a < KH; ++a)
#pragma unroll
        for (int b = 0; b < KW; ++b) w[a][b] = sk[a * KW + b];

    const int cv = p.minor >> 2;
    const int strips = (p.out_h + ROWS - 1) / ROWS;
    const int64_t total = p.major * (int64_t)strips * p.out_w * cv;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        int c = (int)(idx % cv);
        int64_t t = idx / cv;
        int ox = (int)(t % p.out_w);
        t /= p.out_w;
        int strip = (int)(t % strips);
        int64_t n = t / strips;

        const int oy0 = strip * ROWS;
        const int ix0 = ox - p.pad_x0;
        const float* xn = x + n * (int64_t)p.in_h * p.in_w * p.minor + (int64_t)c * 4;
        float4 win[KH][KW];

        auto load_row = [&](int iy, float4 (&row)[KW]) {
            const bool yok = (iy >= 0) && (iy < p.in_h);
#pragma unroll
            for (int b = 0; b < KW; ++b) {
                int ix = ix0 + b;
                if (yok && ix >= 0 && ix < p.in_w)
                    row[b] = __ldg(reinterpret_cast<const float4*>(xn + ((int64_t)iy * p.in_w + ix) * p.minor));
                else
                    row[b] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        // prime the window with the first KH-1 rows
#pragma unroll
        for (int a = 0; a < KH - 1; ++a) load_row(oy0 - p.pad_y0 + a, win[a]);

#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
            const int oy = oy0 + r;
            if (oy >= p.out_h) break;
            load_row(oy - p.pad_y0 + KH - 1, win[KH - 1]);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int a = 0; a < KH; ++a)
#pragma unroll
                for (int b = 0; b < KW; ++b) {
                    acc.x = fmaf(win[a][b].x, w[a][b], acc.x);
                    acc.y = fmaf(win[a][b].y, w[a][b], acc.y);
                    acc.z = fmaf(win[a][b].z, w[a][b], acc.z);
                    acc.w = fmaf(win[a][b].w, w[a][b], acc.w);
                }
            float* dst = out + ((n * p.out_h + oy) * (int64_t)p.out_w + ox) * p.minor + (int64_t)c * 4;
            if (p.round_tf32) { acc.x = rna_tf32(acc.x); acc.y = rna_tf32(acc.y); acc.z = rna_tf32(acc.z); acc.w = rna_tf32(acc.w); }
            *reinterpret_cast<float4*>(dst) = acc;
            // slide the window up by one row
#pragma unroll
            for (int a = 0; a < KH - 1; ++a)
#pragma unroll
                for (int b = 0; b < KW; ++b) win[a][b] = win[a + 1][b];
        }
    }
}

// Separable variant of the strip kernel (every FIR of the networks is an outer product of 1-D taps): the horizontal
// pass runs on the KW loads of the incoming row, the vertical pass on a rolling window of KH already-filtered rows —
// KH float4 of state instead of KH*KW, i.e. ~45 registers instead of 122 and 4-5x the resident warps to hide HBM
// latency.  Taps arrive by value (host arrays), already flipped.
struct SepTaps { float y[8]; float x[8]; };

template <int KH, int KW, int ROWS, int DOWN>
__global__ void __launch_bounds__(256)
fir_sep_strip_kernel(const float* __restrict__ x, float* __restrict__ out, FirParams p, SepTaps taps) {
    const int cv = p.minor >> 2;
    const int strips = (p.out_h + ROWS - 1) / ROWS;
    const uint32_t total = (uint32_t)(p.major * strips * p.out_w * cv);      // host guarantees < 2^32
    for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const uint32_t c = idx % cv;
        uint32_t t = idx / cv;
        const int ox = (int)(t % p.out_w);
        t /= p.out_w;
        const int strip = (int)(t % strips);
        const int64_t n = t / strips;
        const int oy0 = strip * ROWS;
        const int ix0 = ox * DOWN - p.pad_x0;
        const float* xn = x + n * (int64_t)p.in_h * p.in_w * p.minor + (int64_t)c * 4;
        float4 win[KH];

        auto hrow = [&](int iy) -> float4 {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            if (iy < 0 || iy >= p.in_h) return a;
            const float* row = xn + (int64_t)iy * p.in_w * p.minor;
#pragma unroll
            for (int b = 0; b < KW; ++b) {
                const int ix = ix0 + b;
                if (ix >= 0 && ix < p.in_w) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(row + (int64_t)ix * p.minor));
                    a.x = fmaf(v.x, taps.x[b], a.x); a.y = fmaf(v.y, taps.x[b], a.y);
                    a.z = fmaf(v.z, taps.x[b], a.z); a.w = fmaf(v.w, taps.x[b], a.w);
                }
            }
            return a;
        };
        // window rows a = 0..KH-1 hold input rows oy*DOWN - pad + a; each output advances the window by DOWN rows
        constexpr int KEEP = KH > DOWN ? KH - DOWN : 0;
#pragma unroll
        for (int a = 0; a < KEEP; ++a) win[a] = hrow(oy0 * DOWN - p.pad_y0 + a);
#pragma unroll 4
        for (int r = 0; r < ROWS; ++r) {
            const int oy = oy0 + r;
            if (oy >= p.out_h) break;
#pragma unroll
            for (int a = KEEP; a < KH; ++a) win[a] = hrow(oy * DOWN - p.pad_y0 + a);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int a = 0; a < KH; ++a) {
                acc.x = fmaf(win[a].x, taps.y[a], acc.x); acc.y = fmaf(win[a].y, taps.y[a], acc.y);
                acc.z = fmaf(win[a].z, taps.y[a], acc.z); acc.w = fmaf(win[a].w, taps.y[a], acc.w);
            }
            if (p.round_tf32) { acc.x = rna_tf32(acc.x); acc.y = rna_tf32(acc.y); acc.z = rna_tf32(acc.z); acc.w = rna_tf32(acc.w); }
            float* dst = out + ((n * p.out_h + oy) * (int64_t)p.out_w + ox) * p.minor + (int64_t)c * 4;
            *reinterpret_cast<float4*>(dst) = acc;
#pragma unroll
            for (int a = 0; a < KEEP; ++a) win[a] = win[a + DOWN];
        }
    }
}

// TMA-staged separable FIR (up = down = 1, 32-channel blocks): one CTA per 16 x 16 output pixels x 32 channels.  A single
// 4-D bulk tensor load brings the (16+KW-1) x (16+KH-1) pixel window into shared memory — out-of-range rows / columns
// arrive as zeros, which is exactly upfirdn2d's zero padding — so the whole window is in flight with one instruction and
// the threads only read shared memory (each input byte leaves HBM once; the halo is served by L2).  Four CTAs share an SM
// (46 KB each), so loads of three tiles overlap the arithmetic of a fourth.
constexpr int FT_W = 16, FT_H = 16;

// MASK variant (sae_fir_act_backward): the FIR result is the gradient arriving at a fused bias + leaky-ReLU, so the store
// applies that activation's backward — times (act_out > 0 ? 1 : alpha) * scale — and the per-channel sums of the masked
// gradient (the bias gradient) are reduced CTA-wide in shared memory, in a fixed order, and written to the CTA's row of
// partial sums; the caller adds the rows in order (det_reduce).
struct FirMask {
    const float* act_out;     // saved activation output, same shape as the FIR output
    float* grad_bias;         // partial sums [(n * tiles_y + ty) * tiles_x + tx][minor], one row per pixel tile; may be null
    float alpha, scale;
    // MODE 2 (sae_fir_bias_act, forward): out = lrelu(FIR(x) + noise_weight * noise[pixel] + bias[c]) * scale
    const float* bias;        // [minor] or null
    const float* noise;       // one value per output pixel, or null
    const float* noise_weight;
    // activation bit mask, 1 bit per output element: read instead of act_out (MODE 1) / written next to the output (MODE 2)
    uint32_t* act_mask;
};

// MODE: 0 plain FIR, 1 = MASK (activation backward applied to the result), 2 = ACT (noise + bias + leaky-ReLU applied to it)
template <int KH, int KW, int MODE>
__global__ void __launch_bounds__(256)
fir_tma_kernel(const __grid_constant__ CUtensorMap map_x, float* __restrict__ out, FirParams p, SepTaps taps, int tiles_x, int tiles_y,
               int ncb, FirMask mk) {
    constexpr int WW = FT_W + KW - 1, WH = FT_H + KH - 1;
    extern __shared__ uint8_t fir_smem[];
    __shared__ __align__(8) uint64_t bar_storage;
    constexpr bool MASK = MODE == 1;
    __shared__ float bias_part[8][32];     // per warp
    const uint32_t base = (smem_u32(fir_smem) + 127u) & ~127u;
    const float4* win = reinterpret_cast<const float4*>(fir_smem + (base - smem_u32(fir_smem)));
    const uint32_t bar = smem_u32(&bar_storage);

    // 1-D grid, channel block fastest: CTAs that run together cover whole pixel rows (ncb x 128 contiguous bytes per pixel)
    // instead of the same 128-byte slice of far-apart pixels
    // (ncb < 0 selects the old order, channel block slowest: kept for A/B measurements, SAE_FIR_ORDER=0)
    uint32_t t = blockIdx.x;
    int cb;
    if (ncb > 0) { cb = (int)(t % (uint32_t)ncb); t /= (uint32_t)ncb; }
    else { const uint32_t per = (uint32_t)(tiles_x * tiles_y) * (uint32_t)p.major; cb = (int)(t / per); t %= per; }
    const int tx = (int)(t % tiles_x); t /= tiles_x;
    const int ty = (int)(t % tiles_y);
    const int n = (int)(t / tiles_y);
    const int ox0 = tx * FT_W, oy0 = ty * FT_H;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, (uint32_t)(WW * WH * 128));
        tma_load_4d(base, &map_x, bar, cb * 32, ox0 - p.pad_x0, oy0 - p.pad_y0, n);
    }
    mbar_wait(bar, 0);

    const int cvec = threadIdx.x & 7, x = (threadIdx.x >> 3) & 15, r0 = (threadIdx.x >> 7) * (FT_H / 2);
    auto hrow = [&](int wy) -> float4 {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int b = 0; b < KW; ++b) {
            const float4 v = win[(wy * WW + x + b) * 8 + cvec];
            a.x = fmaf(v.x, taps.x[b], a.x); a.y = fmaf(v.y, taps.x[b], a.y);
            a.z = fmaf(v.z, taps.x[b], a.z); a.w = fmaf(v.w, taps.x[b], a.w);
        }
        return a;
    };
    float4 w[KH];
#pragma unroll
    for (int a = 0; a < KH - 1; ++a) w[a] = hrow(r0 + a);
    const int ox = ox0 + x;
    const int64_t off0 = (((int64_t)n * p.out_h + oy0 + r0) * p.out_w + ox) * p.minor + cb * 32 + cvec * 4;
    float* dst = out + off0;
    float4 bsum = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float nw = 0.f;
    if (MODE == 2) {
        if (mk.bias) bias4 = __ldg(reinterpret_cast<const float4*>(mk.bias + cb * 32 + cvec * 4));
        if (mk.noise) nw = __ldg(mk.noise_weight);
    }
#pragma unroll
    for (int r = 0; r < FT_H / 2; ++r) {
        w[KH - 1] = hrow(r0 + r + KH - 1);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int a = 0; a < KH; ++a) {
            acc.x = fmaf(w[a].x, taps.y[a], acc.x); acc.y = fmaf(w[a].y, taps.y[a], acc.y);
            acc.z = fmaf(w[a].z, taps.y[a], acc.z); acc.w = fmaf(w[a].w, taps.y[a], acc.w);
        }
        const bool inside = ox < p.out_w && oy0 + r0 + r < p.out_h;
        if (MASK) {
            if (inside) {
                float4 o;
                if (mk.act_mask) {
                    const uint32_t wd = __ldg(mk.act_mask + ((off0 + (int64_t)r * p.out_w * p.minor) >> 5)) >> (cvec * 4);
                    o = make_float4((wd & 1u) ? 1.f : 0.f, (wd & 2u) ? 1.f : 0.f, (wd & 4u) ? 1.f : 0.f, (wd & 8u) ? 1.f : 0.f);
                } else {
                    o = ldg_stream(reinterpret_cast<const float4*>(mk.act_out + off0 + (int64_t)r * p.out_w * p.minor));
                }
                acc.x *= (o.x > 0.f ? mk.scale : mk.alpha * mk.scale); acc.y *= (o.y > 0.f ? mk.scale : mk.alpha * mk.scale);
                acc.z *= (o.z > 0.f ? mk.scale : mk.alpha * mk.scale); acc.w *= (o.w > 0.f ? mk.scale : mk.alpha * mk.scale);
                bsum.x += acc.x; bsum.y += acc.y; bsum.z += acc.z; bsum.w += acc.w;
            }
        }
        if (MODE == 2) {
            float nz = 0.f;
            if (mk.noise && inside) nz = nw * __ldg(mk.noise + ((int64_t)n * p.out_h + oy0 + r0 + r) * p.out_w + ox);
            acc.x += bias4.x + nz; acc.y += bias4.y + nz; acc.z += bias4.z + nz; acc.w += bias4.w + nz;
            if (mk.act_mask) {
                // the 8 lanes cvec = 0..7 of a pixel hold its 32 channels: OR their 4 sign bits into the pixel's mask word
                uint32_t bits = ((acc.x > 0.f ? 1u : 0u) | (acc.y > 0.f ? 2u : 0u) | (acc.z > 0.f ? 4u : 0u) | (acc.w > 0.f ? 8u : 0u)) << (cvec * 4);
                bits |= __shfl_xor_sync(0xffffffffu, bits, 1); bits |= __shfl_xor_sync(0xffffffffu, bits, 2); bits |= __shfl_xor_sync(0xffffffffu, bits, 4);
                if (inside && cvec == 0) mk.act_mask[(off0 + (int64_t)r * p.out_w * p.minor) >> 5] = bits;
            }
            acc.x = (acc.x > 0.f ? acc.x : acc.x * mk.alpha) * mk.scale; acc.y = (acc.y > 0.f ? acc.y : acc.y * mk.alpha) * mk.scale;
            acc.z = (acc.z > 0.f ? acc.z : acc.z * mk.alpha) * mk.scale; acc.w = (acc.w > 0.f ? acc.w : acc.w * mk.alpha) * mk.scale;
        }
        if (p.round_tf32) { acc.x = rna_tf32(acc.x); acc.y = rna_tf32(acc.y); acc.z = rna_tf32(acc.z); acc.w = rna_tf32(acc.w); }
        if (inside) *reinterpret_cast<float4*>(dst + (int64_t)r * p.out_w * p.minor) = acc;
#pragma unroll
        for (int a = 0; a < KH - 1; ++a) w[a] = w[a + 1];
    }
    if (MASK && mk.grad_bias != nullptr) {
        // the 32 threads that share cvec sit in the lanes {cvec, cvec + 8, cvec + 16, cvec + 24} of every warp: fold those
        // four with shuffles, then one shared-memory slot per warp and channel, summed over the warps in order
#pragma unroll
        for (int o = 8; o < 32; o <<= 1) {
            bsum.x += __shfl_xor_sync(0xffffffffu, bsum.x, o); bsum.y += __shfl_xor_sync(0xffffffffu, bsum.y, o);
            bsum.z += __shfl_xor_sync(0xffffffffu, bsum.z, o); bsum.w += __shfl_xor_sync(0xffffffffu, bsum.w, o);
        }
        if ((threadIdx.x & 31) < 8) {
            float* wp = bias_part[threadIdx.x >> 5];
            wp[cvec * 4 + 0] = bsum.x; wp[cvec * 4 + 1] = bsum.y; wp[cvec * 4 + 2] = bsum.z; wp[cvec * 4 + 3] = bsum.w;
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) v += bias_part[w][threadIdx.x];
            mk.grad_bias[(((int64_t)n * tiles_y + ty) * tiles_x + tx) * p.minor + cb * 32 + threadIdx.x] = v;
        }
    }
}

template <int KH, int KW, int MASK = 0>
static int launch_tma(const float* x, float* out, const FirParams& p, const SepTaps& taps, cudaStream_t st, FirMask mk = FirMask()) {
    constexpr int WW = FT_W + KW - 1, WH = FT_H + KH - 1;
    CUtensorMap mx;
    cuuint64_t dims[4] = {(cuuint64_t)p.minor, (cuuint64_t)p.in_w, (cuuint64_t)p.in_h, (cuuint64_t)p.major};
    cuuint64_t strides[3] = {(cuuint64_t)p.minor * 4, (cuuint64_t)p.in_w * p.minor * 4, (cuuint64_t)p.in_h * p.in_w * p.minor * 4};
    cuuint32_t box[4] = {32, WW, WH, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    int rc = encode_map(&mx, x, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    constexpr int smem = WW * WH * 128 + 128;
    static bool attr_done = false;
    if (!attr_done) {
        SAE_CUDA_TRY(cudaFuncSetAttribute(fir_tma_kernel<KH, KW, MASK>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_done = true;
    }
    const int tiles_x = (p.out_w + FT_W - 1) / FT_W, tiles_y = (p.out_h + FT_H - 1) / FT_H;
    const int ncb = p.minor / 32;
    dim3 grid((unsigned)((int64_t)tiles_x * tiles_y * p.major * ncb));
    static int order = -1;
    if (order < 0) { const char* v = getenv("SAE_FIR_ORDER"); order = (v && v[0] == '0') ? 0 : 1; }
    fir_tma_kernel<KH, KW, MASK><<<grid, 256, smem, st>>>(mx, out, p, taps, tiles_x, tiles_y, order ? ncb : -ncb, mk);
    return SAE_OK;
}

// zero-insert x2 upsampling FIR (the adjoint of the down = 2 filter): output (y, x) only sees the taps whose
// up-sampled position is even — 2 of 4 per axis — so it is a 2 x 2 gather from the low-resolution input
template <int KH, int KW>
__global__ void __launch_bounds__(256)
fir_sep_up2_kernel(const float* __restrict__ x, float* __restrict__ out, FirParams p, SepTaps taps) {
    const int cv = p.minor >> 2;
    const uint32_t total = (uint32_t)(p.major * p.out_h * p.out_w * cv);
    for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const uint32_t c = idx % cv;
        uint32_t t = idx / cv;
        const int ox = (int)(t % p.out_w); t /= p.out_w;
        const int oy = (int)(t % p.out_h);
        const int64_t n = t / p.out_h;
        const float* xn = x + n * (int64_t)p.in_h * p.in_w * p.minor + (int64_t)c * 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        // only taps whose zero-upsampled position (o + tap - pad) is even land on an input sample: per axis that is tap
        // a0 = (pad - o) & 1 and tap a0 + 2 — a 2 x 2 gather, selected without divergent branches or indexed parameters
        const int ay = (p.pad_y0 - oy) & 1, ax = (p.pad_x0 - ox) & 1;
        const float ty[2] = {ay ? taps.y[1] : taps.y[0], ay ? (KH > 3 ? taps.y[3] : 0.f) : (KH > 2 ? taps.y[2] : 0.f)};
        const float tx[2] = {ax ? taps.x[1] : taps.x[0], ax ? (KW > 3 ? taps.x[3] : 0.f) : (KW > 2 ? taps.x[2] : 0.f)};
        const int uy0 = oy + ay - p.pad_y0, ux0 = ox + ax - p.pad_x0;          // both even (possibly negative)
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
            const int iy = (uy0 >> 1) + dy;
            if (ay + 2 * dy >= KH || iy < 0 || iy >= p.in_h) continue;
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
                const int ix = (ux0 >> 1) + dx;
                if (ax + 2 * dx >= KW || ix < 0 || ix >= p.in_w) continue;
                const float w = ty[dy] * tx[dx];
                const float4 v = __ldg(reinterpret_cast<const float4*>(xn + ((int64_t)iy * p.in_w + ix) * p.minor));
                acc.x = fmaf(v.x, w, acc.x); acc.y = fmaf(v.y, w, acc.y); acc.z = fmaf(v.z, w, acc.z); acc.w = fmaf(v.w, w, acc.w);
            }
        }
        if (p.round_tf32) { acc.x = rna_tf32(acc.x); acc.y = rna_tf32(acc.y); acc.z = rna_tf32(acc.z); acc.w = rna_tf32(acc.w); }
        *reinterpret_cast<float4*>(out + (int64_t)idx * 4) = acc;
    }
}

template <int KH, int KW>
static void launch_sep(const float* x, float* out, const FirParams& p, const SepTaps& taps, cudaStream_t st) {
    constexpr int ROWS = 16;
    int64_t total;
    if (p.up_x == 2) total = p.major * (int64_t)p.out_h * p.out_w * (p.minor / 4);
    else total = p.major * (int64_t)((p.out_h + ROWS - 1) / ROWS) * p.out_w * (p.minor / 4);
    int64_t blocks = (total + 255) / 256;
    int64_t cap = (int64_t)sm_count() * 32;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (p.up_x == 2) fir_sep_up2_kernel<KH, KW><<<(unsigned)blocks, 256, 0, st>>>(x, out, p, taps);
    else if (p.down_x == 2) fir_sep_strip_kernel<KH, KW, ROWS, 2><<<(unsigned)blocks, 256, 0, st>>>(x, out, p, taps);
    else fir_sep_strip_kernel<KH, KW, ROWS, 1><<<(unsigned)blocks, 256, 0, st>>>(x, out, p, taps);
}

template <int KH, int KW>
static void launch_strip(const float* x, const float* k, float* out, const FirParams& p, cudaStream_t st) {
    constexpr int ROWS = 8;
    const int strips = (p.out_h + ROWS - 1) / ROWS;
    int64_t total = p.major * (int64_t)strips * p.out_w * (p.minor / 4);
    int64_t blocks = (total + 255) / 256;
    int64_t cap = (int64_t)sm_count() * 32;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    fir_strip_kernel<KH, KW, ROWS><<<(unsigned)blocks, 256, 0, st>>>(x, k, out, p);
}

}  // namespace sae

extern "C" int sae_upfirdn2d(const float* input, const float* kernel, float* out,
                             int64_t major, int in_h, int in_w, int minor,
                             int kernel_h, int kernel_w,
                             int up_x, int up_y, int down_x, int down_y,
                             int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                             int round_tf32, void* stream) {
    using namespace sae;
    if (major == 0) return SAE_OK;                                     // empty batch: nothing to do
    if (!input || !kernel || !out) return fail(SAE_E_INVALID, "upfirdn2d: null pointer");
    if (major < 0 || in_h <= 0 || in_w <= 0 || minor <= 0) return fail(SAE_E_INVALID, "upfirdn2d: bad input shape");
    if (kernel_h <= 0 || kernel_w <= 0 || kernel_h * kernel_w > kMaxTaps)
        return fail(SAE_E_INVALID, "upfirdn2d: kernel %dx%d unsupported (max 32x32)", kernel_h, kernel_w);
    if (up_x <= 0 || up_y <= 0 || down_x <= 0 || down_y <= 0) return fail(SAE_E_INVALID, "upfirdn2d: up/down must be >= 1");
    FirParams p;
    p.major = major; p.in_h = in_h; p.in_w = in_w; p.minor = minor;
    p.kh = kernel_h; p.kw = kernel_w;
    p.up_x = up_x; p.up_y = up_y; p.down_x = down_x; p.down_y = down_y;
    p.pad_x0 = pad_x0; p.pad_y0 = pad_y0; p.round_tf32 = round_tf32;
    int full_h = in_h * up_y + pad_y0 + pad_y1 - kernel_h;
    int full_w = in_w * up_x + pad_x0 + pad_x1 - kernel_w;
    if (full_h < 0 || full_w < 0) return fail(SAE_E_INVALID, "upfirdn2d: kernel larger than padded input");
    p.out_h = full_h / down_y + 1;
    p.out_w = full_w / down_x + 1;
    cudaStream_t st = (cudaStream_t)stream;
    const bool aligned = ((reinterpret_cast<uintptr_t>(input) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    const bool vec = (minor % 4 == 0) && aligned;
    const bool unit = (up_x == 1 && up_y == 1 && down_x == 1 && down_y == 1);
    if (vec && unit && kernel_h == 4 && kernel_w == 4) {
        launch_strip<4, 4>(input, kernel, out, p, st);
    } else if (vec && unit && kernel_h == 3 && kernel_w == 3) {
        launch_strip<3, 3>(input, kernel, out, p, st);
    } else {
        int64_t total = major * (int64_t)p.out_h * p.out_w * (vec ? minor / 4 : minor);
        int64_t blocks = (total + 255) / 256;
        int64_t cap = (int64_t)sm_count() * 32;
        if (blocks > cap) blocks = cap;
        if (blocks < 1) blocks = 1;
        if (vec) fir_generic_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(input, kernel, out, p);
        else     fir_generic_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(input, kernel, out, p);
    }
    return check_launch("upfirdn2d");
}


// Separable fast path: kernel2d[a][b] == taps_y[a] * taps_x[b] (host arrays, NOT flipped — flipping happens here).
// Restricted to up = down = 1, taps <= 4, minor % 4 == 0, < 2^32 work items; callers fall back to sae_upfirdn2d otherwise.
extern "C" int sae_upfirdn2d_separable(const float* input, const float* taps_y, const float* taps_x, float* out,
                                       int64_t major, int in_h, int in_w, int minor, int kernel_h, int kernel_w,
                                       int up, int down, int pad_x0, int pad_x1, int pad_y0, int pad_y1, int round_tf32,
                                       void* stream) {
    using namespace sae;
    if (major == 0) return SAE_OK;
    if (!input || !taps_y || !taps_x || !out) return fail(SAE_E_INVALID, "upfirdn2d_separable: null pointer");
    if (kernel_h < 1 || kernel_h > 4 || kernel_w != kernel_h) return fail(SAE_E_UNSUPPORTED, "upfirdn2d_separable: taps must be 1..4, square");
    if (minor % 4 != 0 || ((reinterpret_cast<uintptr_t>(input) | reinterpret_cast<uintptr_t>(out)) & 15) != 0)
        return fail(SAE_E_UNSUPPORTED, "upfirdn2d_separable: needs minor %% 4 == 0 and 16-byte aligned pointers");
    FirParams p;
    p.major = major; p.in_h = in_h; p.in_w = in_w; p.minor = minor; p.kh = kernel_h; p.kw = kernel_w;
    if (!((up == 1 && (down == 1 || down == 2)) || (up == 2 && down == 1)))
        return fail(SAE_E_UNSUPPORTED, "upfirdn2d_separable: (up, down) must be (1,1), (1,2) or (2,1)");
    p.up_x = p.up_y = up; p.down_x = p.down_y = down; p.pad_x0 = pad_x0; p.pad_y0 = pad_y0; p.round_tf32 = round_tf32;
    const int full_h = in_h * up + pad_y0 + pad_y1 - kernel_h, full_w = in_w * up + pad_x0 + pad_x1 - kernel_w;
    if (full_h < 0 || full_w < 0) return fail(SAE_E_INVALID, "upfirdn2d_separable: kernel larger than padded input");
    p.out_h = full_h / down + 1;
    p.out_w = full_w / down + 1;
    if (major * (int64_t)p.out_h * p.out_w * (minor / 4) >= (int64_t)1 << 32)
        return fail(SAE_E_UNSUPPORTED, "upfirdn2d_separable: too many work items for 32-bit indexing");
    SepTaps t;
    for (int i = 0; i < 8; ++i) { t.y[i] = 0.f; t.x[i] = 0.f; }
    for (int i = 0; i < kernel_h; ++i) t.y[i] = taps_y[kernel_h - 1 - i];
    for (int i = 0; i < kernel_w; ++i) t.x[i] = taps_x[kernel_w - 1 - i];
    cudaStream_t st = (cudaStream_t)stream;
    static int tma_mode = -1;
    if (tma_mode < 0) { const char* v = getenv("SAE_FIR_TMA"); tma_mode = (v && v[0] == '0') ? 0 : 1; }
    // tc_available() also resolves the driver's cuTensorMapEncodeTiled entry point (a FIR can be the first call into the library)
    if (tma_mode && tc_available() && up == 1 && down == 1 && minor % 32 == 0 && (kernel_h == 3 || kernel_h == 4) && p.out_w >= 8 && p.out_h >= 8 &&
        major * (int64_t)((p.out_w + FT_W - 1) / FT_W) * ((p.out_h + FT_H - 1) / FT_H) * (minor / 32) < ((int64_t)1 << 31)) {
        int rc = kernel_h == 3 ? launch_tma<3, 3>(input, out, p, t, st) : launch_tma<4, 4>(input, out, p, t, st);
        if (rc) return rc;
        return check_launch("upfirdn2d_separable(tma)");
    }
    switch (kernel_h) {
        case 1: launch_sep<1, 1>(input, out, p, t, st); break;
        case 2: launch_sep<2, 2>(input, out, p, t, st); break;
        case 3: launch_sep<3, 3>(input, out, p, t, st); break;
        default: launch_sep<4, 4>(input, out, p, t, st); break;
    }
    return check_launch("upfirdn2d_separable");
}

// FIR (up = down = 1, separable 3 or 4 taps) whose result is the gradient arriving at a fused bias + leaky-ReLU:
//   grad_in = FIR(grad) * (act_out > 0 ? 1 : alpha) * scale,   grad_bias[c] += sum over pixels of grad_in
// i.e. sae_upfirdn2d_separable followed by sae_bias_act_backward in ONE pass (the blur adjoint in front of a
// discriminator block's first activation, stylegan2_layers.py:672-693): the blurred gradient is never written to HBM.
// Only the TMA-tiled configuration is implemented (minor % 32 == 0, output >= 8 x 8); anything else returns
// SAE_E_UNSUPPORTED and the caller issues the two separate calls.
extern "C" int sae_fir_act_backward(const float* grad, const float* taps_y, const float* taps_x, const float* act_out,
                                    float* grad_in, float* grad_bias, int64_t major, int in_h, int in_w, int minor,
                                    int kernel_h, int kernel_w, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                                    float alpha, float scale, int round_tf32, const uint32_t* act_mask, void* stream) {
    using namespace sae;
    if (major == 0) return SAE_OK;
    if (!grad || !taps_y || !taps_x || (!act_out && !act_mask) || !grad_in) return fail(SAE_E_INVALID, "fir_act_backward: null pointer");
    if ((kernel_h != 3 && kernel_h != 4) || kernel_w != kernel_h) return fail(SAE_E_UNSUPPORTED, "fir_act_backward: taps must be 3 or 4, square");
    if (minor % 32 != 0 || ((reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(grad_in) | reinterpret_cast<uintptr_t>(act_out)) & 15) != 0)
        return fail(SAE_E_UNSUPPORTED, "fir_act_backward: needs minor %% 32 == 0 and 16-byte aligned pointers");
    FirParams p;
    p.major = major; p.in_h = in_h; p.in_w = in_w; p.minor = minor; p.kh = kernel_h; p.kw = kernel_w;
    p.up_x = p.up_y = 1; p.down_x = p.down_y = 1; p.pad_x0 = pad_x0; p.pad_y0 = pad_y0; p.round_tf32 = round_tf32;
    const int full_h = in_h + pad_y0 + pad_y1 - kernel_h, full_w = in_w + pad_x0 + pad_x1 - kernel_w;
    if (full_h < 0 || full_w < 0) return fail(SAE_E_INVALID, "fir_act_backward: kernel larger than padded input");
    p.out_h = full_h + 1;
    p.out_w = full_w + 1;
    if (!tc_available() || p.out_w < 8 || p.out_h < 8 ||
        major * (int64_t)((p.out_w + FT_W - 1) / FT_W) * ((p.out_h + FT_H - 1) / FT_H) * (minor / 32) >= ((int64_t)1 << 31))
        return fail(SAE_E_UNSUPPORTED, "fir_act_backward: shape outside the TMA-tiled configuration");
    SepTaps t;
    for (int i = 0; i < 8; ++i) { t.y[i] = 0.f; t.x[i] = 0.f; }
    for (int i = 0; i < kernel_h; ++i) t.y[i] = taps_y[kernel_h - 1 - i];
    for (int i = 0; i < kernel_w; ++i) t.x[i] = taps_x[kernel_w - 1 - i];
    FirMask mk;
    mk.act_out = act_out; mk.grad_bias = grad_bias; mk.alpha = alpha; mk.scale = scale; mk.act_mask = const_cast<uint32_t*>(act_mask);
    cudaStream_t st = (cudaStream_t)stream;
    mk.bias = nullptr; mk.noise = nullptr; mk.noise_weight = nullptr;
    const int parts = (int)(major * ((p.out_w + FT_W - 1) / FT_W) * ((p.out_h + FT_H - 1) / FT_H));
    if (grad_bias) {
        mk.grad_bias = det_workspace(det_reduce_floats(minor, parts));
        if (!mk.grad_bias) return SAE_E_CUDA;
    }
    int rc = kernel_h == 3 ? launch_tma<3, 3, 1>(grad, grad_in, p, t, st, mk) : launch_tma<4, 4, 1>(grad, grad_in, p, t, st, mk);
    if (rc) return rc;
    rc = check_launch("fir_act_backward");
    if (rc || !grad_bias) return rc;
    return det_reduce(grad_bias, mk.grad_bias, minor, parts, st);
}

// FIR (up = down = 1, separable 3 or 4 taps) followed by NoiseInjection + bias + leaky-ReLU in ONE pass:
//   out = lrelu(FIR(x) + noise_weight * noise[pixel] + bias[c], alpha) * scale
// the Blur after the generator's transposed convolution and the StyledConv tail behind it
// (stylegan2_layers.py:306-309 -> :398-405): the blurred tensor is never written to HBM.
// Only the TMA-tiled configuration (minor % 32 == 0, output >= 8 x 8); SAE_E_UNSUPPORTED otherwise.
extern "C" int sae_fir_bias_act(const float* x, const float* taps_y, const float* taps_x, const float* bias, const float* noise,
                                const float* noise_weight, float* out, int64_t major, int in_h, int in_w, int minor,
                                int kernel_h, int kernel_w, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                                float alpha, float scale, int round_tf32, uint32_t* act_mask, void* stream) {
    using namespace sae;
    if (major == 0) return SAE_OK;
    if (!x || !taps_y || !taps_x || !out) return fail(SAE_E_INVALID, "fir_bias_act: null pointer");
    if (noise && !noise_weight) return fail(SAE_E_INVALID, "fir_bias_act: noise needs its weight");
    if ((kernel_h != 3 && kernel_h != 4) || kernel_w != kernel_h) return fail(SAE_E_UNSUPPORTED, "fir_bias_act: taps must be 3 or 4, square");
    if (minor % 32 != 0 || ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(bias)) & 15) != 0)
        return fail(SAE_E_UNSUPPORTED, "fir_bias_act: needs minor %% 32 == 0 and 16-byte aligned pointers");
    FirParams p;
    p.major = major; p.in_h = in_h; p.in_w = in_w; p.minor = minor; p.kh = kernel_h; p.kw = kernel_w;
    p.up_x = p.up_y = 1; p.down_x = p.down_y = 1; p.pad_x0 = pad_x0; p.pad_y0 = pad_y0; p.round_tf32 = round_tf32;
    const int full_h = in_h + pad_y0 + pad_y1 - kernel_h, full_w = in_w + pad_x0 + pad_x1 - kernel_w;
    if (full_h < 0 || full_w < 0) return fail(SAE_E_INVALID, "fir_bias_act: kernel larger than padded input");
    p.out_h = full_h + 1;
    p.out_w = full_w + 1;
    if (!tc_available() || p.out_w < 8 || p.out_h < 8 ||
        major * (int64_t)((p.out_w + FT_W - 1) / FT_W) * ((p.out_h + FT_H - 1) / FT_H) * (minor / 32) >= ((int64_t)1 << 31))
        return fail(SAE_E_UNSUPPORTED, "fir_bias_act: shape outside the TMA-tiled configuration");
    SepTaps t;
    for (int i = 0; i < 8; ++i) { t.y[i] = 0.f; t.x[i] = 0.f; }
    for (int i = 0; i < kernel_h; ++i) t.y[i] = taps_y[kernel_h - 1 - i];
    for (int i = 0; i < kernel_w; ++i) t.x[i] = taps_x[kernel_w - 1 - i];
    FirMask mk;
    mk.act_out = nullptr; mk.grad_bias = nullptr; mk.alpha = alpha; mk.scale = scale; mk.act_mask = act_mask;
    mk.bias = bias; mk.noise = noise; mk.noise_weight = noise_weight;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = kernel_h == 3 ? launch_tma<3, 3, 2>(x, out, p, t, st, mk) : launch_tma<4, 4, 2>(x, out, p, t, st, mk);
    if (rc) return rc;
    return check_launch("fir_bias_act");
}
