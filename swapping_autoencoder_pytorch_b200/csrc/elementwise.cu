// HBM-bound pointwise kernels: fused bias + (noise) + leaky-relu forward / backward (with the
// bias-gradient reduction fused in), style modulation forward / backward, gradient bucket
// pack / unpack.  Replaces models/networks/stylegan2_op/fused_bias_act_kernel.cu:19-99 and the
// unfused ATen elementwise kernels listed in SURVEY.md §2.1.
// All kernels: float4 accesses when the channel count allows, grid = multiple of the SM count,
// 64-bit indexing.
#include "common.cuh"

namespace sae {

static inline unsigned grid_for(int64_t work_items, int threads, int per_sm = 8) {
    int64_t blocks = (work_items + threads - 1) / threads;
    int64_t cap = (int64_t)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}

// ----------------------------------------------------------------------------- bias_act forward
template <int VEC, typename IDX>
__global__ void __launch_bounds__(256)
bias_act_kernel(const float* __restrict__ x, const float* __restrict__ b, const float* __restrict__ ref,
                float* __restrict__ out, IDX size_v, IDX step_b, int size_b,
                int act, int grad, float alpha, float scale,
                const float* __restrict__ noise, const float* __restrict__ noise_weight, int64_t noise_div,
                int round_tf32) {
    const float nw = noise ? __ldg(noise_weight) : 0.f;
    for (IDX i = blockIdx.x * (IDX)blockDim.x + threadIdx.x; i < size_v; i += (IDX)gridDim.x * blockDim.x) {
        float v[VEC], r[VEC];
        const IDX e0 = i * VEC;
        if (VEC == 4) {
            float4 t = ldg_stream(reinterpret_cast<const float4*>(x) + i);
            v[0] = t.x; v[1 % VEC] = t.y; v[2 % VEC] = t.z; v[3 % VEC] = t.w;
            if (ref) {
                float4 q = ldg_stream(reinterpret_cast<const float4*>(ref) + i);
                r[0] = q.x; r[1 % VEC] = q.y; r[2 % VEC] = q.z; r[3 % VEC] = q.w;
            }
        } else {
            v[0] = x[e0];
            if (ref) r[0] = ref[e0];
        }
        float nz = 0.f;
        if (noise) nz = nw * __ldg(noise + e0 / (IDX)noise_div);
        // channel of element e0 (+j): one division per vector when channels are innermost (step_b == 1)
        const int cb = b ? (int)((step_b == 1 ? e0 : e0 / step_b) % (IDX)size_b) : 0;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float t = v[j];
            if (b) {
                int ci = cb;
                if (step_b == 1) { ci = cb + j; if (ci >= size_b) ci -= size_b; }
                else if (j > 0) ci = (int)(((e0 + j) / step_b) % (IDX)size_b);
                t += __ldg(b + ci);
            }
            t += nz;
            float y;
            if (act == 3) {
                if (grad == 0)      y = (t > 0.f) ? t : t * alpha;
                else if (grad == 1) y = ((ref ? r[j] : 0.f) > 0.f) ? t : t * alpha;
                else                y = 0.f;
            } else {
                y = (grad == 2) ? 0.f : t;
            }
            v[j] = round_tf32 ? rna_tf32(y * scale) : y * scale;
        }
        if (VEC == 4) reinterpret_cast<float4*>(out)[i] = make_float4(v[0], v[1 % VEC], v[2 % VEC], v[3 % VEC]);
        else out[e0] = v[0];
    }
}

// ---------------------------------------------------------------------------- bias_act backward
// grad_in = grad_out * mask(out) * scale; grad_bias[c] += sum(grad_in); channels innermost.
// Every thread keeps a fixed channel group across its grid-stride loop (stride is a multiple of
// the number of channel groups) and accumulates in registers.  The CTA then sums each channel over its
// threads in thread order and writes the sums (and the noise-weight sum) to its own row part[blockIdx.x][C + 1];
// det_reduce adds the rows in order.
template <int VEC>
__global__ void __launch_bounds__(256)
bias_act_bwd_kernel(const float* __restrict__ go, const float* __restrict__ outp, float* __restrict__ gi,
                    float* __restrict__ part, int want_gb, int64_t size_v, int cv, int64_t stride_v,
                    float alpha, float scale,
                    const float* __restrict__ noise, int64_t noise_div, int round_tf32,
                    const uint32_t* __restrict__ act_mask) {
    extern __shared__ float sthr[];   // [blockDim.x * VEC] per-thread channel sums, then [blockDim.x / 32] warp noise sums
    const int C = cv * VEC;

    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    float bsum[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) bsum[j] = 0.f;
    float nsum = 0.f;
    if (tid < stride_v) {
        for (int64_t i = tid; i < size_v; i += stride_v) {
            float g[VEC], o[VEC];
            if (VEC == 4) {
                float4 t = ldg_stream(reinterpret_cast<const float4*>(go) + i);
                g[0] = t.x; g[1 % VEC] = t.y; g[2 % VEC] = t.z; g[3 % VEC] = t.w;
                if (act_mask) {
                    // 1 bit per element instead of the 4-byte activation output: elements 4i .. 4i+3 are bits (4i & 31) .. of word i >> 3
                    const uint32_t wd = __ldg(act_mask + (i >> 3)) >> (((uint32_t)i & 7u) * 4u);
                    o[0] = (wd & 1u) ? 1.f : 0.f; o[1 % VEC] = (wd & 2u) ? 1.f : 0.f; o[2 % VEC] = (wd & 4u) ? 1.f : 0.f; o[3 % VEC] = (wd & 8u) ? 1.f : 0.f;
                } else {
                    float4 q = ldg_stream(reinterpret_cast<const float4*>(outp) + i);
                    o[0] = q.x; o[1 % VEC] = q.y; o[2 % VEC] = q.z; o[3 % VEC] = q.w;
                }
            } else {
                g[0] = go[i]; o[0] = outp[i];
            }
            float lsum = 0.f;
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                float y = ((o[j] > 0.f) ? g[j] : g[j] * alpha) * scale;
                g[j] = round_tf32 ? rna_tf32(y) : y;
                bsum[j] += y;
                lsum += y;
            }
            if (noise) nsum = fmaf(lsum, __ldg(noise + (i * VEC) / noise_div), nsum);
            if (VEC == 4) reinterpret_cast<float4*>(gi)[i] = make_float4(g[0], g[1 % VEC], g[2 % VEC], g[3 % VEC]);
            else gi[i] = g[0];
        }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) sthr[threadIdx.x * VEC + j] = bsum[j];
    float* swarp = sthr + blockDim.x * VEC;
    nsum = warp_sum(nsum);
    if ((threadIdx.x & 31) == 0) swarp[threadIdx.x >> 5] = nsum;
    __syncthreads();
    float* row = part + (int64_t)blockIdx.x * (C + 1);
    if (want_gb) {
        // thread t of this CTA holds channel group (blockIdx.x * blockDim.x + t) % cv
        const int shift = (int)(((int64_t)blockIdx.x * blockDim.x) % cv);
        for (int i = threadIdx.x; i < C; i += blockDim.x) {
            const int cg = i / VEC, j = i - cg * VEC;
            float v = 0.f;
            for (int t = (cg - shift + cv) % cv; t < (int)blockDim.x; t += cv) v += sthr[t * VEC + j];
            row[i] = v;
        }
    }
    if (noise && threadIdx.x == 0) {
        float v = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += swarp[w];
        row[C] = v;
    }
}

// ------------------------------------------------------------------------------------ modulate
template <typename IDX>
__global__ void __launch_bounds__(256)
modulate_kernel(const float4* __restrict__ x, const float4* __restrict__ s, float4* __restrict__ out,
                IDX total_v, IDX hw, int cv, int round_tf32) {
    for (IDX i = blockIdx.x * (IDX)blockDim.x + threadIdx.x; i < total_v; i += (IDX)gridDim.x * blockDim.x) {
        const IDX pix = i / (IDX)cv;
        const int c = (int)(i - pix * (IDX)cv);
        const IDX n = pix / hw;
        float4 v = ldg_stream(x + i);
        float4 m = __ldg(s + n * cv + c);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
        if (round_tf32) { v.x = rna_tf32(v.x); v.y = rna_tf32(v.y); v.z = rna_tf32(v.z); v.w = rna_tf32(v.w); }
        out[i] = v;
    }
}

__global__ void __launch_bounds__(256)
modulate_scalar_kernel(const float* __restrict__ x, const float* __restrict__ s, float* __restrict__ out,
                       int64_t total, int64_t hw, int c, int round_tf32) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        int ch = (int)(i % c);
        int64_t n = (i / c) / hw;
        float v = x[i] * __ldg(s + n * c + ch);
        out[i] = round_tf32 ? rna_tf32(v) : v;
    }
}

// dx = dy * s;  ds[n, c] += sum_hw dy * x.   grid = (chunks, N); each CTA covers a pixel range of one
// sample; thread keeps a fixed channel group, the CTA sums each channel over its threads in thread order and
// writes the sums to its own row part[blockIdx.x][n][C]; det_reduce adds the rows in order.
template <int VEC>
__global__ void __launch_bounds__(256)
modulate_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ s,
                    float* __restrict__ dx, float* __restrict__ part, int64_t hw, int cv, int64_t pix_per_cta, int round_tf32) {
    extern __shared__ float sthr[];   // [blockDim.x * VEC]
    const int C = cv * VEC;
    const int n = blockIdx.y;
    const int64_t p0 = blockIdx.x * pix_per_cta;
    int64_t p1 = p0 + pix_per_cta;
    if (p1 > hw) p1 = hw;
    const int64_t base_v = (int64_t)n * hw * cv;
    const int64_t lo = p0 * cv, hi = p1 * cv;          // in VEC units inside this sample
    const int64_t stride = (blockDim.x / cv > 0) ? (int64_t)(blockDim.x / cv) * cv : 0;
    float* row = part + ((int64_t)blockIdx.x * gridDim.y + n) * C;
    if (stride > 0) {
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
        if (threadIdx.x < stride) {
            const int c = threadIdx.x % cv;
            float m[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j) m[j] = __ldg(s + (int64_t)n * C + c * VEC + j);
            for (int64_t i = lo + threadIdx.x; i < hi; i += stride) {
                float g[VEC], a[VEC];
                if (VEC == 4) {
                    float4 t = ldg_stream(reinterpret_cast<const float4*>(dy) + base_v + i);
                    float4 q = ldg_stream(reinterpret_cast<const float4*>(x) + base_v + i);
                    g[0] = t.x; g[1 % VEC] = t.y; g[2 % VEC] = t.z; g[3 % VEC] = t.w;
                    a[0] = q.x; a[1 % VEC] = q.y; a[2 % VEC] = q.z; a[3 % VEC] = q.w;
                } else {
                    g[0] = dy[base_v + i]; a[0] = x[base_v + i];
                }
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    acc[j] = fmaf(g[j], a[j], acc[j]);
                    g[j] = round_tf32 ? rna_tf32(g[j] * m[j]) : g[j] * m[j];
                }
                if (VEC == 4) reinterpret_cast<float4*>(dx)[base_v + i] = make_float4(g[0], g[1 % VEC], g[2 % VEC], g[3 % VEC]);
                else dx[base_v + i] = g[0];
            }
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j) sthr[threadIdx.x * VEC + j] = acc[j];
        __syncthreads();
        // thread t < stride holds channel group t % cv
        for (int i = threadIdx.x; i < C; i += blockDim.x) {
            const int cg = i / VEC, j = i - cg * VEC;
            float v = 0.f;
            for (int t = cg; t < stride; t += cv) v += sthr[t * VEC + j];
            row[i] = v;
        }
    } else {
        // more channel groups than threads: each thread owns whole channel groups and walks the pixels of the range
        for (int cc = threadIdx.x; cc < cv; cc += blockDim.x) {
            float acc[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
            for (int64_t pp = p0; pp < p1; ++pp) {
                const int64_t i = pp * cv + cc;
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    int64_t e = (base_v + i) * VEC + j;
                    float g = dy[e], a = x[e];
                    acc[j] = fmaf(g, a, acc[j]);
                    float d = g * __ldg(s + (int64_t)n * C + cc * VEC + j);
                    dx[e] = round_tf32 ? rna_tf32(d) : d;
                }
            }
#pragma unroll
            for (int j = 0; j < VEC; ++j) row[cc * VEC + j] = acc[j];
        }
    }
}

// ------------------------------------------------------------------------- residual merge / rounding
template <int VEC>
__global__ void __launch_bounds__(256)
add_scale_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, int64_t nv, float scale,
                 int round_tf32) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        if (VEC == 4) {
            float4 u = ldg_stream(reinterpret_cast<const float4*>(a) + i);
            if (b) {
                float4 w = ldg_stream(reinterpret_cast<const float4*>(b) + i);
                u.x += w.x; u.y += w.y; u.z += w.z; u.w += w.w;
            }
            u.x *= scale; u.y *= scale; u.z *= scale; u.w *= scale;
            if (round_tf32) { u.x = rna_tf32(u.x); u.y = rna_tf32(u.y); u.z = rna_tf32(u.z); u.w = rna_tf32(u.w); }
            reinterpret_cast<float4*>(out)[i] = u;
        } else {
            float u = a[i];
            if (b) u += b[i];
            u *= scale;
            out[i] = round_tf32 ? rna_tf32(u) : u;
        }
    }
}

// ------------------------------------------------------------ bilinear x2 upsample fused with the residual merge
// out[n,y,x,c] = (bilinear2x(skip)[n,y,x,c] + res[n,y,x,c]) * scale   (align_corners = False, the generator's skip
// branch: F.interpolate(..., scale_factor=2, mode='bilinear') followed by (skip + res) / sqrt(2), generator.py:51-53)
__device__ __forceinline__ void bilin_src(int d, int in_size, int& i0, int& i1, float& l0, float& l1) {
    float src = 0.5f * (d + 0.5f) - 0.5f;          // area_pixel_compute_source_index, scale 1/2
    if (src < 0.f) src = 0.f;
    i0 = (int)src;
    i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    l1 = src - (float)i0;
    l0 = 1.f - l1;
}

__global__ void __launch_bounds__(256)
upsample2x_add_kernel(const float4* __restrict__ skip, const float4* __restrict__ res, float4* __restrict__ out,
                      int64_t total_v, int h, int w, int cv, float scale, int round_tf32) {
    const int oh = 2 * h, ow = 2 * w;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total_v; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cv);
        int64_t t = i / cv;
        const int x = (int)(t % ow); t /= ow;
        const int y = (int)(t % oh);
        const int64_t n = t / oh;
        int y0, y1, x0, x1; float ly0, ly1, lx0, lx1;
        bilin_src(y, h, y0, y1, ly0, ly1);
        bilin_src(x, w, x0, x1, lx0, lx1);
        const float4* sb = skip + n * (int64_t)h * w * cv + c;
        const float4 a = __ldg(sb + ((int64_t)y0 * w + x0) * cv), b = __ldg(sb + ((int64_t)y0 * w + x1) * cv);
        const float4 d = __ldg(sb + ((int64_t)y1 * w + x0) * cv), e = __ldg(sb + ((int64_t)y1 * w + x1) * cv);
        const float4 r = ldg_stream(res + i);
        float4 o;
        o.x = (ly0 * (lx0 * a.x + lx1 * b.x) + ly1 * (lx0 * d.x + lx1 * e.x) + r.x) * scale;
        o.y = (ly0 * (lx0 * a.y + lx1 * b.y) + ly1 * (lx0 * d.y + lx1 * e.y) + r.y) * scale;
        o.z = (ly0 * (lx0 * a.z + lx1 * b.z) + ly1 * (lx0 * d.z + lx1 * e.z) + r.z) * scale;
        o.w = (ly0 * (lx0 * a.w + lx1 * b.w) + ly1 * (lx0 * d.w + lx1 * e.w) + r.w) * scale;
        if (round_tf32) { o.x = rna_tf32(o.x); o.y = rna_tf32(o.y); o.z = rna_tf32(o.z); o.w = rna_tf32(o.w); }
        out[i] = o;
    }
}

// adjoint of the x2 bilinear interpolation, times scale: one thread per low-resolution element gathers the (up to 5x5)
// high-resolution gradients whose interpolation stencil touches it — no atomics
__global__ void __launch_bounds__(256)
upsample2x_bwd_kernel(const float4* __restrict__ dy, float4* __restrict__ dskip, int64_t total_v, int h, int w, int cv,
                      float scale, int round_tf32) {
    const int oh = 2 * h, ow = 2 * w;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total_v; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cv);
        int64_t t = i / cv;
        const int x = (int)(t % w); t /= w;
        const int y = (int)(t % h);
        const int64_t n = t / h;
        const float4* gb = dy + n * (int64_t)oh * ow * cv + c;
        // low-res pixel y is touched by high-res rows 2y-1, 2y, 2y+1, 2y+2 with weights 1/4, 3/4, 3/4, 1/4; the clamped
        // border rows (0 and 2h-1) put their whole weight on the first / last low-res row
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int yy = 2 * y - 1 + a;
            if (yy < 0 || yy >= oh) continue;
            float wy = (a == 0 || a == 3) ? 0.25f : 0.75f;
            if (yy == 0 || yy == oh - 1) wy = 1.0f;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int xx = 2 * x - 1 + b;
                if (xx < 0 || xx >= ow) continue;
                float wx = (b == 0 || b == 3) ? 0.25f : 0.75f;
                if (xx == 0 || xx == ow - 1) wx = 1.0f;
                const float4 g = __ldg(gb + ((int64_t)yy * ow + xx) * cv);
                const float ww = wy * wx;
                acc.x = fmaf(ww, g.x, acc.x); acc.y = fmaf(ww, g.y, acc.y); acc.z = fmaf(ww, g.z, acc.z); acc.w = fmaf(ww, g.w, acc.w);
            }
        }
        acc.x *= scale; acc.y *= scale; acc.z *= scale; acc.w *= scale;
        if (round_tf32) { acc.x = rna_tf32(acc.x); acc.y = rna_tf32(acc.y); acc.z = rna_tf32(acc.z); acc.w = rna_tf32(acc.w); }
        dskip[i] = acc;
    }
}

// out[n, p, 0:c_out] = (x[n, 0:c_in, p], 0 ...): channel zero-padding fused with the NCHW -> NHWC conversion.  One thread per
// output float4; the input is a sliver (3 channels) next to the 32-channel output rows, so the writes set the pace.
__global__ void __launch_bounds__(256)
pad_channels_kernel(const float* __restrict__ x, float4* __restrict__ out, int64_t total_v, int64_t pixels, int c_in, int cv,
                    int64_t sn, int64_t sc, int64_t sp, int round) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total_v; i += (int64_t)gridDim.x * blockDim.x) {
        const int v = (int)(i % cv);
        const int64_t t = i / cv;
        const int64_t pix = t % pixels, n = t / pixels;
        float r[4] = {0.f, 0.f, 0.f, 0.f};
        const int c0 = v * 4;
        if (c0 < c_in) {
            const float* src = x + n * sn + pix * sp;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (c0 + j < c_in) { const float f = __ldg(src + (int64_t)(c0 + j) * sc); r[j] = round ? rna_tf32(f) : f; }
        }
        out[i] = make_float4(r[0], r[1], r[2], r[3]);
    }
}


// ------------------------------------------------------------------------------------ reflection padding (NHWC)
// nn.ReflectionPad2d of the encoder (stylegan2_layers.py:104,642) in one pass over channels-last data; the backward
// gathers, for every input pixel, the (at most 3 x 3) padded positions that mirror onto it — no atomics.
__device__ __forceinline__ int reflect_idx(int i, int len) {
    if (i < 0) i = -i;
    if (i >= len) i = 2 * (len - 1) - i;
    return i;
}

__global__ void __launch_bounds__(256)
reflect_pad_kernel(const float4* __restrict__ x, float4* __restrict__ out, uint32_t total_v, int h, int w, int cv, int oh, int ow,
                   int pl, int pt) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_v; i += gridDim.x * blockDim.x) {
        const uint32_t c = i % cv;
        uint32_t t = i / cv;
        const int ox = (int)(t % ow); t /= ow;
        const int oy = (int)(t % oh);
        const uint32_t n = t / oh;
        const int iy = reflect_idx(oy - pt, h), ix = reflect_idx(ox - pl, w);
        out[i] = ldg_stream(x + (((int64_t)n * h + iy) * w + ix) * cv + c);
    }
}

__global__ void __launch_bounds__(256)
reflect_pad_bwd_kernel(const float4* __restrict__ dy, float4* __restrict__ dx, uint32_t total_v, int h, int w, int cv, int oh, int ow,
                       int pl, int pr, int pt, int pb) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_v; i += gridDim.x * blockDim.x) {
        const uint32_t c = i % cv;
        uint32_t t = i / cv;
        const int ix = (int)(t % w); t /= w;
        const int iy = (int)(t % h);
        const uint32_t n = t / h;
        int ys[3], xs[3], ny = 0, nx = 0;
        ys[ny++] = iy + pt;
        if (iy >= 1 && iy <= pt) ys[ny++] = pt - iy;
        if (iy <= h - 2 && iy >= h - 1 - pb) ys[ny++] = pt + 2 * (h - 1) - iy;
        xs[nx++] = ix + pl;
        if (ix >= 1 && ix <= pl) xs[nx++] = pl - ix;
        if (ix <= w - 2 && ix >= w - 1 - pr) xs[nx++] = pl + 2 * (w - 1) - ix;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int a = 0; a < ny; ++a)
            for (int b = 0; b < nx; ++b) {
                const float4 g = __ldg(dy + (((int64_t)n * oh + ys[a]) * ow + xs[b]) * cv + c);
                acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
            }
        dx[i] = acc;
    }
}

// ------------------------------------------------------------------------------------------ filter preparation
// One pass from the parameter layout [K, C, R, S] to the kernels' layouts: out_krsc[k,r,s,c] (fprop / wgrad) and,
// optionally, out_crsk[c,r,s,k] (dgrad), multiplied by the equalised-lr scale and rounded to TF32 — replaces the
// reference's per-call `weight * scale` (stylegan2_layers.py:138) plus the permute / contiguous / round passes.
__global__ void __launch_bounds__(256)
filter_prep_kernel(const float* __restrict__ w, float* __restrict__ krsc, float* __restrict__ crsk, int K, int C, int RS,
                   float scale, int round_tf32) {
    const int total = K * C * RS;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        // i enumerates the OUTPUT krsc order (c fastest) so the big write is coalesced
        const int c = i % C;
        int t = i / C;
        const int rs = t % RS;
        const int k = t / RS;
        float v = __ldg(w + ((size_t)k * C + c) * RS + rs) * scale;
        if (round_tf32) v = rna_tf32(v);
        krsc[i] = v;
        if (crsk) crsk[((size_t)c * RS + rs) * K + k] = v;
    }
}

// Per-sample filters of the style-modulated convolution (stylegan2_layers.py:284-323): out[n,k,r,s,c] = w[k,r,s,c] * s[n,c]
// (fprop, "KRSC" per image) and out_t[n,c,r,s,k] = the same values transposed (dgrad).  w is the prepared [K,R,S,C] filter
// (scaled, demodulated, TF32-rounded); the product is rounded again.  One block column per image.
__global__ void __launch_bounds__(256)
filter_modulate_kernel(const float* __restrict__ w_krsc, const float* __restrict__ s, float* __restrict__ out, float* __restrict__ out_t,
                       int K, int C, int RS, int round_tf32) {
    const int n = blockIdx.y;
    const int total = K * C * RS;
    const float* sn = s + (size_t)n * C;
    float* on = out ? out + (size_t)n * total : nullptr;
    float* otn = out_t ? out_t + (size_t)n * total : nullptr;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int c = i % C;
        int t = i / C;
        const int rs = t % RS;
        const int k = t / RS;
        float v = __ldg(w_krsc + i) * __ldg(sn + c);
        if (round_tf32) v = rna_tf32(v);
        if (on) on[i] = v;
        if (otn) otn[((size_t)c * RS + rs) * K + k] = v;
    }
}

// adjoint: d_w[k,c,r,s] = scale * d_krsc[k,r,s,c]
__global__ void __launch_bounds__(256)
filter_unprep_kernel(const float* __restrict__ g, float* __restrict__ dw, int K, int C, int RS, float scale) {
    const int total = K * C * RS;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int c = i % C;
        int t = i / C;
        const int rs = t % RS;
        const int k = t / RS;
        dw[((size_t)k * C + c) * RS + rs] = __ldg(g + i) * scale;
    }
}

// --------------------------------------------------------------------------- bucket pack/unpack
__global__ void __launch_bounds__(256)
bucket_copy_kernel(float* const* __restrict__ ptrs, const int64_t* __restrict__ offsets,
                   const int64_t* __restrict__ sizes, float* __restrict__ bucket, float scale, int to_bucket) {
    const int t = blockIdx.y;
    float* p = ptrs[t];
    float* b = bucket + offsets[t];
    const int64_t n = sizes[t];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (to_bucket) b[i] = p[i];
        else p[i] = b[i] * scale;
    }
}

}  // namespace sae

using namespace sae;

extern "C" int sae_fused_bias_act(const float* x, const float* bias, const float* ref, float* out,
                                  int64_t size_x, int64_t step_b, int size_b,
                                  int act, int grad, float alpha, float scale,
                                  const float* noise, const float* noise_weight, int64_t noise_div,
                                  int round_tf32, void* stream) {
    if (size_x == 0) return SAE_OK;
    if (!x || !out || size_x < 0) return fail(SAE_E_INVALID, "fused_bias_act: bad input");
    if (act != 1 && act != 3) return fail(SAE_E_INVALID, "fused_bias_act: act %d unsupported (1 linear, 3 lrelu)", act);
    if (grad < 0 || grad > 2) return fail(SAE_E_INVALID, "fused_bias_act: grad must be 0..2");
    if (bias && (size_b <= 0 || step_b <= 0)) return fail(SAE_E_INVALID, "fused_bias_act: bad bias geometry");
    if (noise && (!noise_weight || noise_div <= 0)) return fail(SAE_E_INVALID, "fused_bias_act: noise needs weight and divisor");
    if (!bias) { size_b = 1; step_b = 1; }
    cudaStream_t st = (cudaStream_t)stream;
    uintptr_t al = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(ref);
    bool vec = (size_x % 4 == 0) && (al % 16 == 0) && (!noise || noise_div % 4 == 0);
    const bool small = size_x < ((int64_t)1 << 31) && step_b < ((int64_t)1 << 31);      // 32-bit index arithmetic
    if (vec) {
        int64_t nv = size_x / 4;
        if (small)
            bias_act_kernel<4, uint32_t><<<grid_for(nv, 256, 16), 256, 0, st>>>(x, bias, ref, out, (uint32_t)nv, (uint32_t)step_b, size_b, act,
                                                                               grad, alpha, scale, noise, noise_weight, noise_div, round_tf32);
        else
            bias_act_kernel<4, int64_t><<<grid_for(nv, 256, 16), 256, 0, st>>>(x, bias, ref, out, nv, step_b, size_b, act, grad, alpha,
                                                                              scale, noise, noise_weight, noise_div, round_tf32);
    } else {
        if (small)
            bias_act_kernel<1, uint32_t><<<grid_for(size_x, 256, 16), 256, 0, st>>>(x, bias, ref, out, (uint32_t)size_x, (uint32_t)step_b, size_b,
                                                                                   act, grad, alpha, scale, noise, noise_weight, noise_div, round_tf32);
        else
            bias_act_kernel<1, int64_t><<<grid_for(size_x, 256, 16), 256, 0, st>>>(x, bias, ref, out, size_x, step_b, size_b, act, grad,
                                                                                  alpha, scale, noise, noise_weight, noise_div, round_tf32);
    }
    return check_launch("fused_bias_act");
}

extern "C" int sae_bias_act_backward(const float* grad_out, const float* out, float* grad_in, float* grad_bias,
                                     int64_t size_x, int size_b, float alpha, float scale,
                                     const float* noise, int64_t noise_div, float* grad_noise_weight,
                                     int round_tf32, const uint32_t* act_mask, void* stream) {
    if (size_x == 0) return SAE_OK;
    if (!grad_out || (!out && !act_mask) || !grad_in || size_b <= 0 || size_x % size_b != 0)
        return fail(SAE_E_INVALID, "bias_act_backward: bad arguments (size_x %% size_b must be 0)");
    if (act_mask && size_b % 32 != 0) return fail(SAE_E_INVALID, "bias_act_backward: the activation bit mask needs a channel count that is a multiple of 32");
    if (noise && (!grad_noise_weight || noise_div <= 0)) return fail(SAE_E_INVALID, "bias_act_backward: noise needs grad slot");
    if (size_b > 12000) return fail(SAE_E_UNSUPPORTED, "bias_act_backward: more than 12000 channels");
    cudaStream_t st = (cudaStream_t)stream;
    uintptr_t al = reinterpret_cast<uintptr_t>(grad_out) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(grad_in);
    bool vec = (size_b % 4 == 0) && (al % 16 == 0) && (!noise || noise_div % 4 == 0);
    if (act_mask && !vec) return fail(SAE_E_INVALID, "bias_act_backward: the activation bit mask needs the vectorised path (16-byte aligned pointers)");
    const int V = vec ? 4 : 1;
    const int cv = size_b / V;
    const int64_t size_v = size_x / V;
    unsigned blocks = grid_for(size_v, 256, 4);
    int64_t threads = (int64_t)blocks * 256;
    // stride must be a multiple of cv so each thread's channel group is loop-invariant
    int64_t stride = (threads / cv) * cv;
    if (stride == 0) {  // fewer threads than channel groups: grow the grid
        blocks = (unsigned)((cv + 255) / 256);
        threads = (int64_t)blocks * 256;
        stride = (threads / cv) * cv;
    }
    float* part = nullptr;
    if (grad_bias || noise) {
        part = det_workspace(det_reduce_floats(size_b + 1, (int)blocks));
        if (!part) return SAE_E_CUDA;
    }
    const size_t smem = (size_t)(256 * V + 256 / 32) * sizeof(float);
    if (vec)
        bias_act_bwd_kernel<4><<<blocks, 256, smem, st>>>(grad_out, out, grad_in, part, grad_bias != nullptr, size_v, cv, stride, alpha,
                                                         scale, noise, noise_div, round_tf32, act_mask);
    else
        bias_act_bwd_kernel<1><<<blocks, 256, smem, st>>>(grad_out, out, grad_in, part, grad_bias != nullptr, size_v, cv, stride, alpha,
                                                         scale, noise, noise_div, round_tf32, nullptr);
    int rc = check_launch("bias_act_backward");
    if (rc || !part) return rc;
    return det_reduce(grad_bias, size_b, noise ? grad_noise_weight : nullptr, part, size_b + 1, (int)blocks, st);
}

extern "C" int sae_modulate(const float* x, const float* s, float* out, int n, int64_t hw, int c, int round_tf32,
                            void* stream) {
    if (n == 0 || hw == 0) return SAE_OK;
    if (!x || !s || !out || n < 0 || hw < 0 || c <= 0) return fail(SAE_E_INVALID, "modulate: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    uintptr_t al = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(s);
    if (c % 4 == 0 && al % 16 == 0) {
        int64_t tv = (int64_t)n * hw * (c / 4);
        if (tv < ((int64_t)1 << 32))
            modulate_kernel<uint32_t><<<grid_for(tv, 256, 16), 256, 0, st>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<const float4*>(s),
                                                                            reinterpret_cast<float4*>(out), (uint32_t)tv, (uint32_t)hw, c / 4, round_tf32);
        else
            modulate_kernel<int64_t><<<grid_for(tv, 256, 16), 256, 0, st>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<const float4*>(s),
                                                                           reinterpret_cast<float4*>(out), tv, hw, c / 4, round_tf32);
    } else {
        int64_t t = (int64_t)n * hw * c;
        modulate_scalar_kernel<<<grid_for(t, 256), 256, 0, st>>>(x, s, out, t, hw, c, round_tf32);
    }
    return check_launch("modulate");
}

extern "C" int sae_modulate_backward(const float* dy, const float* x, const float* s, float* dx, float* ds,
                                     int n, int64_t hw, int c, int round_tf32, void* stream) {
    if (n == 0 || hw == 0) return SAE_OK;
    if (!dy || !x || !s || !dx || !ds || n < 0 || c <= 0) return fail(SAE_E_INVALID, "modulate_backward: bad arguments");
    if (c > 12000) return fail(SAE_E_UNSUPPORTED, "modulate_backward: more than 12000 channels");
    cudaStream_t st = (cudaStream_t)stream;
    uintptr_t al = reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx);
    const bool vec = (c % 4 == 0) && (al % 16 == 0);
    const int V = vec ? 4 : 1;
    // aim for ~4 CTAs per SM over the whole batch
    int64_t want = ((int64_t)sm_count() * 4 + n - 1) / n;
    if (want < 1) want = 1;
    int64_t pix_per_cta = (hw + want - 1) / want;
    if (pix_per_cta < 8) pix_per_cta = 8;
    unsigned chunks = (unsigned)((hw + pix_per_cta - 1) / pix_per_cta);
    dim3 grid(chunks, (unsigned)n);
    float* part = det_workspace(det_reduce_floats((int64_t)n * c, (int)chunks));
    if (!part) return SAE_E_CUDA;
    const size_t smem = (size_t)256 * V * sizeof(float);
    if (vec) modulate_bwd_kernel<4><<<grid, 256, smem, st>>>(dy, x, s, dx, part, hw, c / V, pix_per_cta, round_tf32);
    else     modulate_bwd_kernel<1><<<grid, 256, smem, st>>>(dy, x, s, dx, part, hw, c / V, pix_per_cta, round_tf32);
    int rc = check_launch("modulate_backward");
    if (rc) return rc;
    return det_reduce(ds, part, (int64_t)n * c, (int)chunks, st);
}

extern "C" int sae_add_scale(const float* a, const float* b, float* out, int64_t n, float scale, int round_tf32, void* stream) {
    if (n == 0) return SAE_OK;
    if (!a || !out || n < 0) return fail(SAE_E_INVALID, "add_scale: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    uintptr_t al = reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out);
    if (n % 4 == 0 && al % 16 == 0) add_scale_kernel<4><<<grid_for(n / 4, 256), 256, 0, st>>>(a, b, out, n / 4, scale, round_tf32);
    else add_scale_kernel<1><<<grid_for(n, 256), 256, 0, st>>>(a, b, out, n, scale, round_tf32);
    return check_launch("add_scale");
}

extern "C" int sae_upsample2x_add_scale(const float* skip, const float* res, float* out, int n, int h, int w, int c, float scale,
                                        int round_tf32, void* stream) {
    if (n == 0) return SAE_OK;
    if (!skip || !res || !out || n < 0 || h <= 0 || w <= 0 || c <= 0 || c % 4 != 0)
        return fail(SAE_E_INVALID, "upsample2x_add_scale: bad arguments (channels must be a multiple of 4)");
    if (((reinterpret_cast<uintptr_t>(skip) | reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(out)) & 15) != 0)
        return fail(SAE_E_INVALID, "upsample2x_add_scale: pointers must be 16-byte aligned");
    int64_t tv = (int64_t)n * 4 * h * w * (c / 4);
    upsample2x_add_kernel<<<grid_for(tv, 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(skip), reinterpret_cast<const float4*>(res), reinterpret_cast<float4*>(out), tv, h, w, c / 4,
        scale, round_tf32);
    return check_launch("upsample2x_add_scale");
}

extern "C" int sae_upsample2x_backward(const float* dy, float* dskip, int n, int h, int w, int c, float scale, int round_tf32,
                                       void* stream) {
    if (n == 0) return SAE_OK;
    if (!dy || !dskip || n < 0 || h <= 0 || w <= 0 || c <= 0 || c % 4 != 0)
        return fail(SAE_E_INVALID, "upsample2x_backward: bad arguments (channels must be a multiple of 4)");
    int64_t tv = (int64_t)n * h * w * (c / 4);
    upsample2x_bwd_kernel<<<grid_for(tv, 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(dy), reinterpret_cast<float4*>(dskip), tv, h, w, c / 4, scale, round_tf32);
    return check_launch("upsample2x_backward");
}

extern "C" int sae_pad_channels(const float* x, float* out, int64_t n, int64_t pixels, int c_in, int c_out,
                                int64_t stride_n, int64_t stride_c, int64_t stride_p, int round_tf32, void* stream) {
    using namespace sae;
    if (n == 0 || pixels == 0) return SAE_OK;
    if (!x || !out || n < 0 || pixels < 0 || c_in <= 0 || c_out < c_in || c_out % 4 != 0)
        return fail(SAE_E_INVALID, "pad_channels: bad arguments (0 < c_in <= c_out, c_out %% 4 == 0)");
    if ((reinterpret_cast<uintptr_t>(out) & 15) != 0) return fail(SAE_E_INVALID, "pad_channels: out must be 16-byte aligned");
    const int64_t tv = n * pixels * (c_out / 4);
    pad_channels_kernel<<<grid_for(tv, 256, 16), 256, 0, (cudaStream_t)stream>>>(x, reinterpret_cast<float4*>(out), tv, pixels, c_in,
                                                                                 c_out / 4, stride_n, stride_c, stride_p, round_tf32);
    return check_launch("pad_channels");
}

extern "C" int sae_reflect_pad(const float* x, float* out, int n, int h, int w, int c, int pad_l, int pad_r, int pad_t, int pad_b,
                               void* stream) {
    if (n == 0) return SAE_OK;
    if (!x || !out || n < 0 || h <= 0 || w <= 0 || c <= 0 || c % 4 != 0) return fail(SAE_E_INVALID, "reflect_pad: bad arguments (c %% 4 == 0)");
    if (pad_l < 0 || pad_r < 0 || pad_t < 0 || pad_b < 0 || pad_l >= w || pad_r >= w || pad_t >= h || pad_b >= h)
        return fail(SAE_E_INVALID, "reflect_pad: padding must be non-negative and smaller than the input");
    const int oh = h + pad_t + pad_b, ow = w + pad_l + pad_r;
    int64_t tv = (int64_t)n * oh * ow * (c / 4);
    if (tv >= ((int64_t)1 << 32)) return fail(SAE_E_UNSUPPORTED, "reflect_pad: tensor too large for 32-bit indexing");
    reflect_pad_kernel<<<grid_for(tv, 256, 16), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(out),
                                                                               (uint32_t)tv, h, w, c / 4, oh, ow, pad_l, pad_t);
    return check_launch("reflect_pad");
}

extern "C" int sae_reflect_pad_backward(const float* dy, float* dx, int n, int h, int w, int c, int pad_l, int pad_r, int pad_t,
                                        int pad_b, void* stream) {
    if (n == 0) return SAE_OK;
    if (!dy || !dx || n < 0 || h <= 0 || w <= 0 || c <= 0 || c % 4 != 0) return fail(SAE_E_INVALID, "reflect_pad_backward: bad arguments");
    if (pad_l < 0 || pad_r < 0 || pad_t < 0 || pad_b < 0 || pad_l >= w || pad_r >= w || pad_t >= h || pad_b >= h)
        return fail(SAE_E_INVALID, "reflect_pad_backward: padding must be non-negative and smaller than the input");
    const int oh = h + pad_t + pad_b, ow = w + pad_l + pad_r;
    int64_t tv = (int64_t)n * h * w * (c / 4);
    if ((int64_t)n * oh * ow * (c / 4) >= ((int64_t)1 << 32)) return fail(SAE_E_UNSUPPORTED, "reflect_pad_backward: tensor too large");
    reflect_pad_bwd_kernel<<<grid_for(tv, 256, 16), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(dy), reinterpret_cast<float4*>(dx),
                                                                                   (uint32_t)tv, h, w, c / 4, oh, ow, pad_l, pad_r, pad_t, pad_b);
    return check_launch("reflect_pad_backward");
}

extern "C" int sae_filter_prep(const float* w, float* out_krsc, float* out_crsk, int k, int c, int r, int s_, float scale,
                               int round_tf32, void* stream) {
    if (!w || !out_krsc || k <= 0 || c <= 0 || r <= 0 || s_ <= 0) return fail(SAE_E_INVALID, "filter_prep: bad arguments");
    if ((int64_t)k * c * r * s_ >= ((int64_t)1 << 31)) return fail(SAE_E_UNSUPPORTED, "filter_prep: filter too large");
    filter_prep_kernel<<<grid_for((int64_t)k * c * r * s_, 256), 256, 0, (cudaStream_t)stream>>>(w, out_krsc, out_crsk, k, c, r * s_, scale,
                                                                                               round_tf32);
    return check_launch("filter_prep");
}

extern "C" int sae_filter_modulate(const float* w_krsc, const float* s, float* out_krsc, float* out_crsk, int n, int k, int c,
                                   int r, int s_, int round_tf32, void* stream) {
    if (n == 0) return SAE_OK;
    if (!w_krsc || !s || (!out_krsc && !out_crsk) || n < 0 || k <= 0 || c <= 0 || r <= 0 || s_ <= 0)
        return fail(SAE_E_INVALID, "filter_modulate: bad arguments");
    if ((int64_t)k * c * r * s_ >= ((int64_t)1 << 31) || n > 65535) return fail(SAE_E_UNSUPPORTED, "filter_modulate: too large");
    dim3 grid(grid_for((int64_t)k * c * r * s_, 256, 2), (unsigned)n);
    filter_modulate_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w_krsc, s, out_krsc, out_crsk, k, c, r * s_, round_tf32);
    return check_launch("filter_modulate");
}

extern "C" int sae_filter_unprep(const float* d_krsc, float* d_w, int k, int c, int r, int s_, float scale, void* stream) {
    if (!d_krsc || !d_w || k <= 0 || c <= 0 || r <= 0 || s_ <= 0) return fail(SAE_E_INVALID, "filter_unprep: bad arguments");
    if ((int64_t)k * c * r * s_ >= ((int64_t)1 << 31)) return fail(SAE_E_UNSUPPORTED, "filter_unprep: filter too large");
    filter_unprep_kernel<<<grid_for((int64_t)k * c * r * s_, 256), 256, 0, (cudaStream_t)stream>>>(d_krsc, d_w, k, c, r * s_, scale);
    return check_launch("filter_unprep");
}

extern "C" int sae_round_tf32(const float* x, float* out, int64_t n, void* stream) {
    return sae_add_scale(x, nullptr, out, n, 1.0f, 1, stream);
}

extern "C" int sae_bucket_pack(const float* const* ptrs, const int64_t* offsets, const int64_t* sizes, int n,
                               float* bucket, int64_t total, void* stream) {
    if (n == 0) return SAE_OK;
    if (!ptrs || !offsets || !sizes || !bucket || n < 0 || total < 0) return fail(SAE_E_INVALID, "bucket_pack: bad arguments");
    dim3 grid(64, (unsigned)n);
    bucket_copy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(const_cast<float* const*>(ptrs), offsets, sizes, bucket, 1.f, 1);
    return check_launch("bucket_pack");
}

extern "C" int sae_bucket_unpack(float* const* ptrs, const int64_t* offsets, const int64_t* sizes, int n,
                                 const float* bucket, int64_t total, float scale, void* stream) {
    if (n == 0) return SAE_OK;
    if (!ptrs || !offsets || !sizes || !bucket || n < 0 || total < 0) return fail(SAE_E_INVALID, "bucket_unpack: bad arguments");
    dim3 grid(64, (unsigned)n);
    bucket_copy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ptrs, offsets, sizes, const_cast<float*>(bucket), scale, 0);
    return check_launch("bucket_unpack");
}
