// Generic implicit-GEMM convolution on NHWC fp32 with mma.sync TF32 (m16n8k8) — the shape-complete
// kernel of the conv family (any stride / padding / channel count, forward, data-gradient incl.
// transposed convolution, weight-gradient).  The tcgen05/TMA kernels in conv_tcgen05.cu take over
// for the shapes that carry the FLOPs (SURVEY.md Appendix A); this file covers what they cannot
// tile: Cin = 3 (FromRGB), Cout = 3 / 1 (ToRGB, final linears), 7x7 / 3x3 maps, fractional strides.
//
// fprop / dgrad share one "gather GEMM":  C[m, n] = sum_k A[m, k] * B[n, k]
//   m = output pixel (n_img, oy, ox), k = (tap r,s ; source channel c), A gathered on the fly:
//   iy = (oy*SY + OFFY + r*DY) / DIV  (only if divisible and in range), same in x.
//   fprop: SY = stride, DY = +1, OFF = -pad, DIV = 1;  dgrad: SY = 1, DY = -1, OFF = +pad, DIV = stride.
// wgrad:  dW[o, (r,s,c)] += sum_pixels dy[pixel, o] * x_gathered[pixel, (r,s,c)], split over pixels,
//   each split writes its partial dW to its own workspace slice; det_reduce adds the slices in split order.
// Operands are rounded to TF32 (cvt.rna) when fragments are loaded, accumulation is fp32.
#include "conv_internal.cuh"

namespace sae {

constexpr int BM = 128, BK = 32, LDS_K = BK + 4, STAGES = 3, NTHREADS = 256;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool pred) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    int sz = pred ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

__device__ __forceinline__ uint32_t to_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// ------------------------------------------------------------------------------------------------
template <int BN, bool VEC>
__global__ void __launch_bounds__(NTHREADS)
conv_gather_kernel(const float* __restrict__ src, const float* __restrict__ wmat, float* __restrict__ out,
                   GatherParams p, EpiParams e) {
    extern __shared__ __align__(16) float smem[];
    float* As = smem;                               // [STAGES][BM][LDS_K]
    float* Bs = smem + STAGES * BM * LDS_K;         // [STAGES][BN][LDS_K]

    constexpr int WARPS_N = BN / 32;
    constexpr int WARPS_M = 8 / WARPS_N;
    constexpr int WM = BM / WARPS_M;                // rows per warp
    constexpr int MT = WM / 16;                     // m16 tiles per warp
    constexpr int NT = 4;                           // n8 tiles per warp (32 columns)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp / WARPS_N, wn = warp % WARPS_N;
    const int g = lane >> 2, t = lane & 3;

    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int KB_total = (p.K + BK - 1) / BK;
    // split-K (gridDim.z > 1, small-M GEMMs such as the style / head linears): this CTA reduces k-blocks
    // [kb_begin, kb_begin + KB) and writes its partial tile to slice blockIdx.z of the workspace ``out`` points to
    const int kb_per = (KB_total + (int)gridDim.z - 1) / (int)gridDim.z;
    const int kb_begin = (int)blockIdx.z * kb_per;
    const int KB = max(0, min(kb_per, KB_total - kb_begin));
    const bool split = gridDim.z > 1;

    // per-thread row bookkeeping for the vector loader: rows (tid>>3) + j*32, j = 0..3
    int row_oy[4], row_ox[4];
    int64_t row_base[4];
    bool row_ok[4];
    if (VEC) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int64_t m = m0 + (tid >> 3) + j * 32;
            row_ok[j] = m < p.M;
            int64_t mm = row_ok[j] ? m : 0;
            int ox = (int)(mm % p.OW);
            int64_t q = mm / p.OW;
            int oy = (int)(q % p.OH);
            int64_t ni = q / p.OH;
            row_oy[j] = oy * p.SY + p.OFFY;
            row_ox[j] = ox * p.SY + p.OFFX;
            row_base[j] = ni * (int64_t)p.IH * p.IW;
        }
    }

    auto load_stage = [&](int stage, int kb_rel) {
        const int kb = kb_begin + kb_rel;
        float* as = As + stage * BM * LDS_K;
        float* bs = Bs + stage * BN * LDS_K;
        if (VEC) {
            const int kq = tid & 7;
            const int k = kb * BK + kq * 4;
            const bool kok = k < p.K;
            int tap = kok ? k / p.Cs : 0;
            int c = k - tap * p.Cs;
            int r = tap / p.S, s = tap - r * p.S;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int row = (tid >> 3) + j * 32;
                int iy = row_oy[j] + r * p.DY, ix = row_ox[j] + s * p.DY;
                bool ok = kok && row_ok[j] && iy >= 0 && ix >= 0;
                if (p.DIV > 1) {
                    ok = ok && (iy % p.DIV == 0) && (ix % p.DIV == 0);
                    iy /= p.DIV; ix /= p.DIV;
                }
                ok = ok && iy < p.IH && ix < p.IW;
                const float* gp = ok ? src + (row_base[j] + (int64_t)iy * p.IW + ix) * p.Cs + c : src;
                cp_async16(as + row * LDS_K + kq * 4, gp, ok);
            }
#pragma unroll
            for (int j = 0; j < BN / 32; ++j) {
                int row = (tid >> 3) + j * 32;
                int n = n0 + row;
                bool ok = kok && n < p.Ncol;
                const float* gp = ok ? wmat + (int64_t)n * p.K + k : wmat;
                cp_async16(bs + row * LDS_K + kq * 4, gp, ok);
            }
        } else {
            // scalar path (channel counts that are not multiples of 4): plain loads
            for (int f = tid; f < BM * BK; f += NTHREADS) {
                int row = f >> 5, kk = f & 31;
                int k = kb * BK + kk;
                int64_t m = m0 + row;
                float v = 0.f;
                if (k < p.K && m < p.M) {
                    int tap = k / p.Cs, c = k - tap * p.Cs;
                    int r = tap / p.S, s = tap - r * p.S;
                    int ox = (int)(m % p.OW);
                    int64_t q = m / p.OW;
                    int oy = (int)(q % p.OH);
                    int64_t ni = q / p.OH;
                    int iy = oy * p.SY + p.OFFY + r * p.DY, ix = ox * p.SY + p.OFFX + s * p.DY;
                    bool ok = iy >= 0 && ix >= 0;
                    if (p.DIV > 1) {
                        ok = ok && (iy % p.DIV == 0) && (ix % p.DIV == 0);
                        iy /= p.DIV; ix /= p.DIV;
                    }
                    ok = ok && iy < p.IH && ix < p.IW;
                    if (ok) v = __ldg(src + ((ni * p.IH + iy) * (int64_t)p.IW + ix) * p.Cs + c);
                }
                as[row * LDS_K + kk] = v;
            }
            for (int f = tid; f < BN * BK; f += NTHREADS) {
                int row = f >> 5, kk = f & 31;
                int k = kb * BK + kk, n = n0 + row;
                float v = 0.f;
                if (k < p.K && n < p.Ncol) v = __ldg(wmat + (int64_t)n * p.K + k);
                bs[row * LDS_K + kk] = v;
            }
        }
    };

    float acc[MT][NT][4];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < KB) load_stage(s, s);
        cp_async_commit();
    }
    for (int kb = 0; kb < KB; ++kb) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            int nk = kb + STAGES - 1;
            if (nk < KB) load_stage(nk % STAGES, nk);
            cp_async_commit();
        }
        const float* as = As + (kb % STAGES) * BM * LDS_K + (wm * WM) * LDS_K;
        const float* bs = Bs + (kb % STAGES) * BN * LDS_K + (wn * 32) * LDS_K;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            uint32_t af[MT][4], bf[NT][2];
#pragma unroll
            for (int i = 0; i < MT; ++i) {
                const float* a = as + (i * 16 + g) * LDS_K + ks * 8 + t;
                af[i][0] = to_tf32(a[0]);
                af[i][1] = to_tf32(a[8 * LDS_K]);
                af[i][2] = to_tf32(a[4]);
                af[i][3] = to_tf32(a[8 * LDS_K + 4]);
            }
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                const float* b = bs + (j * 8 + g) * LDS_K + ks * 8 + t;
                bf[j][0] = to_tf32(b[0]);
                bf[j][1] = to_tf32(b[4]);
            }
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < NT; ++j) mma_tf32(acc[i][j], af[i], bf[j]);
        }
    }
    cp_async_wait<0>();

    // epilogue
    if (split) {
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                int64_t m = m0 + wm * WM + i * 16 + g + h * 8;
                if (m >= p.M) continue;
#pragma unroll
                for (int j = 0; j < NT; ++j)
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        int col = n0 + wn * 32 + j * 8 + 2 * t + u;
                        if (col < p.Ncol) out[((int64_t)blockIdx.z * p.M + m) * p.Ncol + col] = acc[i][j][h * 2 + u];
                    }
            }
        return;
    }
    if (p.Ncol % 4 == 0) {
        // stage the tile in shared memory (the pipeline buffers are free now) and write whole rows with float4 stores:
        // the m16n8 fragment layout would otherwise scatter 8-byte stores over 8 rows per instruction
        constexpr int LDC = BN + 4;
        __syncthreads();
        float* cs = smem;
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = wm * WM + i * 16 + g + h * 8;
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    const int c = wn * 32 + j * 8 + 2 * t;
                    *reinterpret_cast<float2*>(cs + r * LDC + c) = make_float2(acc[i][j][h * 2], acc[i][j][h * 2 + 1]);
                }
            }
        __syncthreads();
        constexpr int C4 = BN / 4;
        for (int f = tid; f < BM * C4; f += NTHREADS) {
            const int r = f / C4, c4 = f - r * C4;
            const int64_t m = m0 + r;
            const int col = n0 + c4 * 4;
            if (m >= p.M || col >= p.Ncol) continue;
            float4 v = *reinterpret_cast<const float4*>(cs + r * LDC + c4 * 4);
            v.x = apply_epi(e, v.x, m, col, p.Ncol);
            v.y = apply_epi(e, v.y, m, col + 1, p.Ncol);
            v.z = apply_epi(e, v.z, m, col + 2, p.Ncol);
            v.w = apply_epi(e, v.w, m, col + 3, p.Ncol);
            *reinterpret_cast<float4*>(out + m * p.Ncol + col) = v;
        }
        return;
    }
    const bool even = (p.Ncol % 2 == 0);
#pragma unroll
    for (int i = 0; i < MT; ++i) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int64_t m = m0 + wm * WM + i * 16 + g + h * 8;
            if (m >= p.M) continue;
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                int col = n0 + wn * 32 + j * 8 + 2 * t;
                if (col >= p.Ncol) continue;
                float v0 = apply_epi(e, acc[i][j][h * 2 + 0], m, col, p.Ncol);
                float* dst = out + m * p.Ncol + col;
                if (col + 1 < p.Ncol) {
                    float v1 = apply_epi(e, acc[i][j][h * 2 + 1], m, col + 1, p.Ncol);
                    if (even) *reinterpret_cast<float2*>(dst) = make_float2(v0, v1);
                    else { dst[0] = v0; dst[1] = v1; }
                } else {
                    dst[0] = v0;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// wgrad: C[o, n=(tap,c)] += sum_{pixel} dy[pixel, o] * x[gather(pixel, tap), c]
struct WgradParams {
    int N, H, W, C;       // x
    int Ko, R, S;         // dy channels / filter
    int P, Q;
    int stride, pad_t, pad_l;
    int Ncol;             // R*S*C
    int64_t Mpix;         // N*P*Q
    int64_t chunk;        // pixels per blockIdx.z (multiple of BK)
};
constexpr int LDS_M = 128 + 8;

template <bool VA, bool VB>
__global__ void __launch_bounds__(NTHREADS)
conv_wgrad_kernel(const float* __restrict__ dy, const float* __restrict__ x, float* __restrict__ dw, WgradParams p) {
    extern __shared__ __align__(16) float smem[];
    float* As = smem;                              // [STAGES][BK][LDS_M]   (k = pixel, m = out channel)
    float* Bs = smem + STAGES * BK * LDS_M;        // [STAGES][BK][LDS_M]   (k = pixel, n = (tap, c))

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp >> 2, wn = warp & 3;       // 2 x 4 warps, warp tile 64 x 32
    const int g = lane >> 2, t = lane & 3;
    const int o0 = blockIdx.x * 128;
    const int n0 = blockIdx.y * 128;
    const int64_t pix0 = (int64_t)blockIdx.z * p.chunk;
    int64_t pix1 = pix0 + p.chunk;
    if (pix1 > p.Mpix) pix1 = p.Mpix;
    const int KB = (int)((pix1 - pix0 + BK - 1) / BK);

    // vector loader bookkeeping: this thread always serves column quad (tid & 31)
    const int cq = tid & 31;
    int b_tap_r = 0, b_tap_s = 0, b_c = 0;
    bool b_colok = false;
    if (VB) {
        int n = n0 + cq * 4;
        b_colok = n < p.Ncol;
        int tap = b_colok ? n / p.C : 0;
        b_c = n - tap * p.C;
        b_tap_r = tap / p.S;
        b_tap_s = tap - b_tap_r * p.S;
    }

    auto load_stage = [&](int stage, int kb) {
        float* as = As + stage * BK * LDS_M;
        float* bs = Bs + stage * BK * LDS_M;
        if (VA) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int kp = (tid >> 5) + j * 8;
                int64_t pix = pix0 + (int64_t)kb * BK + kp;
                int o = o0 + cq * 4;
                bool ok = pix < pix1 && o < p.Ko;
                const float* gp = ok ? dy + pix * p.Ko + o : dy;
                cp_async16(as + kp * LDS_M + cq * 4, gp, ok);
            }
        } else {
            for (int f = tid; f < BK * 128; f += NTHREADS) {
                int kp = f >> 7, mm = f & 127;
                int64_t pix = pix0 + (int64_t)kb * BK + kp;
                int o = o0 + mm;
                float v = 0.f;
                if (pix < pix1 && o < p.Ko) v = __ldg(dy + pix * p.Ko + o);
                as[kp * LDS_M + mm] = v;
            }
        }
        if (VB) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int kp = (tid >> 5) + j * 8;
                int64_t pix = pix0 + (int64_t)kb * BK + kp;
                bool ok = b_colok && pix < pix1;
                const float* gp = x;
                if (ok) {
                    int q = (int)(pix % p.Q);
                    int64_t r2 = pix / p.Q;
                    int pp = (int)(r2 % p.P);
                    int64_t ni = r2 / p.P;
                    int iy = pp * p.stride - p.pad_t + b_tap_r;
                    int ix = q * p.stride - p.pad_l + b_tap_s;
                    ok = iy >= 0 && ix >= 0 && iy < p.H && ix < p.W;
                    if (ok) gp = x + ((ni * p.H + iy) * (int64_t)p.W + ix) * p.C + b_c;
                }
                cp_async16(bs + kp * LDS_M + cq * 4, gp, ok);
            }
        } else {
            for (int f = tid; f < BK * 128; f += NTHREADS) {
                int kp = f >> 7, nn = f & 127;
                int64_t pix = pix0 + (int64_t)kb * BK + kp;
                int n = n0 + nn;
                float v = 0.f;
                if (pix < pix1 && n < p.Ncol) {
                    int tap = n / p.C, c = n - tap * p.C;
                    int r = tap / p.S, s = tap - r * p.S;
                    int q = (int)(pix % p.Q);
                    int64_t r2 = pix / p.Q;
                    int pp = (int)(r2 % p.P);
                    int64_t ni = r2 / p.P;
                    int iy = pp * p.stride - p.pad_t + r;
                    int ix = q * p.stride - p.pad_l + s;
                    if (iy >= 0 && ix >= 0 && iy < p.H && ix < p.W)
                        v = __ldg(x + ((ni * p.H + iy) * (int64_t)p.W + ix) * p.C + c);
                }
                bs[kp * LDS_M + nn] = v;
            }
        }
    };

    float acc[4][4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[i][j][q] = 0.f;

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < KB) load_stage(s, s);
        cp_async_commit();
    }
    for (int kb = 0; kb < KB; ++kb) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            int nk = kb + STAGES - 1;
            if (nk < KB) load_stage(nk % STAGES, nk);
            cp_async_commit();
        }
        const float* as = As + (kb % STAGES) * BK * LDS_M + wm * 64;
        const float* bs = Bs + (kb % STAGES) * BK * LDS_M + wn * 32;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            uint32_t af[4][4], bf[4][2];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float* a = as + (ks * 8 + t) * LDS_M + i * 16 + g;
                af[i][0] = to_tf32(a[0]);
                af[i][1] = to_tf32(a[8]);
                af[i][2] = to_tf32(a[4 * LDS_M]);
                af[i][3] = to_tf32(a[4 * LDS_M + 8]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float* b = bs + (ks * 8 + t) * LDS_M + j * 8 + g;
                bf[j][0] = to_tf32(b[0]);
                bf[j][1] = to_tf32(b[4 * LDS_M]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) mma_tf32(acc[i][j], af[i], bf[j]);
        }
    }
    cp_async_wait<0>();

#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int o = o0 + wm * 64 + i * 16 + g + h * 8;
            if (o >= p.Ko) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    int n = n0 + wn * 32 + j * 8 + 2 * t + u;
                    if (n < p.Ncol) dw[((int64_t)blockIdx.z * p.Ko + o) * p.Ncol + n] = acc[i][j][h * 2 + u];
                }
        }
}

// ------------------------------------------------------------------------------------------------
template <int BN, bool VEC>
static int launch_gather(const float* src, const float* wmat, float* out, const GatherParams& p, const EpiParams& e,
                         cudaStream_t st) {
    size_t smem = (size_t)STAGES * (BM + BN) * LDS_K * sizeof(float);
    static bool attr_done = false;   // benign race: idempotent
    if (!attr_done) {
        SAE_CUDA_TRY(cudaFuncSetAttribute(conv_gather_kernel<BN, VEC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = true;
    }
    dim3 grid((unsigned)((p.M + BM - 1) / BM), (unsigned)((p.Ncol + BN - 1) / BN));
    // small-M, deep-K problems (linears): split K so more than a handful of SMs work on them
    const int kblocks = (p.K + BK - 1) / BK;
    const bool plain = !e.bias && !e.noise && !e.residual && e.act == 1 && e.gain == 1.f;
    if (plain && grid.x * grid.y <= 16 && kblocks >= 16) {
        unsigned z = (unsigned)(kblocks / 4);
        if (z > 32) z = 32;
        if (z > 1) grid.z = z;
    }
    if (grid.z == 1) {
        conv_gather_kernel<BN, VEC><<<grid, NTHREADS, smem, st>>>(src, wmat, out, p, e);
        return check_launch("conv_gather");
    }
    // split K: per-split partial tiles, then the output = their sum in split order
    float* part = det_workspace(det_reduce_floats(p.M * p.Ncol, (int)grid.z));
    if (!part) return SAE_E_CUDA;
    SAE_CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)p.M * p.Ncol * sizeof(float), st));
    conv_gather_kernel<BN, VEC><<<grid, NTHREADS, smem, st>>>(src, wmat, part, p, e);
    int rc = check_launch("conv_gather");
    if (rc) return rc;
    return det_reduce(out, part, p.M * p.Ncol, (int)grid.z, st);
}

int conv_gather_dispatch(const float* src, const float* wmat, float* out, const GatherParams& p, const EpiParams& e,
                         cudaStream_t st) {
    if (p.M == 0 || p.Ncol == 0) return SAE_OK;
    const bool aligned = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(wmat)) & 15) == 0;
    const bool vec = (p.Cs % 4 == 0) && aligned;
    if (p.Ncol > 64) return vec ? launch_gather<128, true>(src, wmat, out, p, e, st) : launch_gather<128, false>(src, wmat, out, p, e, st);
    if (p.Ncol > 32) return vec ? launch_gather<64, true>(src, wmat, out, p, e, st) : launch_gather<64, false>(src, wmat, out, p, e, st);
    return vec ? launch_gather<32, true>(src, wmat, out, p, e, st) : launch_gather<32, false>(src, wmat, out, p, e, st);
}

template <bool VA, bool VB>
static int launch_wgrad(const float* dy, const float* x, float* dw, const WgradParams& p, unsigned splits, cudaStream_t st) {
    size_t smem = (size_t)STAGES * 2 * BK * LDS_M * sizeof(float);
    static bool attr_done = false;
    if (!attr_done) {
        SAE_CUDA_TRY(cudaFuncSetAttribute(conv_wgrad_kernel<VA, VB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = true;
    }
    dim3 grid((unsigned)((p.Ko + 127) / 128), (unsigned)((p.Ncol + 127) / 128), splits);
    float* part = det_workspace(det_reduce_floats((int64_t)p.Ko * p.Ncol, (int)splits));
    if (!part) return SAE_E_CUDA;
    conv_wgrad_kernel<VA, VB><<<grid, NTHREADS, smem, st>>>(dy, x, part, p);
    int rc = check_launch("conv_wgrad");
    if (rc) return rc;
    return det_reduce(dw, part, (int64_t)p.Ko * p.Ncol, (int)splits, st);
}

int conv_wgrad_generic(const float* dy, const float* x, float* dw, const sae_conv_geom* g, cudaStream_t st) {
    WgradParams p;
    p.N = g->N; p.H = g->H; p.W = g->W; p.C = g->C; p.Ko = g->K; p.R = g->R; p.S = g->S; p.P = g->P; p.Q = g->Q;
    p.stride = g->stride; p.pad_t = g->pad_t; p.pad_l = g->pad_l;
    p.Ncol = g->R * g->S * g->C;
    p.Mpix = (int64_t)g->N * g->P * g->Q;
    if (p.Mpix == 0 || p.Ko == 0 || p.Ncol == 0) return SAE_OK;
    int64_t tiles = (int64_t)((p.Ko + 127) / 128) * ((p.Ncol + 127) / 128);
    int64_t want = ((int64_t)sm_count() * 2 + tiles - 1) / tiles;      // ~2 CTAs per SM
    int64_t kblocks = (p.Mpix + BK - 1) / BK;
    if (want > kblocks) want = kblocks;
    if (want < 1) want = 1;
    if (want > 2048) want = 2048;
    int64_t kb_per = (kblocks + want - 1) / want;
    p.chunk = kb_per * BK;
    unsigned splits = (unsigned)((p.Mpix + p.chunk - 1) / p.chunk);
    const bool al = ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x)) & 15) == 0;
    const bool va = (p.Ko % 4 == 0) && al, vb = (p.C % 4 == 0) && al;
    if (va && vb) return launch_wgrad<true, true>(dy, x, dw, p, splits, st);
    if (va) return launch_wgrad<true, false>(dy, x, dw, p, splits, st);
    if (vb) return launch_wgrad<false, true>(dy, x, dw, p, splits, st);
    return launch_wgrad<false, false>(dy, x, dw, p, splits, st);
}

}  // namespace sae
