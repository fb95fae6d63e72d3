// Weight-gradient of the convolution on tcgen05 tensor cores (kind::tf32), TMA-fed, split over pixels.
//
//   dW[o, (r,s), c] += sum_{pixels (n,p,q)}  dy[n,p,q,o] * x[n, p*st - pad_t + r, q*st - pad_l + s, c]
//
// GEMM view per filter tap: M = out channels (128 per CTA), N = in channels (128 per CTA), K = pixels.
// Both operands are "MN-major" for the tensor core (the contiguous NHWC dimension is the channel = M resp. N
// dimension, the reduction runs over pixels), which tcgen05 supports for tf32 through the transposed
// (a_major = b_major = MN) shared-memory descriptors — so the NHWC activations are consumed as they are, no
// transposes materialised:
//   * A stage  = dy box of 32 pixels x 128 channels  = four 32-channel sub-tiles of 32 ch x 32 px (SWIZZLE_128B_ATOM_32B — the
//     only layout tcgen05 accepts for MN-major 32-bit operands), fetched by ONE TMA instruction through a 5-D tensor map
//     whose outermost dimension walks the sub-tiles (the single producer thread is issue-bound otherwise, see the kernel)
//   * B stages = for each of the (up to 3) taps of this CTA's tap group, the x box shifted by the tap (one instruction each);
//     out-of-bounds pixels are zero-filled by TMA (= the conv padding), element stride = conv stride
//   * layers with 256 out channels per tile pair run as CTA pairs (cta_group::2, wgrad_tc_kernel<2>): half of every x tile
//     per CTA, a 5-deep ring
//   * one TMEM accumulator (128 x 128 fp32 = 128 columns) per tap; the dy tile is reused by all taps of the group
//   * grid = (M tiles x N tiles, tap groups, pixel splits); every split stores its partial dW straight from the TMEM read
//     into its own workspace slice, and det_reduce adds the slices to dW in split order (no float atomics: the result is
//     the same from run to run).
#include "tc_common.cuh"

namespace sae {

constexpr int WG_THREADS = 192;
constexpr int WG_KPIX = 32;                        // pixels per pipeline stage
constexpr int WG_SUB = WG_KPIX * 128;              // one 32-channel sub-tile: 32 rows x 128 B = 4 KB
constexpr int WG_OPER = 4 * WG_SUB;                // 128 channels: 16 KB
constexpr int WG_MAX_GROUP = 3;
constexpr int WG_STAGES = 3;

struct WgParams {
    int tw, th, tn;                  // pixel box of a K chunk (tw*th*tn == 32)
    int tiles_w, tiles_h, tiles_n;   // over the OUTPUT (dy) pixel space
    int chunks_total, chunks_per_split;
    int stride, pad_t, pad_l;
    int R, S;
    int Ko, C;                       // channels of dy / x
    int group_taps;                  // taps per CTA (tap group); group y covers taps [y*group_taps, ...)
    int ntaps;
    int n_tiles_c;                   // number of 128-wide tiles along C
    int cpt;                         // 32-channel sub-tiles per tap inside an accumulator: min(C,128)/32
                                     // (narrow layers pack 4/cpt taps side by side into the 128 N-columns)
    int shared_b;                    // 1: the 3 horizontal taps of a filter row read ONE 40-pixel x window per sub-tile
                                     //    (descriptor start shifted by s pixel rows) instead of 3 separate 32-pixel boxes
    // style-modulated convolution (stylegan2_layers.py:284-323 as "dense conv of x * s with a shared filter W"): x arrives
    // UNSCALED.  The accumulators are drained once per image n (a CTA's chunk range is cut at image boundaries), and the
    // drain forms both gradients from G_n[k,tap,c] = sum_pixels dy x:   dW[k,tap,c] += s[n,c] G_n,
    // ds[n,c] += sum_{k,tap} W[k,tap,c] G_n.  No modulated copy of x, no per-sample weight-gradient array.
    int chunks_per_image;            // > 0 selects that mode (tn == 1)
    const float* mod_s;              // [N, C]
    const float* mod_w;              // [Ko, taps, C], the filter the forward pass used
    float* mod_ds;                   // partial terms [img][split - first split of img][out tile][tap group][warp][C]
    int ds_kmax, ds_tiles_o;         // extents of those partials: splits per image, 128-row output tiles
    int64_t dw_numel;                // Ko * taps * C: one workspace slice of partial dW
    int five_d;                      // pair mode: the tensor maps are the 5-D views (one TMA instruction per operand tile)
};

constexpr int WG_WIN = 40;                         // pixels per shared window (32 + 2 halo, rounded up to a multiple of 8)
constexpr int WG_WSUB = WG_WIN * 128;              // 5 KB per 32-channel sub-tile

__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t saddr) {
    // MN-major 32-bit operands have exactly one legal shared-memory layout on tcgen05: the 128-byte swizzle with
    // 32-byte atoms (descriptor layout type 1, TMA mode SWIZZLE_128B_ATOM_32B).  Atom = 32 fp32 along M/N (128 B) x 4
    // along K; next atom along M/N: LBO = 4096 B (the next 32-channel sub-tile); next 4 pixels along K: SBO = 512 B.
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(WG_SUB >> 4) << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}

__device__ __forceinline__ uint64_t make_desc_mn_win(uint32_t saddr, int use_base_offset) {
    // same layout, sub-tiles WG_WSUB apart, start address on an arbitrary 128-byte pixel row: the swizzle is a function
    // of the absolute shared-memory address, the descriptor's base-offset field carries the row phase of the start
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(WG_WSUB >> 4) << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    if (use_base_offset) d |= (uint64_t)((saddr >> 7) & 7) << 49;
    d |= (uint64_t)1 << 61;
    return d;
}

// CG = 1: one CTA per (128 out channels x 128 in channels x tap group) tile.
// CG = 2: a CTA pair (tcgen05 cta_group::2) owns 256 out channels x 128 in channels: each CTA loads the dy sub-tiles of ITS
//   128 out channels and HALF of every x tile (64 of the 128 in channels; the M = 256 instruction reads both CTAs' shared
//   memory), so the x bytes per MAC halve — what the stride-2 layers need, whose x tiles are one TMA box per tap (element
//   stride 2): 64 KB -> 40 KB per 32-pixel chunk and CTA, and a 5-deep ring instead of 3.
template <int CG> constexpr int wg_stages() { return CG == 2 ? 5 : WG_STAGES; }
template <int CG> constexpr int wg_stage_bytes() { return WG_OPER + WG_MAX_GROUP * (4 / CG) * WG_SUB; }       // 64 KB / 40 KB
template <int CG> constexpr size_t wg_smem_bytes() { return (size_t)wg_stages<CG>() * wg_stage_bytes<CG>() + 1024 + 256; }

template <int CG>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x,
                float* __restrict__ dw, const WgParams p) {
    constexpr int STAGES = wg_stages<CG>();
    constexpr int STAGE_BYTES = wg_stage_bytes<CG>();
    constexpr int BSUB = 4 / CG;                                   // 32-channel x sub-tiles this CTA loads per tap
    // D fp32, A/B tf32, A and B MN-major (bits 15, 16), N = 128, M = 128 per CTA
    constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((128u >> 3) << 17) | (((128u * CG) >> 4) << 24);
    constexpr uint32_t TMEM_COLS = 512;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_full = base + STAGES * STAGE_BYTES;
    const uint32_t bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_acc = bar_empty + 8 * STAGES;
    const uint32_t bar_drained = bar_acc + 8;          // modulated mode: the epilogue(s) have emptied the accumulators
    const uint32_t tmem_slot = bar_drained + 8;
    uint8_t* smem_gen = smem_raw + (base - smem_u32(smem_raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
    const bool leader = rank == 0;
    const int unit = (int)blockIdx.x / CG;                          // (out-channel tile [pair], in-channel tile)
    const int tile_o = unit / p.n_tiles_c, tile_c = unit % p.n_tiles_c;
    const int o0 = (tile_o * CG + rank) * 128, c0 = tile_c * 128;
    const int tap0 = blockIdx.y * p.group_taps;
    const int ntap = min(p.group_taps, p.ntaps - tap0);       // taps handled by this CTA
    const int tpa = 4 / p.cpt;                                 // taps per accumulator
    const int nacc = (ntap + tpa - 1) / tpa;                   // accumulators in use (<= 3)
    const int nslots = ntap * p.cpt;                           // valid 32-column B sub-tiles (CG = 2: cpt == 4)
    const int chunk_begin = blockIdx.z * p.chunks_per_split;
    const int chunk_end = min(chunk_begin + p.chunks_per_split, p.chunks_total);
    const int KB = chunk_end - chunk_begin;
    // bytes one CTA lands per stage
    const uint32_t stage_tx = p.shared_b ? (uint32_t)(WG_OPER + BSUB * WG_WSUB) : (uint32_t)WG_OPER + (uint32_t)(nslots / CG) * WG_SUB;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_dy) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        mbar_init(bar_acc, 1);
        mbar_init(bar_drained, CG);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if (CG == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));

    // loads: CG = 2 credits the leader's barrier (which expects both CTAs' bytes)
    auto load = [&](uint32_t dst, const CUtensorMap* map, uint32_t bar, int a, int b, int c, int d) {
        if (CG == 2) tma2_load_4d(dst, map, bar, a, b, c, d); else tma_load_4d(dst, map, bar, a, b, c, d);
    };

    if (KB > 0) {
        if (warp == 0) {
            if (elect_one()) {
                // chunk -> (column tile, row tile, image tile), advanced incrementally (three integer divisions per stage
                // were a measurable share of this single thread's issue time at stride 2)
                int tq, tp, tnb;
                { int ch = chunk_begin; tq = ch % p.tiles_w; ch /= p.tiles_w; tp = ch % p.tiles_h; tnb = ch / p.tiles_h; }
                for (int kb = 0; kb < KB; ++kb) {
                    const int s = kb % STAGES;
                    const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1u);
                    const int q0 = tq * p.tw, p0 = tp * p.th, n0 = tnb * p.tn;
                    if (++tq == p.tiles_w) { tq = 0; if (++tp == p.tiles_h) { tp = 0; ++tnb; } }
                    const uint32_t sa = base + (uint32_t)s * STAGE_BYTES;
                    if (leader) mbar_expect_tx(bar_full + 8 * s, CG * stage_tx);
                    if (p.five_d) {
                        // 5-D tensor maps whose outermost dimension walks the 32-channel sub-tiles (128 bytes apart in memory,
                        // WG_SUB / WG_WSUB apart in shared memory): one TMA instruction per operand tile instead of one per
                        // sub-tile — e.g. 4 instead of 10 per stage for a CTA of a pair at stride 2.  The producer is ONE thread; at
                        // ~90 clk of issue per bulk-tensor instruction ten of them filled the 768 clk a stage's MMAs take
                        // (profiles/r2_s2_family_call18.txt: 625 -> 721 TFLOP/s from this alone).
                        auto load5 = [&](uint32_t dst, const CUtensorMap* map, int a, int b, int c, int d, int e) {
                            if (CG == 2) tma2_load_5d(dst, map, bar_full + 8 * s, a, b, c, d, e); else tma_load_5d(dst, map, bar_full + 8 * s, a, b, c, d, e);
                        };
                        load5(sa, &map_dy, 0, q0, p0, n0, o0 / 32);
                        if (p.shared_b) {
                            load5(sa + WG_OPER, &map_x, 0, q0 - p.pad_l, p0 - p.pad_t + tap0 / p.S, n0, c0 / 32 + rank * BSUB);
                        } else {
                            // slot layout: tap-major, the tap's sub-tiles side by side (BSUB of them in pair mode, cpt otherwise:
                            // narrow layers pack 4 / cpt taps into one accumulator) — one box per tap covers them
                            const int xs = CG == 2 ? BSUB : p.cpt;
                            for (int q = 0; q < ntap; ++q) {
                                const int tap = tap0 + q;
                                const int r = tap / p.S, sx = tap - r * p.S;
                                load5(sa + WG_OPER + (uint32_t)(q * xs) * WG_SUB, &map_x, 0, q0 * p.stride - p.pad_l + sx,
                                      p0 * p.stride - p.pad_t + r, n0, c0 / 32 + rank * BSUB);
                            }
                        }
                        continue;
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        load(sa + i * WG_SUB, &map_dy, bar_full + 8 * s, o0 + 32 * i, q0, p0, n0);
                    if (p.shared_b) {
                        // one window of WG_WIN pixels starting at the s = 0 tap position, per 32-channel sub-tile
                        const int r = tap0 / p.S;
#pragma unroll
                        for (int i = 0; i < BSUB; ++i)
                            load(sa + WG_OPER + (uint32_t)i * WG_WSUB, &map_x, bar_full + 8 * s, c0 + 32 * (rank * BSUB + i),
                                 q0 - p.pad_l, p0 - p.pad_t + r, n0);
                    } else if (CG == 2) {
                        for (int q = 0; q < ntap * BSUB; ++q) {
                            // slot q = (tap q / BSUB, this CTA's sub-tile q % BSUB)
                            const int tap = tap0 + q / BSUB;
                            const int r = tap / p.S, sx = tap - r * p.S;
                            load(sa + WG_OPER + (uint32_t)q * WG_SUB, &map_x, bar_full + 8 * s, c0 + 32 * (rank * BSUB + q % BSUB),
                                 q0 * p.stride - p.pad_l + sx, p0 * p.stride - p.pad_t + r, n0);
                        }
                    } else
                    for (int q = 0; q < nslots; ++q) {
                        // slot q = (accumulator q/4, 32-column group q%4) holds tap q/cpt, channels 32*(q%cpt)
                        const int tap = tap0 + q / p.cpt;
                        const int r = tap / p.S, sx = tap - r * p.S;
                        load(sa + WG_OPER + (uint32_t)q * WG_SUB, &map_x, bar_full + 8 * s, c0 + 32 * (q % p.cpt),
                             q0 * p.stride - p.pad_l + sx, p0 * p.stride - p.pad_t + r, n0);
                    }
                }
            }
        } else if (warp == 1) {
            if (leader && elect_one()) {
                auto mma = [&](uint32_t d, uint64_t da, uint64_t db, uint32_t accumulate) {
                    if (CG == 2) umma2_tf32(d, da, db, IDESC, accumulate); else umma_tf32(d, da, db, IDESC, accumulate);
                };
                auto commit = [&](uint32_t bar) { if (CG == 2) umma2_commit(bar); else umma_commit(bar); };
                int seg = 0;
                for (int kb = 0; kb < KB; ++kb) {
                    // modulated mode: a new image starts at this chunk -> hand the finished accumulators to the epilogue and
                    // wait until they are drained; the first MMAs of the segment then overwrite instead of accumulating
                    const bool seg_start = kb == 0 || (p.chunks_per_image > 0 && (chunk_begin + kb) % p.chunks_per_image == 0);
                    if (seg_start && kb > 0) {
                        commit(bar_acc);
                        mbar_wait(bar_drained, (uint32_t)seg & 1u);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        ++seg;
                    }
                    const int s = kb % STAGES;
                    const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
                    mbar_wait(bar_full + 8 * s, ph);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = base + (uint32_t)s * STAGE_BYTES;
                    const uint64_t da = make_desc_mn_sw128(sa);
                    for (int g = 0; g < nacc; ++g) {
                        if (p.shared_b) {
#pragma unroll
                            for (int k = 0; k < WG_KPIX / 8; ++k) {
                                // tap s = g reads window rows [g + 8k, g + 8k + 8)
                                const uint64_t db = make_desc_mn_win(sa + WG_OPER + (uint32_t)(g + 8 * k) * 128u, p.shared_b == 1);
                                mma(tmem_base + (uint32_t)(g * 128), da + (uint64_t)(k * 64), db, (!seg_start || k > 0) ? 1u : 0u);
                            }
                            continue;
                        }
                        const uint64_t db = make_desc_mn_sw128(sa + WG_OPER + (uint32_t)g * (uint32_t)(BSUB * WG_SUB));
#pragma unroll
                        for (int k = 0; k < WG_KPIX / 8; ++k) {
                            // next 8 pixels along K: +1024 B = +64 in the (addr >> 4) field
                            mma(tmem_base + (uint32_t)(g * 128), da + (uint64_t)(k * 64), db + (uint64_t)(k * 64), (!seg_start || k > 0) ? 1u : 0u);
                        }
                    }
                    commit(bar_empty + 8 * s);
                }
                commit(bar_acc);
            }
        } else {
            const int lg = warp & 3;
            const int row = lg * 32 + lane;
            const int o = o0 + row;
            const int64_t ld = (int64_t)p.ntaps * p.C;
            // segments of the chunk range = images (modulated mode) or the whole range
            int seg = 0;
            for (int kb0 = 0; kb0 < KB; ++seg) {
                int kb1 = KB;
                if (p.chunks_per_image > 0) {
                    const int next = ((chunk_begin + kb0) / p.chunks_per_image + 1) * p.chunks_per_image - chunk_begin;
                    if (next < kb1) kb1 = next;
                }
                const int img = p.chunks_per_image > 0 ? (chunk_begin + kb0) / p.chunks_per_image : 0;
                mbar_wait(bar_acc, (uint32_t)seg & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                for (int q = 0; q < nslots; ++q) {
                    float v[32];
                    tmem_ld32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(q * 32), v);
                    const int c = c0 + 32 * (q % p.cpt);
                    const bool in_range = o < p.Ko && c < p.C;
                    const int64_t off = (int64_t)o * ld + (int64_t)(tap0 + q / p.cpt) * p.C + c;
                    if (p.chunks_per_image > 0) {
                        // ds[img, c + j] += sum over this warp's 32 filter rows of W * G; then the row's share of dW, scaled
                        const float* sv = p.mod_s + (int64_t)img * p.C + c;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            float t = in_range ? v[j] * __ldg(p.mod_w + off + j) : 0.f;
                            t = warp_sum(t);
                            if (lane == 0 && c < p.C) {
                                // the first tap of this CTA's group stores, the others add (same thread, fixed order)
                                float* d = p.mod_ds + ((((int64_t)img * p.ds_kmax + (int)blockIdx.z - (int)(((int64_t)img * p.chunks_per_image) / p.chunks_per_split))
                                                        * p.ds_tiles_o + o0 / 128) * gridDim.y + blockIdx.y) * 4 * p.C + (int64_t)lg * p.C + c + j;
                                *d = q < p.cpt ? t : *d + t;
                            }
                            v[j] *= (c < p.C) ? __ldg(sv + j) : 0.f;
                        }
                    }
                    if (in_range) {
                        // this split's slice; later segments (images) of the same CTA add to what the first one stored
                        float4* dst = reinterpret_cast<float4*>(dw + (int64_t)blockIdx.z * p.dw_numel + off);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float4 a = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                            if (seg > 0) {
                                const float4 b = dst[j];
                                a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
                            }
                            dst[j] = a;
                        }
                    }
                }
                kb0 = kb1;
                if (kb0 < KB) {
                    // more segments follow: tell the (leader's) MMA warp that the accumulators may be overwritten
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                    if (warp == 2 && lane == 0) {
                        if (CG == 2) asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_drained & kPeerBitMask) : "memory");
                        else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_drained) : "memory");
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Narrow-input variant (C == 32, stride 1, 3 horizontal taps): the patch discriminator's and the encoder's first
// 32-channel layers.  With only 32 dy channels the kernel above fills a quarter of the 128 M-rows and re-reads the x
// tile once per tap.  Here the operands swap roles:
//   A (M = 128) = the x window of one filter row: M-atom j (32 channels) is the SAME 40-pixel window shifted by j pixel
//                 rows — the descriptor's leading-dimension stride is one 128-byte pixel row, so atoms 0..2 ARE the three
//                 horizontal taps (atom 3 is a fourth, unused shift) and one window load feeds all of them;
//   B (N = Ko)  = the dy tile, 32 pixels x Ko channels;
//   one accumulator per filter row (R x Ko TMEM columns).
// Per 32-pixel chunk: R window loads (5 KB) + Ko/32 dy loads (4 KB) and 4 R MMAs, against 9 x-loads + 4 dy loads and 12
// full-size MMAs before.  Rows of the accumulator are (tap s, channel c), columns are output channels: a warp's 32 lanes
// write 32 consecutive c of dW[k, r, s, :] — coalesced 128-byte reductions.
constexpr int WN_STAGES = 4;

__device__ __forceinline__ uint64_t make_desc_mn_shift(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(128 >> 4) << 16;          // next M-atom = next pixel row of the same window
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}

__global__ void __launch_bounds__(WG_THREADS, 2)
wgrad_narrow_kernel(const __grid_constant__ CUtensorMap map_dy, const __grid_constant__ CUtensorMap map_x,
                    float* __restrict__ dw, const WgParams p, const int tmem_cols) {
    const int nkb = p.Ko / 32;                                  // dy sub-tiles (N = Ko <= 128)
    const uint32_t stage_bytes = (uint32_t)(p.R * WG_WSUB + nkb * WG_SUB);
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.Ko >> 3) << 17) | ((128u >> 4) << 24);

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_full = base + WN_STAGES * stage_bytes;
    const uint32_t bar_empty = bar_full + 8 * WN_STAGES;
    const uint32_t bar_acc = bar_empty + 8 * WN_STAGES;
    const uint32_t tmem_slot = bar_acc + 8;
    uint8_t* smem_gen = smem_raw + (base - smem_u32(smem_raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chunk_begin = blockIdx.x * p.chunks_per_split;
    const int chunk_end = min(chunk_begin + p.chunks_per_split, p.chunks_total);
    const int KB = chunk_end - chunk_begin;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_dy) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        for (int s = 0; s < WN_STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - base));

    if (KB > 0) {
        if (warp == 0) {
            if (elect_one()) {
                for (int kb = 0; kb < KB; ++kb) {
                    const int s = kb % WN_STAGES;
                    const uint32_t ph = (uint32_t)(kb / WN_STAGES) & 1u;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1u);
                    int ch = chunk_begin + kb;
                    const int tq = ch % p.tiles_w; ch /= p.tiles_w;
                    const int p0 = ch % p.tiles_h;
                    const int n0 = ch / p.tiles_h;
                    const int q0 = tq * 32;
                    const uint32_t sa = base + (uint32_t)s * stage_bytes;
                    mbar_expect_tx(bar_full + 8 * s, stage_bytes);
                    for (int r = 0; r < p.R; ++r)
                        tma_load_4d(sa + (uint32_t)r * WG_WSUB, &map_x, bar_full + 8 * s, 0, q0 - p.pad_l, p0 - p.pad_t + r, n0);
                    for (int i = 0; i < nkb; ++i)
                        tma_load_4d(sa + (uint32_t)(p.R * WG_WSUB + i * WG_SUB), &map_dy, bar_full + 8 * s, 32 * i, q0, p0, n0);
                }
            }
        } else if (warp == 1) {
            if (elect_one()) {
                for (int kb = 0; kb < KB; ++kb) {
                    const int s = kb % WN_STAGES;
                    const uint32_t ph = (uint32_t)(kb / WN_STAGES) & 1u;
                    mbar_wait(bar_full + 8 * s, ph);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = base + (uint32_t)s * stage_bytes;
                    const uint64_t db = make_desc_mn_sw128(sa + (uint32_t)(p.R * WG_WSUB));
                    for (int r = 0; r < p.R; ++r) {
#pragma unroll
                        for (int k = 0; k < WG_KPIX / 8; ++k) {
                            const uint64_t da = make_desc_mn_shift(sa + (uint32_t)r * WG_WSUB + (uint32_t)(8 * k) * 128u);
                            umma_tf32(tmem_base + (uint32_t)(r * p.Ko), da, db + (uint64_t)(k * 64), idesc, (kb > 0 || k > 0) ? 1u : 0u);
                        }
                    }
                    umma_commit(bar_empty + 8 * s);
                }
                umma_commit(bar_acc);
            }
        } else {
            const int lg = warp & 3;                 // TMEM lane group = tap s; lane = input channel c
            mbar_wait(bar_acc, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int64_t ld = (int64_t)p.ntaps * p.C;
            for (int r = 0; r < p.R; ++r)
                for (int nb = 0; nb < nkb; ++nb) {
                    float v[32];
                    tmem_ld32(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)(r * p.Ko + nb * 32), v);
                    if (lg < p.S) {
                        float* dst = dw + (int64_t)blockIdx.x * p.dw_numel + (int64_t)(nb * 32) * ld + (int64_t)(r * p.S + lg) * p.C + lane;
#pragma unroll
                        for (int i = 0; i < 32; ++i) dst[(int64_t)i * ld] = v[i];
                    }
                }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

bool tc_wgrad_eligible(const sae_conv_geom* g) {
    if (g->K % 32 != 0 || g->C % 32 != 0) return false;
    if (g->stride != 1 && g->stride != 2) return false;
    if (g->R * g->S > 49) return false;
    int tw = pow2_ceil(g->Q) < 32 ? pow2_ceil(g->Q) : 32;
    if (tw * g->stride > 256) return false;
    if ((int64_t)g->N * g->P * g->Q < 256) return false;      // too few pixels to be worth a tensor-core launch
    return true;
}

bool tc_wgrad_modulated_eligible(const sae_conv_geom* g) {
    // the shared-window configuration of wgrad_tc_kernel with whole 32-pixel chunks inside one image
    return tc_wgrad_eligible(g) && g->stride == 1 && g->Q % 32 == 0 && g->C % 32 == 0 && g->C >= 64 && g->K % 32 == 0;
}

static int tc_wgrad_impl(const float* dy, const float* x, float* dw, const sae_conv_geom* g, cudaStream_t st, const float* mod_s,
                         const float* mod_w, float* mod_ds);

int tc_wgrad(const float* dy, const float* x, float* dw, const sae_conv_geom* g, cudaStream_t st) {
    return tc_wgrad_impl(dy, x, dw, g, st, nullptr, nullptr, nullptr);
}

int tc_wgrad_modulated(const float* dy, const float* x, const float* s, const float* w_krsc, float* dw, float* ds,
                       const sae_conv_geom* g, cudaStream_t st) {
    if (!tc_wgrad_modulated_eligible(g)) return fail(SAE_E_UNSUPPORTED, "modulated wgrad: shape outside the tcgen05 configuration");
    return tc_wgrad_impl(dy, x, dw, g, st, s, w_krsc, ds);
}

// ds[img, c] += the style-gradient terms of every CTA that drained image img, summed in a fixed order: the splits that cover
// the image, then output tiles, tap groups and warps
__global__ void mod_ds_reduce_kernel(const float* __restrict__ part, float* __restrict__ ds, int N, int C, int kmax, int tiles_o,
                                     int groups, int chunks_per_image, int chunks_per_split, int splits) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)N * C) return;
    const int img = (int)(idx / C), c = (int)(idx % C);
    const int first = (int)(((int64_t)img * chunks_per_image) / chunks_per_split);
    int last = (int)(((int64_t)(img + 1) * chunks_per_image - 1) / chunks_per_split);
    if (last > splits - 1) last = splits - 1;
    float v = 0.f;
    for (int k = 0; k <= last - first; ++k)
        for (int o = 0; o < tiles_o; ++o)
            for (int y = 0; y < groups; ++y)
                for (int lg = 0; lg < 4; ++lg)
                    v += part[(((((int64_t)img * kmax + k) * tiles_o + o) * groups + y) * 4 + lg) * C + c];
    ds[idx] += v;
}

static int tc_wgrad_impl(const float* dy, const float* x, float* dw, const sae_conv_geom* g, cudaStream_t st, const float* mod_s,
                         const float* mod_w, float* mod_ds) {
    if (((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dw)) & 15) != 0)
        return fail(SAE_E_INVALID, "conv2d_wgrad(tcgen05): pointers must be 16-byte aligned");
    WgParams p;
    p.chunks_per_image = 0; p.mod_s = mod_s; p.mod_w = mod_w; p.mod_ds = mod_ds; p.five_d = 0;
    p.tw = pow2_ceil(g->Q) < 32 ? pow2_ceil(g->Q) : 32;
    int th = 32 / p.tw;
    if (pow2_ceil(g->P) < th) th = pow2_ceil(g->P);
    p.th = th;
    p.tn = 32 / (p.tw * p.th);
    p.tiles_w = (g->Q + p.tw - 1) / p.tw;
    p.tiles_h = (g->P + p.th - 1) / p.th;
    p.tiles_n = (g->N + p.tn - 1) / p.tn;
    p.chunks_total = p.tiles_w * p.tiles_h * p.tiles_n;
    p.stride = g->stride; p.pad_t = g->pad_t; p.pad_l = g->pad_l; p.R = g->R; p.S = g->S;
    p.Ko = g->K; p.C = g->C;
    p.ntaps = g->R * g->S;
    p.cpt = (g->C >= 128 ? 128 : g->C) / 32;                       // C is a multiple of 32 here: 1, 2, 3 or 4
    if (p.cpt == 3) p.cpt = 4;                                      // C = 96: keep one tap per accumulator (4th slot is OOB zero)
    p.group_taps = WG_MAX_GROUP * (4 / p.cpt);
    if (p.group_taps > p.ntaps) p.group_taps = p.ntaps;
    const int groups = (p.ntaps + p.group_taps - 1) / p.group_taps;
    const int tiles_o = (g->K + 127) / 128;
    p.n_tiles_c = (g->C + 127) / 128;
    const int tiles = tiles_o * p.n_tiles_c * groups;
    // One CTA per SM (192 KB of shared memory each): choose the pixel split so the whole grid is ONE wave
    // (tiles * splits <= SM count); a second, nearly empty wave would double the kernel time.
    int splits = sm_count() / tiles;
    if (splits > p.chunks_total) splits = p.chunks_total;
    if (splits < 1) splits = 1;
    p.chunks_per_split = (p.chunks_total + splits - 1) / splits;
    splits = (p.chunks_total + p.chunks_per_split - 1) / p.chunks_per_split;

    if (mod_s != nullptr) p.chunks_per_image = p.tiles_w * p.tiles_h;       // tn == 1 (Q % 32 == 0)
    p.dw_numel = (int64_t)g->K * p.ntaps * g->C;
    p.ds_kmax = 0;
    p.ds_tiles_o = tiles_o;
    static int narrow_mode = -1;
    if (narrow_mode < 0) { const char* v = getenv("SAE_WGRAD_NARROW"); narrow_mode = (v && v[0] == '0') ? 0 : 1; }
    if (mod_s == nullptr && narrow_mode && g->C == 32 && g->stride == 1 && g->S == 3 && g->R <= 3 && p.tw == 32 && g->K <= 128) {
        // C == 32: x window as the A operand with pixel-shifted M-atoms (see wgrad_narrow_kernel)
        CUtensorMap mdy, mx;
        {
            cuuint64_t dims[4] = {(cuuint64_t)g->K, (cuuint64_t)g->Q, (cuuint64_t)g->P, (cuuint64_t)g->N};
            cuuint64_t strides[3] = {(cuuint64_t)g->K * 4, (cuuint64_t)g->Q * g->K * 4, (cuuint64_t)g->P * g->Q * g->K * 4};
            cuuint32_t box[4] = {32, 32, 1, 1};
            cuuint32_t es[4] = {1, 1, 1, 1};
            int rc = encode_map(&mdy, dy, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
            if (rc) return rc;
        }
        {
            cuuint64_t dims[4] = {(cuuint64_t)g->C, (cuuint64_t)g->W, (cuuint64_t)g->H, (cuuint64_t)g->N};
            cuuint64_t strides[3] = {(cuuint64_t)g->C * 4, (cuuint64_t)g->W * g->C * 4, (cuuint64_t)g->H * g->W * g->C * 4};
            cuuint32_t box[4] = {32, WG_WIN, 1, 1};
            cuuint32_t es[4] = {1, 1, 1, 1};
            int rc = encode_map(&mx, x, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
            if (rc) return rc;
        }
        const int nkb = g->K / 32;
        const size_t stage = (size_t)g->R * WG_WSUB + (size_t)nkb * WG_SUB;
        const size_t smem_n = WN_STAGES * stage + 1024 + 256;
        int cols = 32;
        while (cols < g->R * g->K) cols <<= 1;
        const int per_sm = (cols <= 256 && 2 * smem_n <= 200 * 1024) ? 2 : 1;
        static size_t attr_bytes = 0;
        if (smem_n > attr_bytes) {
            SAE_CUDA_TRY(cudaFuncSetAttribute(wgrad_narrow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_n));
            attr_bytes = smem_n;
        }
        int nsplit = sm_count() * per_sm;
        if (nsplit > p.chunks_total) nsplit = p.chunks_total;
        p.chunks_per_split = (p.chunks_total + nsplit - 1) / nsplit;
        nsplit = (p.chunks_total + p.chunks_per_split - 1) / p.chunks_per_split;
        p.shared_b = 0;
        float* part = det_workspace(det_reduce_floats(p.dw_numel, nsplit));
        if (!part) return SAE_E_CUDA;
        wgrad_narrow_kernel<<<(unsigned)nsplit, WG_THREADS, smem_n, st>>>(mdy, mx, part, p, cols);
        int rc = check_launch("wgrad_narrow");
        if (rc) return rc;
        return det_reduce(dw, part, p.dw_numel, nsplit, st);
    }

    static int win_mode = -1;
    // shared-window mode on by default (2 = plain start address: the swizzle is a function of the absolute shared-memory
    // address, verified on hardware; 1 = additionally set the descriptor's base-offset field — produces wrong results;
    // 0 = off, three separate boxes)
    if (win_mode < 0) { const char* v = getenv("SAE_WGRAD_WINDOW"); win_mode = v ? atoi(v) : 2; }
    p.shared_b = (win_mode >= 1 && p.tw == 32 && g->stride == 1 && g->S == 3 && p.cpt == 4 && p.group_taps == 3) ? win_mode : 0;
    // CTA pairs where the layer has 256 out channels per pair and whole 128-channel x tiles (SAE_WGRAD_PAIR=0: off, A/B runs)
    static int pair_mode = -1;
    if (pair_mode < 0) { const char* v = getenv("SAE_WGRAD_PAIR"); pair_mode = (v && v[0] == '0') ? 0 : 1; }
    const bool pair = pair_mode && g->K % 256 == 0 && g->C % 128 == 0 && p.cpt == 4;

    CUtensorMap mdy, mx;
    {
        cuuint64_t dims[4] = {(cuuint64_t)g->K, (cuuint64_t)g->Q, (cuuint64_t)g->P, (cuuint64_t)g->N};
        cuuint64_t strides[3] = {(cuuint64_t)g->K * 4, (cuuint64_t)g->Q * g->K * 4, (cuuint64_t)g->P * g->Q * g->K * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)p.tw, (cuuint32_t)p.th, (cuuint32_t)p.tn};
        cuuint32_t es[4] = {1, 1, 1, 1};
        int rc = encode_map(&mdy, dy, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
        if (rc) return rc;
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)g->C, (cuuint64_t)g->W, (cuuint64_t)g->H, (cuuint64_t)g->N};
        cuuint64_t strides[3] = {(cuuint64_t)g->C * 4, (cuuint64_t)g->W * g->C * 4, (cuuint64_t)g->H * g->W * g->C * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)(p.tw * g->stride), (cuuint32_t)(p.th * g->stride), (cuuint32_t)p.tn};
        if (p.shared_b) box[1] = WG_WIN;
        cuuint32_t es[4] = {1, (cuuint32_t)g->stride, (cuuint32_t)g->stride, 1};
        int rc = encode_map(&mx, x, 4, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
        if (rc) return rc;
    }
    // 5-D views (32 channels, W, H, N, channel block) — see the producer.  The
    // channel-block dimension has the SMALLEST stride (128 bytes); should a driver refuse such a view, the 4-D maps above stay.
    static int five_d = -1;
    if (five_d < 0) { const char* v = getenv("SAE_WGRAD_5D"); five_d = (v && v[0] == '0') ? 0 : 1; }
    if (five_d && g->C % 32 == 0 && g->K % 32 == 0) {
        CUtensorMap m5dy, m5x;
        cuuint64_t ddims[5] = {32, (cuuint64_t)g->Q, (cuuint64_t)g->P, (cuuint64_t)g->N, (cuuint64_t)(g->K / 32)};
        cuuint64_t dstr[4] = {(cuuint64_t)g->K * 4, (cuuint64_t)g->Q * g->K * 4, (cuuint64_t)g->P * g->Q * g->K * 4, 128};
        cuuint32_t dbox[5] = {32, (cuuint32_t)p.tw, (cuuint32_t)p.th, (cuuint32_t)p.tn, 4};
        cuuint32_t des[5] = {1, 1, 1, 1, 1};
        cuuint64_t xdims[5] = {32, (cuuint64_t)g->W, (cuuint64_t)g->H, (cuuint64_t)g->N, (cuuint64_t)(g->C / 32)};
        cuuint64_t xstr[4] = {(cuuint64_t)g->C * 4, (cuuint64_t)g->W * g->C * 4, (cuuint64_t)g->H * g->W * g->C * 4, 128};
        cuuint32_t xbox[5] = {32, (cuuint32_t)(p.tw * g->stride), (cuuint32_t)(p.th * g->stride), (cuuint32_t)p.tn, pair ? 2u : (cuuint32_t)p.cpt};
        if (p.shared_b) xbox[1] = WG_WIN;
        cuuint32_t xes[5] = {1, (cuuint32_t)g->stride, (cuuint32_t)g->stride, 1, 1};
        if (encode_map(&m5dy, dy, 5, ddims, dstr, dbox, des, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) == SAE_OK &&
            encode_map(&m5x, x, 5, xdims, xstr, xbox, xes, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) == SAE_OK) {
            mdy = m5dy; mx = m5x; p.five_d = 1;
        } else {
            five_d = 0;
        }
    }
    // workspace: the per-split partial dW slices (and det_reduce's scratch behind them), then the style-gradient terms
    const size_t dw_floats = det_reduce_floats(p.dw_numel, splits);
    size_t ds_floats = 0;
    if (mod_s != nullptr) {
        for (int img = 0; img < g->N; ++img) {
            const int first = (int)(((int64_t)img * p.chunks_per_image) / p.chunks_per_split);
            const int last = (int)(((int64_t)(img + 1) * p.chunks_per_image - 1) / p.chunks_per_split);
            if (last - first + 1 > p.ds_kmax) p.ds_kmax = last - first + 1;
        }
        ds_floats = (size_t)g->N * p.ds_kmax * tiles_o * groups * 4 * g->C;
    }
    float* part = det_workspace(dw_floats + ds_floats);
    if (!part) return SAE_E_CUDA;
    if (mod_s != nullptr) p.mod_ds = part + dw_floats;
    int rc;
    if (pair) {
        constexpr size_t smem = wg_smem_bytes<2>();
        static bool attr_done = false;
        if (!attr_done) {
            SAE_CUDA_TRY(cudaFuncSetAttribute(wgrad_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_done = true;
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(tiles_o * p.n_tiles_c), (unsigned)groups, (unsigned)splits);      // tiles_o is even
        cfg.blockDim = dim3(WG_THREADS, 1, 1);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        SAE_CUDA_TRY(cudaLaunchKernelEx(&cfg, wgrad_tc_kernel<2>, mdy, mx, part, p));
        rc = check_launch("wgrad_tc<2>");
    } else {
        constexpr size_t smem = wg_smem_bytes<1>();
        static bool attr_done = false;
        if (!attr_done) {
            SAE_CUDA_TRY(cudaFuncSetAttribute(wgrad_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_done = true;
        }
        dim3 grid((unsigned)(tiles_o * p.n_tiles_c), (unsigned)groups, (unsigned)splits);
        wgrad_tc_kernel<1><<<grid, WG_THREADS, smem, st>>>(mdy, mx, part, p);
        rc = check_launch("wgrad_tc");
    }
    if (rc) return rc;
    rc = det_reduce(dw, part, p.dw_numel, splits, st);
    if (rc || mod_s == nullptr) return rc;
    const int64_t nds = (int64_t)g->N * g->C;
    mod_ds_reduce_kernel<<<(unsigned)((nds + 255) / 256), 256, 0, st>>>(p.mod_ds, mod_ds, g->N, g->C, p.ds_kmax, tiles_o, groups,
                                                                      p.chunks_per_image, p.chunks_per_split, splits);
    return check_launch("mod_ds_reduce");
}

}  // namespace sae
