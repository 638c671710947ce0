// tcgen05 / TMEM / TMA kernels shared by every dense contraction on the VAE/GAN training path.
//
//  igemm_kernel : D[pixels or rows, N] = sum over (tap, k-chunk) A_tap[pixels, k] * B_tap[N, k]^T
//                 A tiles are TMA boxes of an NHWC activation (one box per filter tap -> implicit GEMM),
//                 B tiles are TMA boxes of a tap-major bf16 weight pack. Both K-major, 128B/64B swizzle.
//                 Covers: 5x5 s2 conv fprop, convT dgrad (gather form, 4 stride-parity tensor maps),
//                         5x5 s2 convT fprop, conv dgrad (scatter form, 4 output-parity classes),
//                         5x5 s1 conv, and plain linear layers (1 tap), optional split-K.
//  wgrad_kernel : dW[tap][M, N] = sum over pixels P_dense[pixel, M]^T * P_shift[pixel@tap, N]
//                 both operands MN-major straight out of NHWC (pixels are the reduction dim).
//
// Reference ops replaced: nn.Conv2d / nn.ConvTranspose2d / nn.Linear forward+backward as dispatched by
// /root/reference/models/vae_gan.py:18-21,46-54,79-85,107-121,146-161,199-207,510-521.
#pragma once
#include "ptx.cuh"

namespace fmri {

struct TapDesc {
    int16_t map;   // which A tensor map (stride-parity plane) this tap reads
    int16_t dx;    // pixel offset added to the tile origin (x)
    int16_t dy;    // pixel offset added to the tile origin (y)
    int16_t ncol;  // 0: the MMA covers all BN columns; else (columns / 32) << 8 | (first column / 32): the parity-merged
                   // scatter's weight slab of this coarse tap is zero outside that range (persistent kernel only)
    int32_t brow;  // first row of this tap's weights in the B pack
};

struct TapClass {       // one per blockIdx.z (output-parity class of a transposed conv); 1 class otherwise
    int num_taps;
    int lim_x, lim_y;   // valid extent of the output (sub)grid
    long long out_off;  // element offset of this class' first output pixel
    TapDesc taps[25];
};

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_TANH = 2, ACT_SIGMOID = 3 };

struct IgParams {
    CUtensorMap mapA[4];
    CUtensorMap mapB;
    TapClass cls[4];
    int bw, bh, bn;                 // pixel box of one M tile (bw*bh*bn <= 128 rows)
    int tiles_x, tiles_y, tiles_n;  // M tiles
    int lim_n;                      // images
    int num_chunks;                 // K chunks per tap
    int n_total, n_tiles;           // GEMM N and its tiling
    int splits;                     // split-K factor
    int a_bytes;                    // bytes one A box delivers
    long long out_sn, out_sy, out_sx;
    void* out;
    int out_fp32;    // 0: bf16 store, 1: fp32 store
    int atomic_out;  // fp32 red.add (split-K / accumulate)
    const float* bias;
    int act;
    double* stat_sum;  // optional per-column sum / sum of squares of the stored values
    double* stat_sq;
    // parity-merged scatter (thin-output stride-2 transposed conv / conv data-gradient, Ng = 32): the four output-parity
    // classes become 4 x 32 GEMM columns of ONE gather over the 3x3 neighbourhood of the coarse pixel (taps a class does not
    // use carry zero weights: 36/25 more MACs, but N = 128 instead of 32 and the activation tile is fetched 9x, not 25x).
    // Column group g = col / 32 -> (ph, pw) = (g >> 1, g & 1) is stored at fine pixel (2y + ph, 2x + pw).
    int merge;              // 0 / 1
    const void* mask_y;     // persistent kernel, bf16 output: zero the output where this bf16 tensor (same layout) is <= 0
                            // (ReLU backward of a bias+ReLU layer fused into the data-gradient epilogue)
    const uint32_t* mask_bits;  // same mask as 1 bit per element of a 32-channel pixel (bits[(offset) >> 5]); preferred over mask_y
    int yr;                 // persistent kernel, row-reuse gather (see IgSmem): mapA[plane] boxes are MT*bh+2 rows tall
    int pair;               // persistent kernel: 128-byte-line stores through chunk pairs (dispatch_ig_persistent decides)
    int skip;               // diagnostic (FMRI_IG_SKIP, persistent kernel): bit 0 the producer issues no TMA loads, bit 1 the
                            // epilogue does nothing but hand the accumulators back, bit 2 no MMAs are issued, bit 3 the
                            // epilogue skips only its global stores -- which role bounds a launch (results are garbage)
    int merge_oh, merge_ow; // fine output extent
    long long merge_sy;     // fine row stride (elements)
};

// MT = number of 128-row M sub-tiles one CTA accumulates against the SAME B (weight) tile: the kernels are bound by
// L2 -> shared-memory bandwidth (~43 B/clk/SM measured chip-wide), and MT = 2 halves the weight bytes per FLOP.
//
// YR ("row reuse", stride-2 gather with a thin K side and 32-pixel-wide output rows): the taps kh = py, py+2, py+4 of one
// filter column read the SAME stride-parity plane shifted by whole rows, so ONE tall box of MT*4+2 rows x 32 pixels per
// (kw, py) feeds up to three taps: tap i of sub-tile m starts (4m + i) rows (= a multiple of the swizzle period) into the
// box. 10 boxes of 10 rows instead of 25 x 8 rows: the activation bytes per tile halve, the weights are fetched as before.
// PERS: what the persistent kernel adds behind the stage ring -- a 2 KB per epilogue warp staging buffer through which bf16
// output rows are re-ordered into full 32-byte sectors before they are stored (dropped where it does not fit beside four
// stages, BN = 256).
template <int BN, int KCH, int STAGES, int MT = 1, bool YR = false, bool PERS = false>
struct IgSmem {
    static constexpr int A_SUB = 128 * KCH * 2;
    static constexpr int A_BYTES = YR ? (MT * 4 + 2) * 32 * KCH * 2 : MT * A_SUB;
    static constexpr int B_TAP = BN * KCH * 2;
    static constexpr int B_BYTES = (YR ? 3 : 1) * B_TAP;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
    static constexpr int STAT_OFF = BAR_OFF + (2 * STAGES + 4) * 8 + 16;
    static constexpr int STAT_SLOTS = 8;                        // persistent kernel: one private [2][BN] slot per epilogue warp
    static constexpr int STG_OFF = (STAT_OFF + STAT_SLOTS * 2 * BN * 4 + 127) & ~127;
    static constexpr int STG_BYTES = (PERS && STG_OFF + 8 * 2048 + 1024 <= 227 * 1024) ? 8 * 2048 : 0;
    static constexpr int TOTAL = STG_OFF + STG_BYTES + 1024;  // +1024: manual base alignment
};

// transposing butterfly: on exit lane l holds the sum over the 32 lanes of f[l]
__device__ __forceinline__ float warp_colsum32(float (&f)[32], int lane) {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const bool up = lane & 16;
        const float send = up ? f[j] : f[j + 16];
        const float keep = up ? f[j + 16] : f[j];
        f[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const bool up = lane & 8;
        const float send = up ? f[j] : f[j + 8];
        const float keep = up ? f[j + 8] : f[j];
        f[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const bool up = lane & 4;
        const float send = up ? f[j] : f[j + 4];
        const float keep = up ? f[j + 4] : f[j];
        f[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const bool up = lane & 2;
        const float send = up ? f[j] : f[j + 2];
        const float keep = up ? f[j + 2] : f[j];
        f[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    {
        const bool up = lane & 1;
        const float send = up ? f[0] : f[1];
        const float keep = up ? f[1] : f[0];
        f[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
    return f[0];
}

template <int BN, int KCH, int STAGES, int MT>
__global__ void __launch_bounds__(192) igemm_kernel(const __grid_constant__ IgParams p) {
    using L = IgSmem<BN, KCH, STAGES, MT>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
    float* s_stat = reinterpret_cast<float*>(smem + L::STAT_OFF);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    // ---- which tiles (MT consecutive M tiles share this CTA's weight tiles)
    const TapClass& c = p.cls[blockIdx.z];
    const int total_mt = p.tiles_x * p.tiles_y * p.tiles_n;
    int x0[MT], y0[MT], n0[MT];
    bool live[MT];
    bool any = false;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        const int mt = blockIdx.x * MT + m;
        const int tx = mt % p.tiles_x;
        const int ty = (mt / p.tiles_x) % p.tiles_y;
        const int tn = mt / (p.tiles_x * p.tiles_y);
        x0[m] = tx * p.bw; y0[m] = ty * p.bh; n0[m] = tn * p.bn;
        live[m] = mt < total_mt && x0[m] < c.lim_x && y0[m] < c.lim_y;  // tile inside this parity class' sub-grid
        any |= live[m];
    }
    const int nt = blockIdx.y % p.n_tiles;
    const int split = blockIdx.y / p.n_tiles;
    if (!any) return;
    const int ks_total = c.num_taps * p.num_chunks;
    const int ks_begin = (int)((long long)split * ks_total / p.splits);
    const int ks_end = (int)((long long)(split + 1) * ks_total / p.splits);
    if (ks_begin >= ks_end) return;
    const int nks = ks_end - ks_begin;

    constexpr uint32_t TMEM_COLS = (MT * BN) < 32 ? 32 : (MT * BN);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.mapA[0]);
        tma_prefetch_desc(&p.mapB);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    for (int i = threadIdx.x; i < 4 * 2 * BN; i += blockDim.x) s_stat[i] = 0.f;   // one [2][BN] slot per epilogue warp
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int nlive = 0;
#pragma unroll
            for (int m = 0; m < MT; ++m) nlive += live[m] ? 1 : 0;
            for (int i = 0; i < nks; ++i) {
                const int st = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                mbar_wait(&empty_bar[st], ph ^ 1);
                mbar_arrive_expect_tx(&full_bar[st], nlive * p.a_bytes + L::B_BYTES);
                const int ks = ks_begin + i;
                const int tap = ks / p.num_chunks;
                const int ch = ks - tap * p.num_chunks;
                const TapDesc t = c.taps[tap];
                uint8_t* sa = smem + st * L::STAGE_BYTES;
#pragma unroll
                for (int m = 0; m < MT; ++m)
                    if (live[m])
                        tma_load_4d(sa + m * L::A_SUB, &p.mapA[t.map], &full_bar[st], ch * KCH, x0[m] + t.dx,
                                    y0[m] + t.dy, n0[m]);
                tma_load_2d(sa + L::A_BYTES, &p.mapB, &full_bar[st], ch * KCH, t.brow + nt * BN);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(128, BN, false, false);
            constexpr uint64_t layout = (KCH == 64) ? UMMA_SW128 : UMMA_SW64;
            constexpr uint32_t sbo = 8 * KCH * 2;
            for (int i = 0; i < nks; ++i) {
                const int st = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                mbar_wait(&full_bar[st], ph);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + st * L::STAGE_BYTES);
                const uint64_t bdesc = umma_smem_desc(sa + L::A_BYTES, 16, sbo, layout);
#pragma unroll
                for (int m = 0; m < MT; ++m) {
                    if (!live[m]) continue;
                    const uint64_t adesc = umma_smem_desc(sa + m * L::A_SUB, 16, sbo, layout);
#pragma unroll
                    for (int k = 0; k < KCH / 16; ++k)
                        umma_bf16(tmem_base + m * BN, adesc + 2 * k, bdesc + 2 * k, idesc, (i | k) != 0);
                }
                umma_commit(&empty_bar[st]);  // frees the smem slot once these MMAs retire
            }
            umma_commit(tmem_full);
        }
        __syncwarp();
    } else {
        // ================= epilogue: TMEM -> registers -> global =================
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int q = warp & 3;  // TMEM lane quarter this warp may touch
        const int row = q * 32 + lane;
        const int xi = row % p.bw;
        const int yi = (row / p.bw) % p.bh;
        const int ni = row / (p.bw * p.bh);
        const bool do_stats = p.stat_sum != nullptr;
#pragma unroll 1
        for (int m = 0; m < MT; ++m) {
            if (!live[m]) continue;
            const bool valid = (ni < p.bn) && (n0[m] + ni < p.lim_n) && (y0[m] + yi < c.lim_y) && (x0[m] + xi < c.lim_x);
            const long long off = c.out_off + (long long)(n0[m] + ni) * p.out_sn + (long long)(y0[m] + yi) * p.out_sy +
                                  (long long)(x0[m] + xi) * p.out_sx + (long long)nt * BN;
            const bool valid_tile = valid;
            const long long off_tile = off;
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                bool valid = valid_tile;
                long long off = off_tile;
                int stat_col = c0;
                if (p.merge) {  // 32-column group -> output parity class
                    const int g = (nt * BN + c0) >> 5;
                    const int ph = g >> 1, pw = (g == 0 || g == 3) ? 1 : 0;   // merged column groups: (0,1),(0,0),(1,0),(1,1)
                    valid = valid_tile && (2 * (y0[m] + yi) + ph < p.merge_oh) && (2 * (x0[m] + xi) + pw < p.merge_ow);
                    off = off_tile - (long long)nt * BN + ph * p.merge_sy + pw * 32 - c0;
                    stat_col = 0;
                }
                uint32_t v[32];
                tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + m * BN + c0, v);
                tmem_ld_wait();
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                if (p.bias && split == 0) {  // split-K: exactly one split adds the bias
                    const float* bp = p.bias + (p.merge ? 0 : nt * BN + c0);  // merged: each 32-column group = channels 0..31
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] += __ldg(bp + j);
                }
                if (p.act == ACT_RELU) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
                } else if (p.act == ACT_TANH) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = tanhf(f[j]);
                } else if (p.act == ACT_SIGMOID) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = 1.f / (1.f + __expf(-f[j]));
                }
                if (p.out_fp32) {
                    if (valid) {
                        float* o = reinterpret_cast<float*>(p.out) + off + c0;
                        if (p.atomic_out) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4) red_add_v4(o + j, f[j], f[j + 1], f[j + 2], f[j + 3]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                        }
                    }
                } else {
                    uint32_t pk[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
                    if (valid) {
                        __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + off + c0;
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<uint4*>(o + 8 * j) =
                                make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                    }
                    if (do_stats) {  // statistics of exactly what was stored (bf16-rounded)
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            f[2 * j] = __uint_as_float(pk[j] << 16);
                            f[2 * j + 1] = __uint_as_float(pk[j] & 0xffff0000u);
                        }
                    }
                }
                if (do_stats) {
                    float g[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        f[j] = valid ? f[j] : 0.f;
                        g[j] = f[j] * f[j];
                    }
                    const float s1 = warp_colsum32(f, lane);
                    const float s2 = warp_colsum32(g, lane);
                    float* my_stat = s_stat + q * 2 * BN;   // this warp's slot: no order-dependent shared atomics
                    my_stat[stat_col + lane] += s1;
                    my_stat[BN + stat_col + lane] += s2;
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    tc_fence_after();
    if (p.stat_sum != nullptr) {
        const int ncol = p.merge ? 32 : BN;
        const int cbase = p.merge ? 0 : nt * BN;
        for (int i = threadIdx.x; i < ncol; i += blockDim.x) {
            float a = 0.f, b = 0.f;
            for (int w = 0; w < 4; ++w) {
                a += s_stat[w * 2 * BN + i];
                b += s_stat[w * 2 * BN + BN + i];
            }
            atomicAdd(p.stat_sum + cbase + i, (double)a);
            atomicAdd(p.stat_sq + cbase + i, (double)b);
        }
    }
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// Persistent variant of igemm_kernel (split-K == 1): one CTA per SM walks a list of output tiles; the TMA ring and the MMA
// issue run ahead across tile boundaries and the accumulators are DOUBLE BUFFERED in TMEM (2 x MT x BN <= 512 columns), so the
// epilogue of tile i (TMEM -> registers -> bias/activation -> global, BN statistics) overlaps the main loop of tile i+1.
// The non-persistent kernel leaves the tensor pipe idle during prologue + epilogue (56-64 % busy on the big layers,
// profiles/r1_ncu_full_gemm_kernels_B512.md).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

struct IgTile {
    int cls, nt;
    int x0[2], y0[2], n0[2];
    bool live[2];
    bool any;
};
template <int MT>
__device__ __forceinline__ IgTile ig_decode_tile(const IgParams& p, int t, int m_groups) {
    IgTile r;
    const int per_cls = m_groups * p.n_tiles;
    r.cls = t / per_cls;
    const int rem = t - r.cls * per_cls;
    r.nt = rem / m_groups;
    const int mg = rem - r.nt * m_groups;
    const TapClass& c = p.cls[r.cls];
    const int total_mt = p.tiles_x * p.tiles_y * p.tiles_n;
    r.any = false;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        const int mt = mg * MT + m;
        const int tx = mt % p.tiles_x;
        const int ty = (mt / p.tiles_x) % p.tiles_y;
        const int tn = mt / (p.tiles_x * p.tiles_y);
        r.x0[m] = tx * p.bw; r.y0[m] = ty * p.bh; r.n0[m] = tn * p.bn;
        r.live[m] = mt < total_mt && r.x0[m] < c.lim_x && r.y0[m] < c.lim_y;
        r.any |= r.live[m];
    }
    return r;
}

constexpr int IGP_EPI_WARPS = 8;
constexpr int IGP_THREADS = 64 + 32 * IGP_EPI_WARPS;

// MASK: the fused ReLU-mask epilogue is compiled in; the plain instantiation keeps it out of the register allocation of the
// common case (the epilogue sits at the 168-register cap).
template <int BN, int KCH, int STAGES, int MT, bool MASK = false, bool YR = false>
__global__ void __launch_bounds__(IGP_THREADS) igemm_persistent_kernel(const __grid_constant__ IgParams p, int num_classes) {
    using L = IgSmem<BN, KCH, STAGES, MT, YR, true>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull = empty_bar + STAGES;   // [2] accumulators of buffer b complete (tcgen05.commit)
    uint64_t* tempty = tfull + 2;           // [2] buffer b drained by the 4 epilogue warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* s_stat = reinterpret_cast<float*>(smem + L::STAT_OFF);
    static_assert(2 * MT * BN <= 512, "double-buffered accumulators must fit TMEM");

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int m_groups = (p.tiles_x * p.tiles_y * p.tiles_n + MT - 1) / MT;
    const int total_tiles = m_groups * p.n_tiles * num_classes;
    constexpr uint32_t ACC_COLS = MT * BN;
    constexpr uint32_t TMEM_COLS = (2 * ACC_COLS) < 32 ? 32 : (2 * ACC_COLS);

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.mapA[0]);
        tma_prefetch_desc(&p.mapB);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1);
            mbar_init(&tempty[b], IGP_EPI_WARPS);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    for (int i = threadIdx.x; i < L::STAT_SLOTS * 2 * BN; i += blockDim.x) s_stat[i] = 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        // The whole warp runs the loop converged (warp-uniform operands, elected issue, see ptx.cuh); tap and channel-chunk
        // counters are nested loops instead of a per-stage integer division. A stage of the 32-channel K-chunk layers is
        // only 128-256 tensor-pipe cycles, which the previous single-lane producer (~130 dependent instructions per
        // stage) could not keep up with.
        if constexpr (YR) {   // one tall activation box + the weights of its (up to) three taps per stage
            int it = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const IgTile tl = ig_decode_tile<MT>(p, t, m_groups);
                if (!tl.any) continue;
                const int brow0 = tl.nt * BN;
                for (int g = 0; g < 10; ++g, ++it) {
                    const int kw = g >> 1, py = g & 1, ntap = 3 - py;
                    const int st = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(&empty_bar[st], ph ^ 1);
                    if (p.skip & 1) { mbar_arrive_expect_tx_elect(&full_bar[st], 0); continue; }
                    mbar_arrive_expect_tx_elect(&full_bar[st], p.a_bytes + ntap * L::B_TAP);
                    uint8_t* sa = smem + st * L::STAGE_BYTES;
                    tma_load_4d_elect(sa, &p.mapA[py * 2 + (kw & 1)], &full_bar[st], 0, tl.x0[0] + (kw - 2 - (kw & 1)) / 2,
                                      tl.y0[0] - 1, tl.n0[0]);
                    for (int i = 0; i < ntap; ++i)
                        tma_load_2d_elect(sa + L::A_BYTES + i * L::B_TAP, &p.mapB, &full_bar[st], 0,
                                          ((py + 2 * i) * 5 + kw) * p.n_total + brow0);
                }
            }
        } else {
            int it = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const IgTile tl = ig_decode_tile<MT>(p, t, m_groups);
                if (!tl.any) continue;
                const TapClass& c = p.cls[tl.cls];
                int nlive = 0;
#pragma unroll
                for (int m = 0; m < MT; ++m) nlive += tl.live[m] ? 1 : 0;
                const uint32_t tx_bytes = nlive * p.a_bytes + L::B_BYTES;
                const int brow0 = tl.nt * BN;
                for (int tap = 0; tap < c.num_taps; ++tap) {
                    const TapDesc td = c.taps[tap];
                    const CUtensorMap* mapA = &p.mapA[td.map];
                    for (int ch = 0; ch < p.num_chunks; ++ch, ++it) {
                        const int st = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        mbar_wait(&empty_bar[st], ph ^ 1);
                        if (p.skip & 1) { mbar_arrive_expect_tx_elect(&full_bar[st], 0); continue; }
                        mbar_arrive_expect_tx_elect(&full_bar[st], tx_bytes);
                        uint8_t* sa = smem + st * L::STAGE_BYTES;
#pragma unroll
                        for (int m = 0; m < MT; ++m)
                            if (tl.live[m])
                                tma_load_4d_elect(sa + m * L::A_SUB, mapA, &full_bar[st], ch * KCH, tl.x0[m] + td.dx,
                                                  tl.y0[m] + td.dy, tl.n0[m]);
                        tma_load_2d_elect(sa + L::A_BYTES, &p.mapB, &full_bar[st], ch * KCH, td.brow + brow0);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer =================
        // The whole warp runs the loop converged with warp-uniform operands; one ELECTED lane issues each tcgen05
        // instruction (umma_bf16_elect). Issuing from inside `if (lane == 0)` costs ~15 extra instructions per MMA (an
        // ELECT / R2UR / branch waterfall), which made every N <= 128 launch issue-bound (64-clock MMAs).
        {
            constexpr uint32_t idesc = umma_idesc_bf16(128, BN, false, false);
            constexpr uint64_t layout = (KCH == 64) ? UMMA_SW128 : UMMA_SW64;
            constexpr uint32_t sbo = 8 * KCH * 2;
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
            int it = 0, lt = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const IgTile tl = ig_decode_tile<MT>(p, t, m_groups);
                if (!tl.any) continue;
                const int buf = lt & 1;
                mbar_wait(&tempty[buf], ((lt >> 1) & 1) ^ 1);
                tc_fence_after();
                if constexpr (YR) {
                    for (int g = 0; g < 10; ++g, ++it) {
                        const int ntap = 3 - (g & 1);
                        const int st = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        mbar_wait(&full_bar[st], ph);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(smem + st * L::STAGE_BYTES);
                        for (int i = 0; i < ((p.skip & 4) ? 0 : ntap); ++i) {
                            const uint64_t bdesc = umma_smem_desc(sa + L::A_BYTES + i * L::B_TAP, 16, sbo, layout);
#pragma unroll
                            for (int m = 0; m < MT; ++m) {
                                const uint64_t adesc = umma_smem_desc(sa + (m * 4 + i) * 32 * KCH * 2, 16, sbo, layout);
#pragma unroll
                                for (int k = 0; k < KCH / 16; ++k)
                                    umma_bf16_elect(tmem_u + buf * ACC_COLS + m * BN, adesc + 2 * k, bdesc + 2 * k, idesc,
                                                    (g | i | k) != 0);
                            }
                        }
                        umma_commit_elect(&empty_bar[st]);
                    }
                    umma_commit_elect(&tfull[buf]);
                    ++lt;
                    continue;
                }
                const TapClass& tc_ = p.cls[tl.cls];
                int ks = 0;
                for (int tap = 0; tap < tc_.num_taps; ++tap) {
                    // column range of this tap's MMAs (parity-merged scatter: the rest of its weight slab is zeros)
                    const int nc = tc_.taps[tap].ncol;
                    const uint32_t col0 = nc ? (uint32_t)(nc & 0xff) * 32u : 0u;
                    const uint32_t idesc_t = nc ? umma_idesc_bf16(128, (nc >> 8) * 32, false, false) : idesc;
                    const uint32_t brow_off = (col0 / 8u) * (sbo >> 4);   // descriptor units (16 B) to weight row col0
                    for (int ch = 0; ch < p.num_chunks; ++ch, ++ks, ++it) {
                        const int st = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        mbar_wait(&full_bar[st], ph);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(smem + st * L::STAGE_BYTES);
                        const uint64_t bdesc = umma_smem_desc(sa + L::A_BYTES, 16, sbo, layout) + brow_off;
#pragma unroll
                        for (int m = 0; m < MT; ++m) {
                            if (!tl.live[m] || (p.skip & 4)) continue;
                            const uint64_t adesc = umma_smem_desc(sa + m * L::A_SUB, 16, sbo, layout);
#pragma unroll
                            for (int k = 0; k < KCH / 16; ++k)
                                umma_bf16_elect(tmem_u + buf * ACC_COLS + m * BN + col0, adesc + 2 * k, bdesc + 2 * k, idesc_t,
                                                (ks | k) != 0);
                        }
                        umma_commit_elect(&empty_bar[st]);
                    }
                }
                umma_commit_elect(&tfull[buf]);
                ++lt;
            }
        }
        __syncwarp();
    } else {
        // ================= epilogue =================
        // 8 epilogue warps: two per TMEM lane quarter (a warp may only read lanes 32*(warp%4)..+31); the two warps of a
        // quarter split the tile's 32-column chunks between them (even / odd), halving the epilogue's critical path
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const int xi = row % p.bw;
        const int yi = (row / p.bw) % p.bh;
        const int ni = row / (p.bw * p.bh);
        const bool do_stats = p.stat_sum != nullptr;
        const int etid = threadIdx.x - 64;
        const uint32_t stage_u32 = smem_u32(smem + L::STG_OFF) + (warp - 2) * 2048;   // this warp's store staging (2 KB)
        // BatchNorm statistics of the stored values: with the staging buffer a lane reads ONE COLUMN of the staged chunk
        // (32 two-byte loads, conflict-free) -- no 2 x 32 per-thread accumulators, no transposing shuffle reduction
        constexpr bool SMEM_STATS = L::STG_BYTES > 0;
        // per-channel sums of the tiles processed so far wait in the warps' shared-memory slots and go to the fp64 global
        // accumulators every 16 tiles (or when the column block changes): two named barriers + BN atomics per flush
        int stat_nt = -1, stat_cnt = 0;
        auto flush_stats = [&](int fnt) {
            named_bar_sync(1, 32 * IGP_EPI_WARPS);
            const int ncol = p.merge ? 32 : BN;
            const int cbase = p.merge ? 0 : fnt * BN;
            for (int i = etid; i < ncol; i += 32 * IGP_EPI_WARPS) {
                float a = 0.f, b = 0.f;
#pragma unroll
                for (int w = 0; w < L::STAT_SLOTS; ++w) {
                    a += s_stat[w * 2 * BN + i];
                    b += s_stat[w * 2 * BN + BN + i];
                    s_stat[w * 2 * BN + i] = 0.f;
                    s_stat[w * 2 * BN + BN + i] = 0.f;
                }
                atomicAdd(p.stat_sum + cbase + i, (double)a);
                atomicAdd(p.stat_sq + cbase + i, (double)b);
            }
            named_bar_sync(1, 32 * IGP_EPI_WARPS);
        };
        int lt = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const IgTile tl = ig_decode_tile<MT>(p, t, m_groups);
            if (!tl.any) continue;
            const TapClass& c = p.cls[tl.cls];
            const int buf = lt & 1;
            const int nt = tl.nt;
            if (do_stats && stat_cnt > 0 && (nt != stat_nt || stat_cnt >= 16)) {
                flush_stats(stat_nt);
                stat_cnt = 0;
            }
            stat_nt = nt;
            mbar_wait(&tfull[buf], (lt >> 1) & 1);
            tc_fence_after();
            // BatchNorm statistics: a warp owns the same 32-column chunk in every M sub-tile (and, for the parity-merged
            // scatter, every chunk folds onto the same 32 channels), so the per-thread values are summed in registers
            // first and the 62-shuffle transposing reduction + the shared-memory update run once per chunk (once per tile
            // when merged) instead of once per (chunk, sub-tile). Each warp adds into its own slot: no shared atomics
            // (an ncu capture of the 32->128 discriminator layer showed 37 % of the epilogue in this path, with
            // ATOMS.CAST.SPIN retry loops, and the tensor pipe waiting for TMEM at 32 % busy).
            float sacc[32], qacc[32];
            bool pending = false;
#pragma unroll
            for (int j = 0; j < 32; ++j) sacc[j] = qacc[j] = 0.f;
            float* my_stat = s_stat + (warp - 2) * 2 * BN;
            // PAIR path (bf16 output, BN >= 64): a warp takes two ADJACENT 32-column chunks of its 32 rows, so that a row's
            // 128 contiguous output bytes (for the parity-merged scatter: the two fine pixels 2x, 2x+1 of a coarse pixel) leave
            // as ONE whole 128-byte line written by eight lanes. The 2 KB staging buffer holds 16 rows x 128 B per pass
            // (16-byte pieces XOR-swizzled by row: conflict-free stores, loads and column reads); two passes per pair.
            constexpr bool PAIR = SMEM_STATS && BN >= 64;
            bool pair_done = false;
            if constexpr (PAIR) {
                if (!p.out_fp32 && p.pair) {
                    pair_done = true;
                    constexpr int PPM = BN / 64;        // pairs per M sub-tile
                    constexpr int NP = MT * PPM;
#pragma unroll 1
                    for (int pi = half; pi < ((p.skip & 2) ? 0 : NP); pi += 2) {
                        const int m = pi / PPM;
                        const int c0p = (pi - m * PPM) * 64;
                        if (!tl.live[m]) continue;
                        const bool valid_tile = (ni < p.bn) && (tl.n0[m] + ni < p.lim_n) && (tl.y0[m] + yi < c.lim_y) &&
                                                (tl.x0[m] + xi < c.lim_x);
                        const long long off_tile = c.out_off + (long long)(tl.n0[m] + ni) * p.out_sn +
                                                   (long long)(tl.y0[m] + yi) * p.out_sy +
                                                   (long long)(tl.x0[m] + xi) * p.out_sx + (long long)nt * BN;
                        uint32_t pkA[16], pkB[16];
                        bool vA, vB;
                        long long aA, aB;   // element offset of this row's 32 channels of chunk A / B in the output
                        auto chunk = [&](const int c0, uint32_t (&pk)[16], bool& valid, long long& addr) {
                            valid = valid_tile && !(p.skip & 8);
                            long long off = off_tile;
                            if (p.merge) {
                                const int g = (nt * BN + c0) >> 5;
                                const int ph = g >> 1, pw = (g == 0 || g == 3) ? 1 : 0;
                                valid = valid && (2 * (tl.y0[m] + yi) + ph < p.merge_oh) && (2 * (tl.x0[m] + xi) + pw < p.merge_ow);
                                off = off_tile - (long long)nt * BN + ph * p.merge_sy + pw * 32 - c0;
                            }
                            addr = off + c0;
                            uint32_t mbits = 0xffffffffu;
                            if (MASK && p.mask_bits && valid) mbits = __ldg(p.mask_bits + (addr >> 5));
                            uint32_t v[32];
                            tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * ACC_COLS + m * BN + c0, v);
                            tmem_ld_wait();
                            float f[32];
#pragma unroll
                            for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                            if (p.bias) {
                                const float* bp = p.bias + (p.merge ? 0 : nt * BN + c0);
#pragma unroll
                                for (int j = 0; j < 32; ++j) f[j] += __ldg(bp + j);
                            }
                            if (p.act == ACT_RELU) {
#pragma unroll
                                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
                            } else if (p.act == ACT_TANH) {
#pragma unroll
                                for (int j = 0; j < 32; ++j) f[j] = tanhf(f[j]);
                            } else if (p.act == ACT_SIGMOID) {
#pragma unroll
                                for (int j = 0; j < 32; ++j) f[j] = 1.f / (1.f + __expf(-f[j]));
                            }
                            if (MASK && p.mask_bits) {
#pragma unroll
                                for (int j = 0; j < 32; ++j)
                                    if (!((mbits >> j) & 1u)) f[j] = 0.f;
                            } else if (MASK && p.mask_y && valid) {
                                const __nv_bfloat16* yp = reinterpret_cast<const __nv_bfloat16*>(p.mask_y) + addr;
#pragma unroll
                                for (int j4 = 0; j4 < 4; ++j4) {
                                    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(yp + 8 * j4));
                                    const uint32_t rr[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                                    for (int j = 0; j < 4; ++j) {
                                        if (!(__uint_as_float(rr[j] << 16) > 0.f)) f[8 * j4 + 2 * j] = 0.f;
                                        if (!(__uint_as_float(rr[j] & 0xffff0000u) > 0.f)) f[8 * j4 + 2 * j + 1] = 0.f;
                                    }
                                }
                            }
#pragma unroll
                            for (int j = 0; j < 16; ++j) pk[j] = (do_stats && !valid) ? 0u : pack_bf16x2(f[2 * j], f[2 * j + 1]);
                        };
                        chunk(c0p, pkA, vA, aA);
                        chunk(c0p + 32, pkB, vB, aB);
                        const bool a_first = aA < aB;    // warp-uniform: which chunk holds the lower 64 bytes of the run
                        const long long run = a_first ? aA : aB;
                        const uint32_t vmF = __ballot_sync(0xffffffffu, a_first ? vA : vB);
                        const uint32_t vmS = __ballot_sync(0xffffffffu, a_first ? vB : vA);
                        float sF = 0.f, qF = 0.f, sS = 0.f, qS = 0.f;
#pragma unroll 1
                        for (int ps = 0; ps < 2; ++ps) {
                            if ((lane >> 4) == ps) {
                                const uint32_t x = lane & 7, base = stage_u32 + (lane & 15) * 128;
                                if (a_first) {
#pragma unroll
                                    for (int j = 0; j < 4; ++j) {
                                        sts_v4(base + ((j ^ x) << 4), pkA[4 * j], pkA[4 * j + 1], pkA[4 * j + 2], pkA[4 * j + 3]);
                                        sts_v4(base + (((4 + j) ^ x) << 4), pkB[4 * j], pkB[4 * j + 1], pkB[4 * j + 2], pkB[4 * j + 3]);
                                    }
                                } else {
#pragma unroll
                                    for (int j = 0; j < 4; ++j) {
                                        sts_v4(base + ((j ^ x) << 4), pkB[4 * j], pkB[4 * j + 1], pkB[4 * j + 2], pkB[4 * j + 3]);
                                        sts_v4(base + (((4 + j) ^ x) << 4), pkA[4 * j], pkA[4 * j + 1], pkA[4 * j + 2], pkA[4 * j + 3]);
                                    }
                                }
                            }
                            __syncwarp();
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int r16 = 4 * j + (lane >> 3);
                                const int src = 16 * ps + r16;
                                const int piece = lane & 7;
                                const long long o_r = __shfl_sync(0xffffffffu, run, src);
                                const uint4 v4 = lds_v4(stage_u32 + r16 * 128 + ((piece ^ (r16 & 7)) << 4));
                                if ((((piece < 4) ? vmF : vmS) >> src) & 1u)
                                    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + o_r + piece * 8) = v4;
                            }
                            if (do_stats) {   // lane = column `lane` of the first and of the second chunk
                                const uint32_t cb = stage_u32 + (lane & 7) * 2;
                                const uint32_t ch = lane >> 3;
#pragma unroll
                                for (int r = 0; r < 16; ++r) {
                                    const float a = __uint_as_float(lds_u16(cb + r * 128 + ((ch ^ (r & 7)) << 4)) << 16);
                                    const float b = __uint_as_float(lds_u16(cb + r * 128 + (((4 + ch) ^ (r & 7)) << 4)) << 16);
                                    sF += a;
                                    qF = fmaf(a, a, qF);
                                    sS += b;
                                    qS = fmaf(b, b, qS);
                                }
                            }
                            __syncwarp();
                        }
                        if (do_stats) {
                            if (p.merge) {      // both chunks fold onto channels 0..31
                                my_stat[lane] += sF + sS;
                                my_stat[BN + lane] += qF + qS;
                            } else {            // a_first is true here: first = columns c0p.., second = c0p + 32..
                                my_stat[c0p + lane] += sF;
                                my_stat[BN + c0p + lane] += qF;
                                my_stat[c0p + 32 + lane] += sS;
                                my_stat[BN + c0p + 32 + lane] += qS;
                            }
                        }
                    }
                }
            }
#pragma unroll 1
            for (int c0 = 0; c0 < ((p.skip & 2) || pair_done ? 0 : BN); c0 += 32) {
#pragma unroll 1
                for (int m = 0; m < MT; ++m) {
                    if (!tl.live[m]) continue;
                    if ((((m * (BN / 32)) + (c0 >> 5)) & 1) != half) continue;
                    const bool valid_tile = (ni < p.bn) && (tl.n0[m] + ni < p.lim_n) && (tl.y0[m] + yi < c.lim_y) &&
                                            (tl.x0[m] + xi < c.lim_x);
                    const long long off_tile = c.out_off + (long long)(tl.n0[m] + ni) * p.out_sn +
                                               (long long)(tl.y0[m] + yi) * p.out_sy +
                                               (long long)(tl.x0[m] + xi) * p.out_sx + (long long)nt * BN;
                    bool valid = valid_tile && !(p.skip & 8);
                    long long off = off_tile;
                    int stat_col = c0;
                    if (p.merge) {
                        const int g = (nt * BN + c0) >> 5;
                        const int ph = g >> 1, pw = (g == 0 || g == 3) ? 1 : 0;   // merged column groups: (0,1),(0,0),(1,0),(1,1)
                        valid = valid_tile && !(p.skip & 8) && (2 * (tl.y0[m] + yi) + ph < p.merge_oh) &&
                                (2 * (tl.x0[m] + xi) + pw < p.merge_ow);
                        off = off_tile - (long long)nt * BN + ph * p.merge_sy + pw * 32 - c0;
                        stat_col = 0;
                    }
                    // fused ReLU mask as a bit word (one 4-byte load, issued before the TMEM load so its latency hides)
                    uint32_t mbits = 0xffffffffu;
                    if (MASK && p.mask_bits && valid) mbits = __ldg(p.mask_bits + ((off + c0) >> 5));
                    uint32_t v[32];
                    tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * ACC_COLS + m * BN + c0, v);
                    tmem_ld_wait();
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                    if (p.bias) {
                        const float* bp = p.bias + (p.merge ? 0 : nt * BN + c0);  // merged: each 32-column group = channels 0..31
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] += __ldg(bp + j);
                    }
                    if (p.act == ACT_RELU) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
                    } else if (p.act == ACT_TANH) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = tanhf(f[j]);
                    } else if (p.act == ACT_SIGMOID) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) f[j] = 1.f / (1.f + __expf(-f[j]));
                    }
                    if (MASK && p.mask_bits) {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (!((mbits >> j) & 1u)) f[j] = 0.f;
                    } else if (MASK && p.mask_y && valid) {
                        const __nv_bfloat16* yp = reinterpret_cast<const __nv_bfloat16*>(p.mask_y) + off + c0;
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4) {
                            const uint4 raw = __ldg(reinterpret_cast<const uint4*>(yp + 8 * j4));
                            const uint32_t rr[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                if (!(__uint_as_float(rr[j] << 16) > 0.f)) f[8 * j4 + 2 * j] = 0.f;
                                if (!(__uint_as_float(rr[j] & 0xffff0000u) > 0.f)) f[8 * j4 + 2 * j + 1] = 0.f;
                            }
                        }
                    }
                    if (p.out_fp32) {
                        if (valid) {
                            float* o = reinterpret_cast<float*>(p.out) + off + c0;
                            if (p.atomic_out) {
#pragma unroll
                                for (int j = 0; j < 32; j += 4) red_add_v4(o + j, f[j], f[j + 1], f[j + 2], f[j + 3]);
                            } else {
#pragma unroll
                                for (int j = 0; j < 32; j += 4)
                                    *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                            }
                        }
                    } else {
                        uint32_t pk[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
                        if constexpr (L::STG_BYTES > 0) {
                            // A lane holds 64 contiguous bytes of ONE output row; stored directly, every warp-wide 16-byte
                            // store touches 32 rows = 32 half-written sectors (the L2 write requests, not the bytes, bound the
                            // thin-K launches: switching the stores off took 25-43 % off them). Through the warp's staging
                            // buffer (16-byte chunks XOR-swizzled by row pair: conflict-free both ways) four lanes store one
                            // row's 64 bytes = two whole sectors per row.
                            const uint32_t sw = (lane >> 1) & 3;
                            if (SMEM_STATS && do_stats && !valid) {   // rows outside the output do not count
#pragma unroll
                                for (int j = 0; j < 16; ++j) pk[j] = 0u;
                            }
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                sts_v4(stage_u32 + lane * 64 + ((j ^ sw) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                            const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
                            const long long offc = off + c0;
                            __syncwarp();
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int r = 8 * j + (lane >> 2);
                                const long long o_r = __shfl_sync(0xffffffffu, offc, r);
                                const uint4 v4 = lds_v4(stage_u32 + r * 64 + (((lane & 3) ^ ((r >> 1) & 3)) << 4));
                                if ((vmask >> r) & 1u)
                                    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + o_r + (lane & 3) * 8) = v4;
                            }
                            if (SMEM_STATS && do_stats) {   // lane = column c0 + lane of the staged (= stored) values
                                const uint32_t cb = stage_u32 + (lane & 7) * 2;
                                const uint32_t ch = lane >> 3;
                                float s1 = 0.f, s2 = 0.f;
#pragma unroll
                                for (int r = 0; r < 32; ++r) {
                                    const float v = __uint_as_float(lds_u16(cb + r * 64 + ((ch ^ ((r >> 1) & 3)) << 4)) << 16);
                                    s1 += v;
                                    s2 = fmaf(v, v, s2);
                                }
                                my_stat[stat_col + lane] += s1;
                                my_stat[BN + stat_col + lane] += s2;
                            }
                            __syncwarp();
                        } else if (valid) {
                            __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + off + c0;
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                *reinterpret_cast<uint4*>(o + 8 * j) =
                                    make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                        }
                        if (!SMEM_STATS && do_stats) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                f[2 * j] = __uint_as_float(pk[j] << 16);
                                f[2 * j + 1] = __uint_as_float(pk[j] & 0xffff0000u);
                            }
                        }
                    }
                    if (!SMEM_STATS && do_stats) {
                        float g2[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            f[j] = valid ? f[j] : 0.f;
                            g2[j] = f[j] * f[j];
                        }
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            sacc[j] += f[j];
                            qacc[j] += g2[j];
                        }
                        pending = true;
                    }
                }
                if (!SMEM_STATS && do_stats && pending && !p.merge) {   // this chunk's columns are complete for the tile
                    const float s1 = warp_colsum32(sacc, lane);
                    const float s2 = warp_colsum32(qacc, lane);
                    my_stat[c0 + lane] += s1;
                    my_stat[BN + c0 + lane] += s2;
#pragma unroll
                    for (int j = 0; j < 32; ++j) sacc[j] = qacc[j] = 0.f;
                    pending = false;
                }
            }
            if (!SMEM_STATS && do_stats && pending) {   // merged scatter: every chunk of the tile folded onto channels 0..31
                const float s1 = warp_colsum32(sacc, lane);
                const float s2 = warp_colsum32(qacc, lane);
                my_stat[lane] += s1;
                my_stat[BN + lane] += s2;
            }
            // accumulators of this buffer are in registers / memory: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[buf]);
            if (do_stats) ++stat_cnt;
            ++lt;
        }
        if (do_stats && stat_cnt > 0) flush_stats(stat_nt);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// weight gradient: out[tap][m][n] += sum_pixels D[pixel][m] * S[pixel @ tap][n]
// ------------------------------------------------------------------------------------------------
struct WgParams {
    CUtensorMap mapD;     // dense operand (C, X, Y, N) box (64, bw, bh, bn)
    CUtensorMap mapS[4];  // shifted operand planes, box (NCH, bw, bh, bn)
    TapDesc taps[25];
    int num_taps;
    int rows;  // bw*bh*bn, multiple of 16
    float* out;
    long long split_stride;  // elements between the output slices of consecutive splits (0: all splits add into one)
    int bw, bh, bn;
    int tiles_x, tiles_y, tiles_n;  // pixel tiles (the reduction)
    int m_total, n_total;
    int m_tiles, n_tiles;
    int splits;
};

// TG = filter taps handled by one CTA against the SAME dense-operand tile: with a 32-channel shifted side the dense tile
// (32 KB) dwarfs a tap's shifted tile (8 KB), and one-tap CTAs re-fetch it 25x through L2 (wgrad_kernel<32,32,4> ran at
// 184 TFLOP/s, 12 % tensor pipe). TG = 5 (one filter row) cuts the bytes per MMA-clock 2.9x; the TG accumulators sit side
// by side in TMEM.
template <int BN, int NCH, int STAGES, int TG = 1>
struct WgSmem {
    static constexpr int D_BYTES = 128 * 128 * 2;  // [2 chunks][128 pixels][64 ch]
    static constexpr int S_BYTES = 128 * BN * 2;   // [BN/NCH chunks][128 pixels][NCH ch] per tap
    static constexpr int STAGE_BYTES = D_BYTES + TG * S_BYTES;
    static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
    static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 1) * 8 + 16 + 1024;
};

template <int BN, int NCH, int STAGES, int TG>
__global__ void __launch_bounds__(192) wgrad_kernel(const __grid_constant__ WgParams p) {
    using L = WgSmem<BN, NCH, STAGES, TG>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int tap0 = blockIdx.x * TG;
    const int tg_live = min(TG, p.num_taps - tap0);  // the last group may be short (25 taps, TG = 2)
    const int mtile = blockIdx.y % p.m_tiles;
    const int ntile = blockIdx.y / p.m_tiles;
    const int split = blockIdx.z;
    const int pt_total = p.tiles_x * p.tiles_y * p.tiles_n;
    const int pt_begin = (int)((long long)split * pt_total / p.splits);
    const int pt_end = (int)((long long)(split + 1) * pt_total / p.splits);
    if (pt_begin >= pt_end) return;
    const int npt = pt_end - pt_begin;

    constexpr uint32_t TMEM_COLS = (TG * BN) <= 32 ? 32 : ((TG * BN) <= 64 ? 64 : ((TG * BN) <= 128 ? 128 : ((TG * BN) <= 256 ? 256 : 512)));
    static_assert(TG * BN <= 512, "accumulators must fit TMEM");
    constexpr int S_CHUNKS = BN / NCH;
    const uint32_t d_chunk_bytes = p.rows * 128;
    const uint32_t s_chunk_bytes = p.rows * NCH * 2;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.mapD);
        tma_prefetch_desc(&p.mapS[p.taps[tap0].map]);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        {   // warp-converged producer, elected TMA issue, incremental pixel-tile counters (see igemm_persistent_kernel)
            const int d_chunks_live = (p.m_total - mtile * 128) >= 128 ? 2 : 1;
            const uint32_t tx_bytes = d_chunks_live * d_chunk_bytes + tg_live * S_CHUNKS * s_chunk_bytes;
            int tx = pt_begin % p.tiles_x;
            int ty = (pt_begin / p.tiles_x) % p.tiles_y;
            int tn = pt_begin / (p.tiles_x * p.tiles_y);
            for (int i = 0; i < npt; ++i) {
                const int st = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                mbar_wait(&empty_bar[st], ph ^ 1);
                mbar_arrive_expect_tx_elect(&full_bar[st], tx_bytes);
                const int x0 = tx * p.bw, y0 = ty * p.bh, n0 = tn * p.bn;
                uint8_t* sd = smem + st * L::STAGE_BYTES;
                for (int cchunk = 0; cchunk < d_chunks_live; ++cchunk)
                    tma_load_4d_elect(sd + cchunk * d_chunk_bytes, &p.mapD, &full_bar[st], mtile * 128 + cchunk * 64, x0,
                                      y0, n0);
#pragma unroll
                for (int tg = 0; tg < TG; ++tg) {
                    if (tg >= tg_live) break;
                    const TapDesc t = p.taps[tap0 + tg];
                    uint8_t* ss = sd + L::D_BYTES + tg * L::S_BYTES;
#pragma unroll
                    for (int cchunk = 0; cchunk < S_CHUNKS; ++cchunk)
                        tma_load_4d_elect(ss + cchunk * s_chunk_bytes, &p.mapS[t.map], &full_bar[st],
                                          ntile * BN + cchunk * NCH, x0 + t.dx, y0 + t.dy, n0);
                }
                if (++tx == p.tiles_x) {
                    tx = 0;
                    if (++ty == p.tiles_y) {
                        ty = 0;
                        ++tn;
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        {   // warp-converged issue loop, one elected lane per tcgen05 instruction (see igemm_persistent_kernel)
            constexpr uint32_t idesc = umma_idesc_bf16(128, BN, true, true);
            constexpr uint64_t s_layout = (NCH == 64) ? UMMA_SW128 : UMMA_SW64;
            constexpr uint32_t s_row = NCH * 2;
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
            const int ksteps = p.rows / 16;
            for (int i = 0; i < npt; ++i) {
                const int st = i % STAGES;
                const uint32_t ph = (i / STAGES) & 1;
                mbar_wait(&full_bar[st], ph);
                tc_fence_after();
                const uint32_t sd = smem_u32(smem + st * L::STAGE_BYTES);
                // MN-major: LBO = distance between 64(32)-channel chunks, SBO = 8 pixel rows
                const uint64_t adesc = umma_smem_desc(sd, d_chunk_bytes, 8 * 128, UMMA_SW128);
                if constexpr (TG > 1 && BN == NCH && TG * BN <= 256) {
                    // One channel chunk per tap: the TG shifted tiles sit at a fixed stride in the stage, which is exactly
                    // an MN-major operand whose N-direction atom stride (LBO) is the tile stride. ONE N = TG*BN MMA per
                    // K step instead of TG N = BN ones: the 32-channel layers were issue-bound at 40 N = 32 MMAs per stage.
                    const uint32_t idesc_m = umma_idesc_bf16(128, tg_live * BN, true, true);
                    const uint64_t bdesc = umma_smem_desc(sd + L::D_BYTES, L::S_BYTES, 8 * s_row, s_layout);
                    for (int k = 0; k < ksteps; ++k)
                        umma_bf16_elect(tmem_u, adesc + ((k * 16 * 128) >> 4), bdesc + ((k * 16 * s_row) >> 4), idesc_m,
                                        (i | k) != 0);
                } else {
#pragma unroll
                    for (int tg = 0; tg < TG; ++tg) {
                        if (tg >= tg_live) break;
                        const uint64_t bdesc =
                            umma_smem_desc(sd + L::D_BYTES + tg * L::S_BYTES, s_chunk_bytes, 8 * s_row, s_layout);
                        for (int k = 0; k < ksteps; ++k)
                            umma_bf16_elect(tmem_u + tg * BN, adesc + ((k * 16 * 128) >> 4),
                                            bdesc + ((k * 16 * s_row) >> 4), idesc, (i | k) != 0);
                    }
                }
                umma_commit_elect(&empty_bar[st]);
            }
            umma_commit_elect(tmem_full);
        }
        __syncwarp();
    } else {
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int q = warp & 3;
        const int m = mtile * 128 + q * 32 + lane;
        const bool valid = m < p.m_total;
#pragma unroll 1
        for (int tg = 0; tg < tg_live; ++tg) {
            float* orow = p.out + blockIdx.z * p.split_stride + ((long long)(tap0 + tg) * p.m_total + m) * p.n_total +
                          ntile * BN;
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + tg * BN + c0, v);
                tmem_ld_wait();
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4)
                        red_add_v4(orow + c0 + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                   __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace fmri
