// Halo-tile weight gradient of the 3-channel edge convolutions on tcgen05 ("hwgrad").
//
//   dwk[(ci*25 + tap)*C + c] += sum over pixels p of T[p][c] * img[ci][p + tap - 2]        (stride 1, 5x5, pad 2)
//
// T is the C-channel NHWC bf16 tensor on the convolution's grid (C = 32 / 64: the conv output gradient for a 3 -> C conv, the
// conv input for a C -> 3 conv), img the 3-channel tensor repacked as bf16 NHWC-8 (16 B per pixel, img8_pack_kernel).
// The reduction runs over PIXELS, so both operands are MN-major with the pixel as the K index:
//   A = T tile [K = pixels][M = channels], TMA box (64 ch, PWp columns, bh rows) with 128-byte swizzle; the box is wider than
//       the image (PWp >= PW + 4, bh*PWp a multiple of 16), TMA zero-fills the columns outside, so pixel r = yy*PWp + xx;
//   B = image halo slab [pixel][8 ch = 16 B], no swizzle: for filter row kh ONE MMA covers all five kw taps as N chunks --
//       chunk kw starts one slab row (16 B) after chunk kw-1, i.e. the N-chunk stride of the descriptor is 16 B and the
//       chunks overlap in memory. N = 48 (6 chunks; the 6th is a dummy tap whose accumulator columns are dropped).
// Five accumulators (one per kh, 48 columns) + a 16-column "ones" accumulator for the bias gradient live in TMEM for the
// whole (persistent) CTA and are flushed once with fp32 atomics. CUDA-core version: edge_wgrad_rows_kernel (FMA bound).
//
// Reference ops: weight gradients of Discriminator.conv[0] (vae_gan.py:145) and Decoder.conv[3] (vae_gan.py:118).
#pragma once
#include "ptx.cuh"
#include "hconv_kernels.cuh"

namespace fmri {

struct HwParams {
    CUtensorMap mapT;            // (C, PW, PH, N) box (64, PWp, bh, 1), SWIZZLE_128B
    const __nv_bfloat16* img8;   // [N][IH][IW][8]
    int N, PH, PW, C;
    int PWp, bh;                 // padded tile width, tile rows; rows = bh*PWp (multiple of 16, <= 256: the ones slab)
    int tiles_y;                 // tiles per image
    int slab_rows;               // (bh+4)*PWp + 16, multiple of 8
    float* dwk;                  // [75][C] fp32, +=
    float* dbias;                // [C] fp32 += sum_p T[p][c], nullable
    int flip;                    // write tap 24-tap (C -> 3 conv: T is the conv input, img the output gradient)
    int stages;                  // pipeline depth (<= HW_MAX_STAGES): the tiles are small, so depth hides the L2 latency
    int d_chunk;                 // bytes between the two 64-channel chunks of an A stage (rows*128 rounded up to 1 KB)
    // Stride-2 convolutions run as four launches, one per input parity plane (ph, pw): img8 then holds the plane
    // img[2y + ph][2x + pw] on the T grid, the plane's taps are unit shifts, and virtual tap (kh5, kw5) of this stride-1 kernel
    // is the real tap (2 (kh5 - 1) + ph, 2 (kw5 - 1) + pw). Only filter rows [kh0, kh0 + nkh) are issued and flushed.
    int kh0, nkh;                // filter rows handled (0, 5 for a stride-1 convolution)
    int plane;                   // 0: stride 1; 1: parity-plane launch (remap below)
    int ph, pw;
};

constexpr int HW_MAX_STAGES = 8;
constexpr int HW_THREADS = 384;
constexpr int HW_PRODUCERS = 160;   // warps 2-6
__host__ __device__ inline int hw_stage_bytes(const HwParams& p) { return 2 * p.d_chunk + ((p.slab_rows * 16 + 1023) / 1024) * 1024; }
__host__ __device__ inline int hw_smem_bytes(const HwParams& p) { return p.stages * hw_stage_bytes(p) + 4096 + 256 + 1024; }

__global__ void __launch_bounds__(HW_THREADS) hwgrad_kernel(const __grid_constant__ HwParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int stage_bytes = hw_stage_bytes(p);
    const int HW_STAGES = p.stages;
    uint8_t* s_ones = smem + HW_STAGES * stage_bytes;                 // [256 rows][16 B] of bf16 1.0 (rows = bh*PWp <= 256)
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_ones + 4096);
    uint64_t* full_bar = bars;                    // [STAGES] count = 1 (TMA expect_tx) + producers
    uint64_t* empty_bar = bars + HW_MAX_STAGES;   // [STAGES] count = 2 (one tcgen05.commit per issuing warp)
    uint64_t* tmem_full = bars + 2 * HW_MAX_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * HW_MAX_STAGES + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = p.N * p.tiles_y;
    const int rows = p.bh * p.PWp;
    constexpr uint32_t TMEM_COLS = 256;           // 5 x 48 + 16
    // MMA issuers: one warp per filter row kh (warps 1, 7, 8, 9, 10) + warp 11 for the bias-gradient column. The kernel sat at
    // 54 % tensor-pipe activity with two issuing warps (each tcgen05.mma costs its warp ~40 issue cycles against a 24-cycle
    // dispatch floor for N = 48); warps 8-11 are the epilogue warps, idle until the single flush at the end.
    const int n_issuers = p.nkh + (p.dbias ? 1 : 0);

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&p.mapT);
        for (int s = 0; s < HW_STAGES; ++s) {
            mbar_init(&full_bar[s], 1 + HW_PRODUCERS);
            mbar_init(&empty_bar[s], n_issuers);   // every issuing warp commits
        }
        mbar_init(tmem_full, n_issuers);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    // constant smem: ones slab, zeroed second channel chunk of every A stage (rows 64..127 of M are never loaded) and zeroed
    // slab tails, so no uninitialised (possibly NaN) word ever meets a zero of the other operand
    for (int i = threadIdx.x; i < 4096 / 4; i += HW_THREADS) reinterpret_cast<uint32_t*>(s_ones)[i] = 0x3F803F80u;
    for (int s = 0; s < HW_STAGES; ++s) {
        uint32_t* st = reinterpret_cast<uint32_t*>(smem + s * stage_bytes);
        for (int i = threadIdx.x; i < stage_bytes / 4; i += HW_THREADS) st[i] = 0u;
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer of the T tile =================
        if (lane == 0) {
            int it = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
                const int st = it % HW_STAGES;
                const uint32_t ph = (it / HW_STAGES) & 1;
                const int n = t / p.tiles_y, y0 = (t - n * p.tiles_y) * p.bh;
                mbar_wait(&empty_bar[st], ph ^ 1);
                mbar_arrive_expect_tx(&full_bar[st], rows * 128);
                tma_load_4d(smem + st * stage_bytes, &p.mapT, &full_bar[st], 0, 0, y0, n);
            }
        }
        __syncwarp();
    }
    const int issuer = warp == 1 ? 0 : (warp == 7 ? 1 : (warp >= 8 ? warp - 6 : -1));   // 0..4 = kh, 5 = bias column
    if (issuer >= 0 && issuer < n_issuers) {
        // ================= MMA issuers (warp-converged, elected lane) =================
        // M = 64: the T tile has at most 64 channels, and an M = 128 instruction would read (and multiply) a second, all-zero
        // 64-row half of A from shared memory on every MMA -- the kernel ran at 97 % shared-memory throughput. With M = 64
        // the accumulator row r sits in TMEM lane 32 * (r / 16) + r % 16 (scripts/probes/m64_layout_probe.cu, measured).
        const uint32_t idesc = umma_idesc_bf16(64, 48, true, true);
        const uint32_t idesc1 = umma_idesc_bf16(64, 16, true, true);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        // B (image slab, MN-major, no swizzle): 16-byte N chunks one slab row apart; K advances in 8-pixel groups of 128 B.
        constexpr uint32_t b_lbo = 128, b_sbo = 16;
        const int ksteps = rows / 16;
        int it = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int st = it % HW_STAGES;
            const uint32_t ph = (it / HW_STAGES) & 1;
            mbar_wait(&full_bar[st], ph);
            tc_fence_after();
            const uint32_t sd = smem_u32(smem + st * stage_bytes);
            const uint32_t ss = sd + 2 * p.d_chunk;
            const uint64_t adesc = umma_smem_desc(sd, p.d_chunk, 8 * 128, UMMA_SW128);   // as wgrad_kernel: LBO = 64-channel chunk
            if (issuer < p.nkh) {
                const int kh = p.kh0 + issuer;
                const uint64_t bdesc = umma_smem_desc(ss, b_lbo, b_sbo, 0) + (uint32_t)(kh * p.PWp);
                for (int k = 0; k < ksteps; ++k)
                    umma_bf16_elect(tmem_u + kh * 48, adesc + ((k * 16 * 128) >> 4), bdesc + (uint32_t)(k * 16), idesc,
                                    (it | k) != 0);
            } else {
                const uint64_t odesc = umma_smem_desc(smem_u32(s_ones), b_lbo, b_sbo, 0);
                for (int k = 0; k < ksteps; ++k)
                    umma_bf16_elect(tmem_u + 240, adesc + ((k * 16 * 128) >> 4), odesc + (uint32_t)(k * 16), idesc1, (it | k) != 0);
            }
            umma_commit_elect(&empty_bar[st]);
        }
        umma_commit_elect(tmem_full);
        __syncwarp();
    }
    if (warp == 0 || warp == 1 || warp == 7) {
        // (TMA producer / pure issuer warps: nothing else to do)
    } else if (warp >= 2 && warp < 2 + HW_PRODUCERS / 32) {
        // ================= image halo producers (cp.async 16 B per pixel, zero fill = padding) =================
        const int ptid = threadIdx.x - 64;
        const int halo_px = (p.bh + 4) * p.PWp;
        int it = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int st = it % HW_STAGES;
            const uint32_t ph = (it / HW_STAGES) & 1;
            const int n = t / p.tiles_y, y0 = (t - n * p.tiles_y) * p.bh;
            mbar_wait(&empty_bar[st], ph ^ 1);
            const uint32_t ss = smem_u32(smem + st * stage_bytes) + 2 * p.d_chunk;
            const __nv_bfloat16* In = p.img8 + (size_t)n * p.PH * p.PW * 8;
            int row = ptid;
            int sy = row / p.PWp, sx = row - sy * p.PWp;
            for (; row < halo_px; row += HW_PRODUCERS) {
                const int iy = y0 + sy - 2, ix = sx - 2;
                const bool ok = iy >= 0 && iy < p.PH && ix >= 0 && ix < p.PW;
                cp_async16(ss + row * 16, ok ? In + ((size_t)iy * p.PW + ix) * 8 : In, ok ? 16u : 0u);
                sx += HW_PRODUCERS;
                while (sx >= p.PWp) { sx -= p.PWp; ++sy; }
            }
            cp_async_wait_all();
            fence_proxy_async_smem();
            mbar_arrive(&full_bar[st]);
        }
    }
    if (warp >= 8) {
        // ================= epilogue: one flush of the accumulators =================
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int q = warp & 3;
        const int c = q * 16 + lane;                 // M = 64 layout: lanes 0..15 of quarter q hold rows 16 q .. 16 q + 15
        const bool valid = lane < 16 && c < p.C;
        for (int kh = p.kh0; kh < p.kh0 + p.nkh; ++kh) {
#pragma unroll 1
            for (int part = 0; part < 3; ++part) {   // 48 columns = 3 x 16: chunks (2 part, 2 part + 1) of 8 columns
                uint32_t v[16];
                tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + kh * 48 + part * 16, v);
                tmem_ld_wait();
                if (!valid) continue;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int kw = part * 2 + h;
                    if (kw >= 5) continue;
                    int tap = kh * 5 + kw;
                    if (p.plane) {   // virtual tap of the parity plane -> real tap of the stride-2 filter
                        const int rkh = 2 * (kh - 1) + p.ph, rkw = 2 * (kw - 1) + p.pw;
                        if (kh < 1 || kw < 1 || rkh > 4 || rkw > 4) continue;
                        tap = rkh * 5 + rkw;
                    }
                    if (p.flip) tap = 24 - tap;
#pragma unroll
                    for (int ci = 0; ci < 3; ++ci)
                        atomicAdd(p.dwk + (size_t)blockIdx.x * 75 * p.C + (size_t)(ci * 25 + tap) * p.C + c,
                                  __uint_as_float(v[h * 8 + ci]));
                }
            }
        }
        if (p.dbias) {
            uint32_t v[16];
            tmem_ld16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + 240, v);
            tmem_ld_wait();
            if (valid) atomicAdd(p.dbias + (size_t)blockIdx.x * p.C + c, __uint_as_float(v[0]));
        }
        tc_fence_before();
    }
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);  // the allocating warp
}

}  // namespace fmri
