// Halo-tile implicit-GEMM convolution ("hconv") for the thin-channel 5x5 convolutions at the network edges.
//
// Why: the tap-per-TMA-box kernel (igemm_kernel) re-fetches the activation tile from L2 once per filter tap, and the
// 3-channel image side cannot feed a tensor-core K dimension at all. Here the activation HALO tile of an output tile is
// staged in shared memory ONCE and every tap reads it through a shifted shared-memory descriptor:
//   * the halo tile is stored as "16-byte column slabs": slab j holds channels [8j, 8j+8) of every halo pixel, pixels
//     linearised row-major over the padded tile width PW -> a tcgen05 NO-SWIZZLE K-major operand whose 8x16B core matrices
//     are contiguous 128 B (SBO = 128 B between 8-row groups, LBO = byte distance between the two K halves of an MMA);
//   * output pixel r = yy*PW + xx of the (virtual, padded-width) tile reads halo row r + dy*PW + dx for tap (dy, dx): a tap
//     is just a start-address offset of 16*(dy*PW+dx) bytes. Columns xx >= OW of the virtual tile are computed and dropped;
//   * with >= 16 input channels a K = 16 MMA step takes its two K halves from two adjacent channel slabs (LBO = slab size);
//     with the 3-channel image (padded to 8 bf16 channels = one 16 B slab entry per pixel) a K = 16 step takes its two K
//     halves from TWO DIFFERENT TAPS of the same slab (LBO = the byte distance between the two taps' windows), so the 25 taps
//     of a 5x5 filter are 13 MMA steps;
//   * stride-2 convolutions read four stride-parity planes of the input, each with its own halo slab;
//   * the weights of ALL steps stay resident in shared memory for the life of the (persistent) CTA.
// Roles (384 threads): warps 0-2 = MMA issuers (sub-tile m is issued by warp m % 3: the MMAs here are small, N = 16..64, so
// the kernel is bound by how fast tcgen05.mma can be ISSUED; each issuer runs warp-converged with uniform operands and an
// ELECTED lane, see umma_bf16_elect), the next 5 warps = halo producers (cp.async 16 B with zero fill = conv padding), the last
// 8 warps = epilogue (TMEM -> registers -> bias / activation -> global). Halo slabs and TMEM accumulators are double buffered, so
// producer, tensor pipe and epilogue of consecutive tiles overlap.
//
// Reference ops: Decoder.conv[3] Conv2d(C,3,5,s1,p2)+bias+tanh (/root/reference/models/vae_gan.py:118-121) fprop / dgrad,
// Discriminator.conv[0] Conv2d(3,C,5,s,p2)+bias+ReLU (:145-147) fprop / dgrad, Encoder.conv[0] Conv2d(3,64,5,s2,p2) (:74).
#pragma once
#include "ptx.cuh"

namespace fmri {

struct HcStep {       // one K = 16 MMA step, offsets in 16-byte units
    uint32_t a_off;   // start of the A window inside a halo buffer (plane base + tap offset + channel-slab offset)
    uint32_t a_lbo;   // distance between the two K halves of A
    uint32_t b_off;   // first weight row of this step inside the first K-half slab of B
};
constexpr int HC_MAX_STEPS = 104;

struct HcParams {
    const __nv_bfloat16* X;  // NHWC input [N][H][W][8*chunks]
    int N, H, W;
    int chunks;                  // 8-channel slabs per plane
    int num_planes;
    int pl_ys[4], pl_xs[4];      // input step per halo row / column (1, or 2 for stride-parity planes)
    int pl_yoff[4], pl_xoff[4];  // input y of halo row sy is (oy0 + sy) * ys + yoff, likewise x
    int PW, PH;                  // halo tile width / height (pixels)
    int skip;                    // diagnostic (FMRI_HC_SKIP): bit 0 producers skip the halo copies, bit 1 epilogue skips its global
                                 // stores, bit 2 issuers skip the MMAs -- which role bounds the kernel (results are garbage)
    int slab_rows;               // allocated rows per slab (>= halo rows; 2 mod 8 when there are several channel chunks)
    int num_steps;
    HcStep steps[HC_MAX_STEPS];
    int THt, tiles_y;            // output rows per tile, tiles per image
    int OH, OW;                  // output grid
    int MT;                      // 128-row MMA sub-tiles per tile
    const __nv_bfloat16* Bslab;  // weights in slab layout [2 K-halves][num_steps*BN][8]
    int epi;                     // 0: NCHW fp32, n_out channels (image side); 1: NHWC bf16, BN channels
    void* out;
    const float* bias;           // [n_out] / [BN] or null
    int act;
    int n_out;
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

__device__ __forceinline__ float hc_act(float v, int act) {
    if (act == 1) return fmaxf(v, 0.f);
    if (act == 2) return tanhf(v);
    if (act == 3) return 1.f / (1.f + __expf(-v));
    return v;
}

constexpr int HC_ISSUERS = 5;                       // MMA-issuing warps (one per 128-row sub-tile, MT <= 5)
constexpr int HC_PRODUCERS = 160;                   // the next 5 warps: halo producers
constexpr int HC_EPI_WARPS = 8;                     // two per TMEM lane quarter (quarter = warp % 4): they alternate sub-tiles
constexpr int HC_THREADS = 32 * HC_ISSUERS + HC_PRODUCERS + 32 * HC_EPI_WARPS;

// shared-memory plan (host and device agree through these helpers)
__host__ __device__ inline int hc_slab_bytes(const HcParams& p) { return p.slab_rows * 16; }
__host__ __device__ inline int hc_a_buffer_bytes(const HcParams& p) { return p.num_planes * p.chunks * hc_slab_bytes(p); }
__host__ __device__ inline int hc_b_bytes(const HcParams& p, int BN) { return 2 * p.num_steps * BN * 16; }
__host__ __device__ inline int hc_smem_bytes(const HcParams& p, int BN) {
    return 2 * hc_a_buffer_bytes(p) + hc_b_bytes(p, BN) + 512 + 1024;
}

template <int BN>
__global__ void __launch_bounds__(HC_THREADS, 2) hconv_kernel(const __grid_constant__ HcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int a_buf = hc_a_buffer_bytes(p);
    const int slab = hc_slab_bytes(p);
    const int chunks = p.chunks;
    uint8_t* sA = smem;                      // [2][planes][chunks][slab_rows][16]
    uint8_t* sB = smem + 2 * a_buf;          // [2][num_steps*BN][16]
    const int b_half = p.num_steps * BN * 16;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sB + hc_b_bytes(p, BN));
    uint64_t* slab_full = bars;       // [2] count = producers
    uint64_t* slab_empty = bars + 2;  // [2] count = active issuers (one tcgen05.commit each)
    uint64_t* tmem_full = bars + 4;   // [2] count = active issuers
    uint64_t* tmem_empty = bars + 6;  // [2] count = HC_EPI_WARPS
    uint64_t* b_full = bars + 8;      // count = producers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
    float* s_bias = reinterpret_cast<float*>(bars + 10);   // [64] bias of the NHWC epilogue (zeros when there is none)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 64) s_bias[threadIdx.x] = (p.bias && p.epi == 1 && (int)threadIdx.x < BN) ? p.bias[threadIdx.x] : 0.f;
    const int total_tiles = p.N * p.tiles_y;
    const int acc_cols = p.MT * BN;  // TMEM columns of one accumulator buffer
    const int issuers = p.MT < HC_ISSUERS ? p.MT : HC_ISSUERS;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * acc_cols) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&slab_full[i], HC_PRODUCERS);
            mbar_init(&slab_empty[i], issuers);
            mbar_init(&tmem_full[i], issuers);
            mbar_init(&tmem_empty[i], HC_EPI_WARPS);
        }
        mbar_init(b_full, HC_PRODUCERS);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, tmem_cols);
    // zero both halo buffers once: rows past the halo are never written by the producers, and although only dropped output
    // rows (or zero-weight K halves) ever read them, an uninitialised NaN pattern must not meet a zero of the other operand
    for (int i = threadIdx.x; i < (2 * a_buf) / 16; i += HC_THREADS) reinterpret_cast<uint4*>(sA)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < HC_ISSUERS) {
        // ======================================================== MMA issuers
        // The whole warp runs this loop converged with warp-uniform operands and one ELECTED lane issues each tcgen05
        // instruction. Descriptors are formed by adding a (byte offset >> 4) to a base descriptor -- the 14-bit start-
        // address field never carries into the LBO field (shared memory < 256 KB).
        if (warp < issuers) {
            const uint32_t idesc = umma_idesc_bf16(128, BN, false, false);
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
            mbar_wait(b_full, 0);
            tc_fence_after();
            const uint64_t b_base = umma_smem_desc(smem_u32(sB), b_half, 128, 0);
            int it = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
                const int sb = it & 1;
                const uint32_t par = (it >> 1) & 1;
                mbar_wait(&slab_full[sb], par);
                mbar_wait(&tmem_empty[sb], par ^ 1);
                tc_fence_after();
                const uint64_t a_base = umma_smem_desc(smem_u32(sA + sb * a_buf), 0, 128, 0);  // LBO filled in per step
                const uint32_t d0 = tmem_u + sb * acc_cols;
                uint32_t acc = 0;  // the first step overwrites the accumulators
#pragma unroll 4
                for (int s = 0; s < p.num_steps; ++s) {
                    const HcStep stp = p.steps[s];
                    const uint64_t ad = (a_base | (static_cast<uint64_t>(stp.a_lbo & 0x3FFF) << 16)) + stp.a_off;
                    const uint64_t bd = b_base + stp.b_off;
                    if (p.skip & 4) continue;
                    for (int m = warp; m < p.MT; m += issuers)  // this warp's sub-tiles: independent accumulators
                        umma_bf16_elect(d0 + m * BN, ad + (uint32_t)(m * 128), bd, idesc, acc);
                    acc = 1;
                }
                umma_commit_elect(&slab_empty[sb]);  // halo buffer reusable once these MMAs retire
                umma_commit_elect(&tmem_full[sb]);   // accumulators ready for the epilogue
            }
        }
        __syncwarp();
    } else if (warp < HC_ISSUERS + HC_PRODUCERS / 32) {
        // ======================================================== halo producers (cp.async, zero fill = padding)
        const int ptid = threadIdx.x - 32 * HC_ISSUERS;
        {   // weights once: the global pack already has the slab layout -> straight 16 B copies
            const int n16 = hc_b_bytes(p, BN) / 16;
            const uint32_t b0 = smem_u32(sB);
            for (int i = ptid; i < n16; i += HC_PRODUCERS)
                cp_async16(b0 + i * 16, reinterpret_cast<const uint8_t*>(p.Bslab) + (size_t)i * 16, 16);
            cp_async_wait_all();
            fence_proxy_async_smem();
            mbar_arrive(b_full);
        }
        const int halo_px = p.PH * p.PW;
        const int Cx = chunks * 8;
        int it = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int sb = it & 1;
            const uint32_t par = (it >> 1) & 1;
            const int n = t / p.tiles_y;
            const int oy0 = (t - n * p.tiles_y) * p.THt;
            mbar_wait(&slab_empty[sb], par ^ 1);
            const uint32_t a0 = smem_u32(sA + sb * a_buf);
            const __nv_bfloat16* Xn = p.X + (size_t)n * p.H * p.W * Cx;
            for (int pl = 0; pl < ((p.skip & 1) ? 0 : p.num_planes); ++pl) {
                const int ys = p.pl_ys[pl], xs = p.pl_xs[pl], yo = p.pl_yoff[pl], xo = p.pl_xoff[pl];
                const uint32_t pbase = a0 + pl * chunks * slab;
                // item i = row * chunks + j; HC_PRODUCERS is a multiple of chunks, so j is fixed per thread and the halo
                // pixel advances by a constant number of rows per iteration (no division in the loop)
                const int j = ptid % chunks;
                const int row_step = HC_PRODUCERS / chunks;
                int row = ptid / chunks;
                int sy = row / p.PW, sx = row - sy * p.PW;
                const uint32_t dst0 = pbase + j * slab;
                for (; row < halo_px; row += row_step) {
                    const int iy = (oy0 + sy) * ys + yo, ix = sx * xs + xo;
                    const bool ok = iy >= 0 && iy < p.H && ix >= 0 && ix < p.W;
                    const __nv_bfloat16* src = ok ? Xn + ((size_t)iy * p.W + ix) * Cx + j * 8 : Xn;
                    cp_async16(dst0 + row * 16, src, ok ? 16u : 0u);
                    sx += row_step;
                    while (sx >= p.PW) { sx -= p.PW; ++sy; }
                }
            }
            cp_async_wait_all();
            fence_proxy_async_smem();
            mbar_arrive(&slab_full[sb]);
        }
    } else {
        // ======================================================== epilogue
        // The epilogue is a latency chain per warp (TMEM load -> convert -> store); a probe with the other roles switched off
        // (FMRI_HC_SKIP=7) left hconv_kernel<32> at 80 % of its time. So: two warps per TMEM lane quarter alternate the
        // sub-tiles (at <= 56 registers, so that two CTAs still share an SM), and the bias comes from shared memory.
        const int q = warp & 3;
        const int egrp = (warp - (HC_ISSUERS + HC_PRODUCERS / 32)) >> 2;   // 0 / 1: which of the quarter's two warps
        int it = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
            const int sb = it & 1;
            const uint32_t par = (it >> 1) & 1;
            const int n = t / p.tiles_y;
            const int oy0 = (t - n * p.tiles_y) * p.THt;
            mbar_wait(&tmem_full[sb], par);
            tc_fence_after();
            for (int m = egrp; m < p.MT; m += HC_EPI_WARPS / 4) {
                const int r = m * 128 + q * 32 + lane;
                const int yy = r / p.PW, xx = r - yy * p.PW;
                const bool valid = yy < p.THt && (oy0 + yy) < p.OH && xx < p.OW && !(p.skip & 2);
                const uint32_t tad = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + sb * acc_cols + m * BN;
                if (p.epi == 0) {
                    uint32_t v[16];
                    tmem_ld16(tad, v);
                    tmem_ld_wait();
                    if (valid) {
                        float* o = reinterpret_cast<float*>(p.out) + (((size_t)n * p.n_out) * p.OH + (oy0 + yy)) * p.OW + xx;
                        const size_t cs = (size_t)p.OH * p.OW;
#pragma unroll
                        for (int c = 0; c < 16; ++c) {
                            if (c < p.n_out) {
                                const float f = __uint_as_float(v[c]) + (p.bias ? __ldg(p.bias + c) : 0.f);
                                o[c * cs] = hc_act(f, p.act);
                            }
                        }
                    }
                } else {
                    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) +
                                       (((size_t)n * p.OH + (oy0 + yy)) * p.OW + xx) * BN;
#pragma unroll 1
                    for (int c0 = 0; c0 < BN; c0 += 16) {
                        uint32_t v[16];
                        tmem_ld16(tad + c0, v);
                        tmem_ld_wait();
                        // the epilogue warps' instruction chain is what bounds this kernel: bias and activation are applied
                        // under warp-uniform branches, so the plain data-gradient use (no bias, no activation) pays for neither
                        float f[16];
#pragma unroll
                        for (int c = 0; c < 16; ++c) f[c] = __uint_as_float(v[c]);
                        if (p.bias) {
#pragma unroll
                            for (int c = 0; c < 16; ++c) f[c] += s_bias[c0 + c];
                        }
                        if (p.act == 1) {
#pragma unroll
                            for (int c = 0; c < 16; ++c) f[c] = fmaxf(f[c], 0.f);
                        } else if (p.act != 0) {
#pragma unroll
                            for (int c = 0; c < 16; ++c) f[c] = hc_act(f[c], p.act);
                        }
                        uint32_t pk[8];
#pragma unroll
                        for (int c = 0; c < 8; ++c) pk[c] = pack_bf16x2(f[2 * c], f[2 * c + 1]);
                        if (valid) {
                            *reinterpret_cast<uint4*>(o + c0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                            *reinterpret_cast<uint4*>(o + c0 + 8) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[sb]);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// weights -> slab layout [2 K-halves][num_steps*BN][8]. For step s, half h: tap index tap[s][h] (-1: zeros) and first
// channel cb[s][h]; element e of output channel n:  w[n*s_n + (cb+e)*s_c + tap] when n < n_real and cb+e < c_real.
struct HcPackSpec {
    int16_t tap[HC_MAX_STEPS][2];
    int16_t cb[HC_MAX_STEPS][2];
};
__global__ void hc_pack_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst,
                                       const __grid_constant__ HcPackSpec spec, int num_steps, int BN, int n_real,
                                       int c_real, long long s_n, long long s_c) {
    const int rows = num_steps * BN;
    const int total = 2 * rows * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7;
        const int rr = (i >> 3) % rows;
        const int h = (i >> 3) / rows;
        const int s = rr / BN, n = rr - s * BN;
        const int tap = spec.tap[s][h], c = spec.cb[s][h] + e;
        float v = 0.f;
        if (tap >= 0 && n < n_real && c < c_real) v = __ldg(w + n * s_n + c * s_c + tap);
        dst[i] = __float2bfloat16_rn(v);
    }
}

// 3-channel fp32 NCHW image(s) -> bf16 NHWC with the channels padded to 8 (one 16-byte slab entry per pixel); up to three
// sources are concatenated on the batch axis (the discriminator's torch.cat, vae_gan.py:165).
__global__ void img8_pack_kernel(const float* __restrict__ s0, const float* __restrict__ s1, const float* __restrict__ s2,
                                 int n_per_src, int N, long long HW, __nv_bfloat16* __restrict__ dst) {
    const long long total = (long long)N * HW;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i / HW);
        const long long px = i - (long long)n * HW;
        const int si = n / n_per_src;
        const float* img = (si == 0 ? s0 : (si == 1 ? s1 : s2)) + (long long)(n - si * n_per_src) * 3 * HW + px;
        const uint32_t a = pack_bf16x2(__ldg(img), __ldg(img + HW));
        const uint32_t b = pack_bf16x2(__ldg(img + 2 * HW), 0.f);
        *reinterpret_cast<uint4*>(dst + i * 8) = make_uint4(a, b, 0u, 0u);
    }
}

// One stride-parity plane of 3-channel fp32 NCHW image(s) as bf16 NHWC-8 on the [PH][PW] grid of a stride-2 convolution's
// output: dst[n][y][x][ci] = img[n][ci][2y + ph][2x + pw] (zero outside the image).
__global__ void img8_plane_pack_kernel(const float* __restrict__ s0, const float* __restrict__ s1, const float* __restrict__ s2,
                                       int n_per_src, int N, int IH, int IW, int PH, int PW, int ph, int pw,
                                       __nv_bfloat16* __restrict__ dst) {
    const long long total = (long long)N * PH * PW;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % PW);
        const int y = (int)((i / PW) % PH);
        const int n = (int)(i / ((long long)PW * PH));
        const int iy = 2 * y + ph, ix = 2 * x + pw;
        uint32_t a = 0u, b = 0u;
        if (iy < IH && ix < IW) {
            const int si = n / n_per_src;
            const float* img = (si == 0 ? s0 : (si == 1 ? s1 : s2)) + (long long)(n - si * n_per_src) * 3 * IH * IW +
                               (long long)iy * IW + ix;
            const long long HW = (long long)IH * IW;
            a = pack_bf16x2(__ldg(img), __ldg(img + HW));
            b = pack_bf16x2(__ldg(img + 2 * HW), 0.f);
        }
        *reinterpret_cast<uint4*>(dst + i * 8) = make_uint4(a, b, 0u, 0u);
    }
}

}  // namespace fmri
