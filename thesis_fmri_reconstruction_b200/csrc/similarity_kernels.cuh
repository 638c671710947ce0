// All-pairs similarity matrices and n-way identification (the exhaustive form of the reference's objective_assessment,
// /root/reference/train/train_utils.py:752): for pred [N, C, H, W] and target [M, C, H, W], fp32 NCHW,
//   P[i, j] = PearsonCorrelation()(pred[i:i+1], target[j:j+1])        (train_utils.py:267-293)
//   S[i, j] = StructuralSimilarity()(pred[i:i+1], target[j:j+1])      (train_utils.py:295-425)
// and, from a square matrix X, wins[i] = #{j != i : X[i, i] > X[i, j]} and the expected n-way accuracy
//   acc[n] = (1/N) sum_i C(wins[i], n-1) / C(N-1, n-1).
// CUDA-core fp32 throughout (the metrics are pinned at 1e-5; bf16 / tf32 operand rounding would not hold that), no
// atomics: every output element is written by one thread, after sums in a fixed order, so two calls give the same bits.
#pragma once
#include "eval_kernels.cuh"   // warp_sum_d, SsimWindow

namespace fmri {

// ---- per-image terms ---------------------------------------------------------------------------------------------------

// stats[img] = (mean, sqrt(sum (x - mean)^2)): the mean is rounded to fp32 (the value the GEMM subtracts) and the centred
// norm is taken over exactly the fp32 differences the GEMM multiplies. fp64 sums, thread-strided then a fixed tree.
constexpr int PCC_STAT_THREADS = 256;
__device__ __forceinline__ double block_sum_fixed(double v, double* red) {
    v = warp_sum_d(v);
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) red[w] = v;
    __syncthreads();
    double s = 0.0;
    for (int k = 0; k < PCC_STAT_THREADS / 32; ++k) s += red[k];
    __syncthreads();
    return s;
}
__global__ void __launch_bounds__(PCC_STAT_THREADS) pcc_stats_kernel(const float* __restrict__ x, long long K,
                                                                     double2* __restrict__ stats) {
    __shared__ double red[PCC_STAT_THREADS / 32];
    const float* p = x + (long long)blockIdx.x * K;
    double s = 0.0;
    for (long long k = threadIdx.x; k < K; k += PCC_STAT_THREADS) s += (double)__ldg(p + k);
    const float mean = (float)(block_sum_fixed(s, red) / (double)K);
    double q = 0.0;
    for (long long k = threadIdx.x; k < K; k += PCC_STAT_THREADS) {
        const double d = (double)(__ldg(p + k) - mean);
        q += d * d;
    }
    q = block_sum_fixed(q, red);
    if (threadIdx.x == 0) stats[blockIdx.x] = make_double2((double)mean, sqrt(q));
}

// SSIM maps of one image set: mu = G*x and sig = G*(x^2) - mu^2 per plane, written with a row pitch WP (a multiple of 8,
// zero beyond W) so that the pairwise kernel reads them as aligned float4. The window sum is taken in the separable order
// the pairwise kernel uses for G*(x y): 11 horizontal taps per row, then the 11 rows, each a sequential fp32 FMA chain
// (zero-padded taps add exact zeros), so for x = y the pairwise product term equals this G*(x^2) bit for bit.
__global__ void __launch_bounds__(256) ssim_maps_kernel(const float* __restrict__ x, long long planes, int H, int W, int WP,
                                                        const __grid_constant__ SsimWindow wd, float* __restrict__ mu,
                                                        float* __restrict__ sig) {
    const long long total = planes * H * WP;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % WP);
        const int y = (int)((i / WP) % H);
        const long long pl = i / ((long long)WP * H);
        if (c >= W) {
            mu[i] = 0.f;
            sig[i] = 0.f;
            continue;
        }
        const float* pp = x + pl * H * W;
        float m = 0.f, s = 0.f;
#pragma unroll
        for (int ky = 0; ky < 11; ++ky) {
            const int yy = y + ky - 5;
            float hm = 0.f, hs = 0.f;
            if (yy >= 0 && yy < H) {
#pragma unroll
                for (int kx = 0; kx < 11; ++kx) {
                    const int xx = c + kx - 5;
                    const float v = (xx >= 0 && xx < W) ? __ldg(pp + (long long)yy * W + xx) : 0.f;
                    hm = fmaf(wd.g[kx], v, hm);
                    hs = fmaf(wd.g[kx], v * v, hs);
                }
            }
            m = fmaf(wd.g[ky], hm, m);
            s = fmaf(wd.g[ky], hs, s);
        }
        mu[i] = m;
        sig[i] = s - m * m;
    }
}

// ---- pairwise PCC: P = (Xc Yc^T) / (|xc| |yc|), a tiled CUDA-core GEMM of the centred images ---------------------------
// CTA tile 128 pred x 64 target images, K in chunks of 32 staged in shared memory with each image's mean subtracted as it
// is loaded (rows and K beyond the matrix are zero). A thread owns 8 x 4 outputs: fp32 FMAs within a chunk, folded into
// fp64 accumulators after every chunk.
constexpr int PG_BM = 128, PG_BN = 64, PG_KC = 32, PG_THREADS = 256;
constexpr int PG_SA = PG_BM + 4, PG_SB = PG_BN + 4;   // row pitches: 16-byte aligned, spreads the transposed stores
__global__ void __launch_bounds__(PG_THREADS, 2) pcc_gemm_kernel(const float* __restrict__ a, int N,
                                                                 const float* __restrict__ b, int M, long long K,
                                                                 const double2* __restrict__ sa,
                                                                 const double2* __restrict__ sb, float* __restrict__ out) {
    __shared__ __align__(16) float As[PG_KC][PG_SA];
    __shared__ __align__(16) float Bs[PG_KC][PG_SB];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int i0 = blockIdx.x * PG_BM, j0 = blockIdx.y * PG_BN;
    // loader: lane = k within the chunk (a warp reads 128 contiguous bytes of one image), warp lr loads rows lr + 8q
    __shared__ float mean_a[PG_BM], mean_b[PG_BN];
    if (t < PG_BM) mean_a[t] = i0 + t < N ? (float)sa[i0 + t].x : 0.f;
    else if (t < PG_BM + PG_BN) mean_b[t - PG_BM] = j0 + t - PG_BM < M ? (float)sb[j0 + t - PG_BM].x : 0.f;
    const int lk = t & 31, lr = t >> 5;
    const long long K8 = 8 * K;
    const float* pa = a + (long long)(i0 + lr) * K + lk;
    const float* pb = b + (long long)(j0 + lr) * K + lk;
    double acc[8][4];
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = 0.0;
    __syncthreads();

    for (long long k0 = 0; k0 < K; k0 += PG_KC) {
        const bool kin = k0 + lk < K;
#pragma unroll
        for (int q = 0; q < PG_BM / 8; ++q) {
            const int r = lr + 8 * q;
            As[lk][r] = (kin && i0 + r < N) ? __ldg(pa + q * K8 + k0) - mean_a[r] : 0.f;
        }
#pragma unroll
        for (int q = 0; q < PG_BN / 8; ++q) {
            const int r = lr + 8 * q;
            Bs[lk][r] = (kin && j0 + r < M) ? __ldg(pb + q * K8 + k0) - mean_b[r] : 0.f;
        }
        __syncthreads();
        float f[8][4];
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) f[u][v] = 0.f;
#pragma unroll 8
        for (int kk = 0; kk < PG_KC; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[4] = {b0.x, b0.y, b0.z, b0.w};
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) f[u][v] = fmaf(av[u], bv[v], f[u][v]);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) acc[u][v] += (double)f[u][v];
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const int i = i0 + (u < 4 ? ty * 4 + u : 64 + ty * 4 + u - 4);
        if (i >= N) continue;
        const double na = sa[i].y;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int j = j0 + tx * 4 + v;
            if (j < M) out[(long long)i * M + j] = (float)(acc[u][v] / (na * sb[j].y));
        }
    }
}

// ---- pairwise SSIM ---------------------------------------------------------------------------------------------------
// S[i, j] = mean over C x H x W of ((2 mu_i mu_j + C1)(2 (G*(x_i y_j) - mu_i mu_j) + C2)) /
//                                    ((mu_i^2 + mu_j^2 + C1)(sig_i + sig_j + C2))
// with the mu / sig maps of ssim_maps_kernel. G*(x_i y_j) is the only per-pair convolution.
// A CTA owns SS_TI = 4 pred x SS_TJ = 8 target images: lane = (pred li = lane / 8, target lj = lane % 8), one pair per
// lane, and warp w owns output columns [cg + 8w, cg + 8w + 8) of a column group of at most 64 columns starting at cg
// (wider images are split into equal groups, each a multiple of 8 wide, walked one after the other). The CTA walks each
// plane top to bottom in bands of 11 input rows, staged with their 5-column halos in shared memory by cp.async, two
// bands in flight: the next band is copied in while this one is computed (pitch = 4 mod 32 words, so the 4 pred and
// the 8 target rows a warp reads with one float4 load sit in distinct banks). Per input row a
// thread loads the 18-wide neighbourhood of both images, forms the products and the 8 horizontal 11-tap sums, and keeps
// the last 11 rows of horizontal sums in registers (slot = row mod 11; the band loop is unrolled over the 11 slots, so
// every index is static); with row y' in, output row y' - 5 is complete. The map sum is fp32 within a band (at most
// 88 terms per thread) and fp64 across bands; warps are combined in warp order. No cross-CTA sum, no atomics.
constexpr int SS_TI = 4, SS_TJ = 8, SS_IMGS = SS_TI + SS_TJ, SS_R = 8, SS_BAND = 11, SS_MAXW = 8;
__host__ __device__ constexpr int ss_pitch(int cols) { return ((cols + 27) / 32) * 32 + 4; }   // >= cols, = 4 mod 32
struct SsimPairArgs {
    const float* a;          // pred [N, C, H, W]
    const float* b;          // target [M, C, H, W]
    const float* mu_a;       // [N, C, H, WP]
    const float* sig_a;
    const float* mu_b;       // [M, C, H, WP]
    const float* sig_b;
    int N, M, C, H, W, WP;
    int cols;                // columns of one column group (a multiple of 8, at most SS_MAXW * 8; blockDim = cols / 8 warps)
    int pitch;               // ss_pitch(cols + 10)
    double inv_count;        // 1 / (C H W)
    SsimWindow wd;
    float* out;              // [N, M]
};

// 4-byte asynchronous copy global -> shared; bytes = 0 writes a zero without reading `src`
__device__ __forceinline__ void cp_async4(float* dst, const float* src, int bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_prev() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

__global__ void __launch_bounds__(SS_MAXW * 32) ssim_pair_kernel(const __grid_constant__ SsimPairArgs p) {
    // two band buffers [SS_BAND rows][SS_IMGS][pitch] (band k + 1 is copied in while band k is computed); at the end,
    // [warps][32] doubles
    extern __shared__ __align__(16) float ss_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int li = lane >> 3, lj = lane & 7;
    const int i0 = blockIdx.x * SS_TI, j0 = blockIdx.y * SS_TJ;
    const int ia = min(i0 + li, p.N - 1), jb = min(j0 + lj, p.M - 1);   // clamped: ragged lanes compute, never store
    const int H = p.H, W = p.W, WP = p.WP, pitch = p.pitch;
    const long long HW = (long long)H * W, HWP = (long long)H * WP;
    const int buf_floats = SS_BAND * SS_IMGS * pitch, span = p.cols + 10;
    const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
    double total = 0.0;

    for (int c = 0; c < p.C; ++c) {
        for (int cg = 0; cg < W; cg += p.cols) {
            // input rows yb .. yb + 10 of the 12 images, columns cg - 5 .. cg + cols + 4 (zero outside): one warp per
            // (row, image) line, lanes along the columns
            auto stage = [&](int yb, float* buf) {
                for (int line = warp; line < SS_BAND * SS_IMGS; line += nw) {
                    const int r = line / SS_IMGS, img = line - r * SS_IMGS, y = yb + r;
                    const int n = img < SS_TI ? i0 + img : j0 + img - SS_TI;
                    const bool ok = y < H && n < (img < SS_TI ? p.N : p.M);
                    const float* src = ok ? (img < SS_TI ? p.a : p.b) + ((long long)n * p.C + c) * HW + (long long)y * W
                                          : p.a;
                    for (int col = lane; col < span; col += 32) {
                        const int xx = cg + col - 5;
                        const bool in = ok && xx >= 0 && xx < W;
                        cp_async4(buf + line * pitch + col, in ? src + xx : p.a, in ? 4 : 0);
                    }
                }
                cp_async_commit();
            };
            const int x0 = cg + warp * SS_R;                 // this thread's first output column
            const bool active = x0 < W;
            float ring[SS_BAND][SS_R];
#pragma unroll
            for (int s = 0; s < SS_BAND; ++s)
#pragma unroll
                for (int r = 0; r < SS_R; ++r) ring[s][r] = 0.f;
            const float* mua = p.mu_a + ((long long)ia * p.C + c) * HWP;
            const float* sga = p.sig_a + ((long long)ia * p.C + c) * HWP;
            const float* mub = p.mu_b + ((long long)jb * p.C + c) * HWP;
            const float* sgb = p.sig_b + ((long long)jb * p.C + c) * HWP;
            stage(0, ss_smem);
            for (int yb = 0, bi = 0; yb < H + 5; yb += SS_BAND, bi ^= 1) {
                const float* cur = ss_smem + bi * buf_floats;
                if (yb + SS_BAND < H + 5) stage(yb + SS_BAND, ss_smem + (bi ^ 1) * buf_floats);
                else cp_async_commit();                      // an empty group keeps "all but the newest" meaning this band
                cp_async_wait_prev();
                __syncthreads();
                if (active) {
                    float band = 0.f;
#pragma unroll
                    for (int s = 0; s < SS_BAND; ++s) {
                        const int yin = yb + s;
                        if (yin < H) {   // rows at and beyond H are zero padding: their horizontal sums stay zero
                            const float* ra = cur + (s * SS_IMGS + li) * pitch + warp * SS_R;
                            const float* rb = cur + (s * SS_IMGS + SS_TI + lj) * pitch + warp * SS_R;
                            float pr[SS_R + 10];
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float4 u = *reinterpret_cast<const float4*>(ra + 4 * q);
                                const float4 v = *reinterpret_cast<const float4*>(rb + 4 * q);
                                pr[4 * q] = u.x * v.x; pr[4 * q + 1] = u.y * v.y;
                                pr[4 * q + 2] = u.z * v.z; pr[4 * q + 3] = u.w * v.w;
                            }
                            {
                                const float2 u = *reinterpret_cast<const float2*>(ra + 16);
                                const float2 v = *reinterpret_cast<const float2*>(rb + 16);
                                pr[16] = u.x * v.x; pr[17] = u.y * v.y;
                            }
#pragma unroll
                            for (int r = 0; r < SS_R; ++r) {
                                float h = 0.f;
#pragma unroll
                                for (int k = 0; k < 11; ++k) h = fmaf(p.wd.g[k], pr[r + k], h);
                                ring[s][r] = h;
                            }
                        } else {
#pragma unroll
                            for (int r = 0; r < SS_R; ++r) ring[s][r] = 0.f;
                        }
                        const int y = yin - 5;
                        if (y >= 0 && y < H) {
#pragma unroll
                            for (int q = 0; q < SS_R / 4; ++q) {   // 4 columns at a time: the map values live briefly
                                const long long o = (long long)y * WP + x0 + 4 * q;
                                float ma[4], mb[4], va[4], vb[4];
                                *reinterpret_cast<float4*>(ma) = __ldg(reinterpret_cast<const float4*>(mua + o));
                                *reinterpret_cast<float4*>(mb) = __ldg(reinterpret_cast<const float4*>(mub + o));
                                *reinterpret_cast<float4*>(va) = __ldg(reinterpret_cast<const float4*>(sga + o));
                                *reinterpret_cast<float4*>(vb) = __ldg(reinterpret_cast<const float4*>(sgb + o));
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const int r = 4 * q + e;
                                    float g12 = 0.f;
#pragma unroll
                                    for (int k = 0; k < 11; ++k) g12 = fmaf(p.wd.g[k], ring[(s + 1 + k) % SS_BAND][r], g12);
                                    const float m12 = ma[e] * mb[e];
                                    const float num = (2.f * m12 + C1) * (2.f * (g12 - m12) + C2);
                                    const float den = (ma[e] * ma[e] + mb[e] * mb[e] + C1) * (va[e] + vb[e] + C2);
                                    if (x0 + r < W) band += __fdividef(num, den);
                                }
                            }
                        }
                    }
                    total += (double)band;
                }
                __syncthreads();             // the buffer of this band is the target of the next stage()
            }
        }
    }
    // combine the warps in warp order (one thread per pair writes S[i, j])
    double* red = reinterpret_cast<double*>(ss_smem);
    __syncthreads();
    red[warp * 32 + lane] = total;
    __syncthreads();
    if (warp == 0) {
        double s = 0.0;
        for (int w = 0; w < nw; ++w) s += red[w * 32 + lane];
        const int i = i0 + li, j = j0 + lj;
        if (i < p.N && j < p.M) p.out[(long long)i * p.M + j] = (float)(s * p.inv_count);
    }
}

// ---- identification --------------------------------------------------------------------------------------------------
// wins[i] = #{j != i : X[i, i] > X[i, j]}, one warp per row (a NaN on either side never wins, as with Python's >).
__global__ void __launch_bounds__(256) ident_wins_kernel(const float* __restrict__ X, int N, int* __restrict__ wins) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= N) return;
    const float* r = X + (long long)row * N;
    const float d = r[row];
    int n = 0;
    for (int j = lane; j < N; j += 32) n += (j != row && d > r[j]) ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if (lane == 0) wins[row] = n;
}

// acc[q] = (1/N) sum_i prod_{m < n-1} (wins[i] - m) / (N - 1 - m), n = ns[q]: the probability that row i's own target
// beats n-1 distractors drawn without replacement, averaged over rows. One CTA; rows are thread-strided and the partials
// summed in a fixed tree, all in fp64.
constexpr int IDENT_MAX_NS = 64;
struct IdentNs { int n[IDENT_MAX_NS]; int count; };
__global__ void __launch_bounds__(256) ident_acc_kernel(const int* __restrict__ wins, int N, const __grid_constant__ IdentNs ns,
                                                        double* __restrict__ acc) {
    __shared__ double red[256];
    for (int q = 0; q < ns.count; ++q) {
        const int n1 = ns.n[q] - 1;
        double s = 0.0;
        for (int i = threadIdx.x; i < N; i += 256) {
            const int w = wins[i];
            if (w < n1) continue;
            double pr = 1.0;
            for (int m = 0; m < n1 && pr != 0.0; ++m) pr *= (double)(w - m) / (double)(N - 1 - m);
            s += pr;
        }
        red[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) acc[q] = red[0] / (double)N;
        __syncthreads();
    }
}

}  // namespace fmri
