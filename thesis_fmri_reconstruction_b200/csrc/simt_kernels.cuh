// CUDA-core kernels: the HBM-bound part of the training step (BatchNorm, losses, optimizers, layout/dtype
// packers), the 3-channel edge convolutions, and a generic direct convolution used for the fp32-exact mode
// and for shapes the tensor path does not tile.
#pragma once
#include "ptx.cuh"

namespace fmri {

template <typename T>
__device__ __forceinline__ float ld_f(const T* p);
template <>
__device__ __forceinline__ float ld_f<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ld_f<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T>
__device__ __forceinline__ void st_f(T* p, float v);
template <>
__device__ __forceinline__ void st_f<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void st_f<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == 1) return fmaxf(v, 0.f);
    if (act == 2) return tanhf(v);
    if (act == 3) return 1.f / (1.f + __expf(-v));
    return v;
}

// ------------------------------------------------------------------------------------------------
// Generic 5x5 direct convolution, gather form. Tensors are addressed through element strides so the same
// kernel reads/writes NHWC (internal) and NCHW (module boundary) tensors.
//   transposed == 0 : out[n,oy,ox,co] = sum in[n, oy*s+kh-2, ox*s+kw-2, ci] * w[co*w_so + ci*w_si + kh*5+kw]
//   transposed == 1 : out[n,oy,ox,co] = sum over (kh,kw) with (oy+2-kh) % s == 0 of in[n,(oy+2-kh)/s,..,ci] * w[..]
// (the second form is both ConvTranspose2d forward and Conv2d data-gradient).
// ------------------------------------------------------------------------------------------------
struct DirectConvParams {
    int N, H, W, Cin;       // input
    int OH, OW, Cout;       // output
    int stride, transposed;
    long long in_sn, in_sy, in_sx, in_sc;
    long long out_sn, out_sy, out_sx, out_sc;
    long long w_so, w_si;   // weight element strides for (output channel, input channel); taps are contiguous
    int flip;               // use tap (4-kh, 4-kw) instead of (kh, kw)
    int act;
    int accumulate;         // out += result (fp32 out only)
};

template <typename Tin, typename Tout>
__global__ void direct_conv_kernel(const Tin* __restrict__ in, const float* __restrict__ w,
                                   const float* __restrict__ bias, Tout* __restrict__ out, DirectConvParams p) {
    const long long total = (long long)p.N * p.OH * p.OW * p.Cout;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int co = (int)(idx % p.Cout);
        long long r = idx / p.Cout;
        const int ox = (int)(r % p.OW);
        r /= p.OW;
        const int oy = (int)(r % p.OH);
        const int n = (int)(r / p.OH);
        float acc = bias ? __ldg(bias + co) : 0.f;
        for (int kh = 0; kh < 5; ++kh) {
            int iy;
            if (!p.transposed) {
                iy = oy * p.stride + kh - 2;
            } else {
                const int t = oy + 2 - kh;
                if (t < 0 || (t % p.stride) != 0) continue;
                iy = t / p.stride;
            }
            if (iy < 0 || iy >= p.H) continue;
            for (int kw = 0; kw < 5; ++kw) {
                int ix;
                if (!p.transposed) {
                    ix = ox * p.stride + kw - 2;
                } else {
                    const int t = ox + 2 - kw;
                    if (t < 0 || (t % p.stride) != 0) continue;
                    ix = t / p.stride;
                }
                if (ix < 0 || ix >= p.W) continue;
                const int tap = p.flip ? (4 - kh) * 5 + (4 - kw) : kh * 5 + kw;
                const Tin* ip = in + n * p.in_sn + iy * p.in_sy + ix * p.in_sx;
                const float* wp = w + co * p.w_so + tap;
                for (int ci = 0; ci < p.Cin; ++ci) acc += ld_f(ip + ci * p.in_sc) * __ldg(wp + ci * p.w_si);
            }
        }
        acc = apply_act(acc, p.act);
        Tout* o = out + n * p.out_sn + oy * p.out_sy + ox * p.out_sx + co * p.out_sc;
        st_f(o, acc);
    }
}

// Generic weight gradient: dw[a*w_sa + b*w_sb + tap] (+)= sum_{n,py,px} A[n,py,px,a] * B[n, py*s+kh-2, px*s+kw-2, b]
// A is the tensor on the strided-output side of the convolution, B the one on its input side.
struct DirectWgradParams {
    int N, PH, PW, Ca;   // A grid
    int BH, BW, Cb;      // B grid
    int stride;
    long long a_sn, a_sy, a_sx, a_sc;
    long long b_sn, b_sy, b_sx, b_sc;
    long long w_sa, w_sb;
    int accumulate;
};

template <typename Ta, typename Tb>
__global__ void direct_wgrad_kernel(const Ta* __restrict__ A, const Tb* __restrict__ B, float* __restrict__ dw,
                                    DirectWgradParams p) {
    // one block per (a, b, tap) triple; threads stride over pixels
    const int tap = blockIdx.x % 25;
    const int ab = blockIdx.x / 25;
    const int b = ab % p.Cb;
    const int a = ab / p.Cb;
    const int kh = tap / 5, kw = tap % 5;
    const long long pixels = (long long)p.N * p.PH * p.PW;
    float acc = 0.f;
    for (long long i = threadIdx.x; i < pixels; i += blockDim.x) {
        const int px = (int)(i % p.PW);
        const long long r = i / p.PW;
        const int py = (int)(r % p.PH);
        const int n = (int)(r / p.PH);
        const int by = py * p.stride + kh - 2, bx = px * p.stride + kw - 2;
        if (by < 0 || by >= p.BH || bx < 0 || bx >= p.BW) continue;
        acc += ld_f(A + n * p.a_sn + py * p.a_sy + px * p.a_sx + a * p.a_sc) *
               ld_f(B + n * p.b_sn + by * p.b_sy + bx * p.b_sx + b * p.b_sc);
    }
    __shared__ float red[32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) {
            float* o = dw + a * p.w_sa + b * p.w_sb + tap;
            *o = p.accumulate ? *o + v : v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Edge convolutions with a 3-channel side (image side, NCHW fp32) and a C-channel side (NHWC, C = 32/64).
// ------------------------------------------------------------------------------------------------
// (A) img3 -> C channels. out[n,oy,ox,c] = act(bias[c] + sum_{ci<3,kh,kw} img[n,ci,oy*s+kh-2,ox*s+kw-2] * wk[(ci*25+tap)*C + c])
//     `wk` is a [75][C] fp32 pack staged in shared memory. Up to three source images are concatenated on
//     the batch axis (the discriminator's torch.cat, vae_gan.py:165) without materialising the cat.
template <int C, typename Tout>
__global__ void __launch_bounds__(128) edge3_to_c_kernel(const float* __restrict__ src0, const float* __restrict__ src1,
                                                         const float* __restrict__ src2, int n_per_src,
                                                         const float* __restrict__ wk, const float* __restrict__ bias,
                                                         Tout* __restrict__ out, int N, int H, int W, int OH, int OW,
                                                         int stride, int act) {
    __shared__ float sw[75 * C];
    for (int i = threadIdx.x; i < 75 * C; i += blockDim.x) sw[i] = wk[i];
    __syncthreads();
    const long long pix = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (pix >= (long long)N * OH * OW) return;
    const int ox = (int)(pix % OW);
    const int oy = (int)((pix / OW) % OH);
    const int n = (int)(pix / ((long long)OW * OH));
    const int s = n / n_per_src;
    const float* img = (s == 0 ? src0 : (s == 1 ? src1 : src2)) + (long long)(n - s * n_per_src) * 3 * H * W;
    float acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = bias ? __ldg(bias + c) : 0.f;
    for (int ci = 0; ci < 3; ++ci) {
#pragma unroll
        for (int kh = 0; kh < 5; ++kh) {
            const int iy = oy * stride + kh - 2;
            if (iy < 0 || iy >= H) continue;
#pragma unroll
            for (int kw = 0; kw < 5; ++kw) {
                const int ix = ox * stride + kw - 2;
                if (ix < 0 || ix >= W) continue;
                const float v = __ldg(img + ((long long)ci * H + iy) * W + ix);
                const float4* wr = reinterpret_cast<const float4*>(sw + (ci * 25 + kh * 5 + kw) * C);
#pragma unroll
                for (int c4 = 0; c4 < C / 4; ++c4) {
                    const float4 wv = wr[c4];
                    acc[4 * c4 + 0] += v * wv.x;
                    acc[4 * c4 + 1] += v * wv.y;
                    acc[4 * c4 + 2] += v * wv.z;
                    acc[4 * c4 + 3] += v * wv.w;
                }
            }
        }
    }
    Tout* o = out + pix * C;
    if constexpr (sizeof(Tout) == 2) {
#pragma unroll
        for (int c8 = 0; c8 < C / 8; ++c8) {
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                pk[j] = pack_bf16x2(apply_act(acc[8 * c8 + 2 * j], act), apply_act(acc[8 * c8 + 2 * j + 1], act));
            *reinterpret_cast<uint4*>(o + 8 * c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) st_f(o + c, apply_act(acc[c], act));
    }
}

// (B) C channels -> img3. img[n,co,y,x] = act(bias[co] + sum_{c,taps} in[n, (y,x)@tap, c] * wk[(co*25+tap)*C + c])
//     gather over the C-channel NHWC tensor. `up`: the C-side grid is the stride-s *output* of the forward conv
//     (data gradient of a strided 3->C conv): in pixel = (y+2-kh)/s when divisible.
template <int C, typename Tin>
__global__ void __launch_bounds__(128) edgec_to_3_kernel(const Tin* __restrict__ in, const float* __restrict__ wk,
                                                         const float* __restrict__ bias, float* __restrict__ img,
                                                         int N, int IH, int IW, int OH, int OW, int stride_up,
                                                         int flip, int act, int accumulate) {
    __shared__ float sw[75 * C];
    for (int i = threadIdx.x; i < 75 * C; i += blockDim.x) sw[i] = wk[i];
    __syncthreads();
    const long long pix = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (pix >= (long long)N * OH * OW) return;
    const int ox = (int)(pix % OW);
    const int oy = (int)((pix / OW) % OH);
    const int n = (int)(pix / ((long long)OW * OH));
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    for (int kh = 0; kh < 5; ++kh) {
        int iy;
        if (stride_up == 1) {
            iy = oy + kh - 2;
        } else {
            const int t = oy + 2 - kh;
            if (t < 0 || (t % stride_up)) continue;
            iy = t / stride_up;
        }
        if (iy < 0 || iy >= IH) continue;
        for (int kw = 0; kw < 5; ++kw) {
            int ix;
            if (stride_up == 1) {
                ix = ox + kw - 2;
            } else {
                const int t = ox + 2 - kw;
                if (t < 0 || (t % stride_up)) continue;
                ix = t / stride_up;
            }
            if (ix < 0 || ix >= IW) continue;
            const int tap = flip ? (4 - kh) * 5 + (4 - kw) : kh * 5 + kw;
            const Tin* ip = in + (((long long)n * IH + iy) * IW + ix) * C;
            const float* w0 = sw + (0 * 25 + tap) * C;
            const float* w1 = sw + (1 * 25 + tap) * C;
            const float* w2 = sw + (2 * 25 + tap) * C;
            if constexpr (sizeof(Tin) == 2) {
#pragma unroll
                for (int c8 = 0; c8 < C / 8; ++c8) {
                    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(ip + 8 * c8));
                    const uint32_t rr[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float lo = __uint_as_float(rr[j] << 16), hi = __uint_as_float(rr[j] & 0xffff0000u);
                        const int c = 8 * c8 + 2 * j;
                        a0 += lo * w0[c] + hi * w0[c + 1];
                        a1 += lo * w1[c] + hi * w1[c + 1];
                        a2 += lo * w2[c] + hi * w2[c + 1];
                    }
                }
            } else {
#pragma unroll 8
                for (int c = 0; c < C; ++c) {
                    const float v = ld_f(ip + c);
                    a0 += v * w0[c];
                    a1 += v * w1[c];
                    a2 += v * w2[c];
                }
            }
        }
    }
    if (bias) {
        a0 += __ldg(bias + 0);
        a1 += __ldg(bias + 1);
        a2 += __ldg(bias + 2);
    }
    float* o = img + ((long long)n * 3) * OH * OW + (long long)oy * OW + ox;
    const long long cs = (long long)OH * OW;
    if (accumulate) {
        o[0] += apply_act(a0, act);
        o[cs] += apply_act(a1, act);
        o[2 * cs] += apply_act(a2, act);
    } else {
        o[0] = apply_act(a0, act);
        o[cs] = apply_act(a1, act);
        o[2 * cs] = apply_act(a2, act);
    }
}

// (W) weight gradient with a 3-channel image side: dwk[(c3*25+tap)*C + c] += sum_{n,py,px} T[n,py,px,c] * img[n,c3,py*s+sg*(kh-2),..]
//     T: C-channel NHWC tensor on grid (PH,PW); img: NCHW fp32 on grid (IH,IW). sg = +1 when T is the conv output
//     (3->C conv: img is the input), sg = -1 with s=1 when T is the conv input (C->3 conv: img is dY).
//     grid: blocks stride over pixel chunks; each block reduces into registers then atomics into dwk (fp32 [75][C]).
template <int C, typename Tt>
__global__ void __launch_bounds__(256) edge_wgrad_kernel(const Tt* __restrict__ T, const float* __restrict__ src0,
                                                         const float* __restrict__ src1,
                                                         const float* __restrict__ src2, int n_per_src,
                                                         float* __restrict__ dwk, int N, int PH, int PW, int IH,
                                                         int IW, int stride, int sg, int pix_per_block) {
    // thread -> (channel c, tap-group g); 256 threads = C channels x (256/C) groups
    constexpr int G = 256 / C;
    constexpr int TPG = (75 + G - 1) / G;  // (c3,tap) pairs per group
    const int c = threadIdx.x % C;
    const int g = threadIdx.x / C;
    float acc[TPG];
#pragma unroll
    for (int i = 0; i < TPG; ++i) acc[i] = 0.f;
    __shared__ float patch[8][75];  // 8 pixels staged per iteration
    const long long pixels = (long long)N * PH * PW;
    const long long p_begin = (long long)blockIdx.x * pix_per_block;
    const long long p_end = min(pixels, p_begin + pix_per_block);
    for (long long p0 = p_begin; p0 < p_end; p0 += 8) {
        __syncthreads();
        for (int i = threadIdx.x; i < 8 * 75; i += 256) {
            const int pi = i / 75, j = i % 75;
            const long long pp = p0 + pi;
            float v = 0.f;
            if (pp < p_end) {
                const int px = (int)(pp % PW);
                const int py = (int)((pp / PW) % PH);
                const int n = (int)(pp / ((long long)PW * PH));
                const int c3 = j / 25, tap = j % 25;
                const int iy = py * stride + sg * (tap / 5 - 2), ix = px * stride + sg * (tap % 5 - 2);
                if (iy >= 0 && iy < IH && ix >= 0 && ix < IW) {
                    const int s = n / n_per_src;
                    const float* img = (s == 0 ? src0 : (s == 1 ? src1 : src2)) +
                                       (long long)(n - s * n_per_src) * 3 * IH * IW;
                    v = __ldg(img + ((long long)c3 * IH + iy) * IW + ix);
                }
            }
            patch[pi][j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int pi = 0; pi < 8; ++pi) {
            const long long pp = p0 + pi;
            if (pp >= p_end) break;
            const float tv = ld_f(T + pp * C + c);
#pragma unroll
            for (int i = 0; i < TPG; ++i) {
                const int j = g * TPG + i;
                if (j < 75) acc[i] += tv * patch[pi][j];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < TPG; ++i) {
        const int j = g * TPG + i;
        if (j < 75) atomicAdd(dwk + j * C + c, acc[i]);
    }
}

// (W2) register-tiled version of (W) for T-grid rows of up to 128 pixels (every shape of the 64x64 and 100x100 configs).
//     One block walks `rows_per_block` consecutive (image, row) lines of the T grid. Per line it stages the 15 image
//     rows (3 channels x 5 kh) the line touches and the line of T (as fp32) in shared memory; thread (g, cq, half) owns
//     the 5 kw taps x 4 channels accumulators of patch row g = c3*5+kh for a contiguous half of the line, so the inner
//     loop is 1 LDS.128 (T) + 1..5 LDS.32 (sliding image window) for 20 FMAs. Partial sums go out as fp32 atomics.
//     Optionally also emits dbias[c] += sum_pixels T[pixel][c] (bias gradient of Discriminator.conv[0], vae_gan.py:145).
template <int C, typename Tt>
__global__ void __launch_bounds__(256) edge_wgrad_rows_kernel(const Tt* __restrict__ T, const float* __restrict__ src0,
                                                              const float* __restrict__ src1,
                                                              const float* __restrict__ src2, int n_per_src,
                                                              float* __restrict__ dwk, float* __restrict__ dbias, int N,
                                                              int PH, int PW, int IH, int IW, int stride, int sg,
                                                              int rows_per_block) {
    constexpr int CQ = C / 4;          // channel quads
    constexpr int TPS = 15 * CQ;       // threads per pixel set
    constexpr int PS = 256 / TPS;      // pixel sets (2 for C = 32, 1 for C = 64)
    constexpr int IWS = 144;           // staged image row pitch (>= (PW-1)*stride + 5)
    __shared__ float s_img[15][IWS];
    __shared__ __align__(16) float s_t[128 * C];
    const int tid = threadIdx.x;
    const int set = tid / TPS;
    const int r = tid - set * TPS;
    const int g = r / CQ, cq = r - g * CQ;
    const bool active = set < PS;
    float acc[5][4];
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float bsum[4] = {0.f, 0.f, 0.f, 0.f};
    const long long lines = (long long)N * PH;
    const long long l0 = (long long)blockIdx.x * rows_per_block;
    const long long l1 = min(lines, l0 + rows_per_block);
    const int span = (PW - 1) * stride + 5;  // staged columns: ix = -2 .. (PW-1)*stride + 2
    const int half = (PW + PS - 1) / PS;
    for (long long line = l0; line < l1; ++line) {
        const int n = (int)(line / PH), py = (int)(line - (long long)n * PH);
        const int sidx = n / n_per_src;
        const float* img = (sidx == 0 ? src0 : (sidx == 1 ? src1 : src2)) + (long long)(n - sidx * n_per_src) * 3 * IH * IW;
        __syncthreads();
        for (int i = tid; i < 15 * span; i += 256) {
            const int row = i / span, col = i - row * span;
            const int c3 = row / 5, kh = row - c3 * 5;
            const int iy = py * stride + sg * (kh - 2), ix = col - 2;
            float v = 0.f;
            if (iy >= 0 && iy < IH && ix >= 0 && ix < IW) v = __ldg(img + ((long long)c3 * IH + iy) * IW + ix);
            s_img[row][col] = v;
        }
        const Tt* trow = T + line * (long long)PW * C;
        for (int i = tid; i < PW * C; i += 256) s_t[i] = ld_f(trow + i);
        __syncthreads();
        if (active) {
            const int p0 = set * half, p1 = min(PW, p0 + half);
            const float* ir = s_img[g];
            if (stride == 1) {
                float w0 = ir[p0], w1 = ir[p0 + 1], w2 = ir[p0 + 2], w3 = ir[p0 + 3];
                for (int px = p0; px < p1; ++px) {
                    const float w4 = ir[px + 4];
                    const float4 t = *reinterpret_cast<const float4*>(s_t + px * C + cq * 4);
                    const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc[0][j] += w0 * tv[j];
                        acc[1][j] += w1 * tv[j];
                        acc[2][j] += w2 * tv[j];
                        acc[3][j] += w3 * tv[j];
                        acc[4][j] += w4 * tv[j];
                    }
                    if (g == 0) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) bsum[j] += tv[j];
                    }
                    w0 = w1; w1 = w2; w2 = w3; w3 = w4;
                }
            } else {
                for (int px = p0; px < p1; ++px) {
                    const float* w = ir + px * stride;
                    const float4 t = *reinterpret_cast<const float4*>(s_t + px * C + cq * 4);
                    const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                    for (int k = 0; k < 5; ++k) {
                        const float wv = w[k];
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[k][j] += wv * tv[j];
                    }
                    if (g == 0) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) bsum[j] += tv[j];
                    }
                }
            }
        }
    }
    if (!active) return;
    // staged column k' of the window corresponds to ix = px*stride - 2 + k' = px*stride + sg*(kw-2)  ->  kw = sg > 0 ? k' : 4 - k'
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const int kw = sg > 0 ? k : 4 - k;
        float* o = dwk + (size_t)(g * 5 + kw) * C + cq * 4;  // g = c3*5 + kh -> (c3*25 + kh*5 + kw)
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(o + j, acc[k][j]);
    }
    if (dbias && g == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(dbias + cq * 4 + j, bsum[j]);
    }
}

// ------------------------------------------------------------------------------------------------
// Simple fp32 SIMT GEMM family (exact mode and small shapes): C[M,N] (+)= A[M,K] * B[N,K]^T (+ bias, act)
// with arbitrary element strides so that the transposed products of dgrad / wgrad reuse it.
// ------------------------------------------------------------------------------------------------
template <typename Ta, typename Tb, typename Tc>
__global__ void __launch_bounds__(256) simt_gemm_kernel(const Ta* __restrict__ A, long long a_sm, long long a_sk,
                                                        const Tb* __restrict__ B, long long b_sn, long long b_sk,
                                                        Tc* __restrict__ Cm, long long c_sm, long long c_sn,
                                                        const float* __restrict__ bias, int M, int N, int K, int act,
                                                        int accumulate) {
    __shared__ float sa[16][65];
    __shared__ float sb[16][65];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += 16) {
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            int r, kk;
            // pick the loop order that keeps global reads contiguous
            if (a_sk == 1) { kk = i % 16; r = i / 16; } else { r = i % 64; kk = i / 64; }
            const int m = m0 + r, k = k0 + kk;
            sa[kk][r] = (m < M && k < K) ? ld_f(A + m * a_sm + k * a_sk) : 0.f;
        }
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            int r, kk;
            if (b_sk == 1) { kk = i % 16; r = i / 16; } else { r = i % 64; kk = i / 64; }
            const int n = n0 + r, k = k0 + kk;
            sb[kk][r] = (n < N && k < K) ? ld_f(B + n * b_sn + k * b_sk) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = sa[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) bv[j] = sb[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] += av[i] * bv[j];
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= N) continue;
            float v = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
            v = apply_act(v, act);
            Tc* o = Cm + m * c_sm + n * c_sn;
            if (accumulate) v += ld_f(o);
            st_f(o, v);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// BatchNorm (train mode) on a [rows, C] channels-last matrix (conv: rows = N*H*W; linear: rows = batch)
// ------------------------------------------------------------------------------------------------
// per-channel sum / sum of squares -> double accumulators (used when the producer kernel did not fuse them)
template <typename T>
__global__ void __launch_bounds__(256) colstats_kernel(const T* __restrict__ x, long long rows, int C,
                                                       double* __restrict__ sum, double* __restrict__ sq,
                                                       int rows_per_block) {
    // threads: 256 = cx columns x ry row-lanes, coalesced along C
    const int cx = C >= 256 ? 256 : C;  // C is a power of two multiple of 32 or anything <= 256
    const int ry = 256 / cx;
    const int tc = threadIdx.x % cx, tr = threadIdx.x / cx;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = min(rows, r0 + rows_per_block);
    extern __shared__ float sred[];  // [2][256]
    for (int cb = blockIdx.y * cx; cb < C; cb += gridDim.y * cx) {
        const int col = cb + tc;
        float s = 0.f, q = 0.f;
        if (col < C && tr < ry)
            for (long long r = r0 + tr; r < r1; r += ry) {
                const float v = ld_f(x + r * C + col);
                s += v;
                q += v * v;
            }
        sred[threadIdx.x] = s;
        sred[256 + threadIdx.x] = q;
        __syncthreads();
        if (tr == 0 && col < C) {
            for (int j = 1; j < ry; ++j) {
                s += sred[j * cx + tc];
                q += sred[256 + j * cx + tc];
            }
            atomicAdd(sum + col, (double)s);
            atomicAdd(sq + col, (double)q);
        }
        __syncthreads();
    }
}

// finalize: mean / invstd from the sums, running-stat update (momentum semantic of torch: r = (1-m) r + m * batch,
// unbiased variance for the running estimate), vae_gan.py:21 uses momentum=0.9.
__global__ void bn_finalize_kernel(const double* __restrict__ sum, const double* __restrict__ sq, double count, int C,
                                   float eps, float momentum, float* __restrict__ mean, float* __restrict__ invstd,
                                   float* __restrict__ running_mean, float* __restrict__ running_var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double m = sum[c] / count;
    double var = sq[c] / count - m * m;
    if (var < 0) var = 0;
    mean[c] = (float)m;
    invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) {
        const double unb = count > 1 ? var * count / (count - 1) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
    }
}

// y = relu(gamma * (x - mean) * invstd + beta); 8 elements per thread, channels-last, 128-bit loads/stores. The grid is
// sized so that the grid stride is a multiple of C whenever possible: each thread then sees the same 8 channels in every
// iteration and keeps their (mean, scale, beta) in registers instead of re-reading four per-channel arrays per element.
// Raw 8-element vectors (one or two 128-bit registers quads) so that the NEXT iteration's loads can be issued before the
// current iteration's arithmetic: the BN kernels carry ~50 registers of per-channel coefficients, which limits occupancy, so
// memory-level parallelism has to come from each thread keeping two iterations of loads in flight.
template <typename T> struct Raw8;
template <> struct Raw8<__nv_bfloat16> { uint4 a; };
template <> struct Raw8<float> { float4 a, b; };
__device__ __forceinline__ void raw_ld(const __nv_bfloat16* p, Raw8<__nv_bfloat16>& r) { r.a = *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void raw_ld(const float* p, Raw8<float>& r) {
    r.a = *reinterpret_cast<const float4*>(p);
    r.b = *reinterpret_cast<const float4*>(p + 4);
}
__device__ __forceinline__ void raw_cvt(const Raw8<__nv_bfloat16>& r, float (&v)[8]) {
    const uint32_t rr[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[2 * j] = __uint_as_float(rr[j] << 16);
        v[2 * j + 1] = __uint_as_float(rr[j] & 0xffff0000u);
    }
}
__device__ __forceinline__ void raw_cvt(const Raw8<float>& r, float (&v)[8]) {
    v[0] = r.a.x; v[1] = r.a.y; v[2] = r.a.z; v[3] = r.a.w; v[4] = r.b.x; v[5] = r.b.y; v[6] = r.b.z; v[7] = r.b.w;
}
template <typename T>
__device__ __forceinline__ void bn_ld8(const T* p, float (&v)[8]) {
    if constexpr (sizeof(T) == 2) {
        const uint4 raw = *reinterpret_cast<const uint4*>(p);
        const uint32_t rr[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[2 * j] = __uint_as_float(rr[j] << 16);
            v[2 * j + 1] = __uint_as_float(rr[j] & 0xffff0000u);
        }
    } else {
        const float4 a = *reinterpret_cast<const float4*>(p);
        const float4 b = *reinterpret_cast<const float4*>(p + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
}
template <typename Tin, typename Tout>
__global__ void __launch_bounds__(256) bn_apply_kernel(const Tin* __restrict__ x, Tout* __restrict__ y,
                                                       long long total, int C, const float* __restrict__ mean,
                                                       const float* __restrict__ invstd,
                                                       const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, int relu) {
    const long long step = (long long)gridDim.x * blockDim.x * 8;
    long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8;
    if (i >= total) return;
    const bool hoist = (step % C) == 0;
    float mu[8], sc[8], be[8];
    bool have = false;
    Raw8<Tin> cur, nxt;
    raw_ld(x + i, cur);
    for (; i < total; i += step) {
        if (i + step < total) raw_ld(x + i + step, nxt);  // next iteration's load in flight during this one's math
        if (!hoist || !have) {
            const int c0 = (int)(i % C);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                mu[j] = __ldg(mean + c0 + j);
                sc[j] = __ldg(gamma + c0 + j) * __ldg(invstd + c0 + j);
                be[j] = __ldg(beta + c0 + j);
            }
            have = true;
        }
        float v[8];
        raw_cvt(cur, v);
        cur = nxt;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float o = (v[j] - mu[j]) * sc[j] + be[j];
            v[j] = relu ? fmaxf(o, 0.f) : o;
        }
        if constexpr (sizeof(Tout) == 2) {
            *reinterpret_cast<uint4*>(y + i) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                          pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        } else {
            *reinterpret_cast<float4*>(y + i) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(y + i + 4) = make_float4(v[4], v[5], v[6], v[7]);
        }
    }
}

// backward pass 1: per channel sum(g) and sum(g * xhat), g = dy * (out > 0) where out = gamma*xhat+beta
template <typename Tx, typename Tg>
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const Tx* __restrict__ x, const Tg* __restrict__ dy,
                                                            long long rows, int C, const float* __restrict__ mean,
                                                            const float* __restrict__ invstd,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, int relu,
                                                            double* __restrict__ sum_g, double* __restrict__ sum_gx,
                                                            int rows_per_block) {
    const int cx = C >= 256 ? 256 : C;
    const int ry = 256 / cx;
    const int tc = threadIdx.x % cx, tr = threadIdx.x / cx;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = min(rows, r0 + rows_per_block);
    extern __shared__ float sred[];
    for (int cb = blockIdx.y * cx; cb < C; cb += gridDim.y * cx) {
        const int col = cb + tc;
        float s = 0.f, q = 0.f;
        if (col < C && tr < ry) {
            const float mu = mean[col], is = invstd[col], ga = gamma[col], be = beta[col];
            const float sc = ga * is;
            for (long long r = r0 + tr; r < r1; r += ry) {
                const float xc = ld_f(x + r * C + col) - mu;
                const float xh = xc * is;
                float g = ld_f(dy + r * C + col);
                if (relu && !(xc * sc + be > 0.f)) g = 0.f;  // same expression as bn_apply_kernel -> same mask
                s += g;
                q += g * xh;
            }
        }
        sred[threadIdx.x] = s;
        sred[256 + threadIdx.x] = q;
        __syncthreads();
        if (tr == 0 && col < C) {
            for (int j = 1; j < ry; ++j) {
                s += sred[j * cx + tc];
                q += sred[256 + j * cx + tc];
            }
            atomicAdd(sum_g + col, (double)s);
            atomicAdd(sum_gx + col, (double)q);
        }
        __syncthreads();
    }
}

// vectorised reductions over a channels-last [rows, C] matrix, C % 8 == 0: thread = 8 adjacent channels (one 128-bit load
// per row) x row lane; per-thread fp32 partial sums over its rows, shared-memory reduction over the row lanes, fp64 atomics.
//   MODE 0: per-channel sum(x), sum(x^2)                                            (BatchNorm batch statistics)
//   MODE 1: per-channel sum(g), sum(g*xhat), g = dy masked by the ReLU of the forward (BatchNorm backward, pass 1)
template <int MODE, typename Tx, typename Tg>
__global__ void __launch_bounds__(256) bn_reduce8_kernel(const Tx* __restrict__ x, const Tg* __restrict__ dy, long long rows,
                                                         int C, const float* __restrict__ mean,
                                                         const float* __restrict__ invstd,
                                                         const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, int relu,
                                                         double* __restrict__ out_a, double* __restrict__ out_b,
                                                         int rows_per_block) {
    const int c8 = C >> 3;                      // 8-channel groups per row
    const int cx = c8 >= 256 ? 256 : c8;        // groups handled side by side by one block
    const int ry = 256 / cx;                    // row lanes
    const int tc = threadIdx.x % cx, tr = threadIdx.x / cx;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = min(rows, r0 + rows_per_block);
    __shared__ float sred[2][8][256 + 1];
    for (int gb = blockIdx.y * cx; gb < c8; gb += gridDim.y * cx) {
        const int grp = gb + tc;
        float s[8], q[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
        if (grp < c8 && tr < ry) {
            const int c0 = grp * 8;
            float mu[8], is[8], sc[8], be[8];
            if (MODE == 1) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    mu[j] = mean[c0 + j]; is[j] = invstd[c0 + j]; sc[j] = gamma[c0 + j] * is[j]; be[j] = beta[c0 + j];
                }
            }
            Raw8<Tx> curx;
            Raw8<Tg> curg;
            long long r = r0 + tr;
            if (r < r1) {
                raw_ld(x + r * C + c0, curx);
                if (MODE == 1) raw_ld(dy + r * C + c0, curg);
            }
            for (; r < r1; r += ry) {
                float xv[8];
                raw_cvt(curx, xv);
                float gv[8];
                if (MODE == 1) raw_cvt(curg, gv);
                if (r + ry < r1) {  // next row's loads in flight during this row's math
                    raw_ld(x + (r + ry) * C + c0, curx);
                    if (MODE == 1) raw_ld(dy + (r + ry) * C + c0, curg);
                }
                if (MODE == 0) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) { s[j] += xv[j]; q[j] += xv[j] * xv[j]; }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float xc = xv[j] - mu[j];
                        float g = gv[j];
                        if (relu && !(xc * sc[j] + be[j] > 0.f)) g = 0.f;  // same expression as bn_apply_kernel -> same mask
                        s[j] += g;
                        q[j] += g * (xc * is[j]);
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { sred[0][j][threadIdx.x] = s[j]; sred[1][j][threadIdx.x] = q[j]; }
        __syncthreads();
        if (tr == 0 && grp < c8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float a = s[j], b = q[j];
                for (int l = 1; l < ry; ++l) { a += sred[0][j][l * cx + tc]; b += sred[1][j][l * cx + tc]; }
                atomicAdd(out_a + grp * 8 + j, (double)a);
                atomicAdd(out_b + grp * 8 + j, (double)b);
            }
        }
        __syncthreads();
    }
}

// backward pass 2: dx = gamma*invstd * (g - mean(g) - xhat*mean(g*xhat)). `train`=0 (eval-mode BN: statistics are
// constants): dx = gamma*invstd*g. 8 channels-last elements per thread (C % 8 == 0), 128-bit loads/stores; the
// per-channel means are taken once per channel in fp64 (sum/count) and rounded to fp32.
template <typename T>
__device__ __forceinline__ void ld8(const T* p, float (&v)[8]) {
    if constexpr (sizeof(T) == 2) {
        const uint4 raw = *reinterpret_cast<const uint4*>(p);
        const uint32_t rr[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[2 * j] = __uint_as_float(rr[j] << 16);
            v[2 * j + 1] = __uint_as_float(rr[j] & 0xffff0000u);
        }
    } else {
        const float4 a = *reinterpret_cast<const float4*>(p);
        const float4 b = *reinterpret_cast<const float4*>(p + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
}
template <typename T>
__device__ __forceinline__ void st8(T* p, const float (&v)[8]) {
    if constexpr (sizeof(T) == 2) {
        *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                  pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    } else {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
}
template <typename Tx, typename Tg>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const Tx* __restrict__ x, const Tg* __restrict__ dy,
                                                           Tg* __restrict__ dx, long long total, int C, double count,
                                                           const float* __restrict__ mean,
                                                           const float* __restrict__ invstd,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, int relu, int train,
                                                           const float* __restrict__ mean_g,
                                                           const float* __restrict__ mean_gx) {
    const long long step = (long long)gridDim.x * blockDim.x * 8;
    long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8;
    if (i >= total) return;
    // when step % C == 0 every iteration of this thread sees the same 8 channels: hoist the coefficients
    const bool hoist = (step % C) == 0;
    float mu[8], is[8], sc[8], be[8], mg[8], mgx[8];
    int c0 = -1;
    Raw8<Tx> curx;
    Raw8<Tg> curg;
    raw_ld(x + i, curx);
    raw_ld(dy + i, curg);
    for (; i < total; i += step) {
        const int cc = (int)(i % C);
        if (!hoist || c0 < 0) {
            c0 = cc;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = cc + j;
                mu[j] = mean[c]; is[j] = invstd[c]; sc[j] = gamma[c] * is[j]; be[j] = beta[c];
                mg[j] = train ? mean_g[c] : 0.f;
                mgx[j] = train ? mean_gx[c] : 0.f;
            }
        }
        float xv[8], gv[8], o[8];
        raw_cvt(curx, xv);
        raw_cvt(curg, gv);
        if (i + step < total) {  // next iteration's loads in flight during this one's math
            raw_ld(x + i + step, curx);
            raw_ld(dy + i + step, curg);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float xc = xv[j] - mu[j];
            float g = gv[j];
            if (relu && !(xc * sc[j] + be[j] > 0.f)) g = 0.f;
            o[j] = sc[j] * (g - mg[j] - (xc * is[j]) * mgx[j]);
        }
        st8(dx + i, o);
    }
}

// ---- "channel pair per thread" BatchNorm-backward kernels ---------------------------------------------------------------
// A thread owns TWO adjacent channels (one 4-byte bf16x2 / 8-byte float2 access per row) and walks rows with an unrolled
// stride, so it carries only 2 channels' coefficients (12 registers instead of 48) and keeps 8 independent row accesses in
// flight; a warp's access to one row is one contiguous 128 B (bf16) segment. The 8-channels-per-thread versions above are
// register-bound (84-87 registers, 3 CTAs/SM) and reach 3.7-4.1 TB/s; relu_bwd with the same traffic pattern reaches 6.2.
// raw(): the untouched 32- / 64-bit word (what stays in registers while loads are in flight), cvt(): the two floats
template <typename T> struct Pair;
template <> struct Pair<__nv_bfloat16> {
    using Raw = uint32_t;
    static __device__ __forceinline__ Raw raw(const __nv_bfloat16* p) { return *reinterpret_cast<const uint32_t*>(p); }
    static __device__ __forceinline__ float2 cvt(Raw r) { return make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); }
    static __device__ __forceinline__ float2 ld(const __nv_bfloat16* p) { return cvt(raw(p)); }
    static __device__ __forceinline__ void st(__nv_bfloat16* p, float a, float b) { *reinterpret_cast<uint32_t*>(p) = pack_bf16x2(a, b); }
};
template <> struct Pair<float> {
    using Raw = float2;
    static __device__ __forceinline__ Raw raw(const float* p) { return *reinterpret_cast<const float2*>(p); }
    static __device__ __forceinline__ float2 cvt(Raw r) { return r; }
    static __device__ __forceinline__ float2 ld(const float* p) { return raw(p); }
    static __device__ __forceinline__ void st(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
};

// MODE 1: sums sum(g), sum(g*xhat) per channel; MODE 2: dx = scale*(g - mean_g - xhat*mean_gx)
template <int MODE, typename Tx, typename Tg>
__global__ void __launch_bounds__(256, 4) bn_bwd_cp_kernel(const Tx* __restrict__ x, const Tg* __restrict__ dy, Tg* __restrict__ dx,
                                                        long long rows, int C, const float* __restrict__ mean,
                                                        const float* __restrict__ invstd,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        int relu, int train, const float* __restrict__ mean_g,
                                                        const float* __restrict__ mean_gx, double* __restrict__ sum_g,
                                                        double* __restrict__ sum_gx, int rows_per_block) {
    const int cp = C >> 1;                    // channel pairs per row
    const int tx_n = cp >= 256 ? 256 : cp;    // threads across one row
    const int ry = 256 / tx_n;                // rows handled side by side
    const int tx = threadIdx.x % tx_n, ty = threadIdx.x / tx_n;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = min(rows, r0 + rows_per_block);
    __shared__ float sred[4][256];
    for (int pb = blockIdx.y * tx_n; pb < cp; pb += gridDim.y * tx_n) {
        const int c = (pb + tx) * 2;
        const bool live = (pb + tx) < cp;
        float mu0 = 0, mu1 = 0, is0 = 0, is1 = 0, sc0 = 0, sc1 = 0, be0 = 0, be1 = 0, k10 = 0, k11 = 0, k20 = 0, k21 = 0;
        if (live) {
            mu0 = mean[c]; mu1 = mean[c + 1]; is0 = invstd[c]; is1 = invstd[c + 1];
            sc0 = gamma[c] * is0; sc1 = gamma[c + 1] * is1; be0 = beta[c]; be1 = beta[c + 1];
            if (MODE == 2 && train) {  // dx = sc*g - sc*mean_g - xc*(sc*is*mean_gx): two FMAs per element
                k10 = -sc0 * mean_g[c]; k11 = -sc1 * mean_g[c + 1];
                k20 = -sc0 * is0 * mean_gx[c]; k21 = -sc1 * is1 * mean_gx[c + 1];
            }
        }
        float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
        if (live) {
            long long r = r0 + ty;
            // software pipeline: the raw words of the NEXT 8 rows are in flight while the current 8 are processed (an ncu
            // capture showed the un-pipelined loop latency-bound: 95 % occupancy, 40 % issue utilisation, 4.4 TB/s)
            typename Pair<Tx>::Raw xr[8], xn[8];
            typename Pair<Tg>::Raw gr[8], gn[8];
            bool have = r + 7LL * ry < r1;
            if (have) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    xr[u] = Pair<Tx>::raw(x + (r + (long long)u * ry) * C + c);
                    gr[u] = Pair<Tg>::raw(dy + (r + (long long)u * ry) * C + c);
                }
            }
#pragma unroll 1
            while (have) {
                const long long rn = r + 8LL * ry;
                const bool more = rn + 7LL * ry < r1;
                if (more) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        xn[u] = Pair<Tx>::raw(x + (rn + (long long)u * ry) * C + c);
                        gn[u] = Pair<Tg>::raw(dy + (rn + (long long)u * ry) * C + c);
                    }
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float2 xv = Pair<Tx>::cvt(xr[u]), gv = Pair<Tg>::cvt(gr[u]);
                    const float xc0 = xv.x - mu0, xc1 = xv.y - mu1;
                    float g0 = gv.x, g1 = gv.y;
                    if (relu && !(xc0 * sc0 + be0 > 0.f)) g0 = 0.f;
                    if (relu && !(xc1 * sc1 + be1 > 0.f)) g1 = 0.f;
                    if (MODE == 1) {  // q accumulates g*xc; the invstd factor is applied once at the end
                        s0 += g0; s1 += g1; q0 = fmaf(g0, xc0, q0); q1 = fmaf(g1, xc1, q1);
                    } else {
                        Pair<Tg>::st(dx + (r + (long long)u * ry) * C + c, fmaf(g0, sc0, fmaf(xc0, k20, k10)),
                                     fmaf(g1, sc1, fmaf(xc1, k21, k11)));
                    }
                }
                r = rn;
                have = more;
                if (more) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        xr[u] = xn[u];
                        gr[u] = gn[u];
                    }
                }
            }
            for (; r < r1; r += ry) {
                const float2 xv = Pair<Tx>::ld(x + r * C + c), gv = Pair<Tg>::ld(dy + r * C + c);
                const float xc0 = xv.x - mu0, xc1 = xv.y - mu1;
                float g0 = gv.x, g1 = gv.y;
                if (relu && !(xc0 * sc0 + be0 > 0.f)) g0 = 0.f;
                if (relu && !(xc1 * sc1 + be1 > 0.f)) g1 = 0.f;
                if (MODE == 1) {
                    s0 += g0; s1 += g1; q0 = fmaf(g0, xc0, q0); q1 = fmaf(g1, xc1, q1);
                } else {
                    Pair<Tg>::st(dx + r * C + c, fmaf(g0, sc0, fmaf(xc0, k20, k10)), fmaf(g1, sc1, fmaf(xc1, k21, k11)));
                }
            }
        }
        if (MODE == 1) {
            q0 *= is0; q1 *= is1;
            sred[0][threadIdx.x] = s0; sred[1][threadIdx.x] = s1; sred[2][threadIdx.x] = q0; sred[3][threadIdx.x] = q1;
            __syncthreads();
            if (ty == 0 && live) {
                for (int l = 1; l < ry; ++l) {
                    s0 += sred[0][l * tx_n + tx]; s1 += sred[1][l * tx_n + tx];
                    q0 += sred[2][l * tx_n + tx]; q1 += sred[3][l * tx_n + tx];
                }
                atomicAdd(sum_g + c, (double)s0); atomicAdd(sum_g + c + 1, (double)s1);
                atomicAdd(sum_gx + c, (double)q0); atomicAdd(sum_gx + c + 1, (double)q1);
            }
            __syncthreads();
        }
    }
}

// Two upstreams a, b through ONE train-mode BatchNorm (two backward sweeps over the same saved forward state): the backward is
// linear in its upstream once the forward is fixed, so the two share the reads of x.
//   MODE 1: sums of both upstreams; reads x, dy_a, dy_b (3 passes instead of 4)
//   MODE 2: dx_a and dx_b; reads x, dy_a, dy_b, writes dx_a, dx_b (5 passes instead of 6)
// Per upstream every expression (mask, fmaf order, the row walk of a thread) is that of bn_bwd_cp_kernel: launched with the
// same grid and rows_per_block, each upstream gets the fp32 partial sums, and dx, of a single-upstream call (a thread still
// accumulates its rows in row order; batching the loads does not change that order).
template <int MODE, typename Tx, typename Tg>
__global__ void __launch_bounds__(256, 4) bn_bwd_cp2_kernel(
    const Tx* __restrict__ x, const Tg* __restrict__ dya, const Tg* __restrict__ dyb, Tg* __restrict__ dxa,
    Tg* __restrict__ dxb, long long rows, int C, const float* __restrict__ mean, const float* __restrict__ invstd,
    const float* __restrict__ gamma, const float* __restrict__ beta, int relu, int train, const float* __restrict__ mga,
    const float* __restrict__ mgxa, const float* __restrict__ mgb, const float* __restrict__ mgxb,
    double* __restrict__ sga, double* __restrict__ sgxa, double* __restrict__ sgb, double* __restrict__ sgxb,
    int rows_per_block) {
    constexpr int D = 8;                      // rows per load batch
    const int cp = C >> 1;
    const int tx_n = cp >= 256 ? 256 : cp;
    const int ry = 256 / tx_n;
    const int tx = threadIdx.x % tx_n, ty = threadIdx.x / tx_n;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = min(rows, r0 + rows_per_block);
    __shared__ float sred[8][256];
    for (int pb = blockIdx.y * tx_n; pb < cp; pb += gridDim.y * tx_n) {
        const int c = (pb + tx) * 2;
        const bool live = (pb + tx) < cp;
        float mu0 = 0, mu1 = 0, is0 = 0, is1 = 0, sc0 = 0, sc1 = 0, be0 = 0, be1 = 0;
        float ka10 = 0, ka11 = 0, ka20 = 0, ka21 = 0, kb10 = 0, kb11 = 0, kb20 = 0, kb21 = 0;
        if (live) {
            mu0 = mean[c]; mu1 = mean[c + 1]; is0 = invstd[c]; is1 = invstd[c + 1];
            sc0 = gamma[c] * is0; sc1 = gamma[c + 1] * is1; be0 = beta[c]; be1 = beta[c + 1];
            if (MODE == 2 && train) {
                ka10 = -sc0 * mga[c]; ka11 = -sc1 * mga[c + 1];
                ka20 = -sc0 * is0 * mgxa[c]; ka21 = -sc1 * is1 * mgxa[c + 1];
                kb10 = -sc0 * mgb[c]; kb11 = -sc1 * mgb[c + 1];
                kb20 = -sc0 * is0 * mgxb[c]; kb21 = -sc1 * is1 * mgxb[c + 1];
            }
        }
        float sa0 = 0.f, sa1 = 0.f, qa0 = 0.f, qa1 = 0.f, sb0 = 0.f, sb1 = 0.f, qb0 = 0.f, qb1 = 0.f;
        // one row of this thread's two channels, both upstreams
        auto row = [&](long long r, typename Pair<Tx>::Raw xw, typename Pair<Tg>::Raw aw, typename Pair<Tg>::Raw bw) {
            const float2 xv = Pair<Tx>::cvt(xw), av = Pair<Tg>::cvt(aw), bv = Pair<Tg>::cvt(bw);
            const float xc0 = xv.x - mu0, xc1 = xv.y - mu1;
            const bool z0 = relu && !(xc0 * sc0 + be0 > 0.f), z1 = relu && !(xc1 * sc1 + be1 > 0.f);
            float ga0 = av.x, ga1 = av.y, gb0 = bv.x, gb1 = bv.y;
            if (z0) { ga0 = 0.f; gb0 = 0.f; }
            if (z1) { ga1 = 0.f; gb1 = 0.f; }
            if (MODE == 1) {
                sa0 += ga0; sa1 += ga1; qa0 = fmaf(ga0, xc0, qa0); qa1 = fmaf(ga1, xc1, qa1);
                sb0 += gb0; sb1 += gb1; qb0 = fmaf(gb0, xc0, qb0); qb1 = fmaf(gb1, xc1, qb1);
            } else {
                Pair<Tg>::st(dxa + r * C + c, fmaf(ga0, sc0, fmaf(xc0, ka20, ka10)), fmaf(ga1, sc1, fmaf(xc1, ka21, ka11)));
                Pair<Tg>::st(dxb + r * C + c, fmaf(gb0, sc0, fmaf(xc0, kb20, kb10)), fmaf(gb1, sc1, fmaf(xc1, kb21, kb11)));
            }
        };
        if (live) {
            // batches of D rows: all 3 x D loads of a batch are issued before its math. With three streams a second buffer
            // for the next batch would not fit 64 registers; 32 resident warps per SM keep the loads of other batches in
            // flight while one does its math, and 3 x 8 loads per thread outstanding exceed the single kernel's 2 x 8.
            long long r = r0 + ty;
#pragma unroll 1
            for (; r + (D - 1LL) * ry < r1; r += (long long)D * ry) {
                typename Pair<Tx>::Raw xr[D];
                typename Pair<Tg>::Raw ar[D], br[D];
#pragma unroll
                for (int u = 0; u < D; ++u) {
                    const long long o = (r + (long long)u * ry) * C + c;
                    xr[u] = Pair<Tx>::raw(x + o); ar[u] = Pair<Tg>::raw(dya + o); br[u] = Pair<Tg>::raw(dyb + o);
                }
#pragma unroll
                for (int u = 0; u < D; ++u) row(r + (long long)u * ry, xr[u], ar[u], br[u]);
            }
            for (; r < r1; r += ry)
                row(r, Pair<Tx>::raw(x + r * C + c), Pair<Tg>::raw(dya + r * C + c), Pair<Tg>::raw(dyb + r * C + c));
        }
        if (MODE == 1) {
            qa0 *= is0; qa1 *= is1; qb0 *= is0; qb1 *= is1;
            sred[0][threadIdx.x] = sa0; sred[1][threadIdx.x] = sa1; sred[2][threadIdx.x] = qa0; sred[3][threadIdx.x] = qa1;
            sred[4][threadIdx.x] = sb0; sred[5][threadIdx.x] = sb1; sred[6][threadIdx.x] = qb0; sred[7][threadIdx.x] = qb1;
            __syncthreads();
            if (ty == 0 && live) {
                for (int l = 1; l < ry; ++l) {
                    sa0 += sred[0][l * tx_n + tx]; sa1 += sred[1][l * tx_n + tx];
                    qa0 += sred[2][l * tx_n + tx]; qa1 += sred[3][l * tx_n + tx];
                    sb0 += sred[4][l * tx_n + tx]; sb1 += sred[5][l * tx_n + tx];
                    qb0 += sred[6][l * tx_n + tx]; qb1 += sred[7][l * tx_n + tx];
                }
                atomicAdd(sga + c, (double)sa0); atomicAdd(sga + c + 1, (double)sa1);
                atomicAdd(sgxa + c, (double)qa0); atomicAdd(sgxa + c + 1, (double)qa1);
                atomicAdd(sgb + c, (double)sb0); atomicAdd(sgb + c + 1, (double)sb1);
                atomicAdd(sgxb + c, (double)qb0); atomicAdd(sgxb + c + 1, (double)qb1);
            }
            __syncthreads();
        }
    }
}

// per channel, once: the fp32 means the apply pass needs (one fp64 division per CHANNEL instead of per thread) and the
// parameter gradients dgamma = sum(g*xhat), dbeta = sum(g) (nullable)
__global__ void bn_param_grad_kernel(const double* __restrict__ sum_g, const double* __restrict__ sum_gx, double count,
                                     int C, float* __restrict__ mean_g, float* __restrict__ mean_gx,
                                     float* __restrict__ dgamma, float* __restrict__ dbeta, int accumulate) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    mean_g[c] = (float)(sum_g[c] / count);
    mean_gx[c] = (float)(sum_gx[c] / count);
    if (dgamma) {
        const float dg = (float)sum_gx[c], db = (float)sum_g[c];
        dgamma[c] = accumulate ? dgamma[c] + dg : dg;
        dbeta[c] = accumulate ? dbeta[c] + db : db;
    }
}

// bits[pixel] bit j = (y[pixel][j] > 0) for a channels-last bf16 tensor with exactly 32 channels: the ReLU mask of
// Discriminator.conv[0] in 4 B per pixel instead of 64 B, read back by the data-gradient epilogue that applies the ReLU backward
__global__ void relu_bitmask32_kernel(const __nv_bfloat16* __restrict__ y, uint32_t* __restrict__ bits, long long pixels) {
    // one warp per 32 pixels: lane l loads 16-byte pieces so that the warp reads 2 KB contiguous; ballot-free formulation:
    // thread t of the block handles pixel p = block*256 + t with four 16-byte loads
    const long long px = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= pixels) return;
    const uint4* src = reinterpret_cast<const uint4*>(y + px * 32);
    uint32_t m = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 r = __ldg(src + q);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (__uint_as_float(w[j] << 16) > 0.f) m |= 1u << (q * 8 + 2 * j);
            if (__uint_as_float(w[j] & 0xffff0000u) > 0.f) m |= 1u << (q * 8 + 2 * j + 1);
        }
    }
    bits[px] = m;
}

// relu backward on its own (bias+ReLU layers: discriminator conv0, WAE discriminator MLP): dx = dy * (y > 0);
// 8 elements per thread when n % 8 == 0 (always, for channels-last tensors with C % 8 == 0)
template <typename T>
__global__ void relu_bwd_kernel(const T* __restrict__ y, const T* __restrict__ dy, T* __restrict__ dx, long long n) {
    if ((n & 7) == 0) {
        for (long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 8; i < n;
             i += (long long)gridDim.x * blockDim.x * 8) {
            float a[8], g[8];
            bn_ld8(y + i, a);
            bn_ld8(dy + i, g);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[j] = a[j] > 0.f ? g[j] : 0.f;
            if constexpr (sizeof(T) == 2) {
                *reinterpret_cast<uint4*>(dx + i) = make_uint4(pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]),
                                                               pack_bf16x2(g[4], g[5]), pack_bf16x2(g[6], g[7]));
            } else {
                *reinterpret_cast<float4*>(dx + i) = make_float4(g[0], g[1], g[2], g[3]);
                *reinterpret_cast<float4*>(dx + i + 4) = make_float4(g[4], g[5], g[6], g[7]);
            }
        }
        return;
    }
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        st_f(dx + i, ld_f(y + i) > 0.f ? ld_f(dy + i) : 0.f);
}

// dst[i] += part[0][i] + part[1][i] + ... + part[nparts-1][i], always in this order: the fixed-order replacement for
// atomics where several CTAs contribute to one element (the result must not depend on which CTA finishes first)
template <typename T>
__global__ void ordered_add_kernel(const T* __restrict__ part, int nparts, long long n, T* __restrict__ dst) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        T s = part[i];
        for (int b = 1; b < nparts; ++b) s += part[(long long)b * n + i];
        dst[i] += s;
    }
}

// column sums of a [rows, C] matrix into fp32 (bias gradients)
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, long long rows, int C,
                                                     float* __restrict__ out, int rows_per_block) {
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    const long long r1 = min(rows, r0 + rows_per_block);
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float s = 0.f;
        for (long long r = r0; r < r1; ++r) s += ld_f(x + r * C + c);
        out[(long long)blockIdx.x * C + c] = s;   // this block's partial (summed in block order by ordered_add_kernel)
    }
}

// ------------------------------------------------------------------------------------------------
// layout / dtype packers
// ------------------------------------------------------------------------------------------------
// batched 2-D transpose with dtype conversion through a padded shared-memory tile: dst[n][c][r] (+)= src[n][r][c]
// (the NCHW <-> NHWC flatten / view conversions at the fc boundaries, vae_gan.py:89,127,180). Both sides coalesced.
template <typename Tin, typename Tout>
__global__ void __launch_bounds__(256) transpose_batched_kernel(const Tin* __restrict__ src, Tout* __restrict__ dst, int R,
                                                                int Cc, int accumulate) {
    __shared__ float tile[32][33];
    const long long base = (long long)blockIdx.z * R * Cc;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r = r0 + ty + 8 * k, c = c0 + tx;
        tile[ty + 8 * k][tx] = (r < R && c < Cc) ? ld_f(src + base + (long long)r * Cc + c) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + ty + 8 * k, r = r0 + tx;
        if (c < Cc && r < R) {
            Tout* o = dst + base + (long long)c * R + r;
            float v = tile[tx][ty + 8 * k];
            if (accumulate) v += ld_f(o);
            st_f(o, v);
        }
    }
}

// strided gather copy with dtype conversion: dst[i0,i1,i2,i3] (dense, row-major) = src[i0*s0+i1*s1+i2*s2+i3*s3]
template <typename Tin, typename Tout>
__global__ void permute4_kernel(const Tin* __restrict__ src, Tout* __restrict__ dst, int d0, int d1, int d2, int d3,
                                long long s0, long long s1, long long s2, long long s3, int accumulate) {
    const long long total = (long long)d0 * d1 * d2 * d3;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int i3 = (int)(i % d3);
        long long r = i / d3;
        const int i2 = (int)(r % d2);
        r /= d2;
        const int i1 = (int)(r % d1);
        const int i0 = (int)(r / d1);
        float v = ld_f(src + i0 * s0 + i1 * s1 + i2 * s2 + i3 * s3);
        if (accumulate) v += ld_f(dst + i);
        st_f(dst + i, v);
    }
}
// strided scatter: dst[i0*s0+i1*s1+i2*s2+i3*s3] (+)= src[i0,i1,i2,i3] (dense)
template <typename Tin, typename Tout>
__global__ void scatter4_kernel(const Tin* __restrict__ src, Tout* __restrict__ dst, int d0, int d1, int d2, int d3,
                                long long s0, long long s1, long long s2, long long s3, int accumulate) {
    const long long total = (long long)d0 * d1 * d2 * d3;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int i3 = (int)(i % d3);
        long long r = i / d3;
        const int i2 = (int)(r % d2);
        r /= d2;
        const int i1 = (int)(r % d1);
        const int i0 = (int)(r / d1);
        Tout* o = dst + i0 * s0 + i1 * s1 + i2 * s2 + i3 * s3;
        float v = ld_f(src + i);
        if (accumulate) v += ld_f(o);
        st_f(o, v);
    }
}

// parity-merged scatter pack (see IgParams::merge): dst[(t9*128 + g*32 + n)*Ck + k] = src[((kh*5+kw)*32 + n)*Ck + k] where
// t9 = (dy+1)*3 + (dx+1), g = column group of class (ph,pw) in the order (0,1),(0,0),(1,0),(1,1), kh = ph + 2 - 2*dy, kw = pw + 2 - 2*dx; zero when (kh, kw) falls outside the 5x5 window.
// src is the ordinary tap-major pack [25][32][Ck].
__global__ void merge_pack_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int Ck) {
    const int total = 9 * 128 * Ck;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int k = i % Ck;
        const int r = i / Ck;
        const int n = r & 31, g = (r >> 5) & 3, t9 = r >> 7;
        const int dy = t9 / 3 - 1, dx = t9 % 3 - 1;
        // column groups in the order (ph,pw) = (0,1),(0,0),(1,0),(1,1): the classes with non-zero weights for a coarse tap are
        // then always a CONTIGUOUS column range (dy = -1: groups 0-1, dx = -1: groups 1-2, both: group 1)
        const int ph = g >> 1, pw = (g == 0 || g == 3) ? 1 : 0;
        const int kh = ph + 2 - 2 * dy, kw = pw + 2 - 2 * dx;
        __nv_bfloat16 v = __float2bfloat16_rn(0.f);
        if (kh >= 0 && kh < 5 && kw >= 0 && kw < 5) v = src[((size_t)(kh * 5 + kw) * 32 + n) * Ck + k];
        dst[i] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// losses (vae_gan.py:302-320, train_vgan_stage1.py:369-372, train_wae_stage1.py:281-282,301-303)
// ------------------------------------------------------------------------------------------------
// z = eps*exp(0.5*logvar)+mu ; kl[b] = -0.5 * sum_j (1 + lv - mu^2 - exp(lv)); one warp per row.
// mu / lv have row pitch `ld` (they may be the two halves of one [B, 2Z] head output); z / eps / kl are dense.
__global__ void reparam_kl_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ lv, int ld,
                                      const float* __restrict__ eps, float* __restrict__ z, float* __restrict__ kl,
                                      int B, int Z) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= B) return;
    const int lane = threadIdx.x & 31;
    float s = 0.f;
    for (int j = lane; j < Z; j += 32) {
        const float m = mu[row * (long long)ld + j], l = lv[row * (long long)ld + j];
        const float e = expf(l);
        if (z) z[row * (long long)Z + j] = eps[row * (long long)Z + j] * expf(0.5f * l) + m;
        s += 1.f + l - m * m - e;
    }
    s = warp_sum(s);
    if (lane == 0 && kl) kl[row] = -0.5f * s;
}
// dmu = gz + gkl[b]*mu ; dlv = gz*eps*0.5*exp(0.5 lv) + gkl[b]*0.5*(exp(lv)-1); outputs with row pitch ldd
template <typename Tg>
__global__ void reparam_kl_bwd_kernel(const float* __restrict__ mu, const float* __restrict__ lv, int ld,
                                      const float* __restrict__ eps, const float* __restrict__ gz,
                                      const float* __restrict__ gkl, float gkl_const, Tg* __restrict__ dmu,
                                      Tg* __restrict__ dlv, int ldd, int B, int Z) {
    const long long n = (long long)B * Z;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / Z);
        const int j = (int)(i - (long long)b * Z);
        const float l = lv[(long long)b * ld + j], m = mu[(long long)b * ld + j];
        const float g = gz ? gz[i] : 0.f;
        const float k = gkl ? gkl[b] : gkl_const;
        st_f(dmu + (long long)b * ldd + j, g + k * m);
        st_f(dlv + (long long)b * ldd + j, (gz ? g * eps[i] * 0.5f * expf(0.5f * l) : 0.f) + k * 0.5f * (expf(l) - 1.f));
    }
}
// out[b] = scale * sum_j (a[b,j]-b[b,j])^2 ; one block per row, warp-shuffle reduction, vectorised loads
template <typename T>
__global__ void __launch_bounds__(256) rowsqdiff_fwd_kernel(const T* __restrict__ a, const T* __restrict__ b,
                                                            float* __restrict__ out, long long F, float scale) {
    const long long row = blockIdx.x;
    const T* pa = a + row * F;
    const T* pb = b + row * F;
    float s = 0.f;
    for (long long j = threadIdx.x; j < F; j += blockDim.x) {
        const float d = ld_f(pa + j) - ld_f(pb + j);
        s += d * d;
    }
    __shared__ float red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) out[row] = scale * v;
    }
}
// da = 2*scale*g[b]*(a-b) ; db = -da  (either may be null)
template <typename T>
__global__ void rowsqdiff_bwd_kernel(const T* __restrict__ a, const T* __restrict__ b, const float* __restrict__ g,
                                     T* __restrict__ da, T* __restrict__ db, long long rows, long long F,
                                     float scale) {
    const long long n = rows * F;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = 2.f * scale * g[i / F] * (ld_f(a + i) - ld_f(b + i));
        if (da) st_f(da + i, v);
        if (db) st_f(db + i, -v);
    }
}
// logit head: p = sigmoid(x . w + b) for a [rows, F] matrix and a single output unit (Linear(F,1) + sigmoid);
// one warp per row. vae_gan.py:160,183 and :519-520.
template <typename T>
__global__ void head_sigmoid_fwd_kernel(const T* __restrict__ x, const float* __restrict__ w,
                                        const float* __restrict__ bias, float* __restrict__ p, int rows, int F) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    float s = 0.f;
    for (int j = lane; j < F; j += 32) s += ld_f(x + (long long)row * F + j) * __ldg(w + j);
    s = warp_sum(s);
    if (lane == 0) p[row] = 1.f / (1.f + expf(-(s + bias[0])));
}
// given gp = dL/dp: dlogit = gp*p*(1-p); dx[row,:] = dlogit*w ; dw += sum_rows dlogit*x[row,:] ; db += sum dlogit
template <typename T>
__global__ void __launch_bounds__(256) head_sigmoid_bwd_kernel(const T* __restrict__ x, const float* __restrict__ w,
                                                               const float* __restrict__ p,
                                                               const float* __restrict__ gp, T* __restrict__ dx,
                                                               float* __restrict__ dw, float* __restrict__ db,
                                                               int rows, int F, int rows_per_block) {
    const int r0 = blockIdx.x * rows_per_block;
    const int r1 = min(rows, r0 + rows_per_block);
    for (int j = threadIdx.x; j < F; j += blockDim.x) {
        const float wj = w[j];
        float acc = 0.f;
        for (int r = r0; r < r1; ++r) {
            const float pr = p[r];
            const float dl = gp[r] * pr * (1.f - pr);
            if (dx) st_f(dx + (long long)r * F + j, dl * wj);
            acc += dl * ld_f(x + (long long)r * F + j);
        }
        if (dw) dw[(long long)blockIdx.x * F + j] = acc;   // per-block partials, see colsum_kernel
    }
    if (db && threadIdx.x == 0) {
        float acc = 0.f;
        for (int r = r0; r < r1; ++r) acc += gp[r] * p[r] * (1.f - p[r]);
        db[blockIdx.x] = acc;
    }
}
// bce[i] = -log(sign>0 ? p+1e-3 : 1-p+1e-3) * scale
__global__ void bce_fwd_kernel(const float* __restrict__ p, float* __restrict__ out, int n, int positive,
                               float scale) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = -scale * logf(positive ? p[i] + 1e-3f : 1.f - p[i] + 1e-3f);
}
__global__ void bce_bwd_kernel(const float* __restrict__ p, const float* __restrict__ g, float* __restrict__ dp,
                               int n, int positive, float scale, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = positive ? -scale * g[i] / (p[i] + 1e-3f) : scale * g[i] / (1.f - p[i] + 1e-3f);
    dp[i] = accumulate ? dp[i] + v : v;
}

// ------------------------------------------------------------------------------------------------
// fused multi-tensor optimizers (train_vgan_stage1.py:275-283 RMSprop(alpha=.9, eps=1e-8);
// train_wae_stage1.py:221-224 Adam(betas=(.5,.999))). One launch updates a whole parameter bucket.
// ------------------------------------------------------------------------------------------------
struct MtChunk {
    float* p;
    const float* g;
    float* s1;   // RMSprop: square_avg ; Adam: exp_avg
    float* s2;   // Adam: exp_avg_sq
    long long n;
};
#define FMRI_MT_MAX 48
struct MtArgs {
    MtChunk t[FMRI_MT_MAX];
    int count;
};
// `gate` (nullable): a device flag; the launch is a no-op when *gate == 0 (equilibrium gate decided on the device,
// train_vgan_stage1.py:396-404, so the step needs no host round trip). `lr_dev` (nullable) overrides lr.
__global__ void __launch_bounds__(256) mt_rmsprop_kernel(const __grid_constant__ MtArgs a, float lr, float alpha,
                                                         float eps, float clamp, const float* __restrict__ lr_dev,
                                                         const float* __restrict__ gate) {
    if (gate && *gate == 0.f) return;
    if (lr_dev) lr = *lr_dev;
    const MtChunk t = a.t[blockIdx.y];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < t.n; i += (long long)gridDim.x * blockDim.x) {
        float g = t.g[i];
        if (clamp > 0.f) g = fminf(fmaxf(g, -clamp), clamp);
        const float sq = alpha * t.s1[i] + (1.f - alpha) * g * g;
        t.s1[i] = sq;
        t.p[i] = t.p[i] - lr * g / (sqrtf(sq) + eps);
    }
}
__global__ void __launch_bounds__(256) mt_adam_kernel(const __grid_constant__ MtArgs a, float lr, float beta1,
                                                      float beta2, float eps, float bc1, float bc2, float clamp,
                                                      const float* __restrict__ lr_dev,
                                                      const float* __restrict__ gate, const int* __restrict__ step_dev) {
    if (gate && *gate == 0.f) return;
    if (lr_dev) lr = *lr_dev;
    if (step_dev) {   // step count kept on the device (CUDA-graph replays advance it): bias corrections in double, like the host
        const double st = (double)*step_dev;
        bc1 = (float)(1.0 - pow((double)beta1, st));
        bc2 = (float)(1.0 - pow((double)beta2, st));
    }
    const MtChunk t = a.t[blockIdx.y];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < t.n; i += (long long)gridDim.x * blockDim.x) {
        float g = t.g[i];
        if (clamp > 0.f) g = fminf(fmaxf(g, -clamp), clamp);
        const float m = beta1 * t.s1[i] + (1.f - beta1) * g;
        const float v = beta2 * t.s2[i] + (1.f - beta2) * g * g;
        t.s1[i] = m;
        t.s2[i] = v;
        const float denom = sqrtf(v) / sqrtf(bc2) + eps;
        t.p[i] = t.p[i] - (lr / bc1) * m / denom;
    }
}

__global__ void step_increment_kernel(int* step) { *step += 1; }

// ------------------------------------------------------------------------------------------------
// small glue kernels of the fused training step
// ------------------------------------------------------------------------------------------------
// out = (a*x + b*y) * (img ? 1 - img^2 : 1): gradient mixing (loss_decoder = lambda*mse - (1-lambda)*loss_dis,
// train_vgan_stage1.py:372) fused with the tanh backward of Decoder.conv[3] (vae_gan.py:118-121). y nullable.
__global__ void axpby_tanh_bwd_kernel(float a, const float* __restrict__ x, float b, const float* __restrict__ y,
                                      const float* __restrict__ img, float* __restrict__ out, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = a * x[i] + (y ? b * y[i] : 0.f);
        if (img) {
            const float t = img[i];
            v *= 1.f - t * t;
        }
        out[i] = v;
    }
}
// per-channel sum of an NCHW fp32 tensor (bias gradient of Decoder.conv[3]); one block per (channel, image chunk)
__global__ void __launch_bounds__(256) chansum_nchw_kernel(const float* __restrict__ x, int N, int C, long long HW,
                                                           float* __restrict__ out) {
    const int c = blockIdx.x;
    float s = 0.f;
    for (int n = blockIdx.y; n < N; n += gridDim.y) {
        const float* p = x + ((long long)n * C + c) * HW;
        for (long long i = threadIdx.x; i < HW; i += blockDim.x) s += p[i];
    }
    __shared__ float red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) out[blockIdx.y * C + c] = v;   // per-block partial, see colsum_kernel
    }
}
// out[0] (+)= scale * sum(x[0..n)) in fp64 internally; single block (n is a batch-sized vector of per-sample losses)
__global__ void __launch_bounds__(256) vecsum_kernel(const float* __restrict__ x, long long n, float scale,
                                                     float* __restrict__ out, int accumulate) {
    double s = 0.0;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) s += (double)x[i];
    __shared__ double red[256];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = (accumulate ? out[0] : 0.f) + scale * (float)red[0];
}
// equilibrium gate on the device (train_vgan_stage1.py:396-404): sums[0] = sum bce_original, sums[1] = sum bce_predicted
// over `count` samples (already reduced across ranks); gates[0] = train_dis, gates[1] = train_dec as 0.f / 1.f.
// train_dis_in: the value the loss-mix block leaves in train_dis before the gate (0 in mode 'vae', :387; 1 otherwise)
__global__ void vgan_gate_kernel(const float* __restrict__ sums, float count, float margin, float equilibrium,
                                 int train_dis_in, float* __restrict__ gates) {
    if (threadIdx.x || blockIdx.x) return;
    const float mo = sums[0] / count, mp = sums[1] / count;
    bool dis = train_dis_in != 0, dec = true;
    if (mo < equilibrium - margin || mp < equilibrium - margin) dis = false;
    if (mo > equilibrium + margin || mp > equilibrium + margin) dec = false;
    if (!dis && !dec) dis = dec = true;
    gates[0] = dis ? 1.f : 0.f;
    gates[1] = dec ? 1.f : 0.f;
}
// x[i] *= s over a flat fp32 buffer (elementwise: keeps the step's fixed-order determinism)
__global__ void scale_f32_kernel(float* __restrict__ x, long long n, float s) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        x[i] *= s;
}
// eval-mode BatchNorm: mean / invstd from the running statistics
__global__ void bn_eval_stats_kernel(const float* __restrict__ rm, const float* __restrict__ rv, int C, float eps,
                                     float* __restrict__ mean, float* __restrict__ invstd) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    mean[c] = rm[c];
    invstd[c] = rsqrtf(rv[c] + eps);
}

}  // namespace fmri
