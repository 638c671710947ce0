// Device-side resample as Pillow does it: Image.resize(size, BILINEAR | BICUBIC) on 8-bit L / RGB images (Pillow's
// ImagingResample, libImaging/Resample.c), which torchvision's Resize / CenterCrop / RandomResizedCrop call on PIL images
// (the COCO Stage-I loader's resize, train/train_vgan_stage1.py:161-171, data_preprocessing/data_loader.py:346). Per axis,
// with `in` the source window size and `out` the resized size:
//   scale = in / out, filterscale = max(scale, 1), support = filter_support * filterscale (1 bilinear, 2 bicubic),
//   output index xx: center = (xx + 0.5) scale, xmin = max((int)(center - support + 0.5), 0),
//   xlen = min((int)(center + support + 0.5), in) - xmin, w[x] = filter((x + xmin - center + 0.5) / filterscale)
//   (Pillow multiplies by ss = 1 / filterscale), normalised by their sum unless it is 0, then fixed point with 22
//   fractional bits, (int)(w 2^22 +- 0.5). All of it in IEEE fp64 without FMA contraction (the __d*_rn intrinsics), so the
//   integer taps are those Pillow computes on the host.
// Horizontal pass first (over the source rows the vertical taps read), each value clamp((2^21 + sum src * k) >> 22, 0, 255)
// in int32 and stored as uint8; then the vertical pass over those uint8 rows with the same formula. Image.resize itself
// runs the vertical pass first for an image more than 100 times taller than wide that shrinks vertically, and so does
// this kernel. The shift / flip /
// GreyToColor / normalisation that follow are those of image_pipeline_kernel (eval_kernels.cuh).
#pragma once
#include "ptx.cuh"
#include "../../include/fmri_b200.h"

namespace fmri {

constexpr int RP_THREADS = 256;
constexpr int RP_PREC = 22;   // Pillow's PRECISION_BITS for 8-bit images: 32 - 8 - 2

__host__ __device__ inline int rp_filter_support(int filter) { return filter == FMRI_RESAMPLE_BICUBIC ? 2 : 1; }
// Pillow's per-axis scale, filterscale and support (exact in fp64: in and out are integers below 2^15)
__host__ __device__ inline double rp_scale(int in, int out) { return (double)in / (double)out; }
__host__ __device__ inline double rp_support(int in, int out, int filter) {
    const double s = rp_scale(in, out);
    return rp_filter_support(filter) * (s < 1.0 ? 1.0 : s);
}
// taps per output index: Pillow's ksize = (int)ceil(support) * 2 + 1 (an upper bound of every xlen)
__host__ __device__ inline int rp_ksize(int in, int out, int filter) {
    return (int)ceil(rp_support(in, out, filter)) * 2 + 1;
}
// Source rows of a band of `ty` consecutive resized rows: xmin and xmin + xlen of the first and last row are at least
// center_lo - support - 0.5 and at most center_hi + support + 0.5 apart, center_hi - center_lo = (ty - 1) scale.
__host__ __device__ inline long long rp_band_rows(int Hs, int Hr, int filter, int ty) {
    const long long r = (long long)((ty - 1) * rp_scale(Hs, Hr) + 2.0 * rp_support(Hs, Hr, filter)) + 2;
    return r < Hs ? r : Hs;
}
__host__ __device__ inline long long rp_align16(long long b) { return (b + 15) / 16 * 16; }
// PIL.Image.resize runs the vertical pass first for an image more than 100 times taller than wide that shrinks vertically
__host__ __device__ inline bool rp_vertical_first(const fmri_image_window& d) { return d.H > 100LL * d.W && d.Hr < d.H; }
// Shared memory of one CTA that produces `ty` output rows of an image, in this order: the horizontal taps (W x kx int32)
// and their (xmin, xlen) pairs, the vertical taps of the band (ty x ky int32) and their pairs, and the uint8 first-pass
// values: the rp_band_rows x W horizontal-pass rows of the band, or with the vertical pass first its ty x Ws rows, times
// C. Each part starts on a 16-byte boundary.
__host__ __device__ inline long long rp_smem_bytes(const fmri_image_window& d, int H, int W, int filter, int ty) {
    const long long kx = rp_ksize(d.W, d.Wr, filter), ky = rp_ksize(d.H, d.Hr, filter);
    const long long first = rp_vertical_first(d) ? (long long)ty * d.W : rp_band_rows(d.H, d.Hr, filter, ty) * W;
    return rp_align16(4LL * W * kx) + rp_align16(8LL * W) + rp_align16(4LL * ty * ky) + rp_align16(8LL * ty) + first * d.C;
}

__device__ __forceinline__ double rp_filter(double x, int filter) {
    x = fabs(x);
    if (filter == FMRI_RESAMPLE_BICUBIC) {   // a = -0.5: a + 2 = 1.5, a + 3 = 2.5
        if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(__dmul_rn(1.5, x), 2.5), x), x), 1.0);
        if (x < 2.0) return __dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0), x), 4.0), -0.5);
        return 0.0;
    }
    return x < 1.0 ? __dsub_rn(1.0, x) : 0.0;
}
// Pillow's precompute_coeffs + normalize_coeffs_8bpc for output index xx of an axis in -> out: the fixed-point taps k[0..xlen)
// and (xmin, xlen). The weights are evaluated twice (sum, then divide) rather than held in a scratch array.
__device__ inline int2 rp_coeffs(int in, int out, int filter, int xx, int* __restrict__ k) {
    const double scale = __ddiv_rn((double)in, (double)out), fs = scale < 1.0 ? 1.0 : scale;
    const double support = __dmul_rn((double)rp_filter_support(filter), fs), ss = __ddiv_rn(1.0, fs);
    const double center = __dmul_rn(__dadd_rn((double)xx, 0.5), scale);
    const int xmin = max((int)__dadd_rn(__dsub_rn(center, support), 0.5), 0);
    const int xlen = min((int)__dadd_rn(__dadd_rn(center, support), 0.5), in) - xmin;
    double ww = 0.0;
    for (int x = 0; x < xlen; ++x)
        ww = __dadd_rn(ww, rp_filter(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss), filter));
    for (int x = 0; x < xlen; ++x) {
        double w = rp_filter(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss), filter);
        if (ww != 0.0) w = __ddiv_rn(w, ww);
        const double f = __dmul_rn(w, (double)(1 << RP_PREC));
        k[x] = w < 0.0 ? (int)__dadd_rn(-0.5, f) : (int)__dadd_rn(0.5, f);
    }
    return make_int2(xmin, xlen);
}
__device__ __forceinline__ uint32_t rp_clip8(int s) { return (uint32_t)min(max(s >> RP_PREC, 0), 255); }
// 2^21 + sum_j p[j * stride + ch] k[j] for the C channels at p (global memory through the read-only path when G)
template <bool G>
__device__ __forceinline__ void rp_dot(const uint8_t* p, long long stride, const int* __restrict__ k, int len, int Cs,
                                       int& a0, int& a1, int& a2) {
    a0 = a1 = a2 = 1 << (RP_PREC - 1);
    if (Cs == 3) {
        for (int j = 0; j < len; ++j, p += stride) {
            const int w = k[j];
            a0 += (int)(G ? __ldg(p) : p[0]) * w;
            a1 += (int)(G ? __ldg(p + 1) : p[1]) * w;
            a2 += (int)(G ? __ldg(p + 2) : p[2]) * w;
        }
    } else {
        for (int j = 0; j < len; ++j, p += stride) a0 += (int)(G ? __ldg(p) : p[0]) * k[j];
    }
}

// One CTA = `ty` consecutive output rows of one image (blockIdx.x = image * tiles + tile). dst [N, 3, H, W] fp32:
//   dst[n, c, y, x] = (R[oy + clamp(y - dy), ox + clamp(x' - dx), cs] / 255 - mean[c]) / std[c],
//   x' = flip[n] ? W - 1 - x : x, R = the Hr x Wr Pillow resize of the source window (uint8), cs = c or 0 (grey).
// The CTA computes the taps of its W resized columns and of the (at most ty) resized rows its output rows read, runs the
// horizontal pass over the source rows those vertical taps read (source bytes through L1, the uint8 results in shared
// memory), then the vertical pass and the epilogue per output pixel; or, for the images rp_vertical_first names, the
// vertical pass at those rows over every source column first. Integer sums, no atomics: two calls give the same bits.
__global__ void __launch_bounds__(RP_THREADS, 3) image_resample_kernel(const uint8_t* __restrict__ src,
                                                                    const fmri_image_window* __restrict__ imgs, int H,
                                                                    int W, int filter, int ty, int tiles,
                                                                    const int* __restrict__ flip,
                                                                    const int* __restrict__ shift_xy, float m0, float m1,
                                                                    float m2, float s0, float s1, float s2,
                                                                    float* __restrict__ dst) {
    extern __shared__ __align__(16) uint8_t rp_smem[];
    const int n = blockIdx.x / tiles, tile = blockIdx.x % tiles;
    const fmri_image_window d = imgs[n];
    const int Cs = d.C, kx = rp_ksize(d.W, d.Wr, filter), ky = rp_ksize(d.H, d.Hr, filter);
    int* KX = reinterpret_cast<int*>(rp_smem);
    int2* BX = reinterpret_cast<int2*>(rp_smem + rp_align16(4LL * W * kx));
    int* KY = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(BX) + rp_align16(8LL * W));
    int2* BY = reinterpret_cast<int2*>(reinterpret_cast<uint8_t*>(KY) + rp_align16(4LL * ty * ky));
    uint8_t* T = reinterpret_cast<uint8_t*>(BY) + rp_align16(8LL * ty);

    const int dy = shift_xy ? shift_xy[2 * n] : 0, dx = shift_xy ? shift_xy[2 * n + 1] : 0;
    const int y0 = tile * ty, y1 = min(y0 + ty, H) - 1;
    const int r_lo = min(max(y0 - dy, 0), H - 1), r_hi = min(max(y1 - dy, 0), H - 1);   // window rows of the band
    const int nr = r_hi - r_lo + 1;

    // taps: one thread per resized column of the window, then one per resized row of the band
    for (int i = threadIdx.x; i < W + nr; i += RP_THREADS) {
        if (i < W) BX[i] = rp_coeffs(d.W, d.Wr, filter, d.ox + i, KX + (long long)i * kx);
        else BY[i - W] = rp_coeffs(d.H, d.Hr, filter, d.oy + r_lo + i - W, KY + (long long)(i - W) * ky);
    }
    __syncthreads();

    // first pass into T (uint8, all channels of one value per item), both passes' sums through rp_dot. Horizontal first:
    // the W resized columns of source rows b0 .. b0 + nb - 1. Vertical first (rp_vertical_first): the nr resized rows
    // of the band at every one of the Ws source columns.
    const bool vfirst = rp_vertical_first(d);
    const uint8_t* img = src + d.offset;
    const int b0 = BY[0].x, nb = BY[nr - 1].x + BY[nr - 1].y - b0;
    const int trow = (vfirst ? d.W : W) * Cs;   // bytes per row of T
    for (int it = threadIdx.x; it < (vfirst ? nr * d.W : nb * W); it += RP_THREADS) {
        int a0, a1, a2;
        if (vfirst) {
            const int r = it / d.W, c = it - r * d.W;
            rp_dot<true>(img + (long long)BY[r].x * d.pitch + c * Cs, d.pitch, KY + (long long)r * ky, BY[r].y, Cs, a0, a1, a2);
        } else {
            const int b = it / W, c = it - b * W;
            rp_dot<true>(img + (long long)(b0 + b) * d.pitch + (long long)BX[c].x * Cs, Cs, KX + (long long)c * kx, BX[c].y,
                         Cs, a0, a1, a2);
        }
        uint8_t* t = T + (long long)it * Cs;   // item it is byte it * Cs of T in both orders
        t[0] = (uint8_t)rp_clip8(a0);
        if (Cs == 3) {
            t[1] = (uint8_t)rp_clip8(a1);
            t[2] = (uint8_t)rp_clip8(a2);
        }
    }
    __syncthreads();

    // second pass per output pixel, shift / flip / GreyToColor / normalise
    const int fl = flip ? flip[n] : 0;
    const long long plane = (long long)H * W;
    float* out = dst + (long long)n * 3 * plane;
    for (int it = threadIdx.x; it < (y1 - y0 + 1) * W; it += RP_THREADS) {
        const int y = y0 + it / W, x = it % W;
        const int r = min(max(y - dy, 0), H - 1) - r_lo;
        const int xs = min(max((fl ? W - 1 - x : x) - dx, 0), W - 1);
        int a0, a1, a2;
        if (vfirst)
            rp_dot<false>(T + (long long)r * trow + BX[xs].x * Cs, Cs, KX + (long long)xs * kx, BX[xs].y, Cs, a0, a1, a2);
        else
            rp_dot<false>(T + (long long)(BY[r].x - b0) * trow + xs * Cs, trow, KY + (long long)r * ky, BY[r].y, Cs, a0, a1,
                          a2);
        const float v0 = (float)rp_clip8(a0), v1 = Cs == 3 ? (float)rp_clip8(a1) : v0, v2 = Cs == 3 ? (float)rp_clip8(a2) : v0;
        // (u8 / 255 - mean) / std as image_pipeline_kernel compiles it: one fma of u8, 1/255 and -mean, then the division
        const long long o = (long long)y * W + x;
        out[o] = fmaf(v0, 1.f / 255.f, -m0) / s0;
        out[plane + o] = fmaf(v1, 1.f / 255.f, -m1) / s1;
        out[2 * plane + o] = fmaf(v2, 1.f / 255.f, -m2) / s2;
    }
}

}  // namespace fmri
