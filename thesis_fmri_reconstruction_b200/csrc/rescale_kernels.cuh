// Device-side stimulus rescale: the BOLD5000 stimulus transform of the reference (data_preprocessing/data_loader.py
// Rescale -> RandomShift -> SampleToTensor -> Normalization, train/train_vgan_stage2.py:160-168) on native-resolution uint8
// sources. Rescale calls skimage.transform.resize(img, (H, W)) with its defaults (skimage >= 0.19: order 1, mode 'reflect',
// anti-aliasing when some axis downsamples, float output in [0, 1]); restated per axis with f = in / out:
//   Gaussian pre-filter  sigma = max(0, (f - 1) / 2), radius int(4 sigma + 0.5), normalised exp(-x^2 / 2 sigma^2) taps,
//                        ndimage 'mirror' boundary (d c b | a b c d | c b a); an axis with sigma = 0 is not filtered;
//   linear interpolation at u = (o + 0.5) f - 0.5 (ndi.zoom order 1, grid_mode=True, mode 'mirror', no spline prefilter).
// The shift / flip / GreyToColor / normalisation that follow are those of image_pipeline_kernel (eval_kernels.cuh).
#pragma once
#include "ptx.cuh"
#include "../../include/fmri_b200.h"

namespace fmri {

constexpr int RS_THREADS = 256;

// Per-axis parameters of the resize (host and device compute them with the same double arithmetic).
__host__ __device__ inline double rs_sigma(int in, int out) {
    const double s = ((double)in / (double)out - 1.0) / 2.0;
    return s > 0.0 ? s : 0.0;
}
__host__ __device__ inline int rs_radius(int in, int out) {   // ndimage.gaussian_filter skips sigma <= 1e-15
    const double s = rs_sigma(in, out);
    return s > 1e-15 ? (int)(4.0 * s + 0.5) : 0;
}
// Shared memory of one CTA that produces `ty` output rows of an image: the two tap tables (padded to 16 B), the vertically
// filtered rows (two per resized row, fp32, pitch P = Ws*Cs rounded up to 4) and the uint8 source band (pitch P). The band
// holds the source rows of the bilinear taps +- the vertical radius: floor(u_hi) - floor(u_lo) <= ceil((ty - 1) f) apart,
// so at most ceil((ty - 1) f) + 2 + 2 r rows.
__host__ __device__ inline long long rs_pitch(int Ws, int Cs) { return ((long long)Ws * Cs + 3) / 4 * 4; }
__host__ __device__ inline long long rs_taps_bytes(int ry, int rx) { return ((2LL * ry + 1 + 2LL * rx + 1 + 3) / 4 * 4) * 4; }
__host__ inline long long rs_band_rows(int Hs, int H, int ty) {
    return ((long long)(ty - 1) * Hs + H - 1) / H + 2 + 2LL * rs_radius(Hs, H);
}
__host__ inline long long rs_smem_bytes(int Hs, int Ws, int Cs, int H, int W, int ty) {
    const long long P = rs_pitch(Ws, Cs);
    return rs_taps_bytes(rs_radius(Hs, H), rs_radius(Ws, W)) + 2LL * ty * P * 4 + rs_band_rows(Hs, H, ty) * P;
}

__device__ __forceinline__ int rs_mirror(int i, int n) {
    if (n == 1) return 0;
    const int period = 2 * (n - 1);
    i = abs(i) % period;
    return i < n ? i : period - i;
}
// First of the two source taps i0, i0 + 1 of output coordinate o, and the weight t of the second:
// u = (o + 0.5) in / out - 0.5 = ((2o + 1) in - out) / (2 out) in exact integer arithmetic (sides <= 32768 keep it below
// 2^31), t = remainder * fp32 1 / (2 out) (inv_den). An fp32 u = (o + 0.5f) * f - 0.5f is off by up to o * ulp(f) when
// in / out is not a binary fraction (f = 2.4: 1e-5 of a pixel at o = 100).
__device__ __forceinline__ int rs_tap(int o, int in, int out, float inv_den, float& t) {
    const int num = (2 * o + 1) * in - out, den = 2 * out;
    const int i = num >= 0 ? num / den : -1;   // num >= -out > -den
    t = (float)(num - i * den) * inv_den;
    return i;
}
// byte k of q as an exact float: 2^23 + byte assembled bitwise, minus 2^23 (PRMT + FADD instead of the quarter-rate I2F)
template <int k>
__device__ __forceinline__ float rs_byte(uint32_t q) {
    return __uint_as_float(__byte_perm(q, 0x4B000000u, 0x7540 + k)) - 8388608.f;
}
// normalised Gaussian taps of one axis (fp64, rounded once to fp32), or the single tap 1 when the axis is not filtered
__device__ inline void rs_taps(int in, int out, int r, float* g) {
    if (r == 0) {
        g[0] = 1.f;
        return;
    }
    const double s = rs_sigma(in, out), k = -0.5 / (s * s);
    double sum = 0.0;
    for (int j = -r; j <= r; ++j) sum += exp(k * (double)(j * j));
    for (int j = -r; j <= r; ++j) g[j + r] = (float)(exp(k * (double)(j * j)) / sum);
}
// horizontal taps of a filtered row at source column c, channel ch
__device__ __forceinline__ float rs_hsum(const float* row, int c, int ch, int Ws, int Cs, int rx, const float* gx) {
    float acc = 0.f;
    if (c - rx >= 0 && c + rx < Ws) {
        const float* p = row + (c - rx) * Cs + ch;
        for (int j = 0; j <= 2 * rx; ++j) acc = fmaf(gx[j], p[j * Cs], acc);
    } else {
        for (int j = 0; j <= 2 * rx; ++j) acc = fmaf(gx[j], row[rs_mirror(c - rx + j, Ws) * Cs + ch], acc);
    }
    return acc;
}

// One CTA = `ty` consecutive output rows of one image (blockIdx.x = image * tiles + tile). dst [N, 3, H, W] fp32:
//   dst[n, c, y, x] = (R[clamp(y - dy), clamp(x' - dx), cs] - mean[c]) / std[c],  x' = flip[n] ? W - 1 - x : x,
//   R = resize(src_n) / 255 as above, cs = c (3-channel source) or 0 (grey).
// The CTA needs the resized rows clamp(y - dy) of its output rows (a contiguous range of at most ty rows), i.e. two
// vertically filtered rows each. It stages the uint8 source rows those read (mirrored at the borders), runs the vertical
// taps only at those rows (over all source columns, four bytes per thread), then per output pixel the horizontal taps at
// the two source columns of the bilinear blend, and the blend. fp32 weights and sums, no atomics. When Hs = H and Ws = W
// every tap table is {1} and every blend weight 0, so R = src / 255 with the rounding of image_pipeline_kernel.
__global__ void __launch_bounds__(RS_THREADS) image_rescale_kernel(const uint8_t* __restrict__ src,
                                                                   const fmri_image_src* __restrict__ imgs, int H, int W,
                                                                   int ty, int tiles, const int* __restrict__ flip,
                                                                   const int* __restrict__ shift_xy, float m0, float m1,
                                                                   float m2, float s0, float s1, float s2,
                                                                   float* __restrict__ dst) {
    extern __shared__ __align__(16) uint8_t rs_smem[];
    const int n = blockIdx.x / tiles, tile = blockIdx.x % tiles;
    const fmri_image_src d = imgs[n];
    const int Hs = d.H, Ws = d.W, Cs = d.C;
    const int ry = rs_radius(Hs, H), rx = rs_radius(Ws, W);
    const float iy = 1.f / (float)(2 * H), ix = 1.f / (float)(2 * W);
    const int P = (int)rs_pitch(Ws, Cs);
    float* gy = reinterpret_cast<float*>(rs_smem);
    float* gx = gy + 2 * ry + 1;
    float* V = reinterpret_cast<float*>(rs_smem + rs_taps_bytes(ry, rx));
    uint8_t* band = reinterpret_cast<uint8_t*>(V + 2 * ty * P);

    if (threadIdx.x == 0) rs_taps(Hs, H, ry, gy);
    if (threadIdx.x == 32) rs_taps(Ws, W, rx, gx);

    const int dy = shift_xy ? shift_xy[2 * n] : 0, dx = shift_xy ? shift_xy[2 * n + 1] : 0;
    const int y0 = tile * ty, y1 = min(y0 + ty, H) - 1;
    const int r_lo = min(max(y0 - dy, 0), H - 1), r_hi = min(max(y1 - dy, 0), H - 1);
    float t;
    const int v_lo = rs_tap(r_lo, Hs, H, iy, t) - ry;              // virtual source row of band row 0
    const int nb = rs_tap(r_hi, Hs, H, iy, t) + 1 + ry - v_lo + 1;

    // stage the band: a warp copies 512 bytes of a row per step, 16 loads in flight per lane
    const uint8_t* img = src + d.offset;
    const int row_bytes = Ws * Cs, chunks = (row_bytes + 511) / 512, warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    for (int idx = warp; idx < nb * chunks; idx += RS_THREADS / 32) {
        const int b = idx / chunks, c0 = (idx - b * chunks) * 512 + lane;
        const uint8_t* s = img + (long long)rs_mirror(v_lo + b, Hs) * row_bytes;
        uint8_t* o = band + (long long)b * P;
        uint8_t v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = c0 + 32 * k < row_bytes ? __ldg(s + c0 + 32 * k) : 0;
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (c0 + 32 * k < row_bytes) o[c0 + 32 * k] = v[k];
    }
    __syncthreads();

    // vertical taps at the two source rows of each resized row r_lo..r_hi, four bytes per item
    const int words = P / 4, nv = 2 * (r_hi - r_lo + 1);
    const uint32_t* band32 = reinterpret_cast<const uint32_t*>(band);
    for (int it = threadIdx.x; it < nv * words; it += RS_THREADS) {
        const int k = it / words, w = it - k * words;
        const int vrow = rs_tap(r_lo + k / 2, Hs, H, iy, t) + (k & 1);
        const uint32_t* p = band32 + (long long)(vrow - ry - v_lo) * words + w;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j <= 2 * ry; ++j) {
            const uint32_t q = p[(long long)j * words];
            const float g = gy[j];
            acc.x = fmaf(g, rs_byte<0>(q), acc.x);
            acc.y = fmaf(g, rs_byte<1>(q), acc.y);
            acc.z = fmaf(g, rs_byte<2>(q), acc.z);
            acc.w = fmaf(g, rs_byte<3>(q), acc.w);
        }
        reinterpret_cast<float4*>(V + (long long)k * P)[w] = acc;
    }
    __syncthreads();

    // horizontal taps at the bilinear columns, blend, shift / flip / GreyToColor / normalise
    const int fl = flip ? flip[n] : 0;
    const long long plane = (long long)H * W;
    float* out = dst + (long long)n * 3 * plane;
    for (int it = threadIdx.x; it < (y1 - y0 + 1) * W; it += RS_THREADS) {
        const int y = y0 + it / W, x = it % W;
        const int r = min(max(y - dy, 0), H - 1);
        const int xs = min(max((fl ? W - 1 - x : x) - dx, 0), W - 1);
        float ty_, tx_;
        rs_tap(r, Hs, H, iy, ty_);
        const int c0 = rs_tap(xs, Ws, W, ix, tx_);
        const float* va = V + (long long)(2 * (r - r_lo)) * P;
        const float* vb = va + P;
        auto resized = [&](int ch) {
            const float a0 = rs_hsum(va, c0, ch, Ws, Cs, rx, gx), a1 = rs_hsum(va, c0 + 1, ch, Ws, Cs, rx, gx);
            const float b0 = rs_hsum(vb, c0, ch, Ws, Cs, rx, gx), b1 = rs_hsum(vb, c0 + 1, ch, Ws, Cs, rx, gx);
            const float a = fmaf(tx_, a1 - a0, a0), b = fmaf(tx_, b1 - b0, b0);
            return fmaf(ty_, b - a, a);
        };
        const float v0 = resized(0), v1 = Cs == 3 ? resized(1) : v0, v2 = Cs == 3 ? resized(2) : v0;
        // (R / 255 - mean) / std as image_pipeline_kernel compiles it: one fma of R, 1/255 and -mean, then the division
        const long long o = (long long)y * W + x;
        out[o] = fmaf(v0, 1.f / 255.f, -m0) / s0;
        out[plane + o] = fmaf(v1, 1.f / 255.f, -m1) / s1;
        out[2 * plane + o] = fmaf(v2, 1.f / 255.f, -m2) / s2;
    }
}

}  // namespace fmri
