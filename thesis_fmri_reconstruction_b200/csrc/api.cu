// Host side of libfmri_b200.so: argument checking, tile planning, TMA tensor-map construction and kernel launches
// behind the C ABI declared in include/fmri_b200.h. No torch, no cuDNN/cuBLAS, no CPU fallback.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <algorithm>

#include "../../include/fmri_b200.h"
#include "simt_kernels.cuh"
#include "tc_kernels.cuh"
#include "hconv_kernels.cuh"
#include "hwgrad_kernels.cuh"
#include "cto3_kernels.cuh"
#include "mmd_kernels.cuh"
#include "eval_kernels.cuh"
#include "similarity_kernels.cuh"

using namespace fmri;

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_OK(expr)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) return fail(FMRI_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)
static long long g_launches = 0;  // kernels launched by this library (memsets not counted); host-thread confined
#define LAUNCH_OK()                                                                                    \
    do {                                                                                               \
        ++g_launches;                                                                                  \
        cudaError_t e_ = cudaGetLastError();                                                           \
        if (e_ != cudaSuccess) return fail(FMRI_ERR_CUDA, "launch %s:%d: %s", __FILE__, __LINE__,      \
                                           cudaGetErrorString(e_));                                    \
    } while (0)

extern "C" int fmri_version(void) { return FMRI_ABI_VERSION; }
extern "C" long long fmri_launch_count(int reset) {
    const long long n = g_launches;
    if (reset) g_launches = 0;
    return n;
}
extern "C" const char* fmri_last_error(void) { return g_err; }

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline int grid1d(long long n, int block, int cap = 148 * 16) {
    long long g = (n + block - 1) / block;
    return (int)std::max<long long>(1, std::min<long long>(g, cap));
}

// ---- fixed-order reductions: where several CTAs contribute to one output element, each writes its partial into its own
// slice of a stream-ordered scratch buffer and ordered_add() sums the slices in CTA order onto the output. Atomics made the
// result depend on which CTA finished first: a last-bit difference that bf16 rounding and the optimizer grow step by step.
static void* scratch_alloc(size_t bytes, cudaStream_t st) {
    static bool pool_ready = false;
    if (!pool_ready) {   // keep freed scratch in the pool: no re-mapping from step to step
        int dev = 0;
        cudaMemPool_t pool;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        pool_ready = true;
    }
    void* p = nullptr;
    return cudaMallocAsync(&p, bytes, st) == cudaSuccess ? p : nullptr;
}
#define SCRATCH(ptr, type, count, st)                                                                        \
    type* ptr = reinterpret_cast<type*>(scratch_alloc(sizeof(type) * (size_t)(count), st));                  \
    if (!ptr) return fail(FMRI_ERR_CUDA, "scratch allocation of %zu bytes", sizeof(type) * (size_t)(count))
template <typename T>
static int ordered_add(const T* part, int nparts, long long n, T* dst, cudaStream_t st) {
    ordered_add_kernel<T><<<grid1d(n, 256), 256, 0, st>>>(part, nparts, n, dst);
    LAUNCH_OK();
    return 0;
}

extern "C" int fmri_tensor_path_available(void) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return major == 10 ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------ tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
// bf16 tensor map of rank 2..4. dims/box innermost first; strides in ELEMENTS for dims 1..rank-1.
static int make_map(CUtensorMap* m, const void* base, int rank, const long long* dims, const long long* strides_el,
                    const int* box, int inner_bytes) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(FMRI_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
    cuuint64_t gd[4], gs[3];
    cuuint32_t bx[4], es[4];
    for (int i = 0; i < rank; ++i) {
        gd[i] = (cuuint64_t)dims[i];
        bx[i] = (cuuint32_t)box[i];
        es[i] = 1;
    }
    for (int i = 0; i + 1 < rank; ++i) gs[i] = (cuuint64_t)strides_el[i] * 2;
    const CUtensorMapSwizzle sw = inner_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                     : CU_TENSOR_MAP_SWIZZLE_32B;
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(FMRI_ERR_CUDA,
                    "cuTensorMapEncodeTiled failed (%d): rank %d dims %lld %lld %lld %lld box %d %d %d %d stride0 %lld",
                    (int)r, rank, dims[0], dims[1], rank > 2 ? dims[2] : 0, rank > 3 ? dims[3] : 0, box[0], box[1],
                    rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0, strides_el[0]);
    return 0;
}
// NHWC activation viewed as (C, X, Y, N) with pixel strides (sx, sy, sn) elements.
static int make_act_map(CUtensorMap* m, const void* base, int C, int X, int Y, int N, long long sx, long long sy,
                        long long sn, int box_c, int bw, int bh, int bn) {
    const long long dims[4] = {C, std::max(X, 1), std::max(Y, 1), N};
    const long long st[3] = {sx, sy, sn};
    const int box[4] = {box_c, bw, bh, bn};
    return make_map(m, base, 4, dims, st, box, box_c * 2);
}

// ------------------------------------------------------------------------------------------------ igemm launch
template <int BN, int KCH, int STAGES, int MT>
static int launch_ig(const IgParams& p, int classes, cudaStream_t st) {
    using L = IgSmem<BN, KCH, STAGES, MT>;
    static bool attr_done = false;
    if (!attr_done) {
        CUDA_OK(cudaFuncSetAttribute(igemm_kernel<BN, KCH, STAGES, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     L::TOTAL));
        attr_done = true;
    }
    dim3 grid(cdiv((long long)p.tiles_x * p.tiles_y * p.tiles_n, MT), p.n_tiles * p.splits, classes);
    igemm_kernel<BN, KCH, STAGES, MT><<<grid, 192, L::TOTAL, st>>>(p);
    LAUNCH_OK();
    return 0;
}
template <int BN, int KCH, int STAGES, int MT, bool MASK, bool YR = false>
static int launch_ig_persistent_x(const IgParams& p, int classes, cudaStream_t st) {
    using L = IgSmem<BN, KCH, STAGES, MT, YR, true>;
    static bool attr_done = false;
    if (!attr_done) {
        CUDA_OK(cudaFuncSetAttribute(igemm_persistent_kernel<BN, KCH, STAGES, MT, MASK, YR>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
        attr_done = true;
    }
    const long long m_groups = cdiv((long long)p.tiles_x * p.tiles_y * p.tiles_n, MT);
    const long long tiles = m_groups * p.n_tiles * classes;
    // resident CTAs per SM: TMEM columns, shared memory and registers (asked from the runtime once per instantiation)
    static int occ = 0;
    if (!occ) {
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, igemm_persistent_kernel<BN, KCH, STAGES, MT, MASK, YR>,
                                                              IGP_THREADS, L::TOTAL));
        occ = std::max(1, occ);
    }
    const int per_sm = std::max(1, std::min<int>(std::min(2, 512 / (2 * MT * BN)), occ));
    const int grid = (int)std::min<long long>(tiles, 148LL * per_sm);
    igemm_persistent_kernel<BN, KCH, STAGES, MT, MASK, YR><<<grid, IGP_THREADS, L::TOTAL, st>>>(p, classes);
    LAUNCH_OK();
    return 0;
}
template <int BN, int KCH, int STAGES, int MT, bool YR = false>
static int launch_ig_persistent(const IgParams& p, int classes, cudaStream_t st) {
    // the fused ReLU-mask epilogue lives in its own instantiation (register pressure of the common case)
    if (p.mask_y || p.mask_bits) return launch_ig_persistent_x<BN, KCH, STAGES, MT, true, YR>(p, classes, st);
    return launch_ig_persistent_x<BN, KCH, STAGES, MT, false, YR>(p, classes, st);
}
static bool g_last_ig_was_persistent = false;  // set by dispatch_ig (host-thread confined, like g_launches)
static int dispatch_ig_persistent(const IgParams& p_in, int BN, int KCH, int classes, cudaStream_t st) {
    IgParams p = p_in;
    if (p.stat_sum && p.out_fp32) return fail(FMRI_ERR_UNSUPPORTED, "fused column statistics need a bf16 output");
    static int skip = -1;
    if (skip < 0) {
        const char* e = getenv("FMRI_IG_SKIP");
        skip = e ? atoi(e) : 0;
    }
    p.skip = skip;
    static int force_pair = -1;
    if (force_pair < 0) {
        const char* e = getenv("FMRI_IG_PAIR");
        force_pair = (e && atoi(e) == 2) ? 1 : 0;
    }
    // measured per form (scripts/igemm_probe.py, with and without pairs): 128-byte-line stores take 11 % off the BN = 128
    // gathers (two-pass staging hides behind their short K loop) but cost 5-7 % on the parity-merged scatter and on BN = 256,
    // where holding two chunks before the first store lengthens the epilogue's critical path; FMRI_IG_PAIR=2 forces them
    // everywhere (tests)
    p.pair = (force_pair || (!p.merge && BN == 128)) ? 1 : 0;
    if (p.yr) {   // row-reuse gather (run_gather decided; two M sub-tiles = 8 output rows of one image)
        if (KCH == 32 && BN == 128) return launch_ig_persistent<128, 32, 4, 2, true>(p, classes, st);
        if (KCH == 32 && BN == 64) return launch_ig_persistent<64, 32, 3, 2, true>(p, classes, st);
        return fail(FMRI_ERR_UNSUPPORTED, "row-reuse igemm tile BN=%d KCH=%d not instantiated", BN, KCH);
    }
    if (KCH == 64) {
        switch (BN) {
            case 256: return launch_ig_persistent<256, 64, 4, 1>(p, classes, st);
            case 128: return launch_ig_persistent<128, 64, 4, 2>(p, classes, st);
            case 64: return launch_ig_persistent<64, 64, 4, 2>(p, classes, st);
            case 32: return launch_ig_persistent<32, 64, 4, 2>(p, classes, st);
        }
    } else if (KCH == 32) {
        switch (BN) {
            case 256: return launch_ig_persistent<256, 32, 4, 1>(p, classes, st);
            case 128: return launch_ig_persistent<128, 32, 4, 2>(p, classes, st);
            case 64: return launch_ig_persistent<64, 32, 4, 2>(p, classes, st);
            case 32: return launch_ig_persistent<32, 32, 4, 2>(p, classes, st);
        }
    }
    return fail(FMRI_ERR_UNSUPPORTED, "persistent igemm tile BN=%d KCH=%d not instantiated", BN, KCH);
}
static bool ig_goes_persistent(const IgParams& p, int classes) {
    static int force = -1;   // FMRI_IGEMM_PERSISTENT=2: the persistent kernel for every launch, however small (tests)
    if (force < 0) {
        const char* e = getenv("FMRI_IGEMM_PERSISTENT");
        force = (e && atoi(e) == 2) ? 1 : 0;
    }
    const long long all = (long long)p.tiles_x * p.tiles_y * p.tiles_n * p.n_tiles * classes;
    return p.splits == 1 && (all >= 2 * 148 || force);
}
static int dispatch_ig(const IgParams& p, int BN, int KCH, int classes, cudaStream_t st) {
    {
        g_last_ig_was_persistent = false;
        if (ig_goes_persistent(p, classes)) {
            g_last_ig_was_persistent = true;
            return dispatch_ig_persistent(p, BN, KCH, classes, st);
        }
    }
    // two M sub-tiles per CTA (shared weight tile) once there is more than a few waves of work
    const long long ctas = (long long)p.tiles_x * p.tiles_y * p.tiles_n * p.n_tiles * p.splits * classes;
    const bool mt2 = ctas >= 6 * 148 && p.splits == 1;
    if (KCH == 64) {
        switch (BN) {
            case 256: return mt2 ? launch_ig<256, 64, 3, 2>(p, classes, st) : launch_ig<256, 64, 4, 1>(p, classes, st);
            case 128: return mt2 ? launch_ig<128, 64, 4, 2>(p, classes, st) : launch_ig<128, 64, 4, 1>(p, classes, st);
            case 64: return mt2 ? launch_ig<64, 64, 4, 2>(p, classes, st) : launch_ig<64, 64, 4, 1>(p, classes, st);
            case 32: return mt2 ? launch_ig<32, 64, 4, 2>(p, classes, st) : launch_ig<32, 64, 4, 1>(p, classes, st);
        }
    } else if (KCH == 32) {
        switch (BN) {
            case 256: return mt2 ? launch_ig<256, 32, 4, 2>(p, classes, st) : launch_ig<256, 32, 4, 1>(p, classes, st);
            case 128: return mt2 ? launch_ig<128, 32, 4, 2>(p, classes, st) : launch_ig<128, 32, 4, 1>(p, classes, st);
            case 64: return mt2 ? launch_ig<64, 32, 4, 2>(p, classes, st) : launch_ig<64, 32, 4, 1>(p, classes, st);
            case 32: return mt2 ? launch_ig<32, 32, 4, 2>(p, classes, st) : launch_ig<32, 32, 4, 1>(p, classes, st);
        }
    }
    return fail(FMRI_ERR_UNSUPPORTED, "igemm tile BN=%d KCH=%d not instantiated", BN, KCH);
}
static int pick_bn(int n_total, long long m_tiles_times_classes) {
    if (n_total % 256 == 0 && m_tiles_times_classes * (n_total / 256) >= 148) return 256;
    if (n_total % 128 == 0) return 128;
    if (n_total % 64 == 0) return 64;
    if (n_total % 32 == 0) return 32;
    return 0;
}
static void pick_box(int X, int Y, int N, int* bw, int* bh, int* bn) {
    *bw = std::min(X, 128);
    *bh = std::max(1, std::min(Y, 128 / *bw));
    *bn = std::max(1, std::min(N, 128 / (*bw * *bh)));
}

// power-of-two pixel box (rows = bw*bh*bn is a power of two >= 16 whenever the problem has that many pixels): the weight-
// gradient kernel consumes pixels in K = 16 steps; boxes wider than the grid are zero-filled by TMA on both operands.
static void pick_box_pow2(int X, int Y, int N, int* bw, int* bh, int* bn) {
    auto up = [](int v) { int r = 1; while (r < v) r <<= 1; return r; };
    *bw = std::min(up(X), 128);
    *bh = std::max(1, std::min(up(Y), 128 / *bw));
    *bn = std::max(1, std::min(up(N), 128 / (*bw * *bh)));
}

// Gather-form plan: out[n,oy,ox,:] = sum_taps X[n, oy*s+kh-2, ox*s+kw-2, :] * pack[tap]
// (Conv2d fprop; ConvTranspose2d dgrad). X: [N,H,W,Ck] bf16, out: [N,OH,OW,Ng].
static void apply_mask(IgParams& p, const fmri_relu_mask* m) {   // ReLU backward in the epilogue, see fmri_relu_mask
    if (!m) return;
    p.mask_y = m->y;
    p.mask_bits = m->bits;
}
static int run_gather(const void* X, int N, int H, int W, int Ck, int OH, int OW, int Ng, int stride, const void* pack,
                      const float* bias, int act, void* out, int out_fp32, double* ssum, double* ssq,
                      cudaStream_t st, const fmri_relu_mask* mask = nullptr) {
    if (Ck % 32 || Ng % 32) return fail(FMRI_ERR_UNSUPPORTED, "tensor path needs channels %% 32 == 0 (%d,%d)", Ck, Ng);
    const int KCH = (Ck % 64 == 0) ? 64 : 32;
    IgParams p;
    memset(&p, 0, sizeof(p));
    pick_box(OW, OH, N, &p.bw, &p.bh, &p.bn);
    p.tiles_x = cdiv(OW, p.bw);
    p.tiles_y = cdiv(OH, p.bh);
    p.tiles_n = cdiv(N, p.bn);
    p.lim_n = N;
    const int BN = pick_bn(Ng, (long long)p.tiles_x * p.tiles_y * p.tiles_n);
    if (!BN) return fail(FMRI_ERR_UNSUPPORTED, "no N tile for %d", Ng);
    const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(X);
    // row reuse (IgSmem YR): thin K side, 32-pixel output rows, two vertically adjacent sub-tiles per CTA
    p.n_tiles = Ng / BN;
    p.splits = 1;
    const bool yr = stride == 2 && Ck == 32 && p.bw == 32 && p.bh == 4 && p.bn == 1 && OW == 32 && OH % 8 == 0 &&
                    (BN == 64 || BN == 128) && ig_goes_persistent(p, 1);
    p.yr = yr ? 1 : 0;
    const int box_h = yr ? 2 * p.bh + 2 : p.bh;
    if (stride == 2) {
        for (int ph = 0; ph < 2; ++ph)
            for (int pw = 0; pw < 2; ++pw) {
                const int Wp = (W - pw + 1) / 2, Hp = (H - ph + 1) / 2;
                int rc = make_act_map(&p.mapA[ph * 2 + pw], xb + ((long long)ph * W + pw) * Ck, Ck, Wp, Hp, N,
                                      2LL * Ck, 2LL * W * Ck, (long long)H * W * Ck, KCH, p.bw, box_h, p.bn);
                if (rc) return rc;
            }
    } else {
        int rc = make_act_map(&p.mapA[0], xb, Ck, W, H, N, Ck, (long long)W * Ck, (long long)H * W * Ck, KCH, p.bw,
                              p.bh, p.bn);
        if (rc) return rc;
    }
    {
        const long long dims[2] = {Ck, 25LL * Ng};
        const long long stv[1] = {Ck};
        const int box[2] = {KCH, BN};
        int rc = make_map(&p.mapB, pack, 2, dims, stv, box, KCH * 2);
        if (rc) return rc;
    }
    TapClass& c = p.cls[0];
    c.num_taps = 25;
    c.lim_x = OW;
    c.lim_y = OH;
    c.out_off = 0;
    for (int kh = 0; kh < 5; ++kh)
        for (int kw = 0; kw < 5; ++kw) {
            TapDesc& t = c.taps[kh * 5 + kw];
            if (stride == 2) {
                t.map = (int16_t)((kh & 1) * 2 + (kw & 1));
                t.dy = (int16_t)((kh - 2 - (kh & 1)) / 2);
                t.dx = (int16_t)((kw - 2 - (kw & 1)) / 2);
            } else {
                t.map = 0;
                t.dy = (int16_t)(kh - 2);
                t.dx = (int16_t)(kw - 2);
            }
            t.brow = (kh * 5 + kw) * Ng;
        }
    p.num_chunks = Ck / KCH;
    p.n_total = Ng;
    p.n_tiles = Ng / BN;
    p.splits = 1;
    p.a_bytes = p.bw * box_h * p.bn * KCH * 2;
    p.out_sn = (long long)OH * OW * Ng;
    p.out_sy = (long long)OW * Ng;
    p.out_sx = Ng;
    p.out = out;
    p.out_fp32 = out_fp32;
    p.bias = bias;
    p.act = act;
    p.stat_sum = ssum;
    p.stat_sq = ssq;
    apply_mask(p, mask);
    return dispatch_ig(p, BN, KCH, 1, st);
}

// Scatter-form plan (stride 2): out[n, 2a+ph, 2b+pw, :] = sum_{kh = ph (mod 2), kw = pw (mod 2)} X[n, a+(ph+2-kh)/2, ..] * pack[tap]
// (ConvTranspose2d fprop; Conv2d dgrad). X: [N,H,W,Ck], out: [N,OH,OW,Ng] with OH in {2H-1, 2H}.
static int run_scatter_merged(const void* X, int N, int H, int W, int Ck, int OH, int OW, const void* pack, void* out,
                              double* ssum, double* ssq, cudaStream_t st, const fmri_relu_mask* mask, const float* bias,
                              int act);
static int run_scatter(const void* X, int N, int H, int W, int Ck, int OH, int OW, int Ng, const void* pack, void* out,
                       double* ssum, double* ssq, cudaStream_t st, const fmri_relu_mask* mask = nullptr,
                       const float* bias = nullptr, int act = 0) {
    if (Ck % 32 || Ng % 32) return fail(FMRI_ERR_UNSUPPORTED, "tensor path needs channels %% 32 == 0 (%d,%d)", Ck, Ng);
    if (Ng == 32) return run_scatter_merged(X, N, H, W, Ck, OH, OW, pack, out, ssum, ssq, st, mask, bias, act);
    const int KCH = (Ck % 64 == 0) ? 64 : 32;
    IgParams p;
    memset(&p, 0, sizeof(p));
    const int GX = (OW + 1) / 2, GY = (OH + 1) / 2;  // class (0,0) sub-grid, the largest
    pick_box(GX, GY, N, &p.bw, &p.bh, &p.bn);
    p.tiles_x = cdiv(GX, p.bw);
    p.tiles_y = cdiv(GY, p.bh);
    p.tiles_n = cdiv(N, p.bn);
    p.lim_n = N;
    const int BN = pick_bn(Ng, 4LL * p.tiles_x * p.tiles_y * p.tiles_n);
    if (!BN) return fail(FMRI_ERR_UNSUPPORTED, "no N tile for %d", Ng);
    int rc = make_act_map(&p.mapA[0], X, Ck, W, H, N, Ck, (long long)W * Ck, (long long)H * W * Ck, KCH, p.bw, p.bh,
                          p.bn);
    if (rc) return rc;
    {
        const long long dims[2] = {Ck, 25LL * Ng};
        const long long stv[1] = {Ck};
        const int box[2] = {KCH, BN};
        rc = make_map(&p.mapB, pack, 2, dims, stv, box, KCH * 2);
        if (rc) return rc;
    }
    for (int ph = 0; ph < 2; ++ph)
        for (int pw = 0; pw < 2; ++pw) {
            TapClass& c = p.cls[ph * 2 + pw];
            c.lim_y = (OH - ph + 1) / 2;
            c.lim_x = (OW - pw + 1) / 2;
            c.out_off = ((long long)ph * OW + pw) * Ng;
            int nt = 0;
            for (int kh = ph; kh < 5; kh += 2)
                for (int kw = pw; kw < 5; kw += 2) {
                    TapDesc& t = c.taps[nt++];
                    t.map = 0;
                    t.dy = (int16_t)((ph + 2 - kh) / 2);
                    t.dx = (int16_t)((pw + 2 - kw) / 2);
                    t.brow = (kh * 5 + kw) * Ng;
                }
            c.num_taps = nt;
        }
    p.num_chunks = Ck / KCH;
    p.n_total = Ng;
    p.n_tiles = Ng / BN;
    p.splits = 1;
    p.a_bytes = p.bw * p.bh * p.bn * KCH * 2;
    p.out_sn = (long long)OH * OW * Ng;
    p.out_sy = 2LL * OW * Ng;
    p.out_sx = 2LL * Ng;
    p.out = out;
    p.out_fp32 = 0;
    p.stat_sum = ssum;
    p.stat_sq = ssq;
    p.bias = bias;
    p.act = act;
    apply_mask(p, mask);
    return dispatch_ig(p, BN, KCH, 4, st);
}

// Parity-merged scatter plan for Ng == 32 (IgParams::merge): one gather over the 3x3 coarse neighbourhood, N = 4 x 32.
// `pack` is the ordinary tap-major pack [25][32][Ck] followed by the merged pack [9][128][Ck] (fmri_conv_pack_elems).
static int run_scatter_merged(const void* X, int N, int H, int W, int Ck, int OH, int OW, const void* pack, void* out,
                              double* ssum, double* ssq, cudaStream_t st, const fmri_relu_mask* mask, const float* bias,
                              int act) {
    const int Ng = 32;
    const int KCH = (Ck % 64 == 0) ? 64 : 32;
    IgParams p;
    memset(&p, 0, sizeof(p));
    const int GX = (OW + 1) / 2, GY = (OH + 1) / 2;
    pick_box(GX, GY, N, &p.bw, &p.bh, &p.bn);
    p.tiles_x = cdiv(GX, p.bw);
    p.tiles_y = cdiv(GY, p.bh);
    p.tiles_n = cdiv(N, p.bn);
    p.lim_n = N;
    const int BN = 128;
    int rc = make_act_map(&p.mapA[0], X, Ck, W, H, N, Ck, (long long)W * Ck, (long long)H * W * Ck, KCH, p.bw, p.bh,
                          p.bn);
    if (rc) return rc;
    const __nv_bfloat16* mpack = reinterpret_cast<const __nv_bfloat16*>(pack) + 25LL * Ng * Ck;
    {
        const long long dims[2] = {Ck, 9LL * 128};
        const long long stv[1] = {Ck};
        const int box[2] = {KCH, BN};
        rc = make_map(&p.mapB, mpack, 2, dims, stv, box, KCH * 2);
        if (rc) return rc;
    }
    TapClass& c = p.cls[0];
    c.num_taps = 9;
    c.lim_x = GX;
    c.lim_y = GY;
    c.out_off = 0;
    // Coarse taps, the four full ones first (the first MMA of a tile must initialise every accumulator column). A tap with
    // dy = -1 only feeds the ph = 0 classes and one with dx = -1 only the pw = 0 classes; with the column groups ordered
    // (0,1),(0,0),(1,0),(1,1) (merge_pack_kernel) the live columns are contiguous, and the MMA warp skips the zero slabs:
    // 4 x 128 + 4 x 64 + 1 x 32 = 800 = 25 x 32 columns per K step instead of 9 x 128.
    static const int order[9] = {4, 5, 7, 8, 1, 2, 3, 6, 0};   // t9 = (dy+1)*3 + (dx+1)
    for (int i = 0; i < 9; ++i) {
        const int t9 = order[i], dy = t9 / 3 - 1, dx = t9 % 3 - 1;
        c.taps[i].map = 0;
        c.taps[i].dy = (int16_t)dy;
        c.taps[i].dx = (int16_t)dx;
        c.taps[i].brow = t9 * 128;
        int g0 = 0, ng = 4;                       // column groups [g0, g0 + ng)
        if (dy == -1 && dx == -1) { g0 = 1; ng = 1; }
        else if (dy == -1) { g0 = 0; ng = 2; }
        else if (dx == -1) { g0 = 1; ng = 2; }
        c.taps[i].ncol = (int16_t)(ng < 4 ? ((ng << 8) | g0) : 0);
    }
    p.num_chunks = Ck / KCH;
    p.n_total = 128;
    p.n_tiles = 1;
    p.splits = 1;
    p.a_bytes = p.bw * p.bh * p.bn * KCH * 2;
    p.out_sn = (long long)OH * OW * Ng;
    p.out_sy = 2LL * OW * Ng;
    p.out_sx = 2LL * Ng;
    p.out = out;
    p.out_fp32 = 0;
    p.stat_sum = ssum;
    p.stat_sq = ssq;
    p.bias = bias;   // merged epilogue: every 32-column group is the same 32 output channels (bias index = column % 32)
    p.act = act;
    p.merge = 1;
    p.merge_oh = OH;
    p.merge_ow = OW;
    p.merge_sy = (long long)OW * Ng;
    apply_mask(p, mask);
    return dispatch_ig(p, BN, KCH, 1, st);
}

// Plain GEMM plan: C[M,N] = act(A[M,K] B[N,K]^T + bias), A/B bf16 K-major with pitches, optional split-K into fp32.
static int run_gemm_tn(const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias, int act,
                       void* Cout, int ldc, int c_fp32, int accumulate, cudaStream_t st) {
    if (N % 32) return fail(FMRI_ERR_UNSUPPORTED, "gemm N %% 32 != 0 (%d)", N);
    if ((lda % 8) || (ldb % 8)) return fail(FMRI_ERR_ARG, "gemm pitches must be multiples of 8 elements");
    const int KCH = 64;
    IgParams p;
    memset(&p, 0, sizeof(p));
    p.bw = std::min(128, M);
    p.bh = 1;
    p.bn = 1;
    p.tiles_x = cdiv(M, 128);
    p.tiles_y = 1;
    p.tiles_n = 1;
    p.lim_n = 1;
    int BN = (N % 128 == 0) ? 128 : (N % 64 == 0 ? 64 : 32);
    if (N % 256 == 0 && (long long)p.tiles_x * (N / 256) >= 148) BN = 256;
    int rc = make_act_map(&p.mapA[0], A, K, M, 1, 1, lda, (long long)lda * M, (long long)lda * M, KCH, p.bw, 1, 1);
    if (rc) return rc;
    {
        const long long dims[2] = {K, N};
        const long long stv[1] = {ldb};
        const int box[2] = {KCH, BN};
        rc = make_map(&p.mapB, B, 2, dims, stv, box, KCH * 2);
        if (rc) return rc;
    }
    TapClass& c = p.cls[0];
    c.num_taps = 1;
    c.lim_x = M;
    c.lim_y = 1;
    c.out_off = 0;
    c.taps[0].map = 0;
    c.taps[0].dx = 0;
    c.taps[0].dy = 0;
    c.taps[0].brow = 0;
    p.num_chunks = cdiv(K, KCH);
    p.n_total = N;
    p.n_tiles = N / BN;
    // no split-K: with one writer per output element the result does not depend on CTA completion order (the linear
    // layers are a small share of the step)
    const int splits = 1;
    p.splits = splits;
    p.a_bytes = p.bw * KCH * 2;
    p.out_sn = 0;
    p.out_sy = 0;
    p.out_sx = ldc;
    p.out = Cout;
    p.out_fp32 = c_fp32;
    p.atomic_out = (splits > 1 || accumulate) ? 1 : 0;
    if (p.atomic_out && !c_fp32) return fail(FMRI_ERR_ARG, "accumulating gemm needs fp32 output");
    p.bias = bias;
    p.act = act;
    return dispatch_ig(p, BN, KCH, 1, st);
}

// ------------------------------------------------------------------------------------------------ wgrad launch
template <int BN, int NCH, int STAGES, int TG>
static int launch_wg(const WgParams& p, cudaStream_t st) {
    using L = WgSmem<BN, NCH, STAGES, TG>;
    static bool attr_done = false;
    if (!attr_done) {
        CUDA_OK(cudaFuncSetAttribute(wgrad_kernel<BN, NCH, STAGES, TG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     L::TOTAL));
        attr_done = true;
    }
    dim3 grid(cdiv(p.num_taps, TG), p.m_tiles * p.n_tiles, p.splits);
    wgrad_kernel<BN, NCH, STAGES, TG><<<grid, 192, L::TOTAL, st>>>(p);
    LAUNCH_OK();
    return 0;
}
// Split count for kernels that run ONE CTA per SM (the ~200 KB shared-memory wgrad tiles): pick s so that base * s CTAs fill
// whole waves of 148 (an ncu capture showed 312- and 300-CTA grids = 2.1 waves, i.e. a third round that is 11 % full and
// a 30 % longer kernel). Searches one to three waves, with a small preference for fewer, larger CTAs.
static int wave_splits(long long base, long long max_splits) {
    const long long lo = std::max<long long>(1, (148 + base - 1) / base);
    if (max_splits <= lo) return (int)std::max<long long>(1, max_splits);
    const long long hi = std::min<long long>(max_splits, std::max<long long>(lo, (3 * 148) / base));
    long long best = lo;
    double best_score = -1.0;
    for (long long s = lo; s <= hi; ++s) {
        const long long ctas = base * s, waves = (ctas + 147) / 148;
        const double score = (double)ctas / (148.0 * waves) - 0.01 * waves;
        if (score > best_score) { best_score = score; best = s; }
    }
    return (int)best;
}
static int dispatch_wg(const WgParams& p, int BN, int NCH, cudaStream_t st) {
    if (NCH == 64 && BN == 128) return p.num_taps > 1 ? launch_wg<128, 64, 2, 2>(p, st) : launch_wg<128, 64, 3, 1>(p, st);
    if (NCH == 64 && BN == 64) return launch_wg<64, 64, 4, 1>(p, st);
    if (NCH == 32 && BN == 32) return p.num_taps % 5 == 0 ? launch_wg<32, 32, 3, 5>(p, st) : launch_wg<32, 32, 4, 1>(p, st);
    return fail(FMRI_ERR_UNSUPPORTED, "wgrad tile BN=%d NCH=%d not instantiated", BN, NCH);
}
// ws[tap][m][n] += sum_pixels Dn[pixel][m] * Sh[pixel*stride + tap - 2][n]
//   Dn: [N,PH,PW,Cd] bf16 (dense side), Sh: [N,BH,BW,Cs] bf16 (shifted side; stride-parity planes when stride = 2)
static int run_wgrad_tc(const void* Dn, int N, int PH, int PW, int Cd, const void* Sh, int BH, int BW, int Cs,
                        int stride, int num_taps, float* ws, cudaStream_t st) {
    if (Cd % 64 || Cs % 32) return fail(FMRI_ERR_UNSUPPORTED, "wgrad tensor path needs Cd%%64==0, Cs%%32==0");
    WgParams p;
    memset(&p, 0, sizeof(p));
    pick_box(PW, PH, N, &p.bw, &p.bh, &p.bn);
    if ((p.bw * p.bh * p.bn) % 16) pick_box_pow2(PW, PH, N, &p.bw, &p.bh, &p.bn);
    p.rows = p.bw * p.bh * p.bn;
    if (p.rows % 16) return fail(FMRI_ERR_UNSUPPORTED, "wgrad pixel box %d not a multiple of 16", p.rows);
    p.tiles_x = cdiv(PW, p.bw);
    p.tiles_y = cdiv(PH, p.bh);
    p.tiles_n = cdiv(N, p.bn);
    const int NCH = (Cs % 64 == 0) ? 64 : 32;
    const int BN = (Cs % 128 == 0) ? 128 : (Cs % 64 == 0 ? 64 : 32);
    if (NCH == 32 && BN != 32) return fail(FMRI_ERR_UNSUPPORTED, "wgrad Cs=%d", Cs);
    int rc = make_act_map(&p.mapD, Dn, Cd, PW, PH, N, Cd, (long long)PW * Cd, (long long)PH * PW * Cd, 64, p.bw,
                          p.bh, p.bn);
    if (rc) return rc;
    const __nv_bfloat16* sb = reinterpret_cast<const __nv_bfloat16*>(Sh);
    if (stride == 2) {
        for (int ph = 0; ph < 2; ++ph)
            for (int pw = 0; pw < 2; ++pw) {
                const int Wp = (BW - pw + 1) / 2, Hp = (BH - ph + 1) / 2;
                rc = make_act_map(&p.mapS[ph * 2 + pw], sb + ((long long)ph * BW + pw) * Cs, Cs, Wp, Hp, N, 2LL * Cs,
                                  2LL * BW * Cs, (long long)BH * BW * Cs, NCH, p.bw, p.bh, p.bn);
                if (rc) return rc;
            }
    } else {
        rc = make_act_map(&p.mapS[0], sb, Cs, BW, BH, N, Cs, (long long)BW * Cs, (long long)BH * BW * Cs, NCH, p.bw,
                          p.bh, p.bn);
        if (rc) return rc;
    }
    p.num_taps = num_taps;
    for (int kh = 0; kh < 5; ++kh)
        for (int kw = 0; kw < 5; ++kw) {
            TapDesc& t = p.taps[kh * 5 + kw];
            if (num_taps == 1) {
                t.map = 0;
                t.dx = t.dy = 0;
            } else if (stride == 2) {
                t.map = (int16_t)((kh & 1) * 2 + (kw & 1));
                t.dy = (int16_t)((kh - 2 - (kh & 1)) / 2);
                t.dx = (int16_t)((kw - 2 - (kw & 1)) / 2);
            } else {
                t.map = 0;
                t.dy = (int16_t)(kh - 2);
                t.dx = (int16_t)(kw - 2);
            }
        }
    p.m_total = Cd;
    p.n_total = Cs;
    p.m_tiles = cdiv(Cd, 128);
    p.n_tiles = Cs / BN;
    const long long pt = (long long)p.tiles_x * p.tiles_y * p.tiles_n;
    const int tap_groups = (NCH == 32 && BN == 32 && num_taps % 5 == 0) ? num_taps / 5
                           : ((NCH == 64 && BN == 128 && num_taps > 1) ? (num_taps + 1) / 2 : num_taps);
    const long long base = (long long)tap_groups * p.m_tiles * p.n_tiles;
    p.splits = wave_splits(base, std::max<long long>(1, pt / 4));
    const long long n = (long long)num_taps * Cd * Cs;
    SCRATCH(slices, float, (long long)p.splits * n, st);   // one slice per split
    CUDA_OK(cudaMemsetAsync(slices, 0, sizeof(float) * (size_t)p.splits * n, st));
    p.out = slices;
    p.split_stride = n;
    rc = dispatch_wg(p, BN, NCH, st);
    if (rc) return rc;
    rc = ordered_add(slices, p.splits, n, ws, st);
    CUDA_OK(cudaFreeAsync(slices, st));
    return rc;
}

// ================================================================================================ conv API
extern "C" void fmri_conv_out_hw(const fmri_conv_desc* d, int* OH, int* OW) {
    if (d->transposed) {
        *OH = 2 * d->H - 1 + d->output_pad;
        *OW = 2 * d->W - 1 + d->output_pad;
    } else {
        *OH = (d->H - 1) / d->stride + 1;
        *OW = (d->W - 1) / d->stride + 1;
    }
}
static int check_conv(const fmri_conv_desc* d) {
    if (!d || d->N <= 0 || d->H <= 0 || d->W <= 0 || d->Cin <= 0 || d->Cout <= 0)
        return fail(FMRI_ERR_ARG, "bad conv descriptor");
    if (d->stride != 1 && d->stride != 2) return fail(FMRI_ERR_ARG, "conv stride must be 1 or 2");
    if (d->transposed && d->stride != 2) return fail(FMRI_ERR_ARG, "ConvTranspose2d is stride 2 only");
    if (d->dtype != FMRI_F32 && d->dtype != FMRI_BF16) return fail(FMRI_ERR_ARG, "bad dtype");
    return 0;
}
// reference-layout weight strides: Conv2d [Cout,Cin,25], ConvT [Cin,Cout,25]
static inline long long w_so(const fmri_conv_desc* d) { return d->transposed ? 25LL : 25LL * d->Cin; }
static inline long long w_si(const fmri_conv_desc* d) { return d->transposed ? 25LL * d->Cout : 25LL; }

// elements (bf16) of one pack buffer: the tap-major pack, plus the parity-merged pack when this layer has a 32-channel side
// that a scatter-form launch writes (ConvTranspose2d with Cout == 32: pack_f; stride-2 Conv2d with Cin == 32: pack_d)
extern "C" size_t fmri_conv_pack_elems(const fmri_conv_desc* d) {
    size_t n = 25 * (size_t)d->Cin * d->Cout;
    const int thin = d->transposed ? d->Cout : d->Cin;
    const int other = d->transposed ? d->Cin : d->Cout;
    if (thin == 32 && d->stride == 2) n += 9 * 128 * (size_t)other;
    return n;
}

extern "C" int fmri_conv_pack_weights(const fmri_conv_desc* d, const float* w, void* pack_f, void* pack_d,
                                      void* stream) {
    int rc = check_conv(d);
    if (rc) return rc;
    const long long n = 25LL * d->Cin * d->Cout;
    if (pack_f) {  // [tap][co][ci]
        permute4_kernel<float, __nv_bfloat16><<<grid1d(n, 256), 256, 0, S(stream)>>>(
            w, reinterpret_cast<__nv_bfloat16*>(pack_f), 1, 25, d->Cout, d->Cin, 0, 1, w_so(d), w_si(d), 0);
        LAUNCH_OK();
        if (d->transposed && d->Cout == 32 && d->stride == 2) {  // scatter-form fprop writes the 32-channel side
            __nv_bfloat16* pk = reinterpret_cast<__nv_bfloat16*>(pack_f);
            merge_pack_kernel<<<grid1d(9LL * 128 * d->Cin, 256), 256, 0, S(stream)>>>(pk, pk + n, d->Cin);
            LAUNCH_OK();
        }
    }
    if (pack_d) {  // [tap][ci][co]
        permute4_kernel<float, __nv_bfloat16><<<grid1d(n, 256), 256, 0, S(stream)>>>(
            w, reinterpret_cast<__nv_bfloat16*>(pack_d), 1, 25, d->Cin, d->Cout, 0, 1, w_si(d), w_so(d), 0);
        LAUNCH_OK();
        if (!d->transposed && d->Cin == 32 && d->stride == 2) {  // scatter-form dgrad writes the 32-channel side
            __nv_bfloat16* pk = reinterpret_cast<__nv_bfloat16*>(pack_d);
            merge_pack_kernel<<<grid1d(9LL * 128 * d->Cout, 256), 256, 0, S(stream)>>>(pk, pk + n, d->Cout);
            LAUNCH_OK();
        }
    }
    return 0;
}

template <typename T>
static int direct_conv(const fmri_conv_desc* d, bool backward, const T* in, const float* w, const float* bias, int act,
                       T* out, cudaStream_t st) {
    int OH, OW;
    fmri_conv_out_hw(d, &OH, &OW);
    DirectConvParams p;
    memset(&p, 0, sizeof(p));
    p.N = d->N;
    p.stride = d->stride;
    if (!backward) {
        p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.OH = OH; p.OW = OW; p.Cout = d->Cout;
        p.transposed = d->transposed;
        p.w_so = w_so(d);
        p.w_si = w_si(d);
    } else {  // data gradient: roles of the two grids and of the weight axes swap, gather/scatter form swaps
        p.H = OH; p.W = OW; p.Cin = d->Cout; p.OH = d->H; p.OW = d->W; p.Cout = d->Cin;
        p.transposed = !d->transposed;
        p.w_so = w_si(d);
        p.w_si = w_so(d);
    }
    p.in_sn = (long long)p.H * p.W * p.Cin; p.in_sy = (long long)p.W * p.Cin; p.in_sx = p.Cin; p.in_sc = 1;
    p.out_sn = (long long)p.OH * p.OW * p.Cout; p.out_sy = (long long)p.OW * p.Cout; p.out_sx = p.Cout; p.out_sc = 1;
    p.act = act;
    const long long total = (long long)p.N * p.OH * p.OW * p.Cout;
    direct_conv_kernel<T, T><<<grid1d(total, 256, 148 * 32), 256, 0, st>>>(in, w, bias, out, p);
    LAUNCH_OK();
    return 0;
}

extern "C" int fmri_conv_fprop(const fmri_conv_desc* d, const void* x, const float* w, const void* pack_f,
                               const float* bias, int act, void* y, double* stat_sum, double* stat_sq,
                               void* stream) {
    int rc = check_conv(d);
    if (rc) return rc;
    int OH, OW;
    fmri_conv_out_hw(d, &OH, &OW);
    if (stat_sum) {
        CUDA_OK(cudaMemsetAsync(stat_sum, 0, sizeof(double) * d->Cout, S(stream)));
        CUDA_OK(cudaMemsetAsync(stat_sq, 0, sizeof(double) * d->Cout, S(stream)));
    }
    if (d->dtype == FMRI_BF16) {
        if (!pack_f) return fail(FMRI_ERR_ARG, "bf16 conv needs the packed weights");
        if (d->transposed)   // bias / act: the BatchNorm-folded inference forward (fmri_bn_fold)
            return run_scatter(x, d->N, d->H, d->W, d->Cin, OH, OW, d->Cout, pack_f, y, stat_sum, stat_sq, S(stream), nullptr,
                               bias, act);
        return run_gather(x, d->N, d->H, d->W, d->Cin, OH, OW, d->Cout, d->stride, pack_f, bias, act, y, 0, stat_sum,
                          stat_sq, S(stream));
    }
    rc = direct_conv<float>(d, false, reinterpret_cast<const float*>(x), w, bias, act, reinterpret_cast<float*>(y),
                            S(stream));
    if (rc) return rc;
    if (stat_sum) return fmri_colstats(y, FMRI_F32, (long long)d->N * OH * OW, d->Cout, stat_sum, stat_sq, stream);
    return 0;
}

extern "C" int fmri_conv_dgrad(const fmri_conv_desc* d, const void* dy, const float* w, const void* pack_d, void* dx,
                               const fmri_relu_mask* mask, void* stream) {
    int rc = check_conv(d);
    if (rc) return rc;
    if (mask && !mask->y) return fail(FMRI_ERR_ARG, "conv dgrad: the ReLU mask needs y");
    int OH, OW;
    fmri_conv_out_hw(d, &OH, &OW);
    const long long n_in = (long long)d->N * d->H * d->W * d->Cin;
    if (d->dtype == FMRI_BF16) {
        if (!pack_d) return fail(FMRI_ERR_ARG, "bf16 conv dgrad needs the packed weights");
        fmri_relu_mask m;
        if (mask) {
            m.y = mask->y;
            m.bits = d->Cin == 32 ? mask->bits : nullptr;   // bit words describe 32-channel pixels only
        }
        if (d->transposed)  // gather over dy at stride 2
            rc = run_gather(dy, d->N, OH, OW, d->Cout, d->H, d->W, d->Cin, 2, pack_d, nullptr, 0, dx, 0, nullptr, nullptr,
                            S(stream), mask ? &m : nullptr);
        else if (d->stride == 2)
            rc = run_scatter(dy, d->N, OH, OW, d->Cout, d->H, d->W, d->Cin, pack_d, dx, nullptr, nullptr, S(stream),
                             mask ? &m : nullptr);
        else
            return fail(FMRI_ERR_UNSUPPORTED, "stride-1 conv dgrad on the tensor path");
        if (rc) return rc;
        if (mask && !g_last_ig_was_persistent) {  // small launch (one tile per CTA kernel, no fused mask): mask dx in place
            relu_bwd_kernel<__nv_bfloat16><<<grid1d((n_in + 7) / 8, 256, 148 * 8), 256, 0, S(stream)>>>(
                reinterpret_cast<const __nv_bfloat16*>(mask->y), reinterpret_cast<const __nv_bfloat16*>(dx),
                reinterpret_cast<__nv_bfloat16*>(dx), n_in);
            LAUNCH_OK();
        }
        return 0;
    }
    rc = direct_conv<float>(d, true, reinterpret_cast<const float*>(dy), w, nullptr, 0, reinterpret_cast<float*>(dx),
                            S(stream));
    if (rc) return rc;
    if (mask) {
        relu_bwd_kernel<float><<<grid1d((n_in + 7) / 8, 256, 148 * 8), 256, 0, S(stream)>>>(
            reinterpret_cast<const float*>(mask->y), reinterpret_cast<const float*>(dx), reinterpret_cast<float*>(dx), n_in);
        LAUNCH_OK();
    }
    return 0;
}

extern "C" size_t fmri_conv_wgrad_workspace(const fmri_conv_desc* d) {
    return d->dtype == FMRI_BF16 ? sizeof(float) * 25 * (size_t)d->Cin * d->Cout : 0;
}

extern "C" int fmri_conv_wgrad(const fmri_conv_desc* d, const void* x, const void* dy, float* dw, int accumulate,
                               void* ws, size_t ws_bytes, void* stream) {
    int rc = check_conv(d);
    if (rc) return rc;
    int OH, OW;
    fmri_conv_out_hw(d, &OH, &OW);
    if (d->dtype == FMRI_BF16) {
        const size_t need = fmri_conv_wgrad_workspace(d);
        if (!ws || ws_bytes < need) return fail(FMRI_ERR_WORKSPACE, "conv wgrad workspace %zu < %zu", ws_bytes, need);
        if (d->stride != 2) return fail(FMRI_ERR_UNSUPPORTED, "stride-1 conv wgrad on the tensor path");
        CUDA_OK(cudaMemsetAsync(ws, 0, need, S(stream)));
        float* wsf = reinterpret_cast<float*>(ws);
        int Cd, Cs;
        if (!d->transposed) {  // dense = dy [N,OH,OW,Cout], shifted = x [N,H,W,Cin]
            Cd = d->Cout; Cs = d->Cin;
            rc = run_wgrad_tc(dy, d->N, OH, OW, Cd, x, d->H, d->W, Cs, 2, 25, wsf, S(stream));
        } else {  // dense = x [N,H,W,Cin], shifted = dy [N,OH,OW,Cout]
            Cd = d->Cin; Cs = d->Cout;
            rc = run_wgrad_tc(x, d->N, d->H, d->W, Cd, dy, OH, OW, Cs, 2, 25, wsf, S(stream));
        }
        if (rc) return rc;
        // ws[tap][m][n] -> dw[m][n][tap]
        const long long n = 25LL * Cd * Cs;
        scatter4_kernel<float, float><<<grid1d(n, 256), 256, 0, S(stream)>>>(wsf, dw, 1, 25, Cd, Cs, 0, 1, 25LL * Cs,
                                                                            25, accumulate);
        LAUNCH_OK();
        return 0;
    }
    DirectWgradParams p;
    memset(&p, 0, sizeof(p));
    p.N = d->N;
    p.stride = d->stride;
    p.accumulate = accumulate;
    const float *A, *B;
    if (!d->transposed) {
        A = reinterpret_cast<const float*>(dy); p.PH = OH; p.PW = OW; p.Ca = d->Cout;
        B = reinterpret_cast<const float*>(x); p.BH = d->H; p.BW = d->W; p.Cb = d->Cin;
    } else {
        A = reinterpret_cast<const float*>(x); p.PH = d->H; p.PW = d->W; p.Ca = d->Cin;
        B = reinterpret_cast<const float*>(dy); p.BH = OH; p.BW = OW; p.Cb = d->Cout;
    }
    p.a_sn = (long long)p.PH * p.PW * p.Ca; p.a_sy = (long long)p.PW * p.Ca; p.a_sx = p.Ca; p.a_sc = 1;
    p.b_sn = (long long)p.BH * p.BW * p.Cb; p.b_sy = (long long)p.BW * p.Cb; p.b_sx = p.Cb; p.b_sc = 1;
    p.w_sa = 25LL * p.Cb;
    p.w_sb = 25;
    direct_wgrad_kernel<float, float><<<25 * p.Ca * p.Cb, 128, 0, S(stream)>>>(A, B, dw, p);
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ edge convs
// workspace of the edge convolutions: fp32 [75][C] staging of the CUDA-core kernels, or (tensor-core path) a 64 KB region for
// the bf16 weight slab pack followed by the 3-channel image(s) repacked as bf16 NHWC with 8 channels (16 B per pixel)
static const size_t HC_WS_PACK = 65536;
extern "C" size_t fmri_edge_workspace(const fmri_edge_desc* d) {
    return std::max(sizeof(float) * 75 * (size_t)d->C, HC_WS_PACK + (size_t)d->N * d->H * d->W * 16);
}

// ---- halo-tile tcgen05 convolution (hconv_kernels.cuh): plan + launch -------------------------------------------------
// Builds the tile geometry, the MMA step list and the weight-pack spec for a 5x5 convolution read in gather form from an
// NHWC bf16 input with 8*chunks channels. stride 1: one halo plane; stride 2: four stride-parity planes.
// chunks >= 2: one step per (tap, 16-channel pair of slabs). chunks == 1 (3-channel image padded to 8): one step per PAIR of
// taps (the two K halves of the MMA are two different windows of the same slab).
// Returns false when the shape does not fit (caller falls back to the CUDA-core kernels).
static bool hc_build(HcParams& p, HcPackSpec& spec, int N, int H, int W, int chunks, int stride, int OH, int OW, int BN,
                     bool flip) {
    memset(&p, 0, sizeof(p));
    memset(&spec, 0, sizeof(spec));
    p.N = N; p.H = H; p.W = W; p.chunks = chunks; p.OH = OH; p.OW = OW;
    const int hx = stride == 1 ? 4 : 2;  // halo (columns = rows)
    if (stride == 1) {
        p.num_planes = 1;
        p.pl_ys[0] = p.pl_xs[0] = 1;
        p.pl_yoff[0] = p.pl_xoff[0] = -2;
    } else {
        p.num_planes = 4;
        for (int ph = 0; ph < 2; ++ph)
            for (int pw = 0; pw < 2; ++pw) {
                const int pl = ph * 2 + pw;
                p.pl_ys[pl] = p.pl_xs[pl] = 2;
                p.pl_yoff[pl] = ph - 2;   // halo row sy = 0 is output row offset -1 of this parity plane
                p.pl_xoff[pl] = pw - 2;
            }
    }
    p.PW = OW + hx;
    if (p.PW > 200) return false;
    // Every role of the kernel is a latency-bound single-warp chain (ncu: ~11 cycles per issued instruction per warp), so two
    // co-resident CTAs per SM nearly double the throughput: prefer a plan with <= 256 TMEM columns and <= 110 KB of shared
    // memory; fall back to one big CTA per SM.
    const int max_off = hx * p.PW + hx;
    const int nsteps = chunks >= 2 ? 25 * (chunks / 2) : 13;
    if (nsteps > HC_MAX_STEPS) return false;
    p.num_steps = nsteps;
    // Plan search: rows per tile THt (any value, ragged last tile allowed) maximising the useful fraction of the computed
    // 128-row sub-tiles, first among plans that keep two CTAs per SM (<= 256 TMEM columns, <= 110 KB smem), else one CTA.
    // Windows of dropped rows may run past the last slab into whatever shared memory follows (weights, barriers): those rows
    // only produce dropped outputs, so the slab is allocated for the halo alone.
    bool found = false;
    for (int pass = 0; pass < 2 && !found; ++pass) {
        const int mt_max = std::min(5, (pass == 0 ? 128 : 256) / BN);
        const size_t smem_cap = pass == 0 ? 110 * 1024 : 227 * 1024;
        double best = 0.0;
        for (int tht = std::min(OH, (mt_max * 128) / p.PW); tht >= 1; --tht) {
            HcParams q = p;
            q.THt = tht;
            q.tiles_y = cdiv(OH, tht);
            q.MT = cdiv((long long)tht * q.PW, 128);
            q.PH = tht + hx;
            // rows per channel-chunk slab. With several chunks a producer warp writes lanes (chunk j, pixel r) -> j * slab +
            // r * 16 B; a slab size that is a multiple of 128 B puts all chunks of a pixel on the same banks (ncu: 49
            // shared-memory wavefronts per cp.async instruction instead of 4), so the slab is padded to 32 B mod 128 B.
            q.slab_rows = (q.PH * q.PW + 7) / 8 * 8 + (chunks > 1 ? 2 : 0);
            // the overshoot of the last sub-tile's windows must stay inside the CTA's allocation (it lands in the weight slab)
            const long long overshoot = ((long long)q.MT * 128 + max_off + 1 - q.slab_rows) * 16;
            if (overshoot > 0 && overshoot > hc_b_bytes(q, BN)) continue;
            if ((size_t)hc_smem_bytes(q, BN) > smem_cap) continue;
            const double eff = (double)OH * OW / ((double)q.tiles_y * q.MT * 128);
            if (eff > best + 1e-9) { best = eff; p = q; found = true; }
        }
    }
    if (!found) return false;
    // window offset of every filter tap, in 16-byte rows from the start of a halo buffer
    int woff[25];
    for (int kh = 0; kh < 5; ++kh)
        for (int kw = 0; kw < 5; ++kw) {
            int plane = 0, dyr = kh, dxr = kw;
            if (stride == 2) {
                plane = (kh & 1) * 2 + (kw & 1);
                dyr = (kh - 2 - (kh & 1)) / 2 + 1;
                dxr = (kw - 2 - (kw & 1)) / 2 + 1;
            }
            woff[kh * 5 + kw] = plane * chunks * p.slab_rows + dyr * p.PW + dxr;
        }
    int s = 0;
    if (chunks >= 2) {
        for (int tp = 0; tp < 25; ++tp)
            for (int j = 0; j < chunks / 2; ++j, ++s) {
                p.steps[s].a_off = woff[tp] + 2 * j * p.slab_rows;
                p.steps[s].a_lbo = p.slab_rows;
                p.steps[s].b_off = s * BN;
                spec.tap[s][0] = spec.tap[s][1] = (int16_t)(flip ? 24 - tp : tp);
                spec.cb[s][0] = (int16_t)(16 * j);
                spec.cb[s][1] = (int16_t)(16 * j + 8);
            }
    } else {
        int order[25];
        for (int i = 0; i < 25; ++i) order[i] = i;
        std::sort(order, order + 25, [&](int a, int b) { return woff[a] < woff[b]; });
        // 25 taps = 1 single + 12 pairs. The single is the tap with the SMALLEST window offset: its zero-weight second K half
        // reads the window one row further, which is still inside the halo. (Pairing it at the far end would read one row
        // past the initialised halo, and 0-weight x NaN-garbage = NaN.)
        {
            const int t0 = order[0];
            p.steps[s].a_off = woff[t0];
            p.steps[s].a_lbo = 1;
            p.steps[s].b_off = s * BN;
            spec.tap[s][0] = (int16_t)(flip ? 24 - t0 : t0);
            spec.tap[s][1] = -1;
            spec.cb[s][0] = spec.cb[s][1] = 0;
            ++s;
        }
        for (int i = 1; i < 25; i += 2, ++s) {
            const int t0 = order[i], t1 = order[i + 1];
            p.steps[s].a_off = woff[t0];
            p.steps[s].a_lbo = woff[t1] - woff[t0];
            p.steps[s].b_off = s * BN;
            spec.tap[s][0] = (int16_t)(flip ? 24 - t0 : t0);
            spec.tap[s][1] = (int16_t)(flip ? 24 - t1 : t1);
            spec.cb[s][0] = spec.cb[s][1] = 0;
            if (p.steps[s].a_lbo == 0) return false;
        }
    }
    return true;
}

template <int BN>
static int hc_launch(const HcParams& p_in, cudaStream_t st) {
    HcParams p = p_in;
    static int skip = -1;
    if (skip < 0) {
        const char* e = getenv("FMRI_HC_SKIP");
        skip = e ? atoi(e) : 0;
    }
    p.skip = skip;
    const int smem = hc_smem_bytes(p, BN);
    static int attr_smem = 0;
    if (smem > attr_smem) {
        CUDA_OK(cudaFuncSetAttribute(hconv_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_smem = smem;
    }
    const int total_tiles = p.N * p.tiles_y;
    int tmem = 32;
    while (tmem < 2 * p.MT * BN) tmem <<= 1;
    const int per_sm = std::max(1, std::min(std::min(2, 512 / tmem), (227 * 1024) / smem));
    const int grid = std::min(total_tiles, 148 * per_sm);
    hconv_kernel<BN><<<grid, HC_THREADS, smem, st>>>(p);
    LAUNCH_OK();
    return 0;
}
static int hc_run(HcParams& p, const HcPackSpec& spec, int BN, const float* w, int n_real, int c_real, long long s_n,
                  long long s_c, void* ws, cudaStream_t st) {
    p.Bslab = reinterpret_cast<const __nv_bfloat16*>(ws);
    if ((size_t)hc_b_bytes(p, BN) > HC_WS_PACK) return fail(FMRI_ERR_WORKSPACE, "hconv weight pack exceeds its workspace region");
    hc_pack_weights_kernel<<<cdiv(2LL * p.num_steps * BN * 8, 256), 256, 0, st>>>(
        w, reinterpret_cast<__nv_bfloat16*>(ws), spec, p.num_steps, BN, n_real, c_real, s_n, s_c);
    LAUNCH_OK();
    switch (BN) {
        case 16: return hc_launch<16>(p, st);
        case 32: return hc_launch<32>(p, st);
        case 64: return hc_launch<64>(p, st);
    }
    return fail(FMRI_ERR_UNSUPPORTED, "hconv BN=%d", BN);
}

// C -> 3 convolution as one GEMM per 128-pixel chunk + shift-and-add gather (cto3_kernels.cuh): C = 32, W = 64, enough images
// to give every SM whole images. Returns 1 when the shape does not fit (caller falls back to the halo-tile kernel).
static int cto3_run(const void* X, int N, int H, int W, int C, const float* w, long long s_co, long long s_c, int flip,
                    const float* bias, int act, float* img, void* ws, cudaStream_t st) {
    if (C != 32 || W != C3_W || H < 3 || N < 74) return 1;
    C3Params p;
    memset(&p, 0, sizeof(p));
    __nv_bfloat16* wt = reinterpret_cast<__nv_bfloat16*>(ws);
    c3_pack_weights_kernel<<<cdiv(C3_NB * C, 256), 256, 0, st>>>(w, wt, s_co, s_c, flip, C);
    LAUNCH_OK();
    if (make_act_map(&p.mapX, X, C, H * W, 1, N, C, (long long)H * W * C, (long long)H * W * C, C, 128, 1, 1)) return 1;
    {
        const long long dims[2] = {C, C3_NB};
        const long long stv[1] = {C};
        const int box[2] = {C, C3_NB};
        if (make_map(&p.mapW, wt, 2, dims, stv, box, C * 2)) return 1;
    }
    p.N = N; p.H = H; p.out = img; p.bias = bias; p.act = act;
    static bool attr_done = false;
    if (!attr_done) {
        CUDA_OK(cudaFuncSetAttribute(cto3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, C3_SMEM));
        attr_done = true;
    }
    cto3_kernel<<<std::min(N, 148), C3_THREADS, C3_SMEM, st>>>(p);
    LAUNCH_OK();
    return 0;
}

// C -> 3 convolution, stride 1: img[n,co,y,x] = act(bias + sum_{taps,c} X[n,y+kh-2,x+kw-2,c] * w[co*s_co + c*s_c + tap]);
// flip uses tap 24-tap (data gradient of a 3 -> C convolution). Returns 1 when the shape does not fit (fall back).
static int hconv_c_to_3(const void* X, int N, int H, int W, int C, const float* w, long long s_co, long long s_c, int flip,
                        const float* bias, int act, float* img, void* ws, cudaStream_t st) {
    if (C != 32 && C != 64) return 1;
    {
        const int rc = cto3_run(X, N, H, W, C, w, s_co, s_c, flip, bias, act, img, ws, st);
        if (rc <= 0) return rc;
    }
    HcParams p;
    HcPackSpec spec;
    if (!hc_build(p, spec, N, H, W, C / 8, 1, H, W, 16, flip != 0)) return 1;
    p.X = reinterpret_cast<const __nv_bfloat16*>(X);
    p.epi = 0; p.out = img; p.bias = bias; p.act = act; p.n_out = 3;
    return hc_run(p, spec, 16, w, 3, C, s_co, s_c, ws, st);
}

// 3 -> C convolution (stride 1 or 2) from up to three fp32 NCHW image sources: y[n,oy,ox,c] = act(bias[c] + sum_{taps,ci<3}
// img[n,ci,oy*s+kh-2,ox*s+kw-2] * w[c*s_c + ci*s_ci + tap]); the images are first repacked to bf16 NHWC-8 in the workspace.
static int hconv_3_to_c(const float* i0, const float* i1, const float* i2, int nps, int N, int H, int W, int C, int stride,
                        const float* w, long long s_c, long long s_ci, int flip, const float* bias, int act, void* y,
                        void* ws, cudaStream_t st) {
    if (C != 32 && C != 64) return 1;
    const int OH = (H - 1) / stride + 1, OW = (W - 1) / stride + 1;
    HcParams p;
    HcPackSpec spec;
    if (!hc_build(p, spec, N, H, W, 1, stride, OH, OW, C, flip != 0)) return 1;
    __nv_bfloat16* img8 = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<uint8_t*>(ws) + HC_WS_PACK);
    img8_pack_kernel<<<grid1d((long long)N * H * W, 256), 256, 0, st>>>(i0, i1, i2, nps, N, (long long)H * W, img8);
    LAUNCH_OK();
    p.X = img8;
    p.epi = 1; p.out = y; p.bias = bias; p.act = act; p.n_out = C;
    return hc_run(p, spec, C, w, C, 3, s_c, s_ci, ws, st);
}

// Edge-conv weight gradient on tcgen05 (hwgrad_kernels.cuh), stride 1. T: [N,PH,PW,C] bf16 NHWC; the 3-channel side comes as
// up to three fp32 NCHW sources and is repacked to NHWC-8 in the workspace. dwk: fp32 [75][C] (zeroed by the caller).
// Returns 1 when the shape does not fit (caller falls back to the CUDA-core kernel).
// plane < 0: stride-1 convolution (images packed here). plane = ph * 2 + pw: one stride-parity plane of a stride-2 convolution --
// (IH, IW) is the image, (PH, PW) the T grid = the conv output; see HwParams::plane.
static int hwgrad_run(const void* T, const float* i0, const float* i1, const float* i2, int nps, int N, int PH, int PW, int C,
                      float* dwk, float* dbias, int flip, void* ws, cudaStream_t st, int plane = -1, int IH = 0, int IW = 0) {
    if (C != 32 && C != 64) return 1;
    HwParams p;
    memset(&p, 0, sizeof(p));
    p.N = N; p.PH = PH; p.PW = PW; p.C = C;
    p.PWp = (PW + 4 + 15) / 16 * 16;
    if (p.PWp > 128) return 1;
    // tile rows: every tile re-stages bh + 4 image rows for bh output rows, so taller tiles cut the halo traffic that bounds
    // this kernel reads (5x at bh = 1, 3x at 2, 2.3x at 3) -- which turned out NOT to be its bound; rows = bh * PWp <= 256
    // (ones slab). A ragged last tile is fine: TMA zero-fills the T rows below the image.
    const int bh_cap = 2;  // measured: bh = 2 is 0-3 % faster than 1; bh = 3 needs one CTA per SM and is 10 % slower
    p.bh = std::max(1, std::min(std::min(PH, bh_cap), 256 / p.PWp));
    p.tiles_y = cdiv(PH, p.bh);
    p.slab_rows = ((p.bh + 4) * p.PWp + 16 + 7) / 8 * 8;
    p.d_chunk = (p.bh * p.PWp * 128 + 1023) / 1024 * 1024;
    p.stages = 2;
    if (hw_smem_bytes(p) > 227 * 1024) return 1;
    while (p.stages < HW_MAX_STAGES) {  // two co-resident CTAs per SM (each role is a latency-bound single-warp chain)
        ++p.stages;
        if (hw_smem_bytes(p) > 110 * 1024) { --p.stages; break; }
    }
    const long long dims[4] = {C, PW, PH, N};
    const long long strides[3] = {C, (long long)PW * C, (long long)PH * PW * C};
    const int box[4] = {64, p.PWp, p.bh, 1};
    if (make_map(&p.mapT, T, 4, dims, strides, box, 128)) return 1;  // e.g. a box the driver rejects: CUDA-core fallback
    __nv_bfloat16* img8 = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<uint8_t*>(ws) + HC_WS_PACK);
    p.kh0 = 0; p.nkh = 5;
    if (plane < 0) {
        img8_pack_kernel<<<grid1d((long long)N * PH * PW, 256), 256, 0, st>>>(i0, i1, i2, nps, N, (long long)PH * PW, img8);
    } else {
        p.plane = 1; p.ph = plane >> 1; p.pw = plane & 1;
        p.kh0 = 1; p.nkh = p.ph ? 2 : 3;      // virtual filter rows kh5 = a + 1 with real kh = 2 a + ph <= 4
        img8_plane_pack_kernel<<<grid1d((long long)N * PH * PW, 256), 256, 0, st>>>(i0, i1, i2, nps, N, IH, IW, PH, PW, p.ph,
                                                                                   p.pw, img8);
    }
    LAUNCH_OK();
    p.img8 = img8;
    p.dwk = dwk; p.dbias = dbias; p.flip = flip;
    const int smem = hw_smem_bytes(p);
    static int attr_smem = 0;
    if (smem > attr_smem) {
        CUDA_OK(cudaFuncSetAttribute(hwgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr_smem = smem;
    }
    const int total = N * p.tiles_y;
    const int nb = std::min(total, 148 * (smem <= 110 * 1024 ? 2 : 1));
    const long long nw = 75LL * C;
    SCRATCH(part, float, (long long)nb * (nw + C), st);   // one [75][C] (+ [C] bias) slice per persistent CTA
    CUDA_OK(cudaMemsetAsync(part, 0, sizeof(float) * (size_t)nb * (nw + C), st));
    p.dwk = part;
    p.dbias = dbias ? part + nb * nw : nullptr;
    hwgrad_kernel<<<nb, HW_THREADS, smem, st>>>(p);
    LAUNCH_OK();
    int rc = ordered_add(part, nb, nw, dwk, st);
    if (!rc && dbias) rc = ordered_add(part + nb * nw, nb, C, dbias, st);
    CUDA_OK(cudaFreeAsync(part, st));
    return rc;
}

static int check_edge(const fmri_edge_desc* d, const void* ws, size_t ws_bytes) {
    if (!d || (d->C != 32 && d->C != 64)) return fail(FMRI_ERR_UNSUPPORTED, "edge conv supports C in {32,64}");
    if (d->stride != 1 && d->stride != 2) return fail(FMRI_ERR_ARG, "edge stride");
    if (!ws || ws_bytes < fmri_edge_workspace(d)) return fail(FMRI_ERR_WORKSPACE, "edge workspace too small");
    return 0;
}
// "in" conv weight [C,3,25] -> wk[(ci*25+tap)*C + c]
static int pack_edge_in(const fmri_edge_desc* d, const float* w, float* wk, cudaStream_t st) {
    permute4_kernel<float, float><<<grid1d(75LL * d->C, 256), 256, 0, st>>>(w, wk, 1, 3, 25, d->C, 0, 25, 1, 75, 0);
    LAUNCH_OK();
    return 0;
}
// "out" conv weight [3,C,25] -> wk[(co*25+tap)*C + c] (flip: tap -> 24-tap)
static int pack_edge_out(const fmri_edge_desc* d, const float* w, float* wk, int flip, cudaStream_t st) {
    permute4_kernel<float, float><<<grid1d(75LL * d->C, 256), 256, 0, st>>>(
        flip ? w + 24 : w, wk, 1, 3, 25, d->C, 0, 25LL * d->C, flip ? -1 : 1, 25, 0);
    LAUNCH_OK();
    return 0;
}
template <int C>
static int edge_in_fprop_t(const fmri_edge_desc* d, const float* i0, const float* i1, const float* i2, int nps,
                           const float* wk, const float* bias, int act, void* y, int OH, int OW, cudaStream_t st) {
    const long long pix = (long long)d->N * OH * OW;
    if (d->dtype == FMRI_BF16)
        edge3_to_c_kernel<C, __nv_bfloat16><<<cdiv(pix, 128), 128, 0, st>>>(
            i0, i1, i2, nps, wk, bias, reinterpret_cast<__nv_bfloat16*>(y), d->N, d->H, d->W, OH, OW, d->stride, act);
    else
        edge3_to_c_kernel<C, float><<<cdiv(pix, 128), 128, 0, st>>>(i0, i1, i2, nps, wk, bias,
                                                                   reinterpret_cast<float*>(y), d->N, d->H, d->W, OH,
                                                                   OW, d->stride, act);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_edge_in_fprop(const fmri_edge_desc* d, const float* img0, const float* img1, const float* img2,
                                  int n_per_src, const float* w, const float* bias, int act, void* y, void* ws,
                                  size_t ws_bytes, void* stream) {
    int rc = check_edge(d, ws, ws_bytes);
    if (rc) return rc;
    if (!img1) img1 = img0;
    if (!img2) img2 = img0;
    if (d->dtype == FMRI_BF16 && fmri_tensor_path_available()) {
        // w layout [C][3][25]: y[.., c] = sum img[ci] * w[c*75 + ci*25 + tap]
        rc = hconv_3_to_c(img0, img1, img2, n_per_src, d->N, d->H, d->W, d->C, d->stride, w, 75, 25, 0, bias, act, y, ws,
                          S(stream));
        if (rc <= 0) return rc;
    }
    float* wk = reinterpret_cast<float*>(ws);
    rc = pack_edge_in(d, w, wk, S(stream));
    if (rc) return rc;
    const int OH = (d->H - 1) / d->stride + 1, OW = (d->W - 1) / d->stride + 1;
    return d->C == 32 ? edge_in_fprop_t<32>(d, img0, img1, img2, n_per_src, wk, bias, act, y, OH, OW, S(stream))
                      : edge_in_fprop_t<64>(d, img0, img1, img2, n_per_src, wk, bias, act, y, OH, OW, S(stream));
}
template <int C>
static int edge_to3_t(int dtype, const void* in, const float* wk, const float* bias, float* img, int N, int IH, int IW,
                      int OH, int OW, int stride_up, int flip, int act, cudaStream_t st) {
    const long long pix = (long long)N * OH * OW;
    if (dtype == FMRI_BF16)
        edgec_to_3_kernel<C, __nv_bfloat16><<<cdiv(pix, 128), 128, 0, st>>>(
            reinterpret_cast<const __nv_bfloat16*>(in), wk, bias, img, N, IH, IW, OH, OW, stride_up, flip, act, 0);
    else
        edgec_to_3_kernel<C, float><<<cdiv(pix, 128), 128, 0, st>>>(reinterpret_cast<const float*>(in), wk, bias, img,
                                                                   N, IH, IW, OH, OW, stride_up, flip, act, 0);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_edge_in_dgrad(const fmri_edge_desc* d, const void* dy, const float* w, float* dimg, void* ws,
                                  size_t ws_bytes, void* stream) {
    int rc = check_edge(d, ws, ws_bytes);
    if (rc) return rc;
    const int OH = (d->H - 1) / d->stride + 1, OW = (d->W - 1) / d->stride + 1;
    if (d->dtype == FMRI_BF16 && d->stride == 1 && fmri_tensor_path_available()) {
        // dimg[n,ci,y,x] = sum dy[n,y+kh-2,x+kw-2,c] * w[c][ci][24-tap]  (w layout [C][3][25])
        rc = hconv_c_to_3(dy, d->N, d->H, d->W, d->C, w, 25, 75, 1, nullptr, 0, dimg, ws, S(stream));
        if (rc <= 0) return rc;
    }
    float* wk = reinterpret_cast<float*>(ws);
    rc = pack_edge_in(d, w, wk, S(stream));
    if (rc) return rc;
    // image pixel gathers from the C-side grid (OH,OW); stride 1: flipped taps, stride 2: divisibility form
    const int flip = d->stride == 1 ? 1 : 0;
    return d->C == 32 ? edge_to3_t<32>(d->dtype, dy, wk, nullptr, dimg, d->N, OH, OW, d->H, d->W, d->stride, flip, 0,
                                       S(stream))
                      : edge_to3_t<64>(d->dtype, dy, wk, nullptr, dimg, d->N, OH, OW, d->H, d->W, d->stride, flip, 0,
                                       S(stream));
}
template <int C>
static int edge_wgrad_t(int dtype, const void* T, const float* i0, const float* i1, const float* i2, int nps,
                        float* dwk, float* dbias, int N, int PH, int PW, int IH, int IW, int stride, int sg,
                        cudaStream_t st) {
    if (PW <= 128 && (PW - 1) * stride + 5 <= 144) {
        const long long lines = (long long)N * PH;
        const int rpb = (int)std::max<long long>(1, (lines + 148 * 3 - 1) / (148 * 3));
        const int blocks = cdiv(lines, rpb);
        if (dtype == FMRI_BF16)
            edge_wgrad_rows_kernel<C, __nv_bfloat16><<<blocks, 256, 0, st>>>(
                reinterpret_cast<const __nv_bfloat16*>(T), i0, i1, i2, nps, dwk, dbias, N, PH, PW, IH, IW, stride, sg, rpb);
        else
            edge_wgrad_rows_kernel<C, float><<<blocks, 256, 0, st>>>(reinterpret_cast<const float*>(T), i0, i1, i2, nps,
                                                                    dwk, dbias, N, PH, PW, IH, IW, stride, sg, rpb);
        LAUNCH_OK();
        return 0;
    }
    if (dbias) return fail(FMRI_ERR_UNSUPPORTED, "edge wgrad: fused bias gradient needs rows of <= 128 pixels");
    const long long pix = (long long)N * PH * PW;
    int ppb = (int)std::max<long long>(64, ((pix + 148 * 4 - 1) / (148 * 4) + 7) / 8 * 8);
    const int blocks = cdiv(pix, ppb);
    if (dtype == FMRI_BF16)
        edge_wgrad_kernel<C, __nv_bfloat16><<<blocks, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(T), i0, i1,
                                                                    i2, nps, dwk, N, PH, PW, IH, IW, stride, sg, ppb);
    else
        edge_wgrad_kernel<C, float><<<blocks, 256, 0, st>>>(reinterpret_cast<const float*>(T), i0, i1, i2, nps, dwk, N,
                                                            PH, PW, IH, IW, stride, sg, ppb);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_edge_in_wgrad(const fmri_edge_desc* d, const float* img0, const float* img1, const float* img2,
                                  int n_per_src, const void* dy, float* dw, float* dbias, int accumulate, void* ws,
                                  size_t ws_bytes, void* stream) {
    int rc = check_edge(d, ws, ws_bytes);
    if (rc) return rc;
    float* dwk = reinterpret_cast<float*>(ws);
    CUDA_OK(cudaMemsetAsync(dwk, 0, sizeof(float) * 75 * (size_t)d->C, S(stream)));
    const int OH = (d->H - 1) / d->stride + 1, OW = (d->W - 1) / d->stride + 1;
    if (!img1) img1 = img0;
    if (!img2) img2 = img0;
    if (dbias && !accumulate) CUDA_OK(cudaMemsetAsync(dbias, 0, sizeof(float) * d->C, S(stream)));
    rc = 1;
    if (d->dtype == FMRI_BF16 && d->stride == 1 && fmri_tensor_path_available())
        rc = hwgrad_run(dy, img0, img1, img2, n_per_src, d->N, d->H, d->W, d->C, dwk, dbias, 0, ws, S(stream));
    else if (d->dtype == FMRI_BF16 && d->stride == 2 && !dbias && fmri_tensor_path_available()) {
        // stride 2 (Encoder.conv[0], vae_gan.py:74): four stride-parity planes of the image, each a unit-shift problem
        for (int plane = 0; plane < 4; ++plane) {
            rc = hwgrad_run(dy, img0, img1, img2, n_per_src, d->N, OH, OW, d->C, dwk, nullptr, 0, ws, S(stream), plane, d->H, d->W);
            if (rc) break;
        }
        if (rc == 1) CUDA_OK(cudaMemsetAsync(dwk, 0, sizeof(float) * 75 * (size_t)d->C, S(stream)));   // partial planes: start over
    }
    if (rc == 1)
        rc = d->C == 32 ? edge_wgrad_t<32>(d->dtype, dy, img0, img1, img2, n_per_src, dwk, dbias, d->N, OH, OW, d->H, d->W,
                                           d->stride, 1, S(stream))
                        : edge_wgrad_t<64>(d->dtype, dy, img0, img1, img2, n_per_src, dwk, dbias, d->N, OH, OW, d->H, d->W,
                                           d->stride, 1, S(stream));
    if (rc) return rc;
    // dwk[(ci*25+tap)*C + c] -> dw[c][ci][tap]
    scatter4_kernel<float, float><<<grid1d(75LL * d->C, 256), 256, 0, S(stream)>>>(dwk, dw, 1, 3, 25, d->C, 0, 25, 1,
                                                                                  75, accumulate);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_edge_out_fprop(const fmri_edge_desc* d, const void* x, const float* w, const float* bias, int act,
                                   float* img, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_edge(d, ws, ws_bytes);
    if (rc) return rc;
    if (d->stride != 1) return fail(FMRI_ERR_UNSUPPORTED, "edge out conv is stride 1");
    if (d->dtype == FMRI_BF16 && fmri_tensor_path_available()) {
        // w layout [3][C][25]
        rc = hconv_c_to_3(x, d->N, d->H, d->W, d->C, w, 25LL * d->C, 25, 0, bias, act, img, ws, S(stream));
        if (rc <= 0) return rc;
    }
    float* wk = reinterpret_cast<float*>(ws);
    rc = pack_edge_out(d, w, wk, 0, S(stream));
    if (rc) return rc;
    return d->C == 32
               ? edge_to3_t<32>(d->dtype, x, wk, bias, img, d->N, d->H, d->W, d->H, d->W, 1, 0, act, S(stream))
               : edge_to3_t<64>(d->dtype, x, wk, bias, img, d->N, d->H, d->W, d->H, d->W, 1, 0, act, S(stream));
}
extern "C" int fmri_edge_out_dgrad(const fmri_edge_desc* d, const float* dimg, const float* w, void* dx, void* ws,
                                   size_t ws_bytes, void* stream) {
    int rc = check_edge(d, ws, ws_bytes);
    if (rc) return rc;
    if (d->stride != 1) return fail(FMRI_ERR_UNSUPPORTED, "edge out conv is stride 1");
    if (d->dtype == FMRI_BF16 && fmri_tensor_path_available()) {
        // w layout [3][C][25]: dx[p][c] = sum_{co,tap'} dimg[co][p + tap' - 2] * w[co*25C + c*25 + 24 - tap']
        rc = hconv_3_to_c(dimg, dimg, dimg, d->N, d->N, d->H, d->W, d->C, 1, w, 25, 25LL * d->C, 1, nullptr, 0, dx, ws,
                          S(stream));
        if (rc <= 0) return rc;
    }
    float* wk = reinterpret_cast<float*>(ws);
    // dx[p][c] = sum_{co,tap'} dimg[co][p + tap' - 2] * w[co][c][24 - tap']  -> "3 -> C" form with a flipped pack
    rc = pack_edge_out(d, w, wk, 1, S(stream));
    if (rc) return rc;
    fmri_edge_desc e = *d;
    return e.C == 32 ? edge_in_fprop_t<32>(&e, dimg, dimg, dimg, d->N, wk, nullptr, 0, dx, d->H, d->W, S(stream))
                     : edge_in_fprop_t<64>(&e, dimg, dimg, dimg, d->N, wk, nullptr, 0, dx, d->H, d->W, S(stream));
}
extern "C" int fmri_edge_out_wgrad(const fmri_edge_desc* d, const void* x, const float* dimg, float* dw,
                                   int accumulate, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_edge(d, ws, ws_bytes);
    if (rc) return rc;
    if (d->stride != 1) return fail(FMRI_ERR_UNSUPPORTED, "edge out conv is stride 1");
    float* dwk = reinterpret_cast<float*>(ws);
    CUDA_OK(cudaMemsetAsync(dwk, 0, sizeof(float) * 75 * (size_t)d->C, S(stream)));
    rc = 1;
    if (d->dtype == FMRI_BF16 && fmri_tensor_path_available())
        rc = hwgrad_run(x, dimg, dimg, dimg, d->N, d->N, d->H, d->W, d->C, dwk, nullptr, 1, ws, S(stream));
    if (rc == 1)
        rc = d->C == 32 ? edge_wgrad_t<32>(d->dtype, x, dimg, dimg, dimg, d->N, dwk, nullptr, d->N, d->H, d->W, d->H, d->W,
                                           1, -1, S(stream))
                        : edge_wgrad_t<64>(d->dtype, x, dimg, dimg, dimg, d->N, dwk, nullptr, d->N, d->H, d->W, d->H, d->W,
                                           1, -1, S(stream));
    if (rc) return rc;
    // dwk[(co*25+tap)*C + c] -> dw[co][c][tap]
    scatter4_kernel<float, float><<<grid1d(75LL * d->C, 256), 256, 0, S(stream)>>>(dwk, dw, 1, 3, 25, d->C, 0,
                                                                                  25LL * d->C, 1, 25, accumulate);
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ linear
static int transpose_any(const void* src, int sdt, void* dst, int ddt, int N, int R, int Cc, int accumulate, cudaStream_t st);
extern "C" int fmri_linear_pack_weights(const fmri_linear_desc* d, const float* w, void* wp, int ldw, void* wpt,
                                        int ldwt, void* stream) {
    if (!d || d->M < 0 || d->N <= 0 || d->K <= 0) return fail(FMRI_ERR_ARG, "bad linear descriptor");
    if (wp) {
        if (ldw < d->K) return fail(FMRI_ERR_ARG, "ldw < K");
        int rc = fmri_cast2d(w, FMRI_F32, d->K, wp, FMRI_BF16, ldw, d->N, d->K, stream);
        if (rc) return rc;
    }
    if (wpt) {  // [K][N]
        if (ldwt < d->N) return fail(FMRI_ERR_ARG, "ldwt < N");
        // dst[k][n] (pitch ldwt) = w[n][k]
        if (ldwt == d->N) {  // dense: tiled transpose, both sides coalesced
            int rc = transpose_any(w, FMRI_F32, wpt, FMRI_BF16, 1, d->N, d->K, 0, S(stream));
            if (rc) return rc;
        } else {
            scatter4_kernel<float, __nv_bfloat16><<<grid1d((long long)d->N * d->K, 256), 256, 0, S(stream)>>>(
                w, reinterpret_cast<__nv_bfloat16*>(wpt), 1, 1, d->N, d->K, 0, 0, 1, ldwt, 0);
            LAUNCH_OK();
        }
    }
    return 0;
}

template <typename Ta, typename Tb, typename Tc>
static int simt_gemm(const Ta* A, long long a_sm, long long a_sk, const Tb* B, long long b_sn, long long b_sk, Tc* C,
                     long long c_sm, long long c_sn, const float* bias, int M, int N, int K, int act, int accumulate,
                     cudaStream_t st) {
    dim3 grid(cdiv(N, 64), cdiv(M, 64));
    simt_gemm_kernel<Ta, Tb, Tc><<<grid, 256, 0, st>>>(A, a_sm, a_sk, B, b_sn, b_sk, C, c_sm, c_sn, bias, M, N, K,
                                                      act, accumulate);
    LAUNCH_OK();
    return 0;
}

extern "C" int fmri_linear_fprop(const fmri_linear_desc* d, const void* x, int ldx, const float* w, const void* wp,
                                 int ldw, const float* bias, int act, void* y, int ldy, int y_dtype, void* stream) {
    if (!d || d->M <= 0 || d->N <= 0 || d->K <= 0) return fail(FMRI_ERR_ARG, "bad linear descriptor");
    if (d->dtype == FMRI_BF16) {
        if (!wp) return fail(FMRI_ERR_ARG, "bf16 linear needs packed weights");
        if (d->N % 32 == 0)
            return run_gemm_tn(x, ldx, wp, ldw, d->M, d->N, d->K, bias, act, y, ldy, y_dtype == FMRI_F32, 0, S(stream));
        // narrow outputs (not on the hot path) use the CUDA-core GEMM on the bf16 operands
        if (y_dtype == FMRI_F32)
            return simt_gemm(reinterpret_cast<const __nv_bfloat16*>(x), ldx, 1,
                             reinterpret_cast<const __nv_bfloat16*>(wp), ldw, 1, reinterpret_cast<float*>(y), ldy, 1,
                             bias, d->M, d->N, d->K, act, 0, S(stream));
        return simt_gemm(reinterpret_cast<const __nv_bfloat16*>(x), ldx, 1, reinterpret_cast<const __nv_bfloat16*>(wp),
                         ldw, 1, reinterpret_cast<__nv_bfloat16*>(y), ldy, 1, bias, d->M, d->N, d->K, act, 0,
                         S(stream));
    }
    if (y_dtype != FMRI_F32) return fail(FMRI_ERR_ARG, "fp32 linear writes fp32");
    return simt_gemm(reinterpret_cast<const float*>(x), ldx, 1, w, d->K, 1, reinterpret_cast<float*>(y), ldy, 1, bias,
                     d->M, d->N, d->K, act, 0, S(stream));
}

extern "C" int fmri_linear_dgrad(const fmri_linear_desc* d, const void* dy, int lddy, const float* w, const void* wpt,
                                 int ldwt, void* dx, int lddx, int dx_dtype, int accumulate, void* stream) {
    if (!d || d->M <= 0 || d->N <= 0 || d->K <= 0) return fail(FMRI_ERR_ARG, "bad linear descriptor");
    if (accumulate && dx_dtype != FMRI_F32) return fail(FMRI_ERR_ARG, "accumulating dgrad needs an fp32 dx");
    if (d->dtype == FMRI_BF16) {
        if (!wpt) return fail(FMRI_ERR_ARG, "bf16 linear dgrad needs the transposed pack");
        if (d->K % 32 == 0 && d->N % 8 == 0)  // dx[M,K] = dy[M,N] * wpt[K,N]^T
            return run_gemm_tn(dy, lddy, wpt, ldwt, d->M, d->K, d->N, nullptr, 0, dx, lddx, dx_dtype == FMRI_F32,
                               accumulate, S(stream));
        if (dx_dtype == FMRI_F32)
            return simt_gemm(reinterpret_cast<const __nv_bfloat16*>(dy), lddy, 1,
                             reinterpret_cast<const __nv_bfloat16*>(wpt), ldwt, 1, reinterpret_cast<float*>(dx), lddx,
                             1, nullptr, d->M, d->K, d->N, 0, accumulate, S(stream));
        return simt_gemm(reinterpret_cast<const __nv_bfloat16*>(dy), lddy, 1,
                         reinterpret_cast<const __nv_bfloat16*>(wpt), ldwt, 1, reinterpret_cast<__nv_bfloat16*>(dx),
                         lddx, 1, nullptr, d->M, d->K, d->N, 0, 0, S(stream));
    }
    // dx[m,k] = sum_n dy[m,n] w[n,k] : "B" = w viewed as [K rows (stride 1)] x [N (stride K)]
    return simt_gemm(reinterpret_cast<const float*>(dy), lddy, 1, w, 1, d->K, reinterpret_cast<float*>(dx), lddx, 1,
                     nullptr, d->M, d->K, d->N, 0, accumulate, S(stream));
}

extern "C" int fmri_linear_wgrad(const fmri_linear_desc* d, const void* x, int ldx, const void* dy, int lddy,
                                 float* dw, int accumulate, void* stream) {
    if (!d || d->M <= 0 || d->N <= 0 || d->K <= 0) return fail(FMRI_ERR_ARG, "bad linear descriptor");
    if (d->dtype == FMRI_BF16) {
        // dw[n,k] = sum_m dy[m,n] x[m,k]; tensor path when the tiles fit: N%128 (dense side), K%32, pitch == extent
        const bool tc_ok = (d->N % 128 == 0) && (d->K % 128 == 0 || d->K == 64 || d->K == 32) && (d->M % 16 == 0) &&
                           (lddy % 8 == 0) && (ldx % 8 == 0);
        if (tc_ok) {
            if (!accumulate) CUDA_OK(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)d->N * d->K, S(stream)));
            // reuse the conv wgrad kernel with a [M rows] x 1 x 1 pixel grid; pitches come in through the maps
            WgParams p;
            memset(&p, 0, sizeof(p));
            p.bw = std::min(128, d->M);
            p.bh = p.bn = 1;
            p.rows = p.bw;
            if (p.rows % 16) return fail(FMRI_ERR_UNSUPPORTED, "linear wgrad rows");
            p.tiles_x = cdiv(d->M, p.bw);
            p.tiles_y = p.tiles_n = 1;
            const int NCH = (d->K % 64 == 0) ? 64 : 32;
            const int BN = (d->K % 128 == 0) ? 128 : (d->K % 64 == 0 ? 64 : 32);
            int rc = make_act_map(&p.mapD, dy, d->N, d->M, 1, 1, lddy, (long long)lddy * d->M,
                                  (long long)lddy * d->M, 64, p.bw, 1, 1);
            if (rc) return rc;
            rc = make_act_map(&p.mapS[0], x, d->K, d->M, 1, 1, ldx, (long long)ldx * d->M, (long long)ldx * d->M, NCH,
                              p.bw, 1, 1);
            if (rc) return rc;
            p.num_taps = 1;
            p.m_total = d->N;
            p.n_total = d->K;
            p.m_tiles = d->N / 128;
            p.n_tiles = d->K / BN;
            const long long base = (long long)p.m_tiles * p.n_tiles;
            (void)base;
            p.splits = 1;   // one writer per dw element (see the linear split-K note above)
            p.out = dw;
            return dispatch_wg(p, BN, NCH, S(stream));
        }
        return simt_gemm(reinterpret_cast<const __nv_bfloat16*>(dy), 1, lddy,
                         reinterpret_cast<const __nv_bfloat16*>(x), 1, ldx, dw, d->K, 1, nullptr, d->N, d->K, d->M, 0,
                         accumulate, S(stream));
    }
    return simt_gemm(reinterpret_cast<const float*>(dy), 1, lddy, reinterpret_cast<const float*>(x), 1, ldx, dw, d->K,
                     1, nullptr, d->N, d->K, d->M, 0, accumulate, S(stream));
}

// ================================================================================================ BN / elementwise
static int rows_per_block_for(long long rows) {
    long long target = (rows + 148 * 4 - 1) / (148 * 4);
    return (int)std::max<long long>(8, target);
}
extern "C" int fmri_colstats(const void* x, int dtype, long long rows, int C, double* sum, double* sq, void* stream) {
    if (C <= 0 || rows <= 0) return fail(FMRI_ERR_ARG, "colstats shape");
    if (C < 256 && (256 % C)) return fail(FMRI_ERR_UNSUPPORTED, "colstats C=%d", C);
    const int rpb = rows_per_block_for(rows);
    dim3 grid(cdiv(rows, rpb), std::min(8, cdiv(C, 256)));
    CUDA_OK(cudaMemsetAsync(sum, 0, sizeof(double) * C, S(stream)));
    CUDA_OK(cudaMemsetAsync(sq, 0, sizeof(double) * C, S(stream)));
    if (C % 8 == 0 && ((C / 8) >= 256 ? (C / 8) % 256 == 0 : 256 % (C / 8) == 0)) {
        // wide matrices (the 16384-feature BatchNorm1d of the fc layers): the column blocks already fill the machine, so
        // each block takes more rows -- with 8 rows per block the 2 x 8 fp64 atomics per thread outweighed the loads
        // (4096 x 16384 fp32: 0.36 ms, 0.75 TB/s)
        const int gy = std::max(1, std::min(8, (C / 8) / 256));
        const int rpb8 = (int)std::max<long long>(rpb, cdiv(rows, std::max(1, (148 * 4) / gy)));
        dim3 g8(cdiv(rows, rpb8), gy);
        if (dtype == FMRI_BF16)
            bn_reduce8_kernel<0, __nv_bfloat16, __nv_bfloat16><<<g8, 256, 0, S(stream)>>>(
                reinterpret_cast<const __nv_bfloat16*>(x), nullptr, rows, C, nullptr, nullptr, nullptr, nullptr, 0, sum, sq, rpb8);
        else
            bn_reduce8_kernel<0, float, float><<<g8, 256, 0, S(stream)>>>(reinterpret_cast<const float*>(x), nullptr, rows, C,
                                                                          nullptr, nullptr, nullptr, nullptr, 0, sum, sq, rpb8);
        LAUNCH_OK();
        return 0;
    }
    if (dtype == FMRI_BF16)
        colstats_kernel<__nv_bfloat16><<<grid, 256, 2 * 256 * 4, S(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(x), rows, C, sum, sq, rpb);
    else
        colstats_kernel<float><<<grid, 256, 2 * 256 * 4, S(stream)>>>(reinterpret_cast<const float*>(x), rows, C, sum,
                                                                     sq, rpb);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_bn_finalize(const double* sum, const double* sq, long long rows, int C, float eps, float momentum,
                                float* mean, float* invstd, float* running_mean, float* running_var, void* stream) {
    bn_finalize_kernel<<<cdiv(C, 128), 128, 0, S(stream)>>>(sum, sq, (double)rows, C, eps, momentum, mean, invstd,
                                                           running_mean, running_var);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_bn_apply(const void* x, int x_dtype, void* y, int y_dtype, long long rows, int C, const float* mean,
                             const float* invstd, const float* gamma, const float* beta, int relu, void* stream) {
    if (C % 8) return fail(FMRI_ERR_UNSUPPORTED, "bn_apply needs C %% 8 == 0");
    const long long total = rows * C;
    int g = grid1d((total + 7) / 8, 256, 148 * 8);
    if (C > 2048 && (C % 2048) == 0 && g >= C / 2048) g = g / (C / 2048) * (C / 2048);  // grid stride a multiple of C
    cudaStream_t st = S(stream);
    if (x_dtype == FMRI_BF16 && y_dtype == FMRI_BF16)
        bn_apply_kernel<__nv_bfloat16, __nv_bfloat16><<<g, 256, 0, st>>>(
            reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<__nv_bfloat16*>(y), total, C, mean, invstd,
            gamma, beta, relu);
    else if (x_dtype == FMRI_F32 && y_dtype == FMRI_BF16)
        bn_apply_kernel<float, __nv_bfloat16><<<g, 256, 0, st>>>(reinterpret_cast<const float*>(x),
                                                                reinterpret_cast<__nv_bfloat16*>(y), total, C, mean,
                                                                invstd, gamma, beta, relu);
    else if (x_dtype == FMRI_F32 && y_dtype == FMRI_F32)
        bn_apply_kernel<float, float><<<g, 256, 0, st>>>(reinterpret_cast<const float*>(x), reinterpret_cast<float*>(y),
                                                        total, C, mean, invstd, gamma, beta, relu);
    else
        return fail(FMRI_ERR_UNSUPPORTED, "bn_apply dtype combination");
    LAUNCH_OK();
    return 0;
}
// the channel-pair kernels tile C when a row's channel pairs fill whole 256-thread blocks or divide one evenly
static bool bn_cp_ok(int C) { return C % 2 == 0 && ((C / 2) >= 256 ? (C / 2) % 256 == 0 : 256 % (C / 2) == 0); }
// resident CTAs per SM of a BatchNorm-backward kernel (queried once per instantiation): its grid is exactly one wave
template <typename K>
static int bn_occupancy(K kernel, int& cache) {
    if (!cache) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cache, kernel, 256, 0) != cudaSuccess) return 0;
        cache = std::max(1, cache);
    }
    return cache;
}
static long long bn_cp_rows_per_block(long long rows, int C, int occ) {
    const int ry = std::max(1, 256 / (C / 2));
    return std::max<long long>((long long)ry * 16, (rows + 148 * occ - 1) / (148 * occ));
}
template <typename Tx, typename Tg>
static int bn_cp_reduce_per(long long rows, int C, long long* per) {
    static int occ1 = 0;
    if (!bn_occupancy(bn_bwd_cp_kernel<1, Tx, Tg>, occ1)) return fail(FMRI_ERR_CUDA, "occupancy query of bn_bwd_cp_kernel");
    *per = bn_cp_rows_per_block(rows, C, occ1);
    return 0;
}
template <typename Tx, typename Tg>
static int bn_bwd_reduce_t(const void* x, const void* dy, long long rows, int C, const float* mean, const float* invstd,
                           const float* gamma, const float* beta, int relu, double* ws, cudaStream_t st) {
    const int rpb = rows_per_block_for(rows);
    dim3 grid(cdiv(rows, rpb), std::min(8, cdiv(C, 256)));
    CUDA_OK(cudaMemsetAsync(ws, 0, sizeof(double) * 2 * C, st));
    if (bn_cp_ok(C)) {
        long long per;
        int rc = bn_cp_reduce_per<Tx, Tg>(rows, C, &per);
        if (rc) return rc;
        dim3 gcp(cdiv(rows, per), std::max(1, std::min(8, (C / 2) / 256)));
        bn_bwd_cp_kernel<1, Tx, Tg><<<gcp, 256, 0, st>>>(reinterpret_cast<const Tx*>(x), reinterpret_cast<const Tg*>(dy), nullptr,
                                                       rows, C, mean, invstd, gamma, beta, relu, 1, nullptr, nullptr, ws,
                                                       ws + C, (int)per);
    } else if (C % 8 == 0 && ((C / 8) >= 256 ? (C / 8) % 256 == 0 : 256 % (C / 8) == 0)) {
        dim3 g8(cdiv(rows, rpb), std::max(1, std::min(8, (C / 8) / 256)));
        bn_reduce8_kernel<1, Tx, Tg><<<g8, 256, 0, st>>>(reinterpret_cast<const Tx*>(x), reinterpret_cast<const Tg*>(dy), rows,
                                                       C, mean, invstd, gamma, beta, relu, ws, ws + C, rpb);
    } else {
        bn_bwd_reduce_kernel<Tx, Tg><<<grid, 256, 2 * 256 * 4, st>>>(reinterpret_cast<const Tx*>(x),
                                                                    reinterpret_cast<const Tg*>(dy), rows, C, mean,
                                                                    invstd, gamma, beta, relu, ws, ws + C, rpb);
    }
    LAUNCH_OK();
    return 0;
}
// dx = gamma*invstd * (g - mean_g - xhat*mean_gx) over `rows` rows (x, dy, dx point at the first of them)
template <typename Tx, typename Tg>
static int bn_bwd_apply_t(const void* x, const void* dy, void* dx, long long rows, int C, const float* mean,
                          const float* invstd, const float* gamma, const float* beta, int relu, int train,
                          const float* mean_g, const float* mean_gx, cudaStream_t st) {
    if (rows == 0) return 0;
    if (bn_cp_ok(C)) {
        static int occ2 = 0;
        if (!bn_occupancy(bn_bwd_cp_kernel<2, Tx, Tg>, occ2)) return fail(FMRI_ERR_CUDA, "occupancy query of bn_bwd_cp_kernel");
        const long long per = bn_cp_rows_per_block(rows, C, occ2);
        dim3 gcp(cdiv(rows, per), std::max(1, std::min(8, (C / 2) / 256)));
        bn_bwd_cp_kernel<2, Tx, Tg><<<gcp, 256, 0, st>>>(reinterpret_cast<const Tx*>(x), reinterpret_cast<const Tg*>(dy),
                                                       reinterpret_cast<Tg*>(dx), rows, C, mean, invstd, gamma, beta, relu,
                                                       train, mean_g, mean_gx, nullptr, nullptr, (int)per);
        LAUNCH_OK();
    } else {
        if (C % 8) return fail(FMRI_ERR_UNSUPPORTED, "bn_backward needs C %% 8 == 0");
        bn_bwd_apply_kernel<Tx, Tg><<<grid1d((rows * C + 7) / 8, 256, 148 * 8), 256, 0, st>>>(
            reinterpret_cast<const Tx*>(x), reinterpret_cast<const Tg*>(dy), reinterpret_cast<Tg*>(dx), rows * C, C,
            (double)rows, mean, invstd, gamma, beta, relu, train, mean_g, mean_gx);
        LAUNCH_OK();
    }
    return 0;
}
template <typename Tx, typename Tg>
static int bn_bwd_t(const void* x, const void* dy, void* dx, long long rows, int C, const float* mean,
                    const float* invstd, const float* gamma, const float* beta, int relu, int train, float* dgamma,
                    float* dbeta, int accumulate, double* ws, cudaStream_t st, long long row0 = 0, long long nrows = -1) {
    // [row0, row0 + nrows): the rows dx is produced for (dx points at the first of them); the sums always run over all rows
    int rc = bn_bwd_reduce_t<Tx, Tg>(x, dy, rows, C, mean, invstd, gamma, beta, relu, ws, st);
    if (rc) return rc;
    float* mean_g = reinterpret_cast<float*>(ws + 2 * C);  // third C doubles of the workspace: 2C floats
    float* mean_gx = mean_g + C;
    bn_param_grad_kernel<<<cdiv(C, 128), 128, 0, st>>>(ws, ws + C, (double)rows, C, mean_g, mean_gx, dgamma, dbeta, accumulate);
    LAUNCH_OK();
    if (nrows >= 0) {
        x = reinterpret_cast<const Tx*>(x) + row0 * C;
        dy = reinterpret_cast<const Tg*>(dy) + row0 * C;
        rows = nrows;
    }
    if (!dx) return 0;
    return bn_bwd_apply_t<Tx, Tg>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train, mean_g, mean_gx, st);
}
// Two upstreams a, b through one BatchNorm; dgamma/dbeta (nullable) take upstream a's parameter gradient. dx_a covers all
// rows, dx_b rows [row0, row0 + nrows). ws: 6*C doubles = [sums a | sums b | fp32 means a | fp32 means b].
template <typename Tx, typename Tg>
static int bn_bwd_pair_t(const void* x, const void* dya, const void* dyb, void* dxa, void* dxb, long long rows,
                         long long row0, long long nrows, int C, const float* mean, const float* invstd, const float* gamma,
                         const float* beta, int relu, int train, float* dgamma, float* dbeta, int accumulate, double* ws,
                         cudaStream_t st) {
    if (!bn_cp_ok(C)) {   // shapes the channel-pair kernels do not tile: the two single-upstream passes
        int rc = bn_bwd_t<Tx, Tg>(x, dya, dxa, rows, C, mean, invstd, gamma, beta, relu, train, dgamma, dbeta, accumulate,
                                  ws, st);
        if (rc) return rc;
        return bn_bwd_t<Tx, Tg>(x, dyb, dxb, rows, C, mean, invstd, gamma, beta, relu, train, nullptr, nullptr, 0, ws + 3 * C,
                                st, row0, nrows);
    }
    const Tx* xp = reinterpret_cast<const Tx*>(x);
    const Tg *ap = reinterpret_cast<const Tg*>(dya), *bp = reinterpret_cast<const Tg*>(dyb);
    Tg *dap = reinterpret_cast<Tg*>(dxa), *dbp = reinterpret_cast<Tg*>(dxb);
    // the sums: the grid and rows_per_block of the single-upstream reduce, so that each upstream's partials match it
    long long per;
    int rc = bn_cp_reduce_per<Tx, Tg>(rows, C, &per);
    if (rc) return rc;
    static int occ2 = 0;   // the apply's grid: one wave of the paired kernel
    if (!bn_occupancy(bn_bwd_cp2_kernel<2, Tx, Tg>, occ2)) return fail(FMRI_ERR_CUDA, "occupancy query of bn_bwd_cp2_kernel");
    const int gy = std::max(1, std::min(8, (C / 2) / 256));
    CUDA_OK(cudaMemsetAsync(ws, 0, sizeof(double) * 4 * C, st));
    bn_bwd_cp2_kernel<1, Tx, Tg><<<dim3(cdiv(rows, per), gy), 256, 0, st>>>(
        xp, ap, bp, nullptr, nullptr, rows, C, mean, invstd, gamma, beta, relu, 1, nullptr, nullptr, nullptr, nullptr, ws,
        ws + C, ws + 2 * C, ws + 3 * C, (int)per);
    LAUNCH_OK();
    float* mga = reinterpret_cast<float*>(ws + 4 * C);
    float* mgxa = mga + C;
    float* mgb = mgxa + C;
    float* mgxb = mgb + C;
    bn_param_grad_kernel<<<cdiv(C, 128), 128, 0, st>>>(ws, ws + C, (double)rows, C, mga, mgxa, dgamma, dbeta, accumulate);
    LAUNCH_OK();
    bn_param_grad_kernel<<<cdiv(C, 128), 128, 0, st>>>(ws + 2 * C, ws + 3 * C, (double)rows, C, mgb, mgxb, nullptr, nullptr, 0);
    LAUNCH_OK();
    // the apply: upstream a alone outside the slice, both upstreams on it
    const long long row1 = row0 + nrows;
    if (row0 > 0) {
        rc = bn_bwd_apply_t<Tx, Tg>(xp, ap, dap, row0, C, mean, invstd, gamma, beta, relu, train, mga, mgxa, st);
        if (rc) return rc;
    }
    if (row1 < rows) {
        rc = bn_bwd_apply_t<Tx, Tg>(xp + row1 * C, ap + row1 * C, dap + row1 * C, rows - row1, C, mean, invstd, gamma, beta,
                                    relu, train, mga, mgxa, st);
        if (rc) return rc;
    }
    if (nrows == 0) return 0;
    const long long per2 = bn_cp_rows_per_block(nrows, C, occ2);
    bn_bwd_cp2_kernel<2, Tx, Tg><<<dim3(cdiv(nrows, per2), gy), 256, 0, st>>>(
        xp + row0 * C, ap + row0 * C, bp + row0 * C, dap + row0 * C, dbp, nrows, C, mean, invstd, gamma, beta, relu, train,
        mga, mgxa, mgb, mgxb, nullptr, nullptr, nullptr, nullptr, (int)per2);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_bn_backward(const void* x, int x_dtype, const void* dy, void* dx, int g_dtype, long long rows, int C,
                                const float* mean, const float* invstd, const float* gamma, const float* beta,
                                int relu, int train, float* dgamma, float* dbeta, int accumulate, double* ws, void* stream) {
    if (C < 256 && (256 % C)) return fail(FMRI_ERR_UNSUPPORTED, "bn_backward C=%d", C);
    if (x_dtype == FMRI_BF16 && g_dtype == FMRI_BF16)
        return bn_bwd_t<__nv_bfloat16, __nv_bfloat16>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train,
                                                      dgamma, dbeta, accumulate, ws, S(stream));
    if (x_dtype == FMRI_F32 && g_dtype == FMRI_BF16)
        return bn_bwd_t<float, __nv_bfloat16>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train, dgamma, dbeta,
                                              accumulate, ws, S(stream));
    if (x_dtype == FMRI_F32 && g_dtype == FMRI_F32)
        return bn_bwd_t<float, float>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train, dgamma, dbeta,
                                      accumulate, ws, S(stream));
    return fail(FMRI_ERR_UNSUPPORTED, "bn_backward dtype combination");
}
extern "C" int fmri_bn_backward_slice(const void* x, int x_dtype, const void* dy, void* dx, int g_dtype, long long rows,
                                      long long row0, long long nrows, int C, const float* mean, const float* invstd,
                                      const float* gamma, const float* beta, int relu, int train, float* dgamma,
                                      float* dbeta, int accumulate, double* ws, void* stream) {
    if (C < 256 && (256 % C)) return fail(FMRI_ERR_UNSUPPORTED, "bn_backward C=%d", C);
    if (row0 < 0 || nrows < 0 || row0 + nrows > rows) return fail(FMRI_ERR_ARG, "bn_backward_slice: bad row range");
    if (x_dtype == FMRI_BF16 && g_dtype == FMRI_BF16)
        return bn_bwd_t<__nv_bfloat16, __nv_bfloat16>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train,
                                                      dgamma, dbeta, accumulate, ws, S(stream), row0, nrows);
    if (x_dtype == FMRI_F32 && g_dtype == FMRI_BF16)
        return bn_bwd_t<float, __nv_bfloat16>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train, dgamma, dbeta,
                                              accumulate, ws, S(stream), row0, nrows);
    if (x_dtype == FMRI_F32 && g_dtype == FMRI_F32)
        return bn_bwd_t<float, float>(x, dy, dx, rows, C, mean, invstd, gamma, beta, relu, train, dgamma, dbeta,
                                      accumulate, ws, S(stream), row0, nrows);
    return fail(FMRI_ERR_UNSUPPORTED, "bn_backward dtype combination");
}
static int bn_pair_entry(const void* x, int x_dtype, const void* dya, const void* dyb, void* dxa, void* dxb, int g_dtype,
                         long long rows, long long row0, long long nrows, int C, const float* mean, const float* invstd,
                         const float* gamma, const float* beta, int relu, int train, float* dgamma, float* dbeta,
                         int accumulate, double* ws, void* stream) {
    // every argument is checked before the first launch
    if (C <= 0 || (C < 256 && (256 % C))) return fail(FMRI_ERR_UNSUPPORTED, "bn_backward_pair C=%d", C);
    if (!bn_cp_ok(C) && C % 8) return fail(FMRI_ERR_UNSUPPORTED, "bn_backward_pair needs C %% 8 == 0");
    if (rows < 0 || row0 < 0 || nrows < 0 || row0 + nrows > rows) return fail(FMRI_ERR_ARG, "bn_backward_pair: bad row range");
    if (!x || !dya || !dyb || !dxa || (!dxb && nrows > 0) || !mean || !invstd || !gamma || !beta || !ws)
        return fail(FMRI_ERR_ARG, "bn_backward_pair: null tensor argument");
    if (!dgamma != !dbeta) return fail(FMRI_ERR_ARG, "bn_backward_pair: dgamma and dbeta go together");
    if (dya == dyb || dxa == dxb) return fail(FMRI_ERR_ARG, "bn_backward_pair: the two upstreams need their own buffers");
    if (x_dtype == FMRI_BF16 && g_dtype == FMRI_BF16)
        return bn_bwd_pair_t<__nv_bfloat16, __nv_bfloat16>(x, dya, dyb, dxa, dxb, rows, row0, nrows, C, mean, invstd, gamma,
                                                           beta, relu, train, dgamma, dbeta, accumulate, ws, S(stream));
    if (x_dtype == FMRI_F32 && g_dtype == FMRI_BF16)
        return bn_bwd_pair_t<float, __nv_bfloat16>(x, dya, dyb, dxa, dxb, rows, row0, nrows, C, mean, invstd, gamma, beta,
                                                   relu, train, dgamma, dbeta, accumulate, ws, S(stream));
    if (x_dtype == FMRI_F32 && g_dtype == FMRI_F32)
        return bn_bwd_pair_t<float, float>(x, dya, dyb, dxa, dxb, rows, row0, nrows, C, mean, invstd, gamma, beta, relu,
                                           train, dgamma, dbeta, accumulate, ws, S(stream));
    return fail(FMRI_ERR_UNSUPPORTED, "bn_backward_pair dtype combination");
}
extern "C" int fmri_bn_backward_pair(const void* x, int x_dtype, const void* dy_a, const void* dy_b, void* dx_a, void* dx_b,
                                     int g_dtype, long long rows, int C, const float* mean, const float* invstd,
                                     const float* gamma, const float* beta, int relu, int train, float* dgamma,
                                     float* dbeta, int accumulate, double* ws, void* stream) {
    return bn_pair_entry(x, x_dtype, dy_a, dy_b, dx_a, dx_b, g_dtype, rows, 0, rows, C, mean, invstd, gamma, beta, relu,
                         train, dgamma, dbeta, accumulate, ws, stream);
}
extern "C" int fmri_bn_backward_pair_slice(const void* x, int x_dtype, const void* dy_a, const void* dy_b, void* dx_a,
                                           void* dx_b, int g_dtype, long long rows, long long row0, long long nrows, int C,
                                           const float* mean, const float* invstd, const float* gamma, const float* beta,
                                           int relu, int train, float* dgamma, float* dbeta, int accumulate, double* ws,
                                           void* stream) {
    return bn_pair_entry(x, x_dtype, dy_a, dy_b, dx_a, dx_b, g_dtype, rows, row0, nrows, C, mean, invstd, gamma, beta, relu,
                         train, dgamma, dbeta, accumulate, ws, stream);
}
extern "C" int fmri_relu_backward(const void* y, const void* dy, void* dx, int dtype, long long n, void* stream) {
    if (dtype == FMRI_BF16)
        relu_bwd_kernel<__nv_bfloat16><<<grid1d((n + 7) / 8, 256, 148 * 8), 256, 0, S(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(y), reinterpret_cast<const __nv_bfloat16*>(dy),
            reinterpret_cast<__nv_bfloat16*>(dx), n);
    else
        relu_bwd_kernel<float><<<grid1d((n + 7) / 8, 256, 148 * 8), 256, 0, S(stream)>>>(
            reinterpret_cast<const float*>(y), reinterpret_cast<const float*>(dy), reinterpret_cast<float*>(dx), n);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_relu_bitmask(const void* y, int dtype, long long pixels, int C, unsigned* bits, void* stream) {
    if (dtype != FMRI_BF16 || C != 32) return fail(FMRI_ERR_UNSUPPORTED, "relu_bitmask: bf16 tensors with 32 channels only");
    relu_bitmask32_kernel<<<cdiv(pixels, 256), 256, 0, S(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(y), bits, pixels);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_colsum(const void* x, int dtype, long long rows, int C, float* out, void* stream) {
    const int rpb = rows_per_block_for(rows);
    const int nb = cdiv(rows, rpb);
    SCRATCH(part, float, (long long)nb * C, S(stream));
    if (dtype == FMRI_BF16)
        colsum_kernel<__nv_bfloat16><<<nb, 256, 0, S(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), rows, C, part,
                                                               rpb);
    else
        colsum_kernel<float><<<nb, 256, 0, S(stream)>>>(reinterpret_cast<const float*>(x), rows, C, part, rpb);
    LAUNCH_OK();
    int rc = ordered_add(part, nb, C, out, S(stream));
    CUDA_OK(cudaFreeAsync(part, S(stream)));
    return rc;
}

template <typename TI, typename TO>
static int permute_launch(const void* src, void* dst, int d1, int d2, int d3, long long s1, long long s2, long long s3,
                          int accumulate, cudaStream_t st) {
    const long long n = (long long)d1 * d2 * d3;
    permute4_kernel<TI, TO><<<grid1d(n, 256), 256, 0, st>>>(reinterpret_cast<const TI*>(src),
                                                            reinterpret_cast<TO*>(dst), 1, d1, d2, d3, 0, s1, s2, s3,
                                                            accumulate);
    LAUNCH_OK();
    return 0;
}
static int permute_any(const void* src, int sdt, void* dst, int ddt, int d1, int d2, int d3, long long s1,
                       long long s2, long long s3, int accumulate, cudaStream_t st) {
    if (sdt == FMRI_F32 && ddt == FMRI_F32)
        return permute_launch<float, float>(src, dst, d1, d2, d3, s1, s2, s3, accumulate, st);
    if (sdt == FMRI_F32 && ddt == FMRI_BF16)
        return permute_launch<float, __nv_bfloat16>(src, dst, d1, d2, d3, s1, s2, s3, accumulate, st);
    if (sdt == FMRI_BF16 && ddt == FMRI_F32)
        return permute_launch<__nv_bfloat16, float>(src, dst, d1, d2, d3, s1, s2, s3, accumulate, st);
    if (sdt == FMRI_BF16 && ddt == FMRI_BF16)
        return permute_launch<__nv_bfloat16, __nv_bfloat16>(src, dst, d1, d2, d3, s1, s2, s3, accumulate, st);
    return fail(FMRI_ERR_ARG, "bad dtype");
}
template <typename TI, typename TO>
static int transpose_launch(const void* src, void* dst, int N, int R, int Cc, int accumulate, cudaStream_t st) {
    dim3 grid(cdiv(Cc, 32), cdiv(R, 32), N);
    transpose_batched_kernel<TI, TO><<<grid, 256, 0, st>>>(reinterpret_cast<const TI*>(src), reinterpret_cast<TO*>(dst), R, Cc,
                                                           accumulate);
    LAUNCH_OK();
    return 0;
}
// dst[n][c][r] (+)= src[n][r][c]
static int transpose_any(const void* src, int sdt, void* dst, int ddt, int N, int R, int Cc, int accumulate, cudaStream_t st) {
    if (N > 65535) return fail(FMRI_ERR_UNSUPPORTED, "transpose batch %d > 65535", N);
    if (sdt == FMRI_F32 && ddt == FMRI_F32) return transpose_launch<float, float>(src, dst, N, R, Cc, accumulate, st);
    if (sdt == FMRI_F32 && ddt == FMRI_BF16) return transpose_launch<float, __nv_bfloat16>(src, dst, N, R, Cc, accumulate, st);
    if (sdt == FMRI_BF16 && ddt == FMRI_F32) return transpose_launch<__nv_bfloat16, float>(src, dst, N, R, Cc, accumulate, st);
    if (sdt == FMRI_BF16 && ddt == FMRI_BF16)
        return transpose_launch<__nv_bfloat16, __nv_bfloat16>(src, dst, N, R, Cc, accumulate, st);
    return fail(FMRI_ERR_ARG, "bad dtype");
}
extern "C" int fmri_nchw_to_nhwc(const void* src, int src_dtype, void* dst, int dst_dtype, int N, int C, int H, int W,
                                 void* stream) {
    // dst[n][p][c] = src[n][c][p]: transpose of the [C][HW] matrix of every image
    return transpose_any(src, src_dtype, dst, dst_dtype, N, C, H * W, 0, S(stream));
}
extern "C" int fmri_nhwc_to_nchw(const void* src, int src_dtype, void* dst, int dst_dtype, int N, int C, int H, int W,
                                 int accumulate, void* stream) {
    // dst[n][c][p] = src[n][p][c]
    return transpose_any(src, src_dtype, dst, dst_dtype, N, H * W, C, accumulate, S(stream));
}
extern "C" int fmri_cast2d(const void* src, int src_dtype, int lds, void* dst, int dst_dtype, int ldd, long long rows,
                           int cols, void* stream) {
    const long long n = rows * cols;
    cudaStream_t st = S(stream);
    const int g = grid1d(n, 256);
    // gather from a pitched source into a pitched destination: use scatter4 with dims (1,1,rows,cols) twice-strided
    // dst[r*ldd + c] = src[r*lds + c]  -> implemented as a permute into a dense temp view when ldd == cols
#define CAST_CASE(TI, TO)                                                                                         \
    if (ldd == cols)                                                                                              \
        permute4_kernel<TI, TO><<<g, 256, 0, st>>>(reinterpret_cast<const TI*>(src), reinterpret_cast<TO*>(dst), 1, 1, \
                                                   (int)rows, cols, 0, 0, lds, 1, 0);                             \
    else if (lds == cols)                                                                                         \
        scatter4_kernel<TI, TO><<<g, 256, 0, st>>>(reinterpret_cast<const TI*>(src), reinterpret_cast<TO*>(dst), 1, 1, \
                                                   (int)rows, cols, 0, 0, ldd, 1, 0);                             \
    else                                                                                                          \
        return fail(FMRI_ERR_UNSUPPORTED, "cast2d needs one dense side");
    if (src_dtype == FMRI_F32 && dst_dtype == FMRI_BF16) {
        CAST_CASE(float, __nv_bfloat16)
    } else if (src_dtype == FMRI_BF16 && dst_dtype == FMRI_F32) {
        CAST_CASE(__nv_bfloat16, float)
    } else if (src_dtype == FMRI_F32 && dst_dtype == FMRI_F32) {
        CAST_CASE(float, float)
    } else {
        CAST_CASE(__nv_bfloat16, __nv_bfloat16)
    }
#undef CAST_CASE
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ losses
extern "C" int fmri_reparam_kl_fwd(const float* mu, const float* logvar, int ld, const float* eps, float* z, float* kl,
                                   int B, int Z, void* stream) {
    if (z && !eps) return fail(FMRI_ERR_ARG, "reparam needs eps");
    if (ld < Z) return fail(FMRI_ERR_ARG, "reparam pitch < Z");
    reparam_kl_fwd_kernel<<<cdiv(B, 4), 128, 0, S(stream)>>>(mu, logvar, ld, eps, z, kl, B, Z);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_reparam_kl_bwd(const float* mu, const float* logvar, int ld, const float* eps, const float* gz,
                                   const float* gkl, float gkl_const, void* dmu, void* dlogvar, int ldd, int d_dtype,
                                   int B, int Z, void* stream) {
    if (ld < Z || ldd < Z) return fail(FMRI_ERR_ARG, "reparam pitch < Z");
    const int g = grid1d((long long)B * Z, 256);
    if (d_dtype == FMRI_BF16)
        reparam_kl_bwd_kernel<__nv_bfloat16><<<g, 256, 0, S(stream)>>>(
            mu, logvar, ld, eps, gz, gkl, gkl_const, reinterpret_cast<__nv_bfloat16*>(dmu),
            reinterpret_cast<__nv_bfloat16*>(dlogvar), ldd, B, Z);
    else
        reparam_kl_bwd_kernel<float><<<g, 256, 0, S(stream)>>>(mu, logvar, ld, eps, gz, gkl, gkl_const,
                                                              reinterpret_cast<float*>(dmu),
                                                              reinterpret_cast<float*>(dlogvar), ldd, B, Z);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_rowsqdiff_fwd(const void* a, const void* b, int dtype, float* out, long long rows, long long F,
                                  float scale, void* stream) {
    if (dtype == FMRI_BF16)
        rowsqdiff_fwd_kernel<__nv_bfloat16><<<(unsigned)rows, 256, 0, S(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(a), reinterpret_cast<const __nv_bfloat16*>(b), out, F, scale);
    else
        rowsqdiff_fwd_kernel<float><<<(unsigned)rows, 256, 0, S(stream)>>>(reinterpret_cast<const float*>(a),
                                                                          reinterpret_cast<const float*>(b), out, F,
                                                                          scale);
    LAUNCH_OK();
    return 0;
}
// ------------------------------------------------------------------------------------------------ WAE-MMD (extension)
static size_t mmd_smem() { return sizeof(float) * (size_t)(2 * MMD_T * MMD_LD + MMD_T * (MMD_T + 1)); }
static int mmd_check(int B, int Z) {
    if (B < 2) return fail(FMRI_ERR_ARG, "mmd: the unbiased estimator needs B >= 2 (got %d)", B);
    if (Z < 1 || Z > MMD_KC * MMD_MAXCH) return fail(FMRI_ERR_ARG, "mmd: Z=%d outside [1, %d]", Z, MMD_KC * MMD_MAXCH);
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(mmd_imq_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mmd_smem());
        cudaFuncSetAttribute(mmd_imq_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mmd_smem());
        attr = true;
    }
    return 0;
}
// j-tile slices so that the grid fills the 148 SMs twice over (2 resident CTAs per SM)
static int mmd_splits(int base_ctas, int ntj) { return std::max(1, std::min(ntj, (2 * 148 + base_ctas - 1) / base_ctas)); }
extern "C" int fmri_mmd_imq_fwd(const float* zq, int ldq, const float* zp, int ldp, int B, int Z, float sigma2,
                                float lambda, float* mmd, double* ws, void* stream) {
    if (int rc = mmd_check(B, Z)) return rc;
    if (!zq || !zp || !mmd || !ws) return fail(FMRI_ERR_ARG, "mmd_fwd: null pointer");
    MmdParams P{};
    P.q = zq; P.p = zp; P.ldq = ldq; P.ldp = ldp; P.B = B; P.Z = Z;
    P.cbase = 2.f * (float)Z * sigma2;
    P.stat = ws;
    const int nt = (B + MMD_T - 1) / MMD_T;
    P.nsplit = mmd_splits(2 * nt, nt);
    cudaMemsetAsync(ws, 0, 3 * sizeof(double), S(stream));
    dim3 grid(nt, 2, P.nsplit);
    mmd_imq_kernel<false><<<grid, MMD_THREADS, mmd_smem(), S(stream)>>>(P);
    LAUNCH_OK();
    mmd_finalize_kernel<<<1, 1, 0, S(stream)>>>(ws, B, lambda, mmd);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_mmd_imq_bwd(const float* zq, int ldq, const float* zp, int ldp, int B, int Z, float sigma2,
                                float lambda, float* dzq, int ldd, int accumulate, void* stream) {
    if (int rc = mmd_check(B, Z)) return rc;
    if (!zq || !zp || !dzq) return fail(FMRI_ERR_ARG, "mmd_bwd: null pointer");
    MmdParams P{};
    P.q = zq; P.p = zp; P.ldq = ldq; P.ldp = ldp; P.B = B; P.Z = Z;
    P.cbase = 2.f * (float)Z * sigma2;
    P.dq = dzq; P.ldd = ldd; P.accumulate = accumulate;
    const double b = (double)B;
    P.w_same = (float)(lambda * 4.0 / (b * (b - 1.0)));
    P.w_cross = (float)(-lambda * 4.0 / (b * b));
    const int nt = (B + MMD_T - 1) / MMD_T, nch = (Z + MMD_KC - 1) / MMD_KC;
    P.nsplit = mmd_splits(nt * nch, nt);
    if (P.nsplit > 1 && !accumulate)
        cudaMemset2DAsync(dzq, (size_t)ldd * sizeof(float), 0, (size_t)Z * sizeof(float), (size_t)B, S(stream));
    dim3 grid(nt, 1, P.nsplit * nch);
    mmd_imq_kernel<true><<<grid, MMD_THREADS, mmd_smem(), S(stream)>>>(P);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_rowsqdiff_bwd(const void* a, const void* b, int dtype, const float* g, void* da, void* db,
                                  long long rows, long long F, float scale, void* stream) {
    const int gr = grid1d(rows * F, 256);
    if (dtype == FMRI_BF16)
        rowsqdiff_bwd_kernel<__nv_bfloat16><<<gr, 256, 0, S(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(a), reinterpret_cast<const __nv_bfloat16*>(b), g,
            reinterpret_cast<__nv_bfloat16*>(da), reinterpret_cast<__nv_bfloat16*>(db), rows, F, scale);
    else
        rowsqdiff_bwd_kernel<float><<<gr, 256, 0, S(stream)>>>(reinterpret_cast<const float*>(a),
                                                              reinterpret_cast<const float*>(b), g,
                                                              reinterpret_cast<float*>(da),
                                                              reinterpret_cast<float*>(db), rows, F, scale);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_head_sigmoid_fwd(const void* x, int dtype, const float* w, const float* bias, float* p, int rows,
                                     int F, void* stream) {
    if (dtype == FMRI_BF16)
        head_sigmoid_fwd_kernel<__nv_bfloat16><<<cdiv(rows, 4), 128, 0, S(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(x), w, bias, p, rows, F);
    else
        head_sigmoid_fwd_kernel<float><<<cdiv(rows, 4), 128, 0, S(stream)>>>(reinterpret_cast<const float*>(x), w, bias,
                                                                            p, rows, F);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_head_sigmoid_bwd(const void* x, int dtype, const float* w, const float* p, const float* gp,
                                     void* dx, float* dw, float* db, int rows, int F, void* stream) {
    const int rpb = 16;
    const int nb = cdiv(rows, rpb);
    SCRATCH(part, float, (long long)nb * (F + 1), S(stream));   // per-block dw [nb][F], then db [nb]
    float* pw = dw ? part : nullptr;
    float* pb = db ? part + (long long)nb * F : nullptr;
    if (dtype == FMRI_BF16)
        head_sigmoid_bwd_kernel<__nv_bfloat16><<<nb, 256, 0, S(stream)>>>(
            reinterpret_cast<const __nv_bfloat16*>(x), w, p, gp, reinterpret_cast<__nv_bfloat16*>(dx), pw, pb, rows, F,
            rpb);
    else
        head_sigmoid_bwd_kernel<float><<<nb, 256, 0, S(stream)>>>(
            reinterpret_cast<const float*>(x), w, p, gp, reinterpret_cast<float*>(dx), pw, pb, rows, F, rpb);
    LAUNCH_OK();
    int rc = dw ? ordered_add(pw, nb, F, dw, S(stream)) : 0;
    if (!rc && db) rc = ordered_add(pb, nb, 1, db, S(stream));
    CUDA_OK(cudaFreeAsync(part, S(stream)));
    return rc;
}
extern "C" int fmri_bce_fwd(const float* p, float* out, int n, int positive, float scale, void* stream) {
    bce_fwd_kernel<<<cdiv(n, 256), 256, 0, S(stream)>>>(p, out, n, positive, scale);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_bce_bwd(const float* p, const float* g, float* dp, int n, int positive, float scale,
                            int accumulate, void* stream) {
    bce_bwd_kernel<<<cdiv(n, 256), 256, 0, S(stream)>>>(p, g, dp, n, positive, scale, accumulate);
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ optimizers
static void mt_fill(MtArgs& a, int base, int n, float* const* p, const float* const* g, float* const* s1,
                    float* const* s2, const int64_t* numel, int64_t* mx) {
    a.count = std::min(FMRI_MT_MAX, n - base);
    *mx = 0;
    for (int i = 0; i < a.count; ++i) {
        a.t[i].p = p[base + i];
        a.t[i].g = g[base + i];
        a.t[i].s1 = s1[base + i];
        a.t[i].s2 = s2 ? s2[base + i] : nullptr;
        a.t[i].n = numel[base + i];
        *mx = std::max(*mx, numel[base + i]);
    }
}
extern "C" int fmri_multi_tensor_rmsprop(int n, float* const* p, const float* const* g, float* const* sq,
                                         const int64_t* numel, float lr, float alpha, float eps, float clamp,
                                         const float* lr_dev, const float* gate_dev, void* stream) {
    for (int base = 0; base < n; base += FMRI_MT_MAX) {
        MtArgs a;
        int64_t mx;
        mt_fill(a, base, n, p, g, sq, nullptr, numel, &mx);
        dim3 grid(std::max(1, std::min(148 * 8, cdiv(mx, 256 * 4))), a.count);
        mt_rmsprop_kernel<<<grid, 256, 0, S(stream)>>>(a, lr, alpha, eps, clamp, lr_dev, gate_dev);
        LAUNCH_OK();
    }
    return 0;
}
extern "C" int fmri_multi_tensor_adam(int n, float* const* p, const float* const* g, float* const* m, float* const* v,
                                      const int64_t* numel, float lr, float beta1, float beta2, float eps, int step,
                                      float clamp, const float* lr_dev, const float* gate_dev, void* stream) {
    const float bc1 = (float)(1.0 - pow((double)beta1, (double)step)), bc2 = (float)(1.0 - pow((double)beta2, (double)step));
    for (int base = 0; base < n; base += FMRI_MT_MAX) {
        MtArgs a;
        int64_t mx;
        mt_fill(a, base, n, p, g, m, v, numel, &mx);
        dim3 grid(std::max(1, std::min(148 * 8, cdiv(mx, 256 * 4))), a.count);
        mt_adam_kernel<<<grid, 256, 0, S(stream)>>>(a, lr, beta1, beta2, eps, bc1, bc2, clamp, lr_dev, gate_dev, nullptr);
        LAUNCH_OK();
    }
    return 0;
}
extern "C" int fmri_multi_tensor_adam_dev(int n, float* const* p, const float* const* g, float* const* m, float* const* v,
                                          const int64_t* numel, float lr, float beta1, float beta2, float eps,
                                          const int* step_dev, float clamp, const float* lr_dev, const float* gate_dev,
                                          void* stream) {
    if (!step_dev) return fail(FMRI_ERR_ARG, "multi_tensor_adam_dev needs the device step counter");
    for (int base = 0; base < n; base += FMRI_MT_MAX) {
        MtArgs a;
        int64_t mx;
        mt_fill(a, base, n, p, g, m, v, numel, &mx);
        dim3 grid(std::max(1, std::min(148 * 8, cdiv(mx, 256 * 4))), a.count);
        mt_adam_kernel<<<grid, 256, 0, S(stream)>>>(a, lr, beta1, beta2, eps, 1.f, 1.f, clamp, lr_dev, gate_dev, step_dev);
        LAUNCH_OK();
    }
    return 0;
}
extern "C" int fmri_step_increment(int* step_dev, void* stream) {
    if (!step_dev) return fail(FMRI_ERR_ARG, "step_increment needs a device counter");
    step_increment_kernel<<<1, 1, 0, S(stream)>>>(step_dev);
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ step glue
extern "C" int fmri_axpby_tanh_bwd(float a, const float* x, float b, const float* y, const float* img, float* out,
                                   long long n, void* stream) {
    axpby_tanh_bwd_kernel<<<grid1d(n, 256), 256, 0, S(stream)>>>(a, x, b, y, img, out, n);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_chansum_nchw(const float* x, int N, int C, long long HW, float* out, int accumulate, void* stream) {
    if (!accumulate) CUDA_OK(cudaMemsetAsync(out, 0, sizeof(float) * C, S(stream)));
    dim3 grid(C, std::max(1, std::min(N, 148 * 2 / std::max(C, 1))));
    SCRATCH(part, float, (long long)grid.y * C, S(stream));
    chansum_nchw_kernel<<<grid, 256, 0, S(stream)>>>(x, N, C, HW, part);
    LAUNCH_OK();
    int rc = ordered_add(part, (int)grid.y, C, out, S(stream));
    CUDA_OK(cudaFreeAsync(part, S(stream)));
    return rc;
}
extern "C" int fmri_vecsum(const float* x, long long n, float scale, float* out, int accumulate, void* stream) {
    vecsum_kernel<<<1, 256, 0, S(stream)>>>(x, n, scale, out, accumulate);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_vgan_gate_mix(const float* sums, float count, float margin, float equilibrium, int train_dis_in,
                                  float* gates, void* stream) {
    vgan_gate_kernel<<<1, 32, 0, S(stream)>>>(sums, count, margin, equilibrium, train_dis_in, gates);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_vgan_gate(const float* sums, float count, float margin, float equilibrium, float* gates,
                              void* stream) {
    return fmri_vgan_gate_mix(sums, count, margin, equilibrium, 1, gates, stream);
}
extern "C" int fmri_scale_f32(float* x, long long n, float s, void* stream) {
    if (!x || n < 0) return fail(FMRI_ERR_ARG, "scale_f32 arguments");
    if (n == 0) return 0;
    scale_f32_kernel<<<grid1d(n, 256), 256, 0, S(stream)>>>(x, n, s);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_bn_eval_stats(const float* running_mean, const float* running_var, int C, float eps, float* mean,
                                  float* invstd, void* stream) {
    bn_eval_stats_kernel<<<cdiv(C, 128), 128, 0, S(stream)>>>(running_mean, running_var, C, eps, mean, invstd);
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ inference / metrics / input
extern "C" int fmri_bn_fold(const float* w, long long n, long long inner, int C, const float* running_mean,
                            const float* running_var, const float* gamma, const float* beta, float eps, float* w_out,
                            float* b_out, void* stream) {
    if (!w || !w_out || !b_out || n <= 0 || inner <= 0 || C <= 0) return fail(FMRI_ERR_ARG, "bn_fold arguments");
    bn_fold_kernel<<<grid1d(std::max<long long>(n, C), 256), 256, 0, S(stream)>>>(w, n, inner, C, running_mean, running_var,
                                                                                 gamma, beta, eps, w_out, b_out);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_pearson(const float* a, const float* b, long long n, float* out, double* ws, void* stream) {
    if (!a || !b || !out || !ws || n <= 0) return fail(FMRI_ERR_ARG, "pearson arguments");
    CUDA_OK(cudaMemsetAsync(ws, 0, sizeof(double) * 5, S(stream)));
    pearson_sums_kernel<<<grid1d(n, 256, 148 * 8), 256, 0, S(stream)>>>(a, b, n, ws);
    LAUNCH_OK();
    pearson_final_kernel<<<1, 1, 0, S(stream)>>>(ws, (double)n, out);
    LAUNCH_OK();
    return 0;
}
// gaussian(window_size, 1.5) of train_utils.py:310-323, evaluated in double and rounded to float like torch.Tensor([...]),
// normalised by its fp32 sum; taps beyond `win` are zero. fmri_ssim and fmri_pairwise_similarity share these floats.
static SsimWindow ssim_window(int win) {
    SsimWindow wd;
    double g[11];
    for (int x = 0; x < win; ++x) {
        const double d = x - win / 2;
        g[x] = (double)(float)exp(-(d * d) / (2.0 * 1.5 * 1.5));
    }
    float fs = 0.f;
    for (int x = 0; x < win; ++x) fs += (float)g[x];
    for (int x = 0; x < 11; ++x) wd.g[x] = x < win ? (float)g[x] / fs : 0.f;
    return wd;
}
extern "C" int fmri_ssim(const float* a, const float* b, int N, int C, int H, int W, float* out, double* ws, void* stream) {
    if (!a || !b || !out || !ws || N <= 0 || C <= 0 || H <= 0 || W <= 0) return fail(FMRI_ERR_ARG, "ssim arguments");
    // below 11 pixels the reference pads by 5 around a SMALLER window and its SSIM map outgrows the image (train_utils.py:378-390)
    if (H < 11 || W < 11) return fail(FMRI_ERR_UNSUPPORTED, "ssim: images smaller than the 11 x 11 window (%d x %d)", H, W);
    const int win = std::min(11, std::min(H, W));
    const SsimWindow wd = ssim_window(win);
    CUDA_OK(cudaMemsetAsync(ws, 0, sizeof(double), S(stream)));
    const long long total = (long long)N * C * H * W;
    ssim_kernel<<<grid1d(total, 256, 148 * 8), 256, 0, S(stream)>>>(a, b, N * C, H, W, win, wd, ws);
    LAUNCH_OK();
    scale_d2f_kernel<<<1, 1, 0, S(stream)>>>(ws, 1.0 / (double)total, out);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_image_pipeline(const unsigned char* src, int N, int H, int W, int Csrc, const int* flip,
                                   const int* shift_yx, const float* mean3, const float* std3, float* dst, void* stream) {
    if (!src || !dst || N <= 0 || H <= 0 || W <= 0 || (Csrc != 1 && Csrc != 3)) return fail(FMRI_ERR_ARG, "image_pipeline arguments");
    const float m[3] = {mean3 ? mean3[0] : 0.f, mean3 ? mean3[1] : 0.f, mean3 ? mean3[2] : 0.f};
    const float sd[3] = {std3 ? std3[0] : 1.f, std3 ? std3[1] : 1.f, std3 ? std3[2] : 1.f};
    image_pipeline_kernel<<<grid1d((long long)N * 3 * H * W, 256, 148 * 8), 256, 0, S(stream)>>>(
        src, N, H, W, Csrc, flip, shift_yx, m[0], m[1], m[2], sd[0], sd[1], sd[2], dst);
    LAUNCH_OK();
    return 0;
}

// ================================================================================================ all-pairs similarity
static inline long long ssim_pitch_w(int W) { return ((long long)W + 7) / 8 * 8; }
extern "C" size_t fmri_pairwise_workspace(int N, int M, int C, int H, int W, int metric) {
    if (N <= 0 || M <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
    if (metric == FMRI_METRIC_PCC) return sizeof(double2) * ((size_t)N + (size_t)M);
    if (metric == FMRI_METRIC_SSIM) return sizeof(float) * 2 * ((size_t)N + (size_t)M) * C * H * ssim_pitch_w(W);
    return 0;
}
extern "C" int fmri_pairwise_similarity(const float* pred, int N, const float* target, int M, int C, int H, int W,
                                        int metric, float* out, void* ws, size_t ws_bytes, void* stream) {
    if (!pred || !target || !out || N <= 0 || M <= 0 || C <= 0 || H <= 0 || W <= 0)
        return fail(FMRI_ERR_ARG, "pairwise_similarity arguments");
    if (metric != FMRI_METRIC_PCC && metric != FMRI_METRIC_SSIM) return fail(FMRI_ERR_ARG, "unknown metric %d", metric);
    if (metric == FMRI_METRIC_SSIM && (H < 11 || W < 11))
        return fail(FMRI_ERR_UNSUPPORTED, "ssim: images smaller than the 11 x 11 window (%d x %d)", H, W);
    const size_t need = fmri_pairwise_workspace(N, M, C, H, W, metric);
    if (!ws || ws_bytes < need) return fail(FMRI_ERR_WORKSPACE, "pairwise_similarity workspace %zu < %zu", ws_bytes, need);
    if (reinterpret_cast<uintptr_t>(ws) % 16) return fail(FMRI_ERR_ARG, "pairwise_similarity workspace not 16-byte aligned");
    const long long K = (long long)C * H * W;
    if (metric == FMRI_METRIC_PCC) {
        if (cdiv(M, PG_BN) > 65535) return fail(FMRI_ERR_UNSUPPORTED, "pairwise pcc: M = %d targets", M);
        double2* sa = reinterpret_cast<double2*>(ws);
        double2* sb = sa + N;
        pcc_stats_kernel<<<N, PCC_STAT_THREADS, 0, S(stream)>>>(pred, K, sa);
        LAUNCH_OK();
        pcc_stats_kernel<<<M, PCC_STAT_THREADS, 0, S(stream)>>>(target, K, sb);
        LAUNCH_OK();
        pcc_gemm_kernel<<<dim3(cdiv(N, PG_BM), cdiv(M, PG_BN)), PG_THREADS, 0, S(stream)>>>(pred, N, target, M, K, sa, sb,
                                                                                              out);
        LAUNCH_OK();
        return 0;
    }
    if (cdiv(M, SS_TJ) > 65535) return fail(FMRI_ERR_UNSUPPORTED, "pairwise ssim: M = %d targets", M);
    SsimPairArgs p;
    p.a = pred;
    p.b = target;
    p.N = N, p.M = M, p.C = C, p.H = H, p.W = W, p.WP = (int)ssim_pitch_w(W);
    const long long plane = (long long)H * p.WP;
    float* maps = reinterpret_cast<float*>(ws);
    p.mu_a = maps;
    p.sig_a = maps + (long long)N * C * plane;
    p.mu_b = maps + 2LL * N * C * plane;
    p.sig_b = p.mu_b + (long long)M * C * plane;
    // equal column groups of at most SS_MAXW * 8 columns, each a multiple of 8 wide
    const int groups = cdiv(W, SS_MAXW * SS_R);
    p.cols = cdiv(cdiv(W, groups), SS_R) * SS_R;
    p.pitch = ss_pitch(p.cols + 10);
    p.inv_count = 1.0 / (double)K;
    p.wd = ssim_window(11);
    p.out = out;
    const size_t smem = sizeof(float) * 2 * SS_BAND * SS_IMGS * p.pitch;   // two band buffers
    CUDA_OK(cudaFuncSetAttribute(ssim_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ssim_maps_kernel<<<grid1d((long long)N * C * plane, 256), 256, 0, S(stream)>>>(pred, (long long)N * C, H, W, p.WP, p.wd,
                                                                                     const_cast<float*>(p.mu_a),
                                                                                     const_cast<float*>(p.sig_a));
    LAUNCH_OK();
    ssim_maps_kernel<<<grid1d((long long)M * C * plane, 256), 256, 0, S(stream)>>>(target, (long long)M * C, H, W, p.WP,
                                                                                     p.wd, const_cast<float*>(p.mu_b),
                                                                                     const_cast<float*>(p.sig_b));
    LAUNCH_OK();
    ssim_pair_kernel<<<dim3(cdiv(N, SS_TI), cdiv(M, SS_TJ)), p.cols / SS_R * 32, smem, S(stream)>>>(p);
    LAUNCH_OK();
    return 0;
}
extern "C" int fmri_identification(const float* sim, int N, const int* ns, int n_count, int* wins, double* acc,
                                   void* stream) {
    if (!sim || !wins || N < 2) return fail(FMRI_ERR_ARG, "identification needs an [N, N] matrix with N >= 2 (N = %d)", N);
    if (n_count <= 0 || !ns || !acc) return fail(FMRI_ERR_ARG, "identification: needs n_count >= 1, ns and acc");
    for (int q = 0; q < n_count; ++q)
        if (ns[q] < 2 || ns[q] > N) return fail(FMRI_ERR_ARG, "identification: n = %d outside [2, %d]", ns[q], N);
    ident_wins_kernel<<<cdiv(N, 8), 256, 0, S(stream)>>>(sim, N, wins);
    LAUNCH_OK();
    for (int q0 = 0; q0 < n_count; q0 += IDENT_MAX_NS) {
        IdentNs p;
        p.count = std::min(IDENT_MAX_NS, n_count - q0);
        for (int q = 0; q < p.count; ++q) p.n[q] = ns[q0 + q];
        ident_acc_kernel<<<1, 256, 0, S(stream)>>>(wins, N, p, acc + q0);
        LAUNCH_OK();
    }
    return 0;
}
