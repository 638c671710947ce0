"""ctypes binding of libfmri_b200.so (C ABI in include/fmri_b200.h).

The library is the product: there is no Python/CPU fallback. Loading fails loudly if the shared object is missing
(run ``python -c "import __graft_entry__ as g; g.build()"``), and every wrapper raises ``FmriError`` on a non-zero
status with the library's own message.
"""
from __future__ import annotations

import ctypes as C
import os
import re

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FMRI_B200_LIB", os.path.join(_HERE, "libfmri_b200.so"))  # override: same-box kernel A/B runs
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "fmri_b200.h")

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3
METRIC_PCC, METRIC_SSIM = 0, 1


class FmriError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("N", "H", "W", "Cin", "Cout", "stride", "transposed", "output_pad", "dtype")]


class EdgeDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("N", "H", "W", "C", "stride", "dtype")]


class ReluMask(C.Structure):
    _fields_ = [("y", C.c_void_p), ("bits", C.c_void_p)]


class LinearDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("M", "N", "K", "dtype")]


def header_functions():
    """Names of every function the public header declares (used by the CPU-side export test)."""
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fmri_[a-z0-9_]+)\s*\(", src)))


_lib = None
PROF = None      # list of (entry point, algorithmic flops, start event, end event) while profiling
_FLOPS = 0.0     # algorithmic FLOPs of the next call (set by the conv / linear wrappers)


class _Proxy:
    """Attribute proxy over the CDLL: while profiling is on, brackets every entry point with CUDA events on the
    current stream (the stream the library launches on)."""

    def __init__(self, cdll):
        self._c = cdll

    def __getattr__(self, name):
        f = getattr(self._c, name)
        if PROF is None or name in ("fmri_last_error", "fmri_conv_out_hw", "fmri_conv_wgrad_workspace",
                                    "fmri_edge_workspace", "fmri_launch_count", "fmri_version", "fmri_conv_pack_elems",
                                    "fmri_pairwise_workspace"):
            return f

        def timed(*a):
            global _FLOPS
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = f(*a)
            e1.record()
            PROF.append((name, _FLOPS, e0, e1))
            _FLOPS = 0.0
            return rc

        return timed


def profile_begin():
    global PROF
    PROF = []


def profile_end():
    """Stop profiling; returns {entry point: dict(ms=total device ms, calls=n, flops=total algorithmic flops)}."""
    global PROF
    torch.cuda.synchronize()
    agg = {}
    for name, fl, e0, e1 in PROF or []:
        a = agg.setdefault(name, dict(ms=0.0, calls=0, flops=0.0))
        a["ms"] += e0.elapsed_time(e1)
        a["calls"] += 1
        a["flops"] += fl
    PROF = None
    return agg


def launch_count(reset=False):
    return int(load().fmri_launch_count(int(reset)))


def _conv_flops(d):
    if d.transposed:
        return 2.0 * d.N * d.H * d.W * d.Cin * d.Cout * 25
    oh, ow = (d.H - 1) // d.stride + 1, (d.W - 1) // d.stride + 1
    return 2.0 * d.N * oh * ow * d.Cin * d.Cout * 25


def _note_flops(v):
    global _FLOPS
    if PROF is not None:
        _FLOPS = float(v)


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FmriError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no fallback path."
            )
        c = C.CDLL(LIB_PATH)
        c.fmri_last_error.restype = C.c_char_p
        c.fmri_conv_wgrad_workspace.restype = C.c_size_t
        c.fmri_conv_pack_elems.restype = C.c_size_t
        c.fmri_edge_workspace.restype = C.c_size_t
        c.fmri_pairwise_workspace.restype = C.c_size_t
        c.fmri_conv_out_hw.restype = None
        c.fmri_launch_count.restype = C.c_longlong
        _lib = _Proxy(c)
    return _lib


def _check(rc):
    if rc != 0:
        raise FmriError(f"libfmri_b200 status {rc}: {load().fmri_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dt(t_or_dtype):
    d = t_or_dtype.dtype if isinstance(t_or_dtype, torch.Tensor) else t_or_dtype
    if d == torch.float32:
        return F32
    if d == torch.bfloat16:
        return BF16
    raise FmriError(f"unsupported dtype {d}")


def _ll(v):
    return C.c_longlong(int(v))


def _f(v):
    return C.c_float(float(v))


def _require_cuda(*ts, contiguous=True):
    """contiguous=False for entry points that take explicit row pitches (pitched views are passed by base pointer)."""
    for t in ts:
        if t is not None and not t.is_cuda:
            raise FmriError("libfmri_b200 operates on CUDA tensors only (no CPU fallback)")
        if contiguous and t is not None and not t.is_contiguous():
            raise FmriError("libfmri_b200 expects contiguous tensors")


# ------------------------------------------------------------------------------------------------ convs
def conv_desc(N, H, W, Cin, Cout, stride, transposed, output_pad, dtype):
    return ConvDesc(N, H, W, Cin, Cout, stride, int(transposed), int(output_pad), dt(dtype))


def conv_out_hw(d):
    oh, ow = C.c_int(), C.c_int()
    load().fmri_conv_out_hw(C.byref(d), C.byref(oh), C.byref(ow))
    return oh.value, ow.value


def conv_pack_elems(d):
    return load().fmri_conv_pack_elems(C.byref(d))


def conv_pack_weights(d, w, pack_f, pack_d):
    _require_cuda(w, pack_f, pack_d)
    _check(load().fmri_conv_pack_weights(C.byref(d), ptr(w), ptr(pack_f), ptr(pack_d), stream()))


def conv_fprop(d, x, w, pack_f, bias, act, y, stat_sum=None, stat_sq=None):
    _require_cuda(x, w, pack_f, bias, y, stat_sum, stat_sq)
    _note_flops(_conv_flops(d))
    _check(load().fmri_conv_fprop(C.byref(d), ptr(x), ptr(w), ptr(pack_f), ptr(bias), act, ptr(y), ptr(stat_sum),
                                  ptr(stat_sq), stream()))


def conv_dgrad(d, dy, w, pack_d, dx, relu_mask=None):
    """relu_mask = (y, bits or None): dx is the upstream gradient of a bias+ReLU layer with output y; the call also
    applies its ReLU backward, dx *= (y > 0) (bits: relu_bitmask of y, 32-channel tensors)."""
    _require_cuda(dy, w, pack_d, dx)
    _note_flops(_conv_flops(d))
    m = None
    if relu_mask is not None:
        y, bits = relu_mask
        _require_cuda(y, bits)
        m = ReluMask(ptr(y), ptr(bits))
    _check(load().fmri_conv_dgrad(C.byref(d), ptr(dy), ptr(w), ptr(pack_d), ptr(dx), C.byref(m) if m else None, stream()))


def conv_wgrad_workspace(d):
    return load().fmri_conv_wgrad_workspace(C.byref(d))


def conv_wgrad(d, x, dy, dw, accumulate, ws):
    _require_cuda(x, dy, dw, ws)
    nbytes = ws.numel() * ws.element_size() if ws is not None else 0
    _note_flops(_conv_flops(d))
    _check(load().fmri_conv_wgrad(C.byref(d), ptr(x), ptr(dy), ptr(dw), int(accumulate), ptr(ws), C.c_size_t(nbytes),
                                  stream()))


def edge_desc(N, H, W, Cc, stride, dtype):
    return EdgeDesc(N, H, W, Cc, stride, dt(dtype))


def edge_workspace(d):
    return load().fmri_edge_workspace(C.byref(d))


def _wsb(ws):
    return C.c_size_t(ws.numel() * ws.element_size())


def edge_in_fprop(d, imgs, n_per_src, w, bias, act, y, ws):
    i0, i1, i2 = (list(imgs) + [None, None])[:3]
    _require_cuda(i0, i1, i2, w, bias, y, ws)
    _check(load().fmri_edge_in_fprop(C.byref(d), ptr(i0), ptr(i1), ptr(i2), n_per_src, ptr(w), ptr(bias), act, ptr(y),
                                     ptr(ws), _wsb(ws), stream()))


def edge_in_dgrad(d, dy, w, dimg, ws):
    _require_cuda(dy, w, dimg, ws)
    _check(load().fmri_edge_in_dgrad(C.byref(d), ptr(dy), ptr(w), ptr(dimg), ptr(ws), _wsb(ws), stream()))


def edge_in_wgrad(d, imgs, n_per_src, dy, dw, accumulate, ws, dbias=None):
    i0, i1, i2 = (list(imgs) + [None, None])[:3]
    _require_cuda(i0, i1, i2, dy, dw, ws, dbias)
    _check(load().fmri_edge_in_wgrad(C.byref(d), ptr(i0), ptr(i1), ptr(i2), n_per_src, ptr(dy), ptr(dw), ptr(dbias),
                                     int(accumulate), ptr(ws), _wsb(ws), stream()))


def edge_out_fprop(d, x, w, bias, act, img, ws):
    _require_cuda(x, w, bias, img, ws)
    _check(load().fmri_edge_out_fprop(C.byref(d), ptr(x), ptr(w), ptr(bias), act, ptr(img), ptr(ws), _wsb(ws),
                                      stream()))


def edge_out_dgrad(d, dimg, w, dx, ws):
    _require_cuda(dimg, w, dx, ws)
    _check(load().fmri_edge_out_dgrad(C.byref(d), ptr(dimg), ptr(w), ptr(dx), ptr(ws), _wsb(ws), stream()))


def edge_out_wgrad(d, x, dimg, dw, accumulate, ws):
    _require_cuda(x, dimg, dw, ws)
    _check(load().fmri_edge_out_wgrad(C.byref(d), ptr(x), ptr(dimg), ptr(dw), int(accumulate), ptr(ws), _wsb(ws),
                                      stream()))


# ------------------------------------------------------------------------------------------------ linear
def linear_desc(M, N, K, dtype):
    return LinearDesc(M, N, K, dt(dtype))


def linear_pack_weights(d, w, wp, ldw, wpt, ldwt):
    _require_cuda(w, wp, wpt, contiguous=False)
    _check(load().fmri_linear_pack_weights(C.byref(d), ptr(w), ptr(wp), ldw, ptr(wpt), ldwt, stream()))


def linear_fprop(d, x, ldx, w, wp, ldw, bias, act, y, ldy):
    _require_cuda(x, w, wp, bias, y, contiguous=False)
    _note_flops(2.0 * d.M * d.N * d.K)
    _check(load().fmri_linear_fprop(C.byref(d), ptr(x), ldx, ptr(w), ptr(wp), ldw, ptr(bias), act, ptr(y), ldy,
                                    dt(y), stream()))


def linear_dgrad(d, dy, lddy, w, wpt, ldwt, dx, lddx, accumulate=False):
    _require_cuda(dy, w, wpt, dx, contiguous=False)
    _note_flops(2.0 * d.M * d.N * d.K)
    _check(load().fmri_linear_dgrad(C.byref(d), ptr(dy), lddy, ptr(w), ptr(wpt), ldwt, ptr(dx), lddx, dt(dx),
                                    int(accumulate), stream()))


def linear_wgrad(d, x, ldx, dy, lddy, dw, accumulate):
    _require_cuda(x, dy, dw, contiguous=False)
    _note_flops(2.0 * d.M * d.N * d.K)
    _check(load().fmri_linear_wgrad(C.byref(d), ptr(x), ldx, ptr(dy), lddy, ptr(dw), int(accumulate), stream()))


# ------------------------------------------------------------------------------------------------ BN / elementwise
def colstats(x, rows, Cc, s, q):
    _require_cuda(x, s, q)
    _check(load().fmri_colstats(ptr(x), dt(x), _ll(rows), Cc, ptr(s), ptr(q), stream()))


def bn_finalize(s, q, rows, Cc, eps, momentum, mean, invstd, running_mean, running_var):
    _check(load().fmri_bn_finalize(ptr(s), ptr(q), _ll(rows), Cc, _f(eps), _f(momentum), ptr(mean), ptr(invstd),
                                   ptr(running_mean), ptr(running_var), stream()))


def bn_apply(x, y, rows, Cc, mean, invstd, gamma, beta, relu):
    _require_cuda(x, y, mean, invstd, gamma, beta)
    _check(load().fmri_bn_apply(ptr(x), dt(x), ptr(y), dt(y), _ll(rows), Cc, ptr(mean), ptr(invstd), ptr(gamma),
                                ptr(beta), int(relu), stream()))


def bn_backward(x, dy, dx, rows, Cc, mean, invstd, gamma, beta, relu, train, dgamma, dbeta, accumulate, ws):
    _require_cuda(x, dy, dx, mean, invstd, gamma, beta, dgamma, dbeta, ws)
    _check(load().fmri_bn_backward(ptr(x), dt(x), ptr(dy), ptr(dx), dt(dy), _ll(rows), Cc, ptr(mean), ptr(invstd),
                                   ptr(gamma), ptr(beta), int(relu), int(train), ptr(dgamma), ptr(dbeta),
                                   int(accumulate), ptr(ws), stream()))


def bn_backward_slice(x, dy, dx, rows, row0, nrows, Cc, mean, invstd, gamma, beta, relu, train, ws):
    """BatchNorm backward whose sums run over all `rows` but whose dx is produced for rows [row0, row0 + nrows) only."""
    _require_cuda(x, dy, dx, mean, invstd, gamma, beta, ws)
    _check(load().fmri_bn_backward_slice(ptr(x), dt(x), ptr(dy), ptr(dx), dt(dy), _ll(rows), _ll(row0), _ll(nrows), Cc,
                                         ptr(mean), ptr(invstd), ptr(gamma), ptr(beta), int(relu), int(train), None, None,
                                         0, ptr(ws), stream()))


def _same_grad_dtype(*ts):
    if len({t.dtype for t in ts if t is not None}) > 1:
        raise FmriError("the two upstreams and their gradients share one dtype")


def bn_backward_pair(x, dya, dyb, dxa, dxb, rows, Cc, mean, invstd, gamma, beta, relu, train, dgamma, dbeta, accumulate, ws):
    """Two upstreams through one BatchNorm (x read once for both); dgamma / dbeta take upstream a's. ws: 6*C doubles."""
    _same_grad_dtype(dya, dyb, dxa, dxb)
    _require_cuda(x, dya, dyb, dxa, dxb, mean, invstd, gamma, beta, dgamma, dbeta, ws)
    _check(load().fmri_bn_backward_pair(ptr(x), dt(x), ptr(dya), ptr(dyb), ptr(dxa), ptr(dxb), dt(dya), _ll(rows), Cc,
                                        ptr(mean), ptr(invstd), ptr(gamma), ptr(beta), int(relu), int(train), ptr(dgamma),
                                        ptr(dbeta), int(accumulate), ptr(ws), stream()))


def bn_backward_pair_slice(x, dya, dyb, dxa, dxb, rows, row0, nrows, Cc, mean, invstd, gamma, beta, relu, train, dgamma,
                           dbeta, accumulate, ws):
    """bn_backward_pair with upstream b's dx produced for rows [row0, row0 + nrows) only (dxb holds just those rows)."""
    _same_grad_dtype(dya, dyb, dxa, dxb)
    _require_cuda(x, dya, dyb, dxa, dxb, mean, invstd, gamma, beta, dgamma, dbeta, ws)
    _check(load().fmri_bn_backward_pair_slice(ptr(x), dt(x), ptr(dya), ptr(dyb), ptr(dxa), ptr(dxb), dt(dya), _ll(rows),
                                              _ll(row0), _ll(nrows), Cc, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta),
                                              int(relu), int(train), ptr(dgamma), ptr(dbeta), int(accumulate), ptr(ws),
                                              stream()))


def relu_backward(y, dy, dx):
    _require_cuda(y, dy, dx)
    _check(load().fmri_relu_backward(ptr(y), ptr(dy), ptr(dx), dt(y), _ll(y.numel()), stream()))


def colsum(x, rows, Cc, out):
    _require_cuda(x, out)
    _check(load().fmri_colsum(ptr(x), dt(x), _ll(rows), Cc, ptr(out), stream()))


def nchw_to_nhwc(src, dst, N, Cc, H, W):
    _require_cuda(src, dst)
    _check(load().fmri_nchw_to_nhwc(ptr(src), dt(src), ptr(dst), dt(dst), N, Cc, H, W, stream()))


def nhwc_to_nchw(src, dst, N, Cc, H, W, accumulate=False):
    _require_cuda(src, dst)
    _check(load().fmri_nhwc_to_nchw(ptr(src), dt(src), ptr(dst), dt(dst), N, Cc, H, W, int(accumulate), stream()))


def cast2d(src, lds, dst, ldd, rows, cols):
    _require_cuda(src, dst, contiguous=False)
    _check(load().fmri_cast2d(ptr(src), dt(src), lds, ptr(dst), dt(dst), ldd, _ll(rows), cols, stream()))


# ------------------------------------------------------------------------------------------------ losses
def reparam_kl_fwd(mu, logvar, eps, z, kl, B, Z, ld=None):
    _check(load().fmri_reparam_kl_fwd(ptr(mu), ptr(logvar), ld or Z, ptr(eps), ptr(z), ptr(kl), B, Z, stream()))


def reparam_kl_bwd(mu, logvar, eps, gz, gkl, dmu, dlv, B, Z, ld=None, ldd=None, gkl_const=0.0):
    _check(load().fmri_reparam_kl_bwd(ptr(mu), ptr(logvar), ld or Z, ptr(eps), ptr(gz), ptr(gkl), _f(gkl_const),
                                      ptr(dmu), ptr(dlv), ldd or Z, dt(dmu), B, Z, stream()))


def rowsqdiff_fwd(a, b, out, rows, F, scale):
    _require_cuda(a, b, out)
    _check(load().fmri_rowsqdiff_fwd(ptr(a), ptr(b), dt(a), ptr(out), _ll(rows), _ll(F), _f(scale), stream()))


def rowsqdiff_bwd(a, b, g, da, db, rows, F, scale):
    _require_cuda(a, b, g, da, db)
    _check(load().fmri_rowsqdiff_bwd(ptr(a), ptr(b), dt(a), ptr(g), ptr(da), ptr(db), _ll(rows), _ll(F), _f(scale),
                                     stream()))


def mmd_imq_fwd(zq, zp, B, Z, sigma2, lam, mmd, ws):
    """zq / zp: fp32 [B, Z] views with unit column stride (row pitch taken from .stride(0)); ws: 3 float64."""
    _require_cuda(zq, zp, mmd, ws, contiguous=False)
    _check(load().fmri_mmd_imq_fwd(ptr(zq), zq.stride(0), ptr(zp), zp.stride(0), B, Z, _f(sigma2), _f(lam), ptr(mmd),
                                   ptr(ws), stream()))


def mmd_imq_bwd(zq, zp, B, Z, sigma2, lam, dzq, accumulate=False):
    _require_cuda(zq, zp, dzq, contiguous=False)
    _check(load().fmri_mmd_imq_bwd(ptr(zq), zq.stride(0), ptr(zp), zp.stride(0), B, Z, _f(sigma2), _f(lam), ptr(dzq),
                                   dzq.stride(0), int(accumulate), stream()))


def relu_bitmask(y, pixels, Cc, bits):
    _require_cuda(y, bits)
    _check(load().fmri_relu_bitmask(ptr(y), dt(y), _ll(pixels), Cc, ptr(bits), stream()))


def head_sigmoid_fwd(x, w, bias, p, rows, F):
    _require_cuda(x, w, bias, p)
    _check(load().fmri_head_sigmoid_fwd(ptr(x), dt(x), ptr(w), ptr(bias), ptr(p), rows, F, stream()))


def head_sigmoid_bwd(x, w, p, gp, dx, dw, db, rows, F):
    _require_cuda(x, w, p, gp, dx, dw, db)
    _check(load().fmri_head_sigmoid_bwd(ptr(x), dt(x), ptr(w), ptr(p), ptr(gp), ptr(dx), ptr(dw), ptr(db), rows, F,
                                        stream()))


def bce_fwd(p, out, n, positive, scale):
    _check(load().fmri_bce_fwd(ptr(p), ptr(out), n, int(positive), _f(scale), stream()))


def bce_bwd(p, g, dp, n, positive, scale, accumulate=False):
    _check(load().fmri_bce_bwd(ptr(p), ptr(g), ptr(dp), n, int(positive), _f(scale), int(accumulate), stream()))


# ------------------------------------------------------------------------------------------------ optimizers
def _ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def multi_tensor_rmsprop(params, grads, sqs, lr, alpha, eps, clamp=0.0, lr_dev=None, gate_dev=None):
    n = len(params)
    numel = (C.c_int64 * n)(*[p.numel() for p in params])
    _check(load().fmri_multi_tensor_rmsprop(n, _ptr_array(params), _ptr_array(grads), _ptr_array(sqs), numel, _f(lr),
                                            _f(alpha), _f(eps), _f(clamp), ptr(lr_dev), ptr(gate_dev), stream()))


def multi_tensor_adam(params, grads, ms, vs, lr, beta1, beta2, eps, step, clamp=0.0, lr_dev=None, gate_dev=None):
    n = len(params)
    numel = (C.c_int64 * n)(*[p.numel() for p in params])
    _check(load().fmri_multi_tensor_adam(n, _ptr_array(params), _ptr_array(grads), _ptr_array(ms), _ptr_array(vs),
                                         numel, _f(lr), _f(beta1), _f(beta2), _f(eps), int(step), _f(clamp),
                                         ptr(lr_dev), ptr(gate_dev), stream()))


def multi_tensor_adam_dev(params, grads, ms, vs, lr, beta1, beta2, eps, step_dev, clamp=0.0, lr_dev=None, gate_dev=None):
    """Adam with the step count in a device int32 (see step_increment): capturable in a CUDA graph."""
    n = len(params)
    numel = (C.c_int64 * n)(*[p.numel() for p in params])
    _check(load().fmri_multi_tensor_adam_dev(n, _ptr_array(params), _ptr_array(grads), _ptr_array(ms), _ptr_array(vs),
                                             numel, _f(lr), _f(beta1), _f(beta2), _f(eps), ptr(step_dev), _f(clamp),
                                             ptr(lr_dev), ptr(gate_dev), stream()))


def step_increment(step_dev):
    _check(load().fmri_step_increment(ptr(step_dev), stream()))


# ------------------------------------------------------------------------------------------------ step glue
def axpby_tanh_bwd(a, x, b, y, img, out):
    _require_cuda(x, y, img, out)
    _check(load().fmri_axpby_tanh_bwd(_f(a), ptr(x), _f(b), ptr(y), ptr(img), ptr(out), _ll(out.numel()), stream()))


def chansum_nchw(x, N, Cc, HW, out, accumulate=False):
    _check(load().fmri_chansum_nchw(ptr(x), N, Cc, _ll(HW), ptr(out), int(accumulate), stream()))


def vecsum(x, n, scale, out, accumulate=False):
    _check(load().fmri_vecsum(ptr(x), _ll(n), _f(scale), ptr(out), int(accumulate), stream()))


def vgan_gate(sums, count, margin, equilibrium, gates):
    _check(load().fmri_vgan_gate(ptr(sums), _f(count), _f(margin), _f(equilibrium), ptr(gates), stream()))


def vgan_gate_mix(sums, count, margin, equilibrium, train_dis_in, gates):
    """The gate with the loss mix's pre-gate train_dis (False in mode 'vae', train_vgan_stage1.py:387)."""
    _check(load().fmri_vgan_gate_mix(ptr(sums), _f(count), _f(margin), _f(equilibrium), int(bool(train_dis_in)), ptr(gates),
                                     stream()))


def scale_f32(x, s):
    """x *= s in place (contiguous fp32 CUDA tensor)."""
    _require_cuda(x)
    if x.dtype != torch.float32:
        raise FmriError("scale_f32 expects a float32 tensor")
    _check(load().fmri_scale_f32(ptr(x), _ll(x.numel()), _f(s), stream()))


def bn_eval_stats(rm, rv, Cc, eps, mean, invstd):
    _check(load().fmri_bn_eval_stats(ptr(rm), ptr(rv), Cc, _f(eps), ptr(mean), ptr(invstd), stream()))


# ------------------------------------------------------------------------------------------------ inference / metrics / input
def bn_fold(w, inner, Cc, rm, rv, gamma, beta, eps, w_out, b_out):
    _require_cuda(w, rm, rv, gamma, beta, w_out, b_out)
    _check(load().fmri_bn_fold(ptr(w), _ll(w.numel()), _ll(inner), Cc, ptr(rm), ptr(rv), ptr(gamma), ptr(beta), _f(eps),
                               ptr(w_out), ptr(b_out), stream()))


def pearson(a, b, out, ws):
    _require_cuda(a, b, out, ws)
    _check(load().fmri_pearson(ptr(a), ptr(b), _ll(a.numel()), ptr(out), ptr(ws), stream()))


def ssim(a, b, out, ws):
    _require_cuda(a, b, out, ws)
    N, Cc, H, W = a.shape
    _check(load().fmri_ssim(ptr(a), ptr(b), N, Cc, H, W, ptr(out), ptr(ws), stream()))


def image_pipeline(src_u8, flip, shift_yx, mean3, std3, dst):
    """src_u8: uint8 [N, H, W, C] (C = 1 or 3) on the device; dst: fp32 [N, 3, H, W]."""
    _require_cuda(src_u8, flip, shift_yx, dst)
    N, H, W, Cs = src_u8.shape
    m = (C.c_float * 3)(*[float(v) for v in mean3])
    s = (C.c_float * 3)(*[float(v) for v in std3])
    _check(load().fmri_image_pipeline(ptr(src_u8), N, H, W, Cs, ptr(flip), ptr(shift_yx), m, s, ptr(dst), stream()))


# ------------------------------------------------------------------------------------------------ all-pairs similarity
def pairwise_workspace(N, M, Cc, H, W, metric):
    """Bytes of workspace fmri_pairwise_similarity needs (0 for invalid arguments)."""
    return int(load().fmri_pairwise_workspace(int(N), int(M), int(Cc), int(H), int(W), int(metric)))


def pairwise_similarity(pred, target, metric, out, ws):
    """out[i, j] = metric(pred[i], target[j]) for fp32 NCHW pred [N, C, H, W], target [M, C, H, W]; out fp32 [N, M];
    ws: a device buffer of at least pairwise_workspace(...) bytes."""
    _require_cuda(pred, target, out, ws)
    N, Cc, H, W = pred.shape
    _check(load().fmri_pairwise_similarity(ptr(pred), N, ptr(target), target.shape[0], Cc, H, W, int(metric), ptr(out),
                                           ptr(ws), _wsb(ws) if ws is not None else C.c_size_t(0), stream()))


def identification(sim, ns, wins, acc):
    """wins int32 [N] and acc float64 [len(ns)] from a square fp32 similarity matrix sim [N, N]; ns: host ints."""
    _require_cuda(sim, wins, acc)
    arr = (C.c_int * len(ns))(*[int(n) for n in ns])
    _check(load().fmri_identification(ptr(sim), sim.shape[0], arr, len(ns), ptr(wins), ptr(acc), stream()))
