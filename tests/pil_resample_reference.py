"""numpy restatement of Pillow's 8-bit resampler (PIL.Image.resize with BILINEAR / BICUBIC on L and RGB images:
ImagingResample in libImaging/Resample.c). TEST INFRASTRUCTURE ONLY.

Per axis, with the source window [in0, in1) of an axis of in_size pixels resized to out_size:
    scale = (in1 - in0) / out_size, filterscale = max(scale, 1), support = filter_support * filterscale
    output index xx: center = in0 + (xx + 0.5) scale
        xmin = max(int(center - support + 0.5), 0), xlen = min(int(center + support + 0.5), in_size) - xmin
        w[x] = filter((x + xmin - center + 0.5) * (1 / filterscale)), normalised by their sum unless it is 0
        k[x] = int(w 2^22 + 0.5), or int(w 2^22 - 0.5) for w < 0           (Python floats: IEEE fp64, no FMA)
The horizontal pass runs first, over the source rows the vertical taps read; each value is
clamp((2^21 + sum src * k) >> 22, 0, 255), stored as uint8, and the vertical pass then reads those uint8 rows. Image.resize
itself swaps the order for an image more than 100 times taller than wide that shrinks vertically. The sums are
exact in int64 and equal Pillow's int32 sums, which never overflow for 8-bit inputs.
tests/test_resample_cpu.py checks resize() against PIL.Image.resize byte for byte.
"""
import numpy as np

PREC = 22
SUPPORT = {"bilinear": 1.0, "bicubic": 2.0}


def _bilinear(x):
    x = -x if x < 0.0 else x
    return 1.0 - x if x < 1.0 else 0.0


def _bicubic(x, a=-0.5):
    x = -x if x < 0.0 else x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


FILTERS = {"bilinear": _bilinear, "bicubic": _bicubic}


def coeffs(in_size, in0, in1, out_size, filter):
    """[(xmin, int64 fixed-point taps)] for every output index of one axis."""
    f, scale = FILTERS[filter], (in1 - in0) / out_size
    fs = max(scale, 1.0)
    support, ss = SUPPORT[filter] * fs, 1.0 / fs
    out = []
    for xx in range(out_size):
        center = in0 + (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xlen = min(int(center + support + 0.5), in_size) - xmin
        w = [f((x + xmin - center + 0.5) * ss) for x in range(xlen)]
        ww = 0.0
        for v in w:
            ww += v
        if ww != 0.0:
            w = [v / ww for v in w]
        out.append((xmin, np.array([int(-0.5 + v * (1 << PREC)) if v < 0 else int(0.5 + v * (1 << PREC)) for v in w],
                                   dtype=np.int64)))
    return out


def _clip8(s):
    return np.clip(s >> PREC, 0, 255)


def resize(img_u8, out_hw, filter="bilinear", box=None):
    """uint8 [Hs, Ws] or [Hs, Ws, C] -> uint8 [H, W] or [H, W, C]: PIL.Image.resize((W, H), filter, box) with
    box = (left, upper, right, lower) in source pixels (floats allowed), the whole image by default. Like Image.resize,
    an image more than 100 times taller than wide that shrinks vertically takes the vertical pass first."""
    a = np.asarray(img_u8)
    Hs, Ws = a.shape[:2]
    H, W = (int(v) for v in out_hw)
    x0, y0, x1, y1 = box if box is not None else (0, 0, Ws, Hs)
    if Hs > 100 * Ws and H < Hs:
        return _two_pass(_two_pass(a, (H, Ws), filter, (0, y0, Ws, y1)), (H, W), filter, (x0, 0, x1, H))
    return _two_pass(a, (H, W), filter, (x0, y0, x1, y1))


def _two_pass(a, out_hw, filter, box):
    """Pillow's ImagingResample: the horizontal pass, then the vertical one."""
    Hs, Ws = a.shape[:2]
    H, W = out_hw
    x0, y0, x1, y1 = box
    ch, cv = coeffs(Ws, x0, x1, W, filter), coeffs(Hs, y0, y1, H, filter)
    ya, yb = cv[0][0], cv[-1][0] + len(cv[-1][1])
    src = a.astype(np.int64)
    t = np.empty((yb - ya, W) + a.shape[2:], np.int64)
    for xx, (xm, k) in enumerate(ch):
        t[:, xx] = _clip8((1 << (PREC - 1)) + np.tensordot(k, src[ya:yb, xm:xm + len(k)], axes=([0], [1])))
    o = np.empty((H, W) + a.shape[2:], np.int64)
    for yy, (ym, k) in enumerate(cv):
        o[yy] = _clip8((1 << (PREC - 1)) + np.tensordot(k, t[ym - ya:ym - ya + len(k)], axes=([0], [0])))
    return o.astype(np.uint8)


def resample_window(buf, entry, out_hw, filter):
    """What fmri_image_resample resizes for one descriptor: the window (offset, pitch, h, w, C, Hr, Wr, oy, ox) of the
    flat uint8 buffer `buf`, resized to Hr x Wr, and its out_hw part at (oy, ox). uint8 [H, W, C]."""
    off, pitch, h, w, c, Hr, Wr, oy, ox = (int(v) for v in entry)
    buf = np.asarray(buf)
    win = np.stack([buf[off + y * pitch: off + y * pitch + w * c] for y in range(h)]).reshape(h, w, c)
    H, W = (int(v) for v in out_hw)
    return resize(win, (Hr, Wr), filter)[oy:oy + H, ox:ox + W]
