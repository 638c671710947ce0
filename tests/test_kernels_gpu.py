"""Kernel-level parity: every C-ABI entry point against a plain PyTorch fp32 reference of the same op on the GPU.

Tolerances (rel-L2, stated per test): fp32 path 1e-4 (exact arithmetic, different summation order); bf16 tensor path
3e-3 when the output is stored in bf16 (inputs are pre-rounded to bf16 so only accumulation order and the final
rounding differ), 2e-4 when the output is fp32.
"""
import pytest
import torch
import torch.nn.functional as F

from thesis_fmri_reconstruction_b200 import lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda"


def setup_module(module):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def rel(a, b):
    a = a.float()
    b = b.float()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def nchw(x):
    return x.permute(0, 3, 1, 2).contiguous()


def rnd(x, dtype):
    return x.to(dtype).float()


def tol(dtype, out_bf16=True):
    if dtype == torch.float32:
        return 1e-4
    return 3e-3 if out_bf16 else 2e-4


CONV_CASES = [
    # N, H, W, Cin, Cout
    (4, 16, 16, 64, 128),
    (2, 32, 32, 32, 128),
    (8, 8, 8, 128, 256),
    (3, 16, 16, 256, 256),
    (3, 25, 25, 32, 128),   # 100x100 config: odd grid, 32-channel side -> parity-merged data gradient with ragged classes
    (40, 64, 64, 32, 128),  # Discriminator block 1 at its real grid, >= 296 tiles: the row-reuse gather (tall TMA boxes)
    (5, 64, 64, 32, 128),   # the same below the persistent threshold (row reuse only in the forced-persistent child run)
]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_s2_fprop_stats(case, dtype):
    N, H, W, Cin, Cout = case
    if dtype == torch.float32 and Cin * Cout > 64 * 128:
        pytest.skip("direct fp32 conv is exercised on the small case only")
    g = torch.Generator(device="cpu").manual_seed(1)
    x = rnd(torch.randn(N, Cin, H, W, generator=g).to(DEV), dtype)
    w = rnd((torch.randn(Cout, Cin, 5, 5, generator=g) * 0.05).to(DEV), dtype)
    ref = F.conv2d(x, w, stride=2, padding=2)
    d = L.conv_desc(N, H, W, Cin, Cout, 2, False, 0, dtype)
    OH, OW = L.conv_out_hw(d)
    xs = nhwc(x).to(dtype)
    pack = torch.empty(L.conv_pack_elems(d), dtype=torch.bfloat16, device=DEV)
    L.conv_pack_weights(d, w, pack, None)
    y = torch.full((N, OH, OW, Cout), float("nan"), dtype=dtype, device=DEV)
    ssum = torch.zeros(Cout, dtype=torch.float64, device=DEV)
    ssq = torch.zeros(Cout, dtype=torch.float64, device=DEV)
    L.conv_fprop(d, xs, w, pack, None, L.ACT_NONE, y, ssum, ssq)
    torch.cuda.synchronize()
    assert rel(nchw(y), ref) < tol(dtype)
    yf = y.float().reshape(-1, Cout).double()
    assert rel(ssum, yf.sum(0)) < 1e-5
    assert rel(ssq, (yf * yf).sum(0)) < 1e-5


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_s2_dgrad(case, dtype):
    N, H, W, Cin, Cout = case
    if dtype == torch.float32 and Cin * Cout > 64 * 128:
        pytest.skip("direct fp32 conv is exercised on the small case only")
    g = torch.Generator(device="cpu").manual_seed(2)
    w = rnd((torch.randn(Cout, Cin, 5, 5, generator=g) * 0.05).to(DEV), dtype)
    d = L.conv_desc(N, H, W, Cin, Cout, 2, False, 0, dtype)
    OH, OW = L.conv_out_hw(d)
    dy = rnd(torch.randn(N, Cout, OH, OW, generator=g).to(DEV), dtype)
    ref = torch.nn.grad.conv2d_input((N, Cin, H, W), w, dy, stride=2, padding=2)
    pack_d = torch.empty(L.conv_pack_elems(d), dtype=torch.bfloat16, device=DEV)
    L.conv_pack_weights(d, w, None, pack_d)
    dx = torch.full((N, H, W, Cin), float("nan"), dtype=dtype, device=DEV)
    L.conv_dgrad(d, nhwc(dy).to(dtype), w, pack_d, dx)
    torch.cuda.synchronize()
    assert rel(nchw(dx), ref) < tol(dtype)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_s2_wgrad(case, dtype):
    N, H, W, Cin, Cout = case
    if dtype == torch.float32:
        if Cin * Cout > 64 * 128:
            pytest.skip("direct fp32 wgrad is exercised on the small case only")
    g = torch.Generator(device="cpu").manual_seed(3)
    x = rnd(torch.randn(N, Cin, H, W, generator=g).to(DEV), dtype)
    d = L.conv_desc(N, H, W, Cin, Cout, 2, False, 0, dtype)
    OH, OW = L.conv_out_hw(d)
    dy = rnd(torch.randn(N, Cout, OH, OW, generator=g).to(DEV), dtype)
    ref = torch.nn.grad.conv2d_weight(x, (Cout, Cin, 5, 5), dy, stride=2, padding=2)
    ws = torch.empty(max(1, L.conv_wgrad_workspace(d)), dtype=torch.uint8, device=DEV)
    dw = torch.full((Cout, Cin, 5, 5), float("nan"), dtype=torch.float32, device=DEV)
    L.conv_wgrad(d, nhwc(x).to(dtype), nhwc(dy).to(dtype), dw, False, ws)
    torch.cuda.synchronize()
    assert rel(dw, ref) < tol(dtype, out_bf16=False)
    L.conv_wgrad(d, nhwc(x).to(dtype), nhwc(dy).to(dtype), dw, True, ws)
    torch.cuda.synchronize()
    assert rel(dw, 2 * ref) < tol(dtype, out_bf16=False)


CONVT_CASES = [
    # N, H, W, Cin, Cout, output_pad
    (4, 8, 8, 256, 256, 1),
    (2, 16, 16, 256, 128, 1),
    (2, 32, 32, 128, 32, 1),
    (3, 13, 13, 64, 64, 0),
    (3, 13, 13, 128, 32, 0),  # odd output (25x25) through the parity-merged scatter
    (40, 32, 32, 64, 32, 1),  # Decoder block 3 at its real grid: its data gradient is a row-reuse gather with N = 64
]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("case", CONVT_CASES)
def test_convT_fprop_dgrad_wgrad(case, dtype):
    N, H, W, Cin, Cout, op = case
    if dtype == torch.float32 and Cin * Cout > 64 * 64:
        pytest.skip("direct fp32 conv is exercised on the small case only")
    g = torch.Generator(device="cpu").manual_seed(4)
    x = rnd(torch.randn(N, Cin, H, W, generator=g).to(DEV), dtype).requires_grad_(True)
    w = rnd((torch.randn(Cin, Cout, 5, 5, generator=g) * 0.05).to(DEV), dtype).requires_grad_(True)
    ref = F.conv_transpose2d(x, w, stride=2, padding=2, output_padding=op)
    d = L.conv_desc(N, H, W, Cin, Cout, 2, True, op, dtype)
    OH, OW = L.conv_out_hw(d)
    assert (OH, OW) == tuple(ref.shape[2:])
    dyr = rnd(torch.randn(N, Cout, OH, OW, generator=g).to(DEV), dtype)
    gx, gw = torch.autograd.grad(ref, (x, w), dyr)
    pack_f = torch.empty(L.conv_pack_elems(d), dtype=torch.bfloat16, device=DEV)
    pack_d = torch.empty(L.conv_pack_elems(d), dtype=torch.bfloat16, device=DEV)
    wd = w.detach()
    L.conv_pack_weights(d, wd, pack_f, pack_d)
    xs = nhwc(x.detach()).to(dtype)
    y = torch.full((N, OH, OW, Cout), float("nan"), dtype=dtype, device=DEV)
    ssum = torch.zeros(Cout, dtype=torch.float64, device=DEV)
    ssq = torch.zeros(Cout, dtype=torch.float64, device=DEV)
    L.conv_fprop(d, xs, wd, pack_f, None, L.ACT_NONE, y, ssum, ssq)
    torch.cuda.synchronize()
    assert rel(nchw(y), ref) < tol(dtype)
    yf = y.float().reshape(-1, Cout).double()
    assert rel(ssum, yf.sum(0)) < 1e-5
    assert rel(ssq, (yf * yf).sum(0)) < 1e-5
    dys = nhwc(dyr).to(dtype)
    dx = torch.full((N, H, W, Cin), float("nan"), dtype=dtype, device=DEV)
    L.conv_dgrad(d, dys, wd, pack_d, dx)
    torch.cuda.synchronize()
    assert rel(nchw(dx), gx) < tol(dtype)
    ws = torch.empty(max(1, L.conv_wgrad_workspace(d)), dtype=torch.uint8, device=DEV)
    dw = torch.full((Cin, Cout, 5, 5), float("nan"), dtype=torch.float32, device=DEV)
    L.conv_wgrad(d, xs, dys, dw, False, ws)
    torch.cuda.synchronize()
    assert rel(dw, gw) < tol(dtype, out_bf16=False)


LIN_CASES = [
    # M, N, K
    (64, 1024, 16384),  # encoder fc (split-K)
    (192, 512, 16384),  # discriminator fc
    (64, 16384, 128),   # decoder fc
    (256, 256, 1024),   # fused mu/logvar heads
    (96, 1024, 3620),   # cognitive encoder (K padded to the TMA pitch)
    (128, 512, 512),    # WAE discriminator hidden layer
]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("case", LIN_CASES)
def test_linear(case, dtype):
    M, N, K = case
    g = torch.Generator(device="cpu").manual_seed(5)
    x = rnd(torch.randn(M, K, generator=g).to(DEV), dtype)
    w = rnd((torch.randn(N, K, generator=g) * 0.02).to(DEV), dtype)
    b = torch.randn(N, generator=g).to(DEV)
    dy = rnd(torch.randn(M, N, generator=g).to(DEV), dtype)
    d = L.linear_desc(M, N, K, dtype)
    Kp = (K + 7) // 8 * 8
    if dtype == torch.bfloat16:
        xs = torch.zeros(M, Kp, dtype=dtype, device=DEV)
        xs[:, :K] = x.to(dtype)
        wp = torch.empty(N, Kp, dtype=dtype, device=DEV)
        wpt = torch.empty(K, N, dtype=dtype, device=DEV)
        L.linear_pack_weights(d, w, wp, Kp, wpt, N)
    else:
        xs, wp, wpt, Kp = x.contiguous(), None, None, K
    # fp32 output, no bias (split-K eligible)
    y = torch.full((M, N), float("nan"), dtype=torch.float32, device=DEV)
    L.linear_fprop(d, xs, Kp, w, wp, Kp, None, L.ACT_NONE, y, N)
    torch.cuda.synchronize()
    assert rel(y, x @ w.t()) < tol(dtype, out_bf16=False)
    # bias + relu, activation dtype output
    y2 = torch.full((M, N), float("nan"), dtype=dtype, device=DEV)
    L.linear_fprop(d, xs, Kp, w, wp, Kp, b, L.ACT_RELU, y2, N)
    torch.cuda.synchronize()
    assert rel(y2, torch.relu(x @ w.t() + b)) < tol(dtype)
    # dgrad
    dys = dy.to(dtype).contiguous()
    dx = torch.full((M, Kp), float("nan"), dtype=dtype, device=DEV)
    L.linear_dgrad(d, dys, N, w, wpt, N, dx, Kp)
    torch.cuda.synchronize()
    assert rel(dx[:, :K], dy @ w) < tol(dtype)
    # wgrad (+ accumulate)
    dw = torch.full((N, K), float("nan"), dtype=torch.float32, device=DEV)
    L.linear_wgrad(d, xs, Kp, dys, N, dw, False)
    torch.cuda.synchronize()
    assert rel(dw, dy.t() @ x) < tol(dtype, out_bf16=False)
    L.linear_wgrad(d, xs, Kp, dys, N, dw, True)
    torch.cuda.synchronize()
    assert rel(dw, 2 * (dy.t() @ x)) < tol(dtype, out_bf16=False)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("C,stride", [(32, 1), (64, 2), (32, 2)])
def test_edge_in(C, stride, dtype):
    N, H, W = 6, 16, 16
    g = torch.Generator(device="cpu").manual_seed(6)
    # the tensor path repacks the 3-channel side to bf16 (NHWC-8): pre-round it like every other bf16 operand
    imgs = [rnd(torch.randn(N // 3, 3, H, W, generator=g).to(DEV), dtype).requires_grad_(True) for _ in range(3)]
    # weights pre-rounded to the compute dtype: the tensor path consumes bf16 weight packs (as in the conv tests above)
    w = rnd((torch.randn(C, 3, 5, 5, generator=g) * 0.1).to(DEV), dtype).requires_grad_(True)
    b = torch.randn(C, generator=g).to(DEV)
    ref = torch.relu(F.conv2d(torch.cat(imgs, 0).double(), w.double(), b.double(), stride=stride, padding=2))
    d = L.edge_desc(N, H, W, C, stride, dtype)
    ws = torch.empty(L.edge_workspace(d), dtype=torch.uint8, device=DEV)
    OH = (H - 1) // stride + 1
    y = torch.full((N, OH, OH, C), float("nan"), dtype=dtype, device=DEV)
    L.edge_in_fprop(d, [t.detach() for t in imgs], N // 3, w.detach(), b, L.ACT_RELU, y, ws)
    torch.cuda.synchronize()
    assert rel(nchw(y), ref) < tol(dtype)
    # backward of the pre-activation conv
    pre = F.conv2d(torch.cat(imgs, 0).double(), w.double(), b.double(), stride=stride, padding=2)
    dyr = rnd(torch.randn_like(pre).float(), dtype)
    grads = torch.autograd.grad(pre, imgs + [w], dyr.double())
    dys = nhwc(dyr).to(dtype)
    dimg = torch.full((N, 3, H, W), float("nan"), dtype=torch.float32, device=DEV)
    L.edge_in_dgrad(d, dys, w.detach(), dimg, ws)
    torch.cuda.synchronize()
    assert rel(dimg, torch.cat(grads[:3], 0)) < tol(dtype, out_bf16=False)
    dw = torch.full((C, 3, 5, 5), float("nan"), dtype=torch.float32, device=DEV)
    L.edge_in_wgrad(d, [t.detach() for t in imgs], N // 3, dys, dw, False, ws)
    torch.cuda.synchronize()
    assert rel(dw, grads[3]) < tol(dtype, out_bf16=False)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("C", [32, 64])
def test_edge_out(C, dtype):
    N, H, W = 4, 16, 16
    g = torch.Generator(device="cpu").manual_seed(7)
    x = rnd(torch.randn(N, C, H, W, generator=g).to(DEV), dtype).requires_grad_(True)
    w = rnd((torch.randn(3, C, 5, 5, generator=g) * 0.1).to(DEV), dtype).requires_grad_(True)
    b = torch.randn(3, generator=g).to(DEV)
    # fp64 reference: cuDNN may pick an FFT/Winograd algorithm for a 5x5 stride-1 fp32 conv (1e-3 noise)
    pre = F.conv2d(x.double(), w.double(), b.double(), stride=1, padding=2)
    ref = torch.tanh(pre)
    d = L.edge_desc(N, H, W, C, 1, dtype)
    ws = torch.empty(L.edge_workspace(d), dtype=torch.uint8, device=DEV)
    xs = nhwc(x.detach()).to(dtype)
    img = torch.full((N, 3, H, W), float("nan"), dtype=torch.float32, device=DEV)
    L.edge_out_fprop(d, xs, w.detach(), b, L.ACT_TANH, img, ws)
    torch.cuda.synchronize()
    assert rel(img, ref) < tol(dtype, out_bf16=False)
    dimg = rnd(torch.randn_like(pre).float(), dtype)
    gx, gw = torch.autograd.grad(pre, (x, w), dimg.double())
    dx = torch.full((N, H, W, C), float("nan"), dtype=dtype, device=DEV)
    L.edge_out_dgrad(d, dimg, w.detach(), dx, ws)
    torch.cuda.synchronize()
    assert rel(nchw(dx), gx) < tol(dtype)
    dw = torch.full((3, C, 5, 5), float("nan"), dtype=torch.float32, device=DEV)
    L.edge_out_wgrad(d, xs, dimg, dw, False, ws)
    torch.cuda.synchronize()
    assert rel(dw, gw) < tol(dtype, out_bf16=False)


@pytest.mark.parametrize("xdtype,gdtype", [(torch.bfloat16, torch.bfloat16), (torch.float32, torch.bfloat16),
                                           (torch.float32, torch.float32)])
@pytest.mark.parametrize("rows,C", [(4 * 16 * 16, 128), (64, 1024), (96, 16384), (2 * 64 * 64, 32)])
def test_batchnorm_relu(rows, C, xdtype, gdtype):
    g = torch.Generator(device="cpu").manual_seed(8)
    x = rnd((torch.randn(rows, C, generator=g) * 2 + 0.5).to(DEV), xdtype).requires_grad_(True)
    gamma = (torch.rand(C, generator=g) + 0.5).to(DEV).requires_grad_(True)
    beta = (torch.randn(C, generator=g) * 0.1).to(DEV).requires_grad_(True)
    rm = torch.zeros(C, device=DEV)
    rv = torch.ones(C, device=DEV)
    ref = torch.relu(F.batch_norm(x, rm, rv, gamma, beta, True, 0.9, 1e-5))
    xs = x.detach().to(xdtype)
    s = torch.zeros(C, dtype=torch.float64, device=DEV)
    q = torch.zeros(C, dtype=torch.float64, device=DEV)
    L.colstats(xs, rows, C, s, q)
    mean = torch.empty(C, device=DEV)
    invstd = torch.empty(C, device=DEV)
    rm2 = torch.zeros(C, device=DEV)
    rv2 = torch.ones(C, device=DEV)
    L.bn_finalize(s, q, rows, C, 1e-5, 0.9, mean, invstd, rm2, rv2)
    y = torch.empty(rows, C, dtype=gdtype, device=DEV)
    L.bn_apply(xs, y, rows, C, mean, invstd, gamma.detach(), beta.detach(), True)
    torch.cuda.synchronize()
    out_bf16 = gdtype == torch.bfloat16
    assert rel(y, ref) < (3e-3 if out_bf16 else 1e-5)
    assert rel(rm2, rm) < 1e-5 and rel(rv2, rv) < 1e-4
    dy = rnd(torch.randn(rows, C, generator=g).to(DEV), gdtype)
    gx, gg, gb = torch.autograd.grad(ref, (x, gamma, beta), dy)
    dx = torch.empty(rows, C, dtype=gdtype, device=DEV)
    dgamma = torch.empty(C, device=DEV)
    dbeta = torch.empty(C, device=DEV)
    ws = torch.empty(3 * C, dtype=torch.float64, device=DEV)
    L.bn_backward(xs, dy.to(gdtype), dx, rows, C, mean, invstd, gamma.detach(), beta.detach(), True, True, dgamma,
                  dbeta, False, ws)
    torch.cuda.synchronize()
    assert rel(dx, gx) < (4e-3 if out_bf16 else 1e-4)
    assert rel(dgamma, gg) < 1e-4 and rel(dbeta, gb) < 1e-4


def test_losses():
    g = torch.Generator(device="cpu").manual_seed(9)
    B, Z, Fe = 48, 128, 16384
    mu = torch.randn(B, Z, generator=g).to(DEV).requires_grad_(True)
    lv = (torch.randn(B, Z, generator=g) * 0.3).to(DEV).requires_grad_(True)
    eps = torch.randn(B, Z, generator=g).to(DEV)
    z_ref = eps * torch.exp(0.5 * lv) + mu
    kl_ref = -0.5 * torch.sum(-lv.exp() - mu.pow(2) + lv + 1, 1)
    z = torch.empty(B, Z, device=DEV)
    kl = torch.empty(B, device=DEV)
    L.reparam_kl_fwd(mu.detach(), lv.detach(), eps, z, kl, B, Z)
    torch.cuda.synchronize()
    assert rel(z, z_ref) < 1e-6 and rel(kl, kl_ref) < 1e-5
    gz = torch.randn(B, Z, generator=g).to(DEV)
    gk = torch.randn(B, generator=g).to(DEV)
    rmu, rlv = torch.autograd.grad((z_ref * gz).sum() + (kl_ref * gk).sum(), (mu, lv))
    dmu = torch.empty(B, Z, device=DEV)
    dlv = torch.empty(B, Z, device=DEV)
    L.reparam_kl_bwd(mu.detach(), lv.detach(), eps, gz, gk, dmu, dlv, B, Z)
    torch.cuda.synchronize()
    assert rel(dmu, rmu) < 1e-6 and rel(dlv, rlv) < 1e-5
    for dtype in (torch.float32, torch.bfloat16):
        a = rnd(torch.randn(B, Fe, generator=g).to(DEV), dtype).requires_grad_(True)
        b = rnd(torch.randn(B, Fe, generator=g).to(DEV), dtype).requires_grad_(True)
        ref = torch.sum(0.5 * (a - b) ** 2, 1)
        out = torch.empty(B, device=DEV)
        L.rowsqdiff_fwd(a.detach().to(dtype), b.detach().to(dtype), out, B, Fe, 0.5)
        torch.cuda.synchronize()
        assert rel(out, ref) < 1e-5
        go = torch.randn(B, generator=g).to(DEV)
        ra, rb = torch.autograd.grad((ref * go).sum(), (a, b))
        da = torch.empty(B, Fe, dtype=dtype, device=DEV)
        db = torch.empty(B, Fe, dtype=dtype, device=DEV)
        L.rowsqdiff_bwd(a.detach().to(dtype), b.detach().to(dtype), go, da, db, B, Fe, 0.5)
        torch.cuda.synchronize()
        assert rel(da, ra) < tol(dtype) and rel(db, rb) < tol(dtype)
    # sigmoid head + BCE
    Fh = 512
    x = torch.randn(B, Fh, generator=g).to(DEV).requires_grad_(True)
    w = (torch.randn(1, Fh, generator=g) * 0.05).to(DEV).requires_grad_(True)
    bias = torch.randn(1, generator=g).to(DEV).requires_grad_(True)
    p_ref = torch.sigmoid(x @ w.t() + bias)
    p = torch.empty(B, 1, device=DEV)
    L.head_sigmoid_fwd(x.detach(), w.detach(), bias.detach(), p, B, Fh)
    torch.cuda.synchronize()
    assert rel(p, p_ref) < 1e-5
    for positive in (True, False):
        bce_ref = -torch.log(p_ref + 1e-3) if positive else -torch.log(1 - p_ref + 1e-3)
        bce = torch.empty(B, 1, device=DEV)
        L.bce_fwd(p, bce, B, positive, 1.0)
        torch.cuda.synchronize()
        assert rel(bce, bce_ref) < 1e-5
        gb = torch.randn(B, 1, generator=g).to(DEV)
        rx, rw, rb = torch.autograd.grad((bce_ref * gb).sum(), (x, w, bias), retain_graph=True)
        dp = torch.empty(B, 1, device=DEV)
        L.bce_bwd(p, gb, dp, B, positive, 1.0)
        dx = torch.empty(B, Fh, device=DEV)
        dw = torch.zeros(1, Fh, device=DEV)
        dbias = torch.zeros(1, device=DEV)
        L.head_sigmoid_bwd(x.detach(), w.detach(), p, dp, dx, dw, dbias, B, Fh)
        torch.cuda.synchronize()
        assert rel(dx, rx) < 1e-5 and rel(dw, rw) < 1e-5 and rel(dbias, rb) < 1e-5


def test_optimizers_match_torch():
    g = torch.Generator(device="cpu").manual_seed(10)
    shapes = [(1024, 300), (77,), (64, 3, 5, 5), (1,)]
    for kind in ("rmsprop", "adam"):
        ps = [torch.randn(*s, generator=g).to(DEV) for s in shapes]
        ref_ps = [p.clone().requires_grad_(True) for p in ps]
        if kind == "rmsprop":
            opt = torch.optim.RMSprop(ref_ps, lr=1e-4, alpha=0.9, eps=1e-8)
            st1 = [torch.zeros_like(p) for p in ps]
        else:
            opt = torch.optim.Adam(ref_ps, lr=1e-4, betas=(0.5, 0.999))
            st1 = [torch.zeros_like(p) for p in ps]
            st2 = [torch.zeros_like(p) for p in ps]
        for step in range(1, 4):
            gs = [torch.randn(*s, generator=g).to(DEV) for s in shapes]
            for rp, gg in zip(ref_ps, gs):
                rp.grad = gg.clone()
            opt.step()
            if kind == "rmsprop":
                L.multi_tensor_rmsprop(ps, gs, st1, 1e-4, 0.9, 1e-8)
            else:
                L.multi_tensor_adam(ps, gs, st1, st2, 1e-4, 0.5, 0.999, 1e-8, step)
            torch.cuda.synchronize()
            for p, rp in zip(ps, ref_ps):
                assert rel(p, rp.detach()) < 1e-6


def test_layout_converters():
    g = torch.Generator(device="cpu").manual_seed(11)
    x = torch.randn(3, 5, 7, 9, generator=g).to(DEV)
    for dtype in (torch.float32, torch.bfloat16):
        y = torch.empty(3, 7, 9, 5, dtype=dtype, device=DEV)
        L.nchw_to_nhwc(x, y, 3, 5, 7, 9)
        torch.cuda.synchronize()
        assert torch.equal(y, nhwc(x).to(dtype))
        back = torch.empty(3, 5, 7, 9, device=DEV)
        L.nhwc_to_nchw(y, back, 3, 5, 7, 9)
        torch.cuda.synchronize()
        assert torch.equal(back, x.to(dtype).float())
    src = torch.randn(10, 3620, generator=g).to(DEV)
    dst = torch.zeros(10, 3624, dtype=torch.bfloat16, device=DEV)
    L.cast2d(src, 3620, dst, 3624, 10, 3620)
    torch.cuda.synchronize()
    assert torch.equal(dst[:, :3620], src.to(torch.bfloat16)) and float(dst[:, 3620:].abs().sum()) == 0.0


@pytest.mark.parametrize("mode", ["bf16", "bf16_bits", "fp32"])
@pytest.mark.parametrize("case", [(40, 64, 64, 32, 128), (3, 25, 25, 32, 128)])
def test_conv_dgrad_fused_relu_mask(case, mode):
    """fmri_conv_dgrad with fmri_relu_mask: dx also goes through the ReLU backward of the bias+ReLU layer below, dx *= (y > 0)
    (Discriminator.conv[0] under block 1). Cases: block 1 at its real grid (>= 296 tiles: the mask is applied in the
    persistent kernel's epilogue) and the ragged 100x100 grid (a small launch: the mask is applied in place after the
    one-tile kernel; the forced-persistent child run of test_persistent_path_subprocess takes it through the epilogue too).
    y holds exact zeros, negatives and positives; bits = NULL or fmri_relu_bitmask(y). Tolerance as test_conv_s2_dgrad."""
    N, H, W, Cin, Cout = case
    dtype = torch.float32 if mode == "fp32" else torch.bfloat16
    g = torch.Generator(device="cpu").manual_seed(23)
    w = rnd((torch.randn(Cout, Cin, 5, 5, generator=g) * 0.05).to(DEV), dtype)
    d = L.conv_desc(N, H, W, Cin, Cout, 2, False, 0, dtype)
    OH, OW = L.conv_out_hw(d)
    dy = rnd(torch.randn(N, Cout, OH, OW, generator=g).to(DEV), dtype)
    y = torch.randn(N, H, W, Cin, generator=g)
    y[y.abs() < 0.4] = 0.0                                  # about a third exact zeros, the rest split between signs
    y = y.to(DEV).to(dtype)
    bits = None
    if mode == "bf16_bits":
        bits = torch.empty(N * H * W, dtype=torch.int32, device=DEV)
        L.relu_bitmask(y, N * H * W, Cin, bits)
    pack_d = torch.empty(L.conv_pack_elems(d), dtype=torch.bfloat16, device=DEV)
    L.conv_pack_weights(d, w, None, pack_d)
    dx = torch.full((N, H, W, Cin), float("nan"), dtype=dtype, device=DEV)
    L.conv_dgrad(d, nhwc(dy).to(dtype), w, pack_d, dx, relu_mask=(y, bits))
    torch.cuda.synchronize()
    ref = torch.nn.grad.conv2d_input((N, Cin, H, W), w, dy, stride=2, padding=2) * (nchw(y).float() > 0)
    assert rel(nchw(dx), ref) < tol(dtype)
    assert not bool(torch.isnan(dx).any())


@pytest.mark.parametrize("B,Z", [(2, 128), (7, 128), (64, 128), (100, 96), (300, 128), (37, 512)])
def test_mmd_imq_fwd_bwd(B, Z):
    """fmri_mmd_imq_{fwd,bwd} against oracle/mmd.py in fp64 (extension: the reference has no MMD; parity unpinned).
    Tolerance 1e-5 relative (fp32 pairwise sums, fp64 accumulation across tiles); ragged B / Z exercise the tile masks."""
    from oracle.mmd import mmd_imq

    g = torch.Generator().manual_seed(B * 1000 + Z)
    ycat = torch.randn(B, 2 * Z, generator=g)          # zq is the mu half of a [B, 2Z] head output (pitched view)
    zp = torch.randn(B, Z, generator=g) * 0.5
    lam, sigma2 = 10.0, 0.25
    q64 = ycat[:, :Z].double().requires_grad_(True)
    ref = lam * mmd_imq(q64, zp.double(), sigma2)
    ref.backward()
    yc = ycat.cuda()
    zq_d, zp_d = yc[:, :Z], zp.cuda()
    out, ws = torch.empty(1, device="cuda"), torch.empty(3, device="cuda", dtype=torch.float64)
    L.mmd_imq_fwd(zq_d, zp_d, B, Z, sigma2, lam, out, ws)
    dq = torch.full((B, Z), 7.0, device="cuda")
    L.mmd_imq_bwd(zq_d, zp_d, B, Z, sigma2, lam, dq)
    base = 1e-3   # same magnitude as the gradient, so that fp32 accumulation onto it keeps the 1e-5 resolution
    dq2 = torch.full((B, Z), base, device="cuda")
    L.mmd_imq_bwd(zq_d, zp_d, B, Z, sigma2, lam, dq2, accumulate=True)
    torch.cuda.synchronize()
    # the estimate is a difference of kernel sums of magnitude ~ 7 * lam: the bound is relative to that magnitude
    assert abs(out.item() - ref.item()) <= 1e-5 * abs(ref.item()) + 2e-6 * 7 * lam, (out.item(), ref.item())
    gr = q64.grad.float()
    assert rel(dq.cpu(), gr) < 1e-5, rel(dq.cpu(), gr)
    assert rel(dq2.cpu() - base, gr) < 1e-4


def test_persistent_path_subprocess():
    """The persistent implicit-GEMM kernel (double-buffered TMEM accumulators, warp-converged producer, per-tap column ranges
    of the parity-merged scatter) only takes over at >= 296 tiles, which the kernel-level cases above do not reach. The library
    reads FMRI_IGEMM_PERSISTENT once per process, so the conv / convT cases are re-run in a child process with the
    persistent kernel forced for every launch (value 2), at the same tolerances. The child also forces the chunk-pair
    (128-byte-line) store path of the epilogue for every form (FMRI_IG_PAIR=2; by default only the BN = 128 gathers take it)."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, FMRI_IGEMM_PERSISTENT="2", FMRI_IG_PAIR="2")   # and the 128-byte-line store path in every form
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_kernels_gpu.py"), "-m", "gpu", "-q",
                        "-x", "-p", "no:cacheprovider", "-k",
                        "conv_s2_dgrad or convT_fprop or conv_s2_fprop or fused_relu"],
                       cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " passed" in r.stdout


@pytest.mark.parametrize("N,H", [(80, 7), (148, 2), (75, 64), (200, 5)])
def test_edge_c_to_3_gemm_gather_path(N, H):
    """The GEMM + shift-and-add kernel of the C -> 3 convolutions (cto3_kernels.cuh; taken for C = 32, W = 64, N >= 74) on
    shapes the full-size tests do not reach: odd heights (a last chunk of one image row, H*W not a multiple of the 128-pixel
    chunk), images shorter than the 5x5 window, more images than CTAs. Forward (bias + tanh) and the flipped-tap data-gradient
    use, against fp64 torch; fp32 outputs, tolerance 2e-4."""
    C, W = 32, 64
    dtype = torch.bfloat16
    g = torch.Generator(device="cpu").manual_seed(70 + H)
    x = rnd(torch.randn(N, C, H, W, generator=g).to(DEV), dtype)
    w = rnd((torch.randn(3, C, 5, 5, generator=g) * 0.1).to(DEV), dtype)
    b = torch.randn(3, generator=g).to(DEV)
    d = L.edge_desc(N, H, W, C, 1, dtype)
    ws = torch.empty(L.edge_workspace(d), dtype=torch.uint8, device=DEV)
    img = torch.full((N, 3, H, W), float("nan"), dtype=torch.float32, device=DEV)
    L.edge_out_fprop(d, nhwc(x).to(dtype), w, b, L.ACT_TANH, img, ws)
    torch.cuda.synchronize()
    ref = torch.tanh(F.conv2d(x.double(), w.double(), b.double(), stride=1, padding=2))
    assert rel(img, ref) < 2e-4
    # data gradient of a 3 -> C convolution: dimg = conv_transpose(dy, w_in) -- same kernel, flipped taps, other weight layout
    w_in = rnd((torch.randn(C, 3, 5, 5, generator=g) * 0.1).to(DEV), dtype)
    dy = rnd(torch.randn(N, C, H, W, generator=g).to(DEV), dtype)
    dimg = torch.full((N, 3, H, W), float("nan"), dtype=torch.float32, device=DEV)
    L.edge_in_dgrad(d, nhwc(dy).to(dtype), w_in, dimg, ws)
    torch.cuda.synchronize()
    ref_d = torch.nn.grad.conv2d_input((N, 3, H, W), w_in.double(), dy.double(), stride=1, padding=2)
    assert rel(dimg, ref_d) < 2e-4
