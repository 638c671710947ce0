"""Paired backward sweeps: two upstreams through one saved forward state.

* fmri_bn_backward_pair / _pair_slice against two single fmri_bn_backward / _slice calls: dx bit for bit, the fp32 means
  (seen through dgamma / dbeta) equal up to the order of the fp64 atomics behind them;
* the conv data gradient over two upstreams stacked along the batch against two separate launches, bit for bit;
* VaeGanStage1.backward (paired sweeps) against the four-sweep sequence assembled from the single-upstream methods on the
  same saved forward state: every gradient bucket, dz and the image gradients, bit for bit;
* argument errors raise FmriError before any launch.
"""
import pytest
import torch

from oracle import vaegan as O
from thesis_fmri_reconstruction_b200 import engine, hp
from thesis_fmri_reconstruction_b200 import lib as L
from thesis_fmri_reconstruction_b200 import nets as NN

pytestmark = pytest.mark.gpu
DEV = "cuda"
F32, BF16, F64 = torch.float32, torch.bfloat16, torch.float64


def _bn_state(rows, C, xdtype, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = ((torch.randn(rows, C, generator=g) * 2 + 0.5).to(DEV)).to(xdtype)
    gamma = (torch.rand(C, generator=g) + 0.5).to(DEV)
    beta = (torch.randn(C, generator=g) * 0.1).to(DEV)
    s, q = torch.zeros(C, dtype=F64, device=DEV), torch.zeros(C, dtype=F64, device=DEV)
    L.colstats(x, rows, C, s, q)
    mean, invstd = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    L.bn_finalize(s, q, rows, C, 1e-5, 0.9, mean, invstd, None, None)
    dya = torch.randn(rows, C, generator=g).to(DEV).to(xdtype if xdtype == BF16 else F32)
    dyb = torch.randn(rows, C, generator=g).to(DEV)
    dyb[torch.rand(rows, C, generator=g).to(DEV) < 0.3] = 0.0      # exact zeros in one upstream
    return x, gamma, beta, mean, invstd, dya, dyb


# the Stage-I layer shapes (discriminator blocks 2 / 1, decoder blocks, decoder fc) at small batches, a ragged row count,
# and a channel count the channel-pair kernels do not tile
SHAPES = [(3 * 4 * 16 * 16, 256), (3 * 4 * 32 * 32, 128), (2 * 64 * 64, 32), (24, 16384), (1001, 256), (3 * 333, 128),
          (300, 768)]
DTYPES = [(BF16, BF16), (F32, BF16), (F32, F32)]


@pytest.mark.parametrize("rows,C", SHAPES)
@pytest.mark.parametrize("xdtype,gdtype", DTYPES)
@pytest.mark.parametrize("relu,train", [(1, 1), (0, 1), (1, 0)])
def test_bn_backward_pair_matches_two_single_calls(rows, C, xdtype, gdtype, relu, train):
    x, gamma, beta, mean, invstd, dya, dyb = _bn_state(rows, C, xdtype, seed=rows + C)
    dya, dyb = dya.to(gdtype).contiguous(), dyb.to(gdtype).contiguous()
    ws = torch.empty(3 * C, dtype=F64, device=DEV)
    ref_a, ref_b = torch.empty_like(dya), torch.empty_like(dyb)
    dg_r, db_r = torch.full((C,), 0.25, device=DEV), torch.full((C,), -0.5, device=DEV)
    L.bn_backward(x, dya, ref_a, rows, C, mean, invstd, gamma, beta, relu, train, dg_r, db_r, True, ws)
    L.bn_backward(x, dyb, ref_b, rows, C, mean, invstd, gamma, beta, relu, train, None, None, False, ws)
    ws2 = torch.empty(6 * C, dtype=F64, device=DEV)
    out = torch.empty(2 * rows, C, dtype=gdtype, device=DEV)
    dg, db = torch.full((C,), 0.25, device=DEV), torch.full((C,), -0.5, device=DEV)
    L.bn_backward_pair(x, dya, dyb, out[:rows], out[rows:], rows, C, mean, invstd, gamma, beta, relu, train, dg, db, True,
                       ws2)
    torch.cuda.synchronize()
    assert torch.equal(out[:rows], ref_a)
    assert torch.equal(out[rows:], ref_b)
    torch.testing.assert_close(dg, dg_r, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(db, db_r, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("rows,C,row0,nrows", [(3 * 4 * 32 * 32, 128, 4 * 32 * 32, 4 * 32 * 32), (1001, 256, 0, 300),
                                               (1001, 256, 701, 300), (1001, 256, 100, 0), (900, 768, 300, 300)])
@pytest.mark.parametrize("xdtype,gdtype", DTYPES)
@pytest.mark.parametrize("relu,train", [(1, 1), (0, 0)])
def test_bn_backward_pair_slice_matches_single_calls(rows, C, row0, nrows, xdtype, gdtype, relu, train):
    x, gamma, beta, mean, invstd, dya, dyb = _bn_state(rows, C, xdtype, seed=7 * rows + C)
    dya, dyb = dya.to(gdtype).contiguous(), dyb.to(gdtype).contiguous()
    ws = torch.empty(3 * C, dtype=F64, device=DEV)
    ref_a, ref_b = torch.empty_like(dya), torch.empty(nrows, C, dtype=gdtype, device=DEV)
    dg_r, db_r = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    L.bn_backward(x, dya, ref_a, rows, C, mean, invstd, gamma, beta, relu, train, dg_r, db_r, False, ws)
    L.bn_backward_slice(x, dyb, ref_b, rows, row0, nrows, C, mean, invstd, gamma, beta, relu, train, ws)
    ws2 = torch.empty(6 * C, dtype=F64, device=DEV)
    out = torch.empty(rows + nrows, C, dtype=gdtype, device=DEV)
    dg, db = torch.empty(C, device=DEV), torch.empty(C, device=DEV)
    L.bn_backward_pair_slice(x, dya, dyb, out[:rows], out[rows:], rows, row0, nrows, C, mean, invstd, gamma, beta, relu,
                             train, dg, db, False, ws2)
    torch.cuda.synchronize()
    assert torch.equal(out[:rows], ref_a)
    assert torch.equal(out[rows:], ref_b)
    torch.testing.assert_close(dg, dg_r, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(db, db_r, rtol=1e-6, atol=1e-6)


def test_bn_backward_pair_argument_errors_launch_nothing():
    rows, C = 512, 128
    x, gamma, beta, mean, invstd, dya, dyb = _bn_state(rows, C, BF16, seed=3)
    dyb = dyb.to(BF16)
    ws2 = torch.empty(6 * C, dtype=F64, device=DEV)
    dxa, dxb = torch.empty_like(dya), torch.empty_like(dyb)
    g = torch.empty(C, device=DEV)
    bad = [
        lambda: L.bn_backward_pair(x, dya, dyb, dxa, dxb, rows, 96, mean, invstd, gamma, beta, 1, 1, None, None, 0, ws2),
        lambda: L.bn_backward_pair(x, dya, dyb, dxa, dxb, rows, C, mean, invstd, gamma, beta, 1, 1, g, None, 0, ws2),
        lambda: L.bn_backward_pair(x, dya, None, dxa, dxb, rows, C, mean, invstd, gamma, beta, 1, 1, None, None, 0, ws2),
        lambda: L.bn_backward_pair(x, dya, dyb, dxa, dxb, rows, C, mean, invstd, gamma, beta, 1, 1, None, None, 0, None),
        lambda: L.bn_backward_pair(x, dya, dya, dxa, dxb, rows, C, mean, invstd, gamma, beta, 1, 1, None, None, 0, ws2),
        lambda: L.bn_backward_pair(x, dya, dyb.float(), dxa, dxb, rows, C, mean, invstd, gamma, beta, 1, 1, None, None, 0,
                                   ws2),
        lambda: L.bn_backward_pair_slice(x, dya, dyb, dxa, dxb, rows, 400, 200, C, mean, invstd, gamma, beta, 1, 1, None,
                                         None, 0, ws2),
        lambda: L.bn_backward_pair_slice(x, dya, dyb, dxa, dxb, rows, -1, 10, C, mean, invstd, gamma, beta, 1, 1, None,
                                         None, 0, ws2),
    ]
    torch.cuda.synchronize()
    for call in bad:
        L.launch_count(reset=True)
        with pytest.raises(L.FmriError):
            call()
        assert L.launch_count() == 0


def _dgrad_pair(d_single, d_stacked, dya, dyb, w, pack, dx_shape):
    ref = torch.empty((2 * dx_shape[0],) + tuple(dx_shape[1:]), dtype=BF16, device=DEV)
    L.conv_dgrad(d_single, dya, w, pack, ref[:dx_shape[0]])
    L.conv_dgrad(d_single, dyb, w, pack, ref[dx_shape[0]:])
    got = torch.empty_like(ref)
    L.conv_dgrad(d_stacked, torch.cat([dya, dyb]), w, pack, got)
    torch.cuda.synchronize()
    return got, ref


@pytest.mark.parametrize("N", [4, 64, 256])
@pytest.mark.parametrize("layer", ["dec0", "dec1", "dec2", "dis2"])
def test_stacked_conv_dgrad_matches_two_launches(N, layer):
    cfg = hp.CFG64
    dc, ch = cfg["decoder_channels"], cfg["discrim_channels"]
    spec = {"dec0": (256, 256, True, cfg["output_pad_dec"][0], 8), "dec1": (256, dc[1], True, cfg["output_pad_dec"][1], 16),
            "dec2": (dc[1], dc[2], True, cfg["output_pad_dec"][2], 32), "dis2": (ch[1], ch[2], False, 0, 32)}[layer]
    Cin, Cout, tr, op, H = spec
    blk = NN.ConvBlock("", Cin, Cout, tr, op, BF16)
    g = torch.Generator(device="cpu").manual_seed(11)
    P = {"conv.weight": (torch.randn(*((Cin, Cout) if tr else (Cout, Cin)), 5, 5, generator=g) * 0.05).to(DEV)}
    blk.refresh(P)
    d = blk.desc(N, H, H)
    OH, OW = L.conv_out_hw(d)
    dya = torch.randn(N, OH, OW, Cout, generator=g).to(DEV).to(BF16)
    dyb = torch.randn(N, OH, OW, Cout, generator=g).to(DEV).to(BF16)
    got, ref = _dgrad_pair(d, blk.desc(2 * N, H, H), dya, dyb, P["conv.weight"], blk.pack_d, (N, H, H, Cin))
    assert torch.equal(got, ref)


def _four_sweeps(tr, st):
    """The Stage-I backward as four single-upstream sweeps (the sequence the paired backward replaces)."""
    hp_, B = tr.hp, st.B
    lam = float(hp_["lambda_mse"])
    bd, bc = tr.buckets["decoder."], tr.buckets["discriminator."]
    cd1, cd2, cc, raw3, p = st.cd1, st.cd2, st.cc, st.raw3, st.p
    Fd = raw3[0].numel()
    gp = torch.empty(3 * B, device=DEV)
    ones = tr._ones(3 * B)
    L.bce_bwd(p[:B], ones, gp[:B], B, True, 1.0)
    L.bce_bwd(p[B:], ones, gp[B:], 2 * B, False, 1.0)
    dimg_bce = tr.dis.backward_gan(bc.P, cc, gp, bc.G, False, True, (1, 3))
    draw3 = torch.empty_like(raw3)
    draw3[2 * B:].zero_()
    L.rowsqdiff_bwd(raw3[:B], raw3[B:2 * B], ones, draw3[:B], draw3[B:2 * B], B, Fd, 0.5)
    dimg_mse = tr.dis.backward_rec(bc.P, cc, draw3, None, False, False, (1, 2), live=(0, 2))
    tr.dec.backward(bd.P, cd1, lam, dimg_mse, -(1.0 - lam), dimg_bce[:B], bd.G, False, True, False)
    tr.dec.backward(bd.P, cd2, -(1.0 - lam), dimg_bce[B:], 0.0, None, bd.G, True, True, False)
    dz = tr.dec.backward(bd.P, cd1, 1.0, dimg_mse, 0.0, None, None, False, False, True)
    dycat = tr._encoder_backward(st, dz)
    st.sweeps = dict(dimg_bce=dimg_bce, dimg_mse=dimg_mse, dz=dz, dycat=dycat)


@pytest.mark.parametrize("B", [8, 64])
def test_paired_stage1_backward_matches_four_sweeps(B):
    P, S = O.make_vaegan(O.CFG64, seed=77)
    x = O.synthetic_images(B, seed=77).cuda()
    eps, z_p = (t.cuda() for t in O.synthetic_noise(B, 128, seed=77))
    tr = engine.VaeGanStage1(P, S, hp.CFG64, 128, BF16)
    st = tr.forward(x, eps, z_p)
    results = []
    for run in (tr.backward, lambda s: _four_sweeps(tr, s)):
        run(st)
        NN.join_side()
        torch.cuda.synchronize()
        results.append(({k: b.flat_g.clone() for k, b in tr.buckets.items()},
                        {k: v.clone() for k, v in st.sweeps.items()}))
    (g1, s1), (g0, s0) = results
    for k in g0:
        assert torch.equal(g1[k], g0[k]), k
    for k in ("dimg_bce", "dimg_mse", "dz", "dycat"):
        assert torch.equal(s1[k], s0[k]), k
