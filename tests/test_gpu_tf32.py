"""-m gpu: fp32 storage with SPC_ALGO_TF32 (tcgen05 kind::tf32) against cuDNN fp32 with TF32 off.

Full-size parity: every distinct BASELINE conv shape the TF32 path covers, at the N=1 tile and at the N=4 tile with halo
strips on every exchanged side, reference built as in test_gpu_fullsize_parity.py.  Two input sets:

* TF32-representable inputs (x, w, gy, strips rounded to a 10-bit mantissa): every product is exact in fp32, so only
  the summation order differs.  Tolerance 2^-14 |ref| + 2^-14 rms(ref) for y / dx, two orders of magnitude below the bf16
  test's 2^-7 / 2^-8.  The same comparison with the result replaced by the reference of bf16-rounded inputs must FAIL,
  so a path that silently went through bf16 would not pass.
* Random fp32 inputs.  The tensor cores read each operand truncated to its top 19 bits (10-bit mantissa; measured,
  profiles/r3_tf32_mma_probe.txt), a relative error in [0, 2^-10) per operand, so each product carries a relative error
  in [0, 2^-9): a bias of about 2^-10 of the result plus a random part whose standard deviation is about
  2^-11.3 * sqrt(sum of squared products) ~ 2^-11.3 rms(ref).  Hence  |got - ref| <= 2^-8 |ref| + 2^-8 rms(ref)  (bias
  4x inside, noise ~10 sigma inside).  Where a few large products dominate one output the noise can exceed that, so the
  rigorous worst case  2^-9 (1 + 2^-3) * sum_i |a_i b_i|  (computed by the same convolution of |x| and |w|) is also
  accepted: an element fails only if it exceeds both.  dw is checked the same way against conv2d_weight of |x|, |gy|.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import gpu_util as gu
from tests.test_gpu_fullsize_parity import CONVS, DEV, _cid, _padded

pytestmark = pytest.mark.gpu

TF32_CONVS = [c for c in CONVS if not (c[1]["R"] * c[1]["S"] > 1 and c[1]["stride_h"] == 2)]


@pytest.fixture(autouse=True)
def _no_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    import gc

    gc.collect()
    torch.cuda.empty_cache()


def tf32_round(t):
    """Round fp32 to the nearest value with a 10-bit mantissa (exactly representable as TF32)."""
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _violations(got, ref, rel, floor, bound=None):
    """(count, worst excess, rms) of |got - ref| > max(rel |ref| + floor rms(ref), bound); a few channels at a time, so
    the temporaries of a 14 GB tensor stay small."""
    rms = float(ref.double().square().mean().sqrt()) if ref.dim() < 2 else \
        float(sum(float(ref[:, i:i + 8].double().square().sum()) for i in range(0, ref.shape[1], 8)) / ref.numel()) ** 0.5
    n, worst = 0, -float("inf")
    for i in range(0, ref.shape[1] if ref.dim() >= 2 else 1, 8):
        sl = (slice(None), slice(i, i + 8)) if ref.dim() >= 2 else (slice(None),)
        r = ref[sl].float()
        tol = r.abs() * rel + floor * rms
        if bound is not None:
            tol = torch.maximum(tol, bound[sl])
        viol = (got[sl].float() - r).abs_() - tol
        n += int((viol > 0).sum())
        worst = max(worst, float(viol.max()))
        del r, tol, viol
    return n, worst, rms


def _check(got, ref, name, rel, floor, bound=None):
    assert got.shape == ref.shape, (name, tuple(got.shape), tuple(ref.shape))
    n, worst, rms = _violations(got, ref, rel, floor, bound)
    assert n == 0, "%s: %d elements out of tolerance, worst excess %.3g (rms %.3g)" % (name, n, worst, rms)


def _strips(N, Cc, H, W, hh, hw, gen, rnd):
    strips = [None] * 9
    dirs = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 0), (0, 1), (1, -1), (1, 0), (1, 1)]
    for i, (dr, dc) in enumerate(dirs):
        if i == 4 or (dr != 0 and hh == 0) or (dc != 0 and hw == 0):
            continue
        shp = (N, Cc, H if dr == 0 else hh, W if dc == 0 else hw)
        strips[i] = rnd(torch.randn(shp, device=DEV, generator=gen))
    return strips


def _wgrad(L, d, x, strips, gy, K, wshape):
    from mpi4dl_b200 import _lib

    dw = torch.empty(wshape, dtype=torch.float32, device=DEV)
    nb = L.spc_conv_workspace_bytes(C.byref(d), 2)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
    halo = _lib.make_halo(strips)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.spc_conv2d_wgrad(C.byref(d), C.c_void_p(x.data_ptr()), C.byref(halo), C.c_void_p(gy.data_ptr()),
                                  C.c_void_p(dw.data_ptr()), None, 0, C.c_void_p(ws.data_ptr()), nb, st), "wgrad")
    return dw


@pytest.mark.parametrize("inputs", ["representable", "random"])
@pytest.mark.parametrize("tile", ["n1", "n4"])
@pytest.mark.parametrize("case", TF32_CONVS, ids=_cid)
def test_tf32_fullsize_vs_cudnn_fp32(case, tile, inputs):
    from mpi4dl_b200 import _lib
    from mpi4dl_b200.torchgems.spatial import _ConvSpatialFn

    tag, l, first = case
    L = _lib.lib()
    div = 1 if tile == "n1" else 2
    Cc, K, R, S = l["C"], l["K"], l["R"], l["S"]
    H, W = l["H"] // div, l["W"] // div
    sh, sw, hh, hw = l["stride_h"], l["stride_w"], l["pad_h"], l["pad_w"]
    rnd = tf32_round if inputs == "representable" else (lambda t: t)
    gen = torch.Generator(device=DEV).manual_seed(3000 + Cc * 7 + K * 3 + R * 11 + S + H)
    x = rnd(torch.randn((1, Cc, H, W), device=DEV, generator=gen))
    w = rnd(torch.randn((K, Cc, R, S), device=DEV, generator=gen) / (Cc * R * S) ** 0.5)
    b = rnd(torch.randn(K, device=DEV, generator=gen)) if l.get("bias") else None
    strips = _strips(1, Cc, H, W, hh, hw, gen, rnd) if tile == "n4" else [None] * 9
    desc = (1, Cc, H, W, K, R, S, sh, sw, hh, hw, _lib.SPC_F32, _lib.SPC_ALGO_TF32)
    d = _lib.ConvDesc(*desc)
    assert L.spc_conv_uses_tcgen05(C.byref(d), 0) and L.spc_conv_uses_tcgen05(C.byref(d), 2)

    exact = inputs == "representable"
    rel, floor = (2.0 ** -14, 2.0 ** -14) if exact else (2.0 ** -8, 2.0 ** -8)
    slack = 2.0 ** -9 * (1 + 2.0 ** -3)

    xg = x.clone().requires_grad_(not first)
    y = _ConvSpatialFn.apply(xg, w, b, desc, *strips)
    gy = rnd(torch.randn(y.shape, device=DEV, generator=gen) * 0.25)
    xp = _padded(x, strips, hh, hw)
    with torch.no_grad():
        ref = F.conv2d(xp, w, b, stride=(sh, sw), padding=0)
        bound = None if exact else slack * F.conv2d(xp.abs(), w.abs(), None, stride=(sh, sw), padding=0)
        torch.cuda.empty_cache()
        _check(y.detach(), ref, "y", rel, floor, bound)
        if exact:
            # a bf16 path would not pass: the reference of bf16-rounded operands is far outside this tolerance
            ref_bf = F.conv2d(xp.bfloat16().float(), w.bfloat16().float(), b, stride=(sh, sw), padding=0)
            n, _, _ = _violations(ref_bf, ref, rel, floor)
            assert n > 0, "tolerance cannot tell TF32 from bf16"
            del ref_bf
        del ref, bound
    if not first:
        y.backward(gy)
        with torch.no_grad():
            dxp = torch.nn.grad.conv2d_input(xp.shape, w, gy, stride=(sh, sw), padding=0)
            bound = None if exact else slack * torch.nn.grad.conv2d_input(xp.shape, w.abs(), gy.abs(), stride=(sh, sw),
                                                                          padding=0)[:, :, hh:hh + H, hw:hw + W]
            _check(xg.grad, dxp[:, :, hh:hh + H, hw:hw + W], "dx", rel, floor, bound)
            del dxp, bound
    del y, xg
    torch.cuda.empty_cache()
    with torch.no_grad():
        dw_ref = torch.nn.grad.conv2d_weight(xp, w.shape, gy, stride=(sh, sw), padding=0)
        dw = _wgrad(L, d, x, strips, gy, K, w.shape)
        if exact:
            # exact products; what differs is the fp32 summation order of up to 6.7e7 pixels, as in the bf16 test
            err = float((dw - dw_ref).abs().max())
            tol = 1e-3 * float(dw_ref.abs().max())
            assert err <= tol, "dw: max err %.3g > %.3g" % (err, tol)
        else:
            bound = slack * torch.nn.grad.conv2d_weight(xp.abs(), w.shape, gy.abs(), stride=(sh, sw), padding=0)
            _check(dw, dw_ref, "dw", 2.0 ** -8, 2.0 ** -8, bound)


# ---- the small oracle cases of test_gpu_parity.py (multi-rank tiles, odd shapes on the direct kernel, stride 2) ----
from tests.test_gpu_parity import CONV_CASES  # noqa: E402


@pytest.mark.parametrize("case", CONV_CASES)
def test_tf32_against_oracle_seeded(case):
    from mpi4dl_b200 import _lib
    from oracle import spatial_oracle as so

    Cc, K, (R, S), stride, H, W, bias = case
    rng = np.random.default_rng(hash((Cc, K, R, S, H, W, "tf32")) % (2 ** 31))
    hh, hw = (R - 1) // 2, (S - 1) // 2
    x = rng.standard_normal((2, Cc, H, W)).astype(np.float32)
    w = (rng.standard_normal((K, Cc, R, S)) / np.sqrt(Cc * R * S)).astype(np.float32)
    b = rng.standard_normal(K).astype(np.float32) if bias else None
    xp = np.pad(x, ((0, 0), (0, 0), (hh, hh), (hw, hw)))
    halo_vals = rng.standard_normal(xp.shape).astype(np.float32)
    inner = np.zeros(xp.shape, dtype=bool)
    inner[:, :, hh:hh + H, hw:hw + W] = True
    xp = np.where(inner, xp, halo_vals)
    mask = [1, 1, 1, 1, 0, 1, 1, 1, 1]
    if R == 1:
        mask = [0, 0, 0, 1, 0, 1, 0, 0, 0]
    if S == 1:
        mask = [0, 1, 0, 0, 0, 0, 0, 1, 0] if R > 1 else [0] * 9
    strips = gu.strips_from_padded(xp, mask, hh, hw, torch.float32)
    y_ref = so.conv2d_fwd(xp, w, b, stride)
    gy = rng.standard_normal(y_ref.shape).astype(np.float32)
    dxp, dw_ref, db_ref = so.conv2d_bwd(xp, w, gy, stride, need_db=bias)
    out = gu.conv_tile(x, w, b, gy, strips, stride, torch.float32, algo=_lib.SPC_ALGO_TF32)
    # per element: TF32 worst case 2^-9 * sum |products| (<= 2^-9 * sqrt(n) * ||.||) -> 2e-3 of max|ref| plus 2e-3 relative
    for name, got, ref in (("y", out["y"], y_ref), ("dx", out["dx"], so.crop(dxp, hh, hw)), ("dw", out["dw"], dw_ref)):
        np.testing.assert_allclose(got, ref, rtol=4e-3, atol=4e-3 * np.abs(ref).max(), err_msg=name)
    if bias:
        np.testing.assert_allclose(out["db"], db_ref, rtol=1e-4, atol=1e-4 * np.abs(db_ref).max())


# ---- module level ------------------------------------------------------------------------------------------------
def _c_abi_conv(x, w, b, algo):
    from mpi4dl_b200 import _lib
    from mpi4dl_b200.torchgems.spatial import _ConvSpatialFn

    N, Cc, H, W = x.shape
    K, _, R, S = w.shape
    xg = x.clone().requires_grad_(True)
    wg = w.clone().requires_grad_(True)
    bg = b.clone().requires_grad_(True)
    desc = (N, Cc, H, W, K, R, S, 1, 1, (R - 1) // 2, (S - 1) // 2, _lib.SPC_F32, algo)
    y = _ConvSpatialFn.apply(xg, wg, bg, desc, *([None] * 9))
    return y, xg, wg, bg


@pytest.mark.parametrize("kind", ["conv_spatial", "local_conv2d"])
@pytest.mark.parametrize("k", [1, 3, (1, 7)])
def test_module_follows_fp32_math(kind, k):
    from mpi4dl_b200 import _lib
    from mpi4dl_b200.torchgems import spatial

    kh, kw = (k, k) if isinstance(k, int) else k
    pad = ((kh - 1) // 2, (kw - 1) // 2)
    torch.manual_seed(5)
    if kind == "conv_spatial":
        m = spatial.conv_spatial(0, 1, 1, 64, 96, (kh, kw), padding=pad).cuda()
    else:
        m = spatial.local_conv2d(64, 96, (kh, kw), padding=pad).cuda()
    x = torch.randn(2, 64, 32, 128, device=DEV)
    gy = torch.randn(2, 96, 32, 128, device=DEV)
    old = spatial.get_fp32_math()
    try:
        for mode, algo in (("tf32", _lib.SPC_ALGO_TF32), ("ieee", _lib.SPC_ALGO_DIRECT)):
            spatial.set_fp32_math(mode)
            m.zero_grad()
            xg = x.clone().requires_grad_(True)
            y = m(xg)
            y.backward(gy)
            yr, xr, wr, br = _c_abi_conv(x, m.weight.detach(), m.bias.detach(), algo)
            yr.backward(gy)
            assert torch.equal(y, yr), mode
            assert torch.equal(xg.grad, xr.grad), mode
            # wgrad adds partial sums with atomics in a run-dependent order
            torch.testing.assert_close(m.weight.grad, wr.grad, rtol=1e-5, atol=1e-5 * float(wr.grad.abs().max()))
            torch.testing.assert_close(m.bias.grad, br.grad, rtol=1e-5, atol=1e-5 * float(br.grad.abs().max()))
        # an explicit algo is left alone
        spatial.set_fp32_math("tf32")
        m.algo = _lib.SPC_ALGO_DIRECT
        y = m(x)
        yr, _, _, _ = _c_abi_conv(x, m.weight.detach(), m.bias.detach(), _lib.SPC_ALGO_DIRECT)
        assert torch.equal(y, yr)
    finally:
        spatial.set_fp32_math(old)
