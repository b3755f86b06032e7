"""CPU-only: which path SPC_ALGO_TF32 selects (libspconv.so dispatch queries, no kernel runs) and the fp32 math switch
of torchgems.spatial (set_fp32_math / SPCONV_FP32_MATH)."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

from mpi4dl_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _distinct_convs():
    out, seen = [], set()
    for fn in ("layers_amoebanetd_sp4.json", "layers_resnet101_sp2.json"):
        for l in json.load(open(os.path.join(ROOT, "tests", "golden", fn)))["layers"]:
            if l["op"] != "conv":
                continue
            key = tuple(l[k] for k in ("C", "K", "R", "S", "stride_h", "stride_w", "pad_h", "pad_w", "H", "W"))
            if key not in seen:
                seen.add(key)
                out.append(key)
    return out


CONVS = _distinct_convs()


def _desc(key, dtype, algo, N=1):
    Cc, K, R, S, sh, sw, ph, pw, H, W = key
    return _lib.ConvDesc(N, Cc, H, W, K, R, S, sh, sw, ph, pw, dtype, algo)


def _cid(key):
    return "%dto%d-%dx%d-s%d-%d" % (key[0], key[1], key[2], key[3], key[4], key[8])


def test_layer_lists_have_both_kinds_of_shape():
    assert len(CONVS) >= 25
    assert any(k[2] * k[3] > 1 and k[4] == 2 for k in CONVS)
    assert any(k[2] * k[3] > 1 and k[4] == 1 for k in CONVS)


@pytest.mark.parametrize("op", [0, 1, 2])
@pytest.mark.parametrize("key", CONVS, ids=_cid)
def test_tf32_dispatch(key, op):
    L = _lib.lib()
    uses = lambda dt, algo: L.spc_conv_uses_tcgen05(C.byref(_desc(key, dt, algo)), op)
    ws = lambda dt, algo: L.spc_conv_workspace_bytes(C.byref(_desc(key, dt, algo)), op)
    # the default is unchanged: fp32 with AUTO runs in exact fp32 on the direct kernel
    assert uses(_lib.SPC_F32, _lib.SPC_ALGO_AUTO) == 0
    assert ws(_lib.SPC_F32, _lib.SPC_ALGO_AUTO) == 0
    # TF32 covers every shape but the 3x3 stride-2 ones, which stay on the direct kernel in fp32
    s2_tap = key[2] * key[3] > 1 and key[4] == 2
    assert uses(_lib.SPC_F32, _lib.SPC_ALGO_TF32) == (0 if s2_tap else 1)
    if not s2_tap:
        assert ws(_lib.SPC_F32, _lib.SPC_ALGO_TF32) > 0
    # with bf16 storage TF32 is AUTO
    assert uses(_lib.SPC_BF16, _lib.SPC_ALGO_TF32) == uses(_lib.SPC_BF16, _lib.SPC_ALGO_AUTO)
    assert ws(_lib.SPC_BF16, _lib.SPC_ALGO_TF32) == ws(_lib.SPC_BF16, _lib.SPC_ALGO_AUTO)


def test_tf32_workspace_uses_four_byte_elements():
    """1x1 104->208: the repacked filter is [Mpad=256][Cpad] in the storage type (Cpad = 128 channels for fp32's
    32-channel stages, 128 for bf16's 64-channel stages): twice the bytes in fp32."""
    L = _lib.lib()
    key = (104, 208, 1, 1, 1, 1, 0, 0, 1024, 1024)
    f32 = L.spc_conv_workspace_bytes(C.byref(_desc(key, _lib.SPC_F32, _lib.SPC_ALGO_TF32)), 0)
    bf = L.spc_conv_workspace_bytes(C.byref(_desc(key, _lib.SPC_BF16, _lib.SPC_ALGO_AUTO)), 0)
    assert f32 >= 256 * 128 * 4 and bf >= 256 * 128 * 2 and f32 > bf


def test_explicit_algos_ignore_tf32_mode():
    """DIRECT stays direct; TCGEN05 with fp32 is still refused (not silently TF32)."""
    L = _lib.lib()
    key = (104, 208, 1, 1, 1, 1, 0, 0, 1024, 1024)
    for op in range(3):
        assert L.spc_conv_uses_tcgen05(C.byref(_desc(key, _lib.SPC_F32, _lib.SPC_ALGO_DIRECT)), op) == 0
        assert L.spc_conv_uses_tcgen05(C.byref(_desc(key, _lib.SPC_F32, _lib.SPC_ALGO_TCGEN05)), op) == 0


def test_set_fp32_math_and_algo_selection():
    import torch

    from mpi4dl_b200.torchgems import spatial

    old = spatial.get_fp32_math()
    try:
        spatial.set_fp32_math("ieee")
        assert spatial.get_fp32_math() == "ieee"
        assert spatial._algo_for(_lib.SPC_ALGO_AUTO, torch.float32) == _lib.SPC_ALGO_AUTO
        spatial.set_fp32_math("tf32")
        assert spatial.get_fp32_math() == "tf32"
        assert spatial._algo_for(_lib.SPC_ALGO_AUTO, torch.float32) == _lib.SPC_ALGO_TF32
        assert spatial._algo_for(_lib.SPC_ALGO_AUTO, torch.bfloat16) == _lib.SPC_ALGO_AUTO
        assert spatial._algo_for(_lib.SPC_ALGO_DIRECT, torch.float32) == _lib.SPC_ALGO_DIRECT
        assert spatial._algo_for(_lib.SPC_ALGO_TCGEN05, torch.float32) == _lib.SPC_ALGO_TCGEN05
        for bad in ("TF32", "fp32", "", None):
            with pytest.raises(ValueError):
                spatial.set_fp32_math(bad)
        assert spatial.get_fp32_math() == "tf32"
    finally:
        spatial.set_fp32_math(old)


def _import_mode(env_value):
    env = dict(os.environ)
    env.pop("SPCONV_FP32_MATH", None)
    if env_value is not None:
        env["SPCONV_FP32_MATH"] = env_value
    code = "from mpi4dl_b200.torchgems import spatial; print(spatial.get_fp32_math())"
    return subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True)


@pytest.mark.parametrize("value,expect", [(None, "ieee"), ("ieee", "ieee"), ("tf32", "tf32")])
def test_env_initial_value(value, expect):
    r = _import_mode(value)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip().splitlines()[-1] == expect


def test_env_bad_value_raises():
    r = _import_mode("fast")
    assert r.returncode != 0
    assert "SPCONV_FP32_MATH" in r.stderr and "fast" in r.stderr
