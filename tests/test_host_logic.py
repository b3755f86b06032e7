"""CPU-only: host-side mirror of torchgems.spatial -- topology, constructor contracts, and the
"no CPU fallback" rule."""
import pytest
import torch

from mpi4dl_b200.torchgems import spatial
from oracle import spatial_oracle as so

GRIDS = [("square", 4), ("square", 9), ("square", 16), ("vertical", 2), ("vertical", 4), ("vertical", 8),
         ("horizontal", 2), ("horizontal", 4), ("horizontal", 8)]


@pytest.mark.parametrize("method,P", GRIDS)
@pytest.mark.parametrize("k", [(3, 3), (1, 7), (7, 1), (5, 5)])
def test_conv_neighbours_match_oracle(method, P, k):
    for rank in range(P):
        m = spatial.conv_spatial(rank, 1, P, 2, 2, k, padding=((k[0] - 1) // 2, (k[1] - 1) // 2), slice_method=method)
        mask = so.neighbour_mask(method, P, rank, k[0], k[1])
        assert m.neighbours == mask
        assert m.rank_neighbours == so.neighbour_ranks(method, P, rank, mask)


@pytest.mark.parametrize("method,P", GRIDS)
def test_halo_layer_and_pool_neighbours(method, P):
    for rank in range(P):
        h = spatial.halo_exchange_layer(rank, 1, P, 2, slice_method=method)
        mask = so.neighbour_mask(method, P, rank)
        assert h.neighbours == mask and h.rank_neighbours == so.neighbour_ranks(method, P, rank, mask)
        p = spatial.Pool(rank, 1, P, 3, 1, 1, slice_method=method, operation="AvgPool2d")
        assert p.neighbours == mask
        p2 = spatial.Pool(rank, 1, P, 2, 2, 0, slice_method=method, operation="MaxPool2d")
        assert p2.neighbours is None and p2.halo_len == 0


def test_list_num_spatial_parts():
    m = spatial.conv_spatial(5, 2, [4, 2], 2, 2, 3, padding=1, slice_method="vertical")
    assert (m.spatial_local_rank, m.num_spatial_parts) == (1, 2)
    assert m.neighbours == [0, 0, 0, 1, 0, 0, 0, 0, 0]
    assert m.rank_neighbours[3] == 4


def test_conv_spatial_is_a_conv2d_with_reference_state_dict():
    m = spatial.conv_spatial(0, 1, 4, 3, 8, 3, stride=2, padding=1, bias=True)
    assert isinstance(m, torch.nn.Conv2d)
    assert list(m.state_dict().keys()) == ["weight", "bias"]
    assert m.weight.shape == (8, 3, 3, 3) and m.padding == (0, 0) and m.stride == (2, 2)
    assert (m.halo_len_height, m.halo_len_width) == (1, 1)
    ref = torch.nn.Conv2d(3, 8, 3, stride=2)
    ref.load_state_dict(m.state_dict())


def test_reference_assertions():
    with pytest.raises(AssertionError, match="Spatial not supported yet"):
        spatial.conv_spatial(0, 1, 4, 3, 8, 3, padding=0)
    with pytest.raises(AssertionError, match="halo_len should be equal to padding"):
        spatial.Pool(0, 1, 4, 3, 1, 0, operation="AvgPool2d")
    with pytest.raises(AssertionError, match="operation is none"):
        spatial.Pool(0, 1, 4, 3, 1, 1)
    with pytest.raises(AssertionError, match="Only MaxPool2d and AvgPool2d"):
        spatial.Pool(0, 1, 4, 3, 1, 1, operation="LPPool2d")
    with pytest.raises(AssertionError, match="Custom Halo Len"):
        spatial.conv_spatial(0, 1, 4, 3, 8, 3, padding=1, halo_len=1)


def test_fused_halo_variant_border_sides():
    """conv_spatial(halo_len=0): padding only on true image borders (reference table spatial.py:76-104
    for the 2x2 grid: rank0 pads left/top, rank1 right/top, rank2 left/bottom, rank3 right/bottom)."""
    inner = {r: spatial.conv_spatial(r, 1, 4, 3, 8, 3, padding=1, halo_len=0)._inner_sides for r in range(4)}
    # (top, bottom, left, right) sides that face a neighbour
    assert inner[0] == (False, True, False, True)
    assert inner[1] == (False, True, True, False)
    assert inner[2] == (True, False, False, True)
    assert inner[3] == (True, False, True, False)
    m = spatial.conv_spatial(0, 1, 4, 3, 8, 3, padding=1, halo_len=0)
    assert m.neighbours is None   # never exchanges


def test_no_cpu_fallback():
    m = spatial.conv_spatial(0, 1, 1, 3, 4, 3, padding=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        spatial.Pool(0, 1, 1, 3, 1, 1, operation="AvgPool2d")(torch.zeros(1, 3, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        spatial.halo_exchange_layer(0, 1, 1, 1)(torch.zeros(1, 3, 8, 8))


def test_north_star_aliases():
    assert spatial.pool_spatial is spatial.Pool and spatial.halo_exchange is spatial.halo_exchange_layer


def test_dropin_import_shim_resolves_reference_imports():
    """The import lines of the reference's benchmark scripts, unmodified, with mpi4dl_b200/dropin on
    the path (fresh interpreter so sys.modules of this process stays clean)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys; sys.path[:0] = [%r, %r]\n"
        "from torchgems import parser\n"
        "from torchgems.mp_pipeline import model_generator\n"
        "from torchgems.train_spatial import train_model_spatial, split_input, get_shapes_spatial, verify_spatial_config\n"
        "from torchgems.train_spatial_master import train_spatial_model_master, verify_spatial_master_config\n"
        "from torchgems.gems_master import train_model_master\n"
        "import torchgems.comm as gems_comm\n"
        "from torchgems.spatial import conv_spatial, halo_exchange_layer, Pool\n"
        "from models import resnet, resnet_spatial, amoebanet, amoebanet_d2, resnet_spatial_d2\n"
        "from utils import get_depth, isPowerTwo\n"
        "import mpi4dl_b200.torchgems.train_spatial as mine\n"
        "assert train_model_spatial is mine.train_model_spatial and gems_comm.MPIComm.__module__.startswith('mpi4dl_b200')\n"
        "assert get_depth(2, 12) == 110 and parser.get_parser().parse_args([]).split_size == 2\n"
        "print('ok')\n") % (os.path.join(root, "mpi4dl_b200", "dropin"), root)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stderr[-2000:]


def test_halo_benchmark_known_answers_match_the_oracle():
    """benchmarks/communication/halo/halo_common.py (numpy fixtures of the self-checking halo benchmarks)
    against the oracle: exchanged padded tiles and the ones-weights convolution, every grid."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "benchmarks", "communication", "halo"))
    import halo_common as hc
    import numpy as np

    from oracle import spatial_oracle as so
    full = hc.full_image(2, 3, 16)
    for method, P in (("square", 4), ("vertical", 4), ("horizontal", 2), ("vertical", 2)):
        tiles = so.split(full, method, P)
        for halo in (1, 3):
            padded = so.halo_exchange_layer(tiles, method, halo)
            for r in range(P):
                assert np.array_equal(hc.tile(full, method, P, r), tiles[r])
                got = padded[r]["y"] if isinstance(padded[r], dict) else padded[r]
                assert np.array_equal(hc.expected_padded_tile(full, method, P, r, halo), got), (method, P, halo, r)
        for kh, kw in ((3, 3), (1, 7), (7, 1)):
            w = np.ones((4, 3, kh, kw), np.float32)
            ref = so.conv_spatial(tiles, w, np.ones(4, np.float32), method, (1, 1), None)
            for r in range(P):
                assert np.array_equal(hc.expected_conv_tile(full, method, P, r, kh, kw, 4), ref[r]["y"].astype(np.float64)), \
                    (method, P, kh, kw, r)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver's second arm): one JSON line with the contract's keys, produced on the
    host by the oracle port alone; under torchrun only rank 0 prints, the other ranks exit 0 without work."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", SPCONV_BENCH_CPU_BUDGET_S="0.01")
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-scale", "128"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and "8192" in d["config"]["workload"] and d["vs_baseline"] is None
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=120, cwd=root,
                           env=dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert other.returncode == 0 and other.stdout.strip() == "", (other.stdout, other.stderr[-500:])


@pytest.mark.parametrize("extra,msg", [(["--steps", "0"], "--steps"),
                                       (["--impl", "reference", "--dump-outputs", "out"], "--dump-outputs")])
def test_bench_rejects_bad_arguments(extra, msg, tmp_path):
    """No timed steps, or a dump the CPU reference arm cannot make, is a usage error before any work starts."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + extra, capture_output=True, text=True,
                         timeout=120, cwd=tmp_path, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 2 and msg in out.stderr and out.stdout == "", out.stderr[-500:]
    assert os.listdir(tmp_path) == []
