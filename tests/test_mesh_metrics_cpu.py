"""CPU: the fp64 oracle of the paper's mesh metrics (oracle/mesh_metrics.compare_meshes_with) on known answers, the cross-rank
mean of sharding.reduce_mesh_metrics in a world-2 gloo run, and the C ABI of the new entry points."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cubify_np
from oracle import mesh_metrics as om

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAUS = (0.1, 0.2, 0.3, 0.4, 0.5)


def _draws(f_index, n, seed):
    g = torch.Generator().manual_seed(seed)
    fi = torch.stack([torch.randint(0, max(int(f), 1), (n,), generator=g) for f in f_index])
    return fi, torch.rand(len(f_index), n, generator=g, dtype=torch.float64), torch.rand(len(f_index), n, generator=g,
                                                                                      dtype=torch.float64)


def _square(z):
    v = torch.tensor([[0, 0, z], [10, 0, z], [10, 10, z], [0, 10, z]], dtype=torch.float64)
    return v, torch.tensor([[0, 1, 2], [0, 2, 3]])


def test_identical_meshes_give_perfect_scores():
    from meshrcnn_b200 import synthetic
    v, vi, f, fi, _ = cubify_np.cubify(synthetic.blob_voxels(2, 8, 3).numpy(), 0.2)
    v, f = torch.from_numpy(v).double(), torch.from_numpy(f)
    rnd = _draws(fi, 500, 0)
    res = om.compare_meshes_with(v, f, vi, fi, v, f, vi, fi, rnd, rnd, thresholds=TAUS)
    for row in res:
        assert float(row["Chamfer-L2"]) == 0.0
        assert float(row["NormalConsistency"]) == pytest.approx(1.0, abs=1e-12)
        assert float(row["AbsNormalConsistency"]) == pytest.approx(1.0, abs=1e-12)
        for tau in TAUS:
            assert float(row["F1@%g" % tau]) == pytest.approx(100.0, abs=1e-6)


def test_parallel_squares_analytic():
    h = 0.25
    pv, pf = _square(0.0)
    gv, gf = _square(h)
    rnd = _draws([2], 2000, 1)
    for scale in ("gt-10", None):                                  # the square's longest side is already 10
        row = om.compare_meshes_with(pv, pf, [4], [2], gv, gf, [4], [2], rnd, rnd, scale=scale, thresholds=TAUS)[0]
        assert float(row["Chamfer-L2"]) == pytest.approx(2 * h * h, rel=1e-6)
        assert float(row["NormalConsistency"]) == pytest.approx(1.0, abs=1e-12)
        for tau in TAUS:
            assert float(row["F1@%g" % tau]) == pytest.approx(100.0 if tau > h else 0.0, abs=1e-6)


def test_gt10_scale_makes_longest_side_ten():
    from meshrcnn_b200 import synthetic
    v, vi, f, fi, _ = cubify_np.cubify(synthetic.blob_voxels(3, 10, 5).numpy(), 0.2)
    v = torch.from_numpy(v).double() * torch.tensor([0.3, 1.7, 0.9], dtype=torch.float64)     # anisotropic extent
    for part in v.split(vi):
        scaled = om.gt_scale(part) * part
        assert float((scaled.max(0).values - scaled.min(0).values).max()) == pytest.approx(10.0, rel=1e-12)


def test_empty_predicted_mesh_row():
    pv, pf = _square(0.0)
    gv, gf = _square(0.1)
    rnd = _draws([2, 2], 100, 2)
    rows = om.compare_meshes_with(pv, pf, [4], [2], torch.cat([gv, gv]), torch.cat([gf, gf]), [4, 4], [2, 2], rnd,
                                        rnd, thresholds=TAUS)
    assert np.isnan(float(rows[1]["Chamfer-L2"])) and np.isnan(float(rows[1]["NormalConsistency"]))
    assert all(float(rows[1]["%s@%g" % (k, t)]) == 0.0 for k in ("Precision", "Recall", "F1") for t in TAUS)
    assert np.isfinite(float(rows[0]["Chamfer-L2"]))


_GLOO_WORKER = r"""
import sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from meshrcnn_b200.sharding import reduce_mesh_metrics
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()

def per_mesh(r):
    g = torch.Generator().manual_seed(100 + r)
    B = 3 + 2 * r
    valid = torch.rand(B, generator=g) > 0.3
    valid[0] = True
    d = {"Chamfer-L2": torch.rand(B, generator=g), "F1@0.3": 100 * torch.rand(B, generator=g)}
    d["Chamfer-L2"][~valid] = float("nan")
    d["F1@0.3"][~valid] = 0.0
    d["valid"] = valid
    return d

mine = per_mesh(rank)
before = {k: v.clone() for k, v in mine.items()}
got = reduce_mesh_metrics(mine)
assert all(torch.equal(before[k], mine[k]) if k == "valid" else torch.allclose(before[k], mine[k], equal_nan=True)
           for k in mine)                                                        # input left as it was
allv = [per_mesh(r) for r in range(world)]
valid = torch.cat([a["valid"] for a in allv])
assert got["num_valid"] == int(valid.sum())
for k in ("Chamfer-L2", "F1@0.3"):
    want = torch.cat([a[k] for a in allv]).double()[valid].mean()
    assert abs(float(got[k]) - float(want)) <= 1e-6 * abs(float(want)), (k, float(got[k]), float(want))
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_world_size_2_gloo_reduce_mesh_metrics(tmp_path):
    script = tmp_path / "gloo_metrics_worker.py"
    script.write_text(_GLOO_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29547", str(script)],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok") == 2


def test_reduce_mesh_metrics_without_process_group_is_the_local_mean():
    from meshrcnn_b200.sharding import reduce_mesh_metrics
    d = {"Chamfer-L2": torch.tensor([1.0, float("nan"), 3.0]), "valid": torch.tensor([True, False, True])}
    got = reduce_mesh_metrics(d)
    assert got["num_valid"] == 2 and float(got["Chamfer-L2"]) == 2.0
    assert np.isnan(float(d["Chamfer-L2"][1]))


def test_new_entry_points_parse_and_export(lib):
    import ctypes
    from meshrcnn_b200 import _lib
    sig = _lib.SIGNATURES
    assert sig["mrb_sample_surface_fwd"] == ("i", "pppppiippppLppppp")
    assert sig["mrb_mesh_gt_scale"] == ("i", "ppifpp")
    assert sig["mrb_mesh_metrics"] == ("i", "ppppppiiipipp")
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("mrb_sample_surface_fwd", "mrb_mesh_gt_scale", "mrb_mesh_metrics"):
        assert hasattr(raw, name)
    if _lib._fast_call is not None:                   # pointer / integer arguments only: bound through the call shim
        assert "mrb_sample_surface_fwd" in _lib._FAST and "mrb_mesh_metrics" in _lib._FAST
        assert "mrb_mesh_gt_scale" not in _lib._FAST
    # argument checks run before any device work
    assert lib.mrb_mesh_metrics(None, None, None, None, None, None, 1, 1, 1, None, 0, None, None) != 0
    taus = (ctypes.c_float * 9)(*([0.1] * 9))
    p = ctypes.c_void_p(16)
    assert lib.mrb_mesh_metrics(p, p, p, p, p, p, 1, 1, 1, taus, 9, p, None) != 0
    assert b"thresholds" in lib.mrb_last_error()
