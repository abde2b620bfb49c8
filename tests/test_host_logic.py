"""CPU: host-side logic (sharding, synthetic generators, module / state-dict surface) and the world_size-2 gloo path."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_split_to_n_matches_reference_semantics():
    from meshrcnn_b200.sharding import balanced_split, split_to_n
    assert split_to_n(10, 4) == [(0, 3), (3, 6), (6, 8), (8, 10)]      # first len % n chunks get one extra
    assert split_to_n(256, 8) == [(32 * r, 32 * r + 32) for r in range(8)]
    assert split_to_n(3, 4) == [(0, 1), (1, 2), (2, 3), (3, 3)]
    parts = balanced_split([5, 3, 8, 1, 2, 7], 2)
    assert sorted(sum(parts, [])) == list(range(6))
    loads = [sum([5, 3, 8, 1, 2, 7][i] for i in p) for p in parts]
    assert abs(loads[0] - loads[1]) <= 2
    costs = [float(c) for c in np.random.RandomState(0).randint(1500, 2600, size=64)]
    eq = balanced_split(costs, 8, equal_counts=True)                    # snake deal: equal counts, near-equal sums
    assert sorted(sum(eq, [])) == list(range(64)) and all(len(p) == 8 for p in eq)
    sums = [sum(costs[i] for i in p) for p in eq]
    naive = [sum(costs[8 * r:8 * r + 8]) for r in range(8)]
    assert max(sums) - min(sums) < 0.25 * (max(naive) - min(naive))
    assert balanced_split(costs[:32], 1, equal_counts=True) == [list(range(32))]


def test_flat_grad_bucket_survives_zero_grad_set_to_none():
    """ADVICE r1: zero_grad(set_to_none=True) drops the bucket views; all_reduce()/zero() must re-attach them instead of
    silently exchanging a stale buffer."""
    from meshrcnn_b200.sharding import FlatGradBucket, StagedGradBuckets
    torch.manual_seed(0)
    lin = torch.nn.Sequential(torch.nn.Linear(5, 4, bias=False), torch.nn.Linear(4, 2, bias=False))
    bucket = FlatGradBucket(lin.parameters())
    x = torch.randn(3, 5)
    lin(x).pow(2).sum().backward()
    want = bucket.flat.clone()
    assert float(want.abs().sum()) > 0
    lin.zero_grad(set_to_none=True)                                     # the views are gone
    lin(x).pow(2).sum().backward()                                      # fresh .grad tensors, bucket untouched
    assert bucket.sync_views() == 2
    assert torch.allclose(bucket.flat, want) and lin[0].weight.grad.data_ptr() == bucket.flat.data_ptr()
    bucket.zero()
    assert float(bucket.flat.abs().sum()) == 0 and float(lin[1].weight.grad.abs().sum()) == 0
    lin.zero_grad(set_to_none=True)
    bucket.zero()                                                       # re-binds
    lin(x).pow(2).sum().backward()
    assert torch.allclose(bucket.flat, want)
    # staged buckets: gradients start as None (no accumulate kernels), hooks count the parameters of a group; without a
    # process group nothing is packed or exchanged and the gradients stay where autograd put them
    sb = StagedGradBuckets([list(lin[0].parameters()), list(lin[1].parameters())])
    assert all(p.grad is None for p in lin.parameters())
    lin(x).pow(2).sum().backward()
    assert sb._pending == [0, 0] and sb._issued == [True, True]
    sb.finish()
    assert torch.allclose(torch.cat([p.grad.flatten() for p in lin.parameters()]), want)
    sb._pack(0); sb._pack(1)                                             # what a multi-GPU run does before its all-reduce
    assert torch.allclose(torch.cat(sb.flats), want)
    sb.zero()
    assert sb._pending == [1, 1] and sb._issued == [False, False] and lin[0].weight.grad is None


def test_synthetic_inputs_are_deterministic_and_sized():
    from meshrcnn_b200 import synthetic
    a, b = synthetic.blob_voxels(4, 32, 0), synthetic.blob_voxels(4, 32, 0)
    assert torch.equal(a, b) and a.shape == (4, 32, 32, 32)
    occ = float((a > 0.2).float().mean())
    assert 0.12 < occ < 0.25                                            # ~18.5 % (SURVEY 8d)
    pos = synthetic.in_frustum_positions(1000, 224, 0)
    h = 248 * (pos[:, 1] / pos[:, 2]) + 111.5
    w = 248 * (pos[:, 0] / -pos[:, 2]) + 111.5
    assert bool(((h > 0) & (h < 223) & (w > 0) & (w < 223)).all())


def test_module_surface_and_state_dict_keys():
    """Names, constructor arguments and state-dict keys of reference meshRCNN/layers.py (SURVEY 8b / section 5)."""
    import inspect
    import meshrcnn_b200.layers as L
    from meshrcnn_b200.pipeline import RefinementHead
    head = RefinementHead("shapenet_residual")
    keys = set(head.state_dict())
    assert {"cubify.kernel", "cubify.deltas", "refineStages.0.linear.weight", "refineStages.0.resGraphConv0.conv0.w0",
            "refineStages.0.resGraphConv0.projection.weight", "refineStages.2.graphConv.w1"} <= keys
    assert head.cubify.kernel.shape == (6, 1, 3, 3, 3) and head.cubify.deltas.shape == (6, 4, 5)
    assert head.refineStages[0].resGraphConv0.conv0.w0.shape == (131, 128)      # stored in x out
    assert head.refineStages[1].resGraphConv0.conv0.w0.shape == (259, 128)
    assert sum(p.numel() for p in head.parameters()) == 2217600                 # SURVEY 8e
    assert sum(p.numel() for p in RefinementHead("pix3d").parameters()) == 466843
    sig = inspect.signature(L.ResVertixRefineShapenet.forward)
    assert list(sig.parameters)[1:] == ["vertice_index", "img_feature_maps", "vertex_adjacency", "vertex_positions",
                                        "image_sizes", "vertex_features", "mesh_index"]
    sig = inspect.signature(L.VertixRefinePix3D.forward)
    assert list(sig.parameters)[1:] == ["vertice_index", "back_bone_features", "vertex_adjacency", "vertex_positions",
                                        "image_sizes", "mesh_index", "vertex_features"]
    k = L.Cubify(0.5).kernel
    assert k[2, 0, 1, 1, 1] == 1 and k[2, 0, 1, 2, 1] == -1 and float(k[2].sum()) == 0
    d = L.Cubify(0.5).deltas
    assert d[2, 0].tolist() == [0, 0, 0.5, -0.5, -0.5] and d[4, 1].tolist() == [0, 0, -0.5, -0.5, -0.5]


def test_sharded_losses_recombine_like_reference_dp():
    """Chamfer / normal terms are batch sums, so per-shard values add up to the unsharded value; the edge loss is a
    per-replica mean that the reference DP sums over replicas (gather.py:109-112) -- SURVEY 8e."""
    from oracle import cubify_np, mesh_ops
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.sharding import split_to_n
    B, n, k = 4, 200, 4
    verts, vi, faces, fi, adj = cubify_np.cubify(synthetic.blob_voxels(B, 8, 0).numpy(), 0.2)
    gverts, gvi, gfaces, gfi, _ = cubify_np.cubify(synthetic.blob_voxels(B, 8, 1000).numpy(), 0.5)
    pos = torch.from_numpy(verts).double() * 0.1
    gpos = torch.from_numpy(gverts).double() * 0.1
    faces, gfaces, adj = torch.from_numpy(faces), torch.from_numpy(gfaces), torch.from_numpy(adj)
    u, x2, x1 = synthetic.sampling_randomness(B, n, 1)
    fi_p = torch.stack([mesh_ops.face_cdf_draw(v, f, u[b]) for b, (v, f) in enumerate(zip(pos.split(vi), faces.split(fi)))])
    fi_g = torch.stack([mesh_ops.face_cdf_draw(v, f, u[b]) for b, (v, f) in enumerate(zip(gpos.split(gvi), gfaces.split(gfi)))])
    full = mesh_ops.mesh_loss_with(pos, faces, adj, vi, fi, gpos, gfaces, gvi, gfi, (fi_p, x2.double(), x1.double()),
                                   (fi_g, x2.double(), x1.double()), float(n), k)
    ch = nl = 0.0
    edges = []
    for lo, hi in split_to_n(B, 2):
        vo, fo, gvo, gfo = sum(vi[:lo]), sum(fi[:lo]), sum(gvi[:lo]), sum(gfi[:lo])
        vn, fn, gvn, gfn = sum(vi[lo:hi]), sum(fi[lo:hi]), sum(gvi[lo:hi]), sum(gfi[lo:hi])
        sel = (adj[0] >= vo) & (adj[0] < vo + vn)
        part = mesh_ops.mesh_loss_with(pos[vo:vo + vn], faces[fo:fo + fn], adj[:, sel] - vo, vi[lo:hi], fi[lo:hi],
                                       gpos[gvo:gvo + gvn], gfaces[gfo:gfo + gfn], gvi[lo:hi], gfi[lo:hi],
                                       (fi_p[lo:hi], x2[lo:hi].double(), x1[lo:hi].double()),
                                       (fi_g[lo:hi], x2[lo:hi].double(), x1[lo:hi].double()), float(n), k)
        ch, nl = ch + part[0], nl + part[1]
        edges.append((part[2], int(sel.sum())))
    assert torch.allclose(ch, full[0], rtol=1e-12) and torch.allclose(nl, full[1], rtol=1e-9)
    recombined = sum(e * m for e, m in edges) / sum(m for _, m in edges)
    assert torch.allclose(recombined, full[2], rtol=1e-12)


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from meshrcnn_b200.sharding import FlatGradBucket, StagedGradBuckets, all_reduce_losses, split_to_n
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
torch.manual_seed(0)
lin = torch.nn.Sequential(torch.nn.Linear(5, 4, bias=False), torch.nn.Linear(4, 2, bias=False))
bucket = FlatGradBucket(lin.parameters())
data = torch.arange(40.).reshape(8, 5) / 10
lo, hi = split_to_n(8, world)[rank]
bucket.zero()
lin(data[lo:hi]).pow(2).sum().backward()
assert lin[0].weight.grad.data_ptr() == bucket.flat.data_ptr()          # grads accumulate straight into the bucket
bucket.all_reduce()
ref = torch.nn.Sequential(torch.nn.Linear(5, 4, bias=False), torch.nn.Linear(4, 2, bias=False))
ref.load_state_dict(lin.state_dict())
ref(data).pow(2).sum().backward()                                       # SUM over shards == unsharded gradient
for p, q in zip(lin.parameters(), ref.parameters()):
    assert torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-6), (rank, p.grad, q.grad)
# overlapped exchange: one bucket per layer, all-reduce issued from the post-accumulate-grad hooks during backward
lin2 = torch.nn.Sequential(torch.nn.Linear(5, 4, bias=False), torch.nn.Linear(4, 2, bias=False))
lin2.load_state_dict(ref.state_dict())
sb = StagedGradBuckets([list(lin2[0].parameters()), list(lin2[1].parameters())])
for _ in range(2):                                                      # two steps: counters / handles reset correctly
    sb.zero()
    lin2(data[lo:hi]).pow(2).sum().backward()
    assert sb._issued == [True, True]                                   # both exchanges were issued inside backward
    sb.finish()
    for p, q in zip(lin2.parameters(), ref.parameters()):
        assert torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-6), (rank, p.grad, q.grad)
sb.enabled = False                                                      # rank-local steps (time-based loops) issue nothing
sb.zero()
lin2(data[lo:hi]).pow(2).sum().backward()
assert sb._issued == [False, False]
sb.finish(exchange=False)
# eval outputs: ragged gather with the edge ids re-offset (reference gather.py:65-92)
from meshrcnn_b200.sharding import gather_eval_outputs
nv = [3, 2] if rank == 0 else [4]
SV = sum(nv)
mine = {"vertex_positions": [torch.full((SV, 3), float(rank)), torch.full((SV, 3), 10.0 + rank)],
        "edge_index": torch.tensor([[0, SV - 1], [SV - 1, 0]]), "faces": torch.tensor([[0, 1, 2]] * (rank + 1)),
        "vertice_index": nv, "face_index": [1] * len(nv), "mesh_index": [1] * len(nv)}
g = gather_eval_outputs(mine)
assert g["vertice_index"] == [3, 2, 4] and g["mesh_index"] == [1, 1, 1] and g["faces"].shape == (3, 3)
assert g["vertex_positions"][0].shape == (9, 3) and float(g["vertex_positions"][1][5:].mean()) == 11.0
assert g["edge_index"].tolist() == [[0, 4, 5, 8], [4, 0, 8, 5]], g["edge_index"].tolist()
tot = all_reduce_losses({"chamfer_loss": torch.tensor(float(rank + 1)), "edge_loss": torch.tensor(2.0)})
assert float(tot["chamfer_loss"]) == sum(range(1, world + 1)) and float(tot["edge_loss"]) == 2.0 * world
# identically seeded ranks must still draw different surface-sampling seeds
from meshrcnn_b200.functional import _next_seed
torch.manual_seed(123)
seeds = [None] * world
dist.all_gather_object(seeds, _next_seed())
assert len(set(seeds)) == world, seeds
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_world_size_2_gloo_gradient_allreduce(tmp_path):
    script = tmp_path / "gloo_worker.py"
    script.write_text(_GLOO_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("ok") == 2


def test_batched_seed_draw_equals_single_draws():
    """functional._next_seeds(n): one randint call, the values of n single draws (the refinement head pre-draws the seeds of all
    stages; the lazy path draws them one by one)."""
    from meshrcnn_b200.functional import _next_seed, _next_seeds
    torch.manual_seed(77)
    single = [_next_seed() for _ in range(6)] + [_next_seed()]
    torch.manual_seed(77)
    batched = _next_seeds(6) + [_next_seed()]
    assert single == batched and len(set(single)) == 7


def test_bench_reference_arm_extra_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bench_time_based_loops_issue_no_collective():
    """A loop bounded by wall-clock time runs a different number of iterations on every rank, so it must not contain the
    step's NCCL all-reduce (bench.py's start-up phase once did: deadlock at N > 1)."""
    import ast
    src = open(os.path.join(ROOT, "bench.py")).read()
    tree = ast.parse(src)
    checked = 0
    for node in ast.walk(tree):
        if isinstance(node, ast.While) and "perf_counter" in ast.get_source_segment(src, node.test):
            for call in ast.walk(node):
                if isinstance(call, ast.Call) and "step" in (getattr(call.func, "id", None), getattr(call.func, "attr", None)):
                    kw = {k.arg: k.value for k in call.keywords}
                    assert "exchange" in kw and isinstance(kw["exchange"], ast.Constant) and kw["exchange"].value is False
                    checked += 1
    assert checked >= 1


def test_bench_reference_arm_line_keeps_the_contract():
    """`bench.py --impl reference` (the reference's own CPU path from oracle/_ref, else the oracle port) prints ONE JSON
    line with the contract's keys and the CUDA arm's workload string."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "meshes/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    from oracle import ref_import
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_import.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "BASELINE configs[1]" in d["config"]["workload"] and "1 mesh" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "meshes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.parametrize("argv, message", [
    (["--steps", "0"], "--steps must be at least 1"),
    (["--impl", "reference", "--dump-outputs", "d"], "does not go with --check or --impl reference"),
    (["--check", "--dump-outputs", "d"], "does not go with --check or --impl reference")])
def test_bench_rejects_bad_arguments(argv, message):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and message in r.stderr and r.stdout.strip() == ""


def test_bench_refuses_a_library_not_built_from_the_tree(lib, monkeypatch):
    """bench.py compiles nothing; a library whose recorded source digest differs from the tree's sources (an edited .cu
    file) is refused instead of being timed and dumped as if it were the current code."""
    import bench
    from meshrcnn_b200 import build
    assert not build.needs_build() and bench.load_built_library() is lib
    monkeypatch.setattr(build, "source_digest", lambda: "0" * 64)
    assert build.needs_build()
    with pytest.raises(SystemExit, match="run build"):
        bench.load_built_library()


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """`bench.py --dump-outputs DIR` writes the last timed step's losses and gradients as float32 .npy files.  The timed steps
    start from a fixed seed, so the same step recomputed here from the same workload gives the same arrays (up to the order
    of floating-point sums), while the step before it, which draws other surface samples, does not."""
    import json
    import bench
    d = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout)["steps"] == 2
    got = {p.name[:-4]: np.load(p) for p in d.iterdir()}
    assert sum(x.nbytes for x in got.values()) <= 64 << 20

    wl = bench.HeadWorkload("pix3d", torch.device("cuda", 0), 0, 1)
    torch.manual_seed(0)
    first = {k: float(v) for k, v in wl.step().items()}
    losses = wl.step()
    want = {k: v.detach().cpu().numpy() for k, v in losses.items()}
    want["feature_map0.grad"] = wl.fmaps_d[0].grad.cpu().numpy()
    want.update({n + ".grad": p.grad.cpu().numpy() for n, p in wl.head.named_parameters()})
    assert len(want) == 3 + 1 + 21 and set(got) == set(want)
    for k, w in want.items():
        assert got[k].dtype == np.float32 and got[k].shape == w.shape and np.isfinite(got[k]).all(), k
        np.testing.assert_allclose(got[k], w, rtol=1e-4, atol=1e-5 * float(np.abs(w).max()), err_msg=k)
    assert abs(first["chamfer_loss"] - float(got["chamfer_loss"])) > 1e-4 * abs(first["chamfer_loss"])
