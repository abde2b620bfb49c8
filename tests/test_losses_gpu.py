"""Sampling + chamfer / normal / edge losses: CUDA path vs the reference's outputs (tests/golden) and the fp64
oracle.  Tolerances: fp32 rtol 1e-4 (north star); k-NN / NN index sets compared exactly away from fp32 ties.

Normal loss (see DESIGN.md): the reference takes a *row* of the eigenvector matrix, whose value depends on
LAPACK's unspecified eigenvector signs; the kernel uses a documented canonical sign rule and is compared with the
oracle under the same rule (``canonical_signs=True``); everything else (k-NN sets, scatter matrices, eigenvectors up
to sign, backward) is compared directly."""
import numpy as np
import pytest
import torch

from oracle import mesh_ops
from tests.test_layers_gpu import close, cuda

pytestmark = pytest.mark.gpu


class FakeBatch:
    def __init__(self, meshes, vertice_index, face_index):
        self.meshes, self.vertice_index, self.face_index = meshes, vertice_index, face_index


def test_known_answers_from_reference_tests(lib):
    """tests/test_loss_functions.py:14-55,59-72,76-96,100-125 of the reference, through the fused kernels."""
    from meshrcnn_b200 import loss_functions as LF
    from meshrcnn_b200.mesh_sampling import surface_areas, sample
    from meshrcnn_b200.utils import dummy
    # chamfer sums 300 / 21 and 600 / 42 (exact ==)
    pt0, pt1 = dummy(1, 10, 3).cuda(), (dummy(1, 7, 3) + 1).cuda()
    l0, i0, l1, i1 = LF.chamfer_distance(pt0, pt1)
    assert i0.shape == (1, 10) and i1.shape == (1, 7) and l0.item() == 300 and l1.item() == 21
    l0, i0, l1, i1 = LF.chamfer_distance(pt0.expand(2, 10, 3).contiguous(), pt1.expand(2, 7, 3).contiguous())
    assert l0.item() == 600 and l1.item() == 42
    d = LF.batched_point2point_distance(pt0, pt1)
    r0, ri0, r1, ri1 = LF.batched_chamfer_distance(d)
    assert r0.item() == 300 and r1.item() == 21 and torch.equal(ri0, i0[:1]) and torch.equal(ri1, i1[:1])
    # edge length (test_edge_length)
    pos = dummy(1, 10, 3).squeeze().cuda()
    adj = torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]]).cuda()
    p2p = LF.batched_point2point_distance(pos).squeeze()
    want = (p2p[0, 1] + p2p[1, 0] + p2p[1, 2] + p2p[2, 1]) / 4
    assert torch.allclose(LF.edge_length(pos, adj), want)
    assert torch.allclose(LF.total_edge_length(p2p, adj), want)
    # triangle areas [1.22474, 4, 3.5, 8.3666]
    v = torch.tensor([[0, 0, 0], [1, 0, 0], [1, 1, 1], [0, 0, 2], [0, 2, 0], [0, 1, 5], [2, 2, 2], [2, 7, 0],
                      [2, 3, 5], [2, 7, 8], [0, 3, 2]], dtype=torch.float32).cuda()
    f = torch.tensor([[1, 2, 8], [3, 4, 5], [0, 1, 7], [6, 9, 10]]).cuda()
    assert torch.allclose(surface_areas(v, f).cpu(), torch.tensor([1.22474, 4.0, 3.5, 8.3666]), rtol=1e-5)
    assert sample(v, f, num_points=2000).shape == (2000, 3)


def _load(golden):
    g = golden("sampling_losses")
    t = lambda k: torch.as_tensor(g[k])
    return g, t


def test_areas_and_sampling_match_reference(lib, golden):
    from meshrcnn_b200 import functional as F_
    g, t = _load(golden)
    v_index, f_index = g["v_index"].tolist(), g["f_index"].tolist()
    pos = cuda(g["pos"], grad=True)
    faces = cuda(g["faces"]).long()
    close(F_.face_areas(pos, faces, v_index, f_index), g["f64__areas"], what="areas")
    # injected face indices + barycentric draws == the reference's sample() under the same draws
    cloud, fidx = F_.sample_points(pos, faces, v_index, f_index, int(g["n_points"]), face_idx=cuda(g["fi_p"]).long(),
                                   xi2=cuda(g["xi2_p"]), xi1=cuda(g["xi1_p"]))
    close(cloud, g["f64__cloud"], what="cloud")
    (cloud * cuda(g["f64__gcloud"])).sum().backward()
    close(pos.grad, g["f64__cloud_gpos"], what="cloud grad")
    # the kernel's own inverse-CDF draw from injected uniforms == oracle face_cdf_draw
    cloud2, fidx2 = F_.sample_points(pos.detach(), faces, v_index, f_index, int(g["n_points"]), u=cuda(g["u_p"]),
                                     xi2=cuda(g["xi2_p"]), xi1=cuda(g["xi1_p"]))
    f_off = np.concatenate([[0], np.cumsum(f_index)])[:-1]
    local = fidx2.cpu().numpy() - f_off[:, None]
    mism = (local != g["fi_p"]).mean()
    assert mism < 2e-3, mism          # fp32 areas vs fp64 oracle areas can move a draw that sits on a CDF boundary
    if mism == 0:
        close(cloud2, g["f64__cloud"], what="cloud (cdf draw)")


def test_philox_sampling_distribution(lib):
    """Own-RNG path: faces are drawn proportionally to area (chi-square), points lie on their triangles,
    reproducible under torch.manual_seed."""
    from meshrcnn_b200 import functional as F_
    v = torch.tensor([[0, 0, 0], [1, 0, 0], [0, 1, 0], [3, 0, 0], [0, 3, 0], [0, 0, 0.5]], dtype=torch.float32).cuda()
    f = torch.tensor([[0, 1, 2], [0, 3, 4], [0, 1, 5]]).cuda()
    areas = mesh_ops.surface_areas(v.cpu().double(), f.cpu())
    n = 200000
    torch.manual_seed(7)
    cloud, fidx = F_.sample_points(v, f, [6], [3], n)
    torch.manual_seed(7)
    cloud_b, fidx_b = F_.sample_points(v, f, [6], [3], n)
    assert torch.equal(cloud, cloud_b) and torch.equal(fidx, fidx_b)
    counts = torch.bincount(fidx.flatten().long().cpu(), minlength=3).double()
    expect = areas / areas.sum() * n
    chi2 = float(((counts - expect) ** 2 / expect).sum())
    assert chi2 < 20.0, (chi2, counts, expect)          # 2 dof; P(chi2 > 20) ~ 5e-5
    assert abs(float(cloud.mean())) < 1e-3              # centred


def test_chamfer_knn_vs_oracle(lib, golden):
    from meshrcnn_b200 import functional as F_
    g, t = _load(golden)
    p, q = cuda(g["f64__cloud"], grad=True), cuda(g["f64__cloud_gt"])
    k = int(g["k"])
    l1, l2, ip, iq, kp, kq = F_.chamfer_knn(p, q, k)
    assert np.array_equal(ip.cpu().numpy(), g["f64__idx_p"]) and np.array_equal(iq.cpu().numpy(), g["f64__idx_gt"])
    assert np.array_equal(kp.sort(-1).values.cpu().numpy(), g["f64__knn_p"])
    assert np.array_equal(kq.sort(-1).values.cpu().numpy(), g["f64__knn_gt"])
    d = mesh_ops.p2p_distance(t("f64__cloud"), t("f64__cloud_gt"))
    w1, _, w2, _ = mesh_ops.chamfer(d)
    close(l1, w1, what="loss_1")
    close(l2, w2, what="loss_2")


@pytest.mark.parametrize("B,P,Q,k", [(2, 1000, 1000, 10), (3, 777, 1301, 4), (1, 5, 2049, 0), (2, 130, 64, 16)])
def test_knn_ragged_sizes_vs_oracle(lib, B, P, Q, k):
    from meshrcnn_b200 import functional as F_
    gen = torch.Generator().manual_seed(B * 1000 + P)
    p, q = torch.rand(B, P, 3, generator=gen) - 0.5, torch.rand(B, Q, 3, generator=gen) - 0.5
    pc, qc = p.cuda().requires_grad_(), q.cuda().requires_grad_()
    l1, l2, ip, iq, kp, kq = F_.chamfer_knn(pc, qc, k)
    _, ip_t, kp_t, _, iq_t, kq_t = F_.knn_search(p.cuda(), q.cuda(), k, algo="tiled")
    assert torch.equal(ip, ip_t) and torch.equal(iq, iq_t) and (not k or (torch.equal(kp, kp_t) and torch.equal(kq, kq_t)))
    p64, q64 = p.double().requires_grad_(), q.double().requires_grad_()
    d = mesh_ops.p2p_distance(p64, q64)
    w1, wi1, w2, wi2 = mesh_ops.chamfer(d)
    close(l1, w1.detach(), what="l1")
    close(l2, w2.detach(), what="l2")
    assert torch.equal(ip.cpu().long(), wi1) and torch.equal(iq.cpu().long(), wi2)
    # gradients of both sums through the dense fp64 matrix (P != Q: the two scatter directions must not be swapped)
    gp, gq = torch.autograd.grad(0.7 * l1 + 1.3 * l2, [pc, qc])
    hp, hq = torch.autograd.grad(0.7 * w1 + 1.3 * w2, [p64, q64])
    close(gp, hp, what="grad p")
    close(gq, hq, what="grad q")
    d = d.detach()
    if k:
        for got, dd in ((kp, d), (kq, d.transpose(1, 2))):
            want = dd.topk(k, dim=2, largest=False).indices.sort(-1).values
            assert torch.equal(got.cpu().long().sort(-1).values, want)


def _knn_clouds(kind, B, P, Q, seed):
    gen = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.rand(*s, generator=gen)
    if kind == "cube":
        return r(B, P, 3) - 0.5, r(B, Q, 3) - 0.5
    if kind == "sphere":                                   # points on two different surfaces
        a, b = torch.randn(B, P, 3, generator=gen), torch.randn(B, Q, 3, generator=gen)
        return a / a.norm(dim=2, keepdim=True), 0.7 * b / b.norm(dim=2, keepdim=True) * torch.tensor([1.0, 0.6, 1.4])
    if kind == "far":                                      # queries far outside the other cloud's bounding box
        return r(B, P, 3) + 5.0, r(B, Q, 3) * 0.1
    if kind == "plane":                                    # degenerate axis (z extent 0) and an x-y lattice full of ties
        a = torch.stack([torch.randint(0, 12, (B, P), generator=gen).float(),
                         torch.randint(0, 12, (B, P), generator=gen).float(), torch.zeros(B, P)], 2)
        b = torch.stack([torch.randint(0, 12, (B, Q), generator=gen).float(),
                         torch.randint(0, 12, (B, Q), generator=gen).float(), torch.zeros(B, Q)], 2)
        return a, b
    if kind == "point":                                    # every candidate identical
        return r(B, P, 3), torch.full((B, Q, 3), 0.25)
    if kind == "clusters":                                 # two tight clusters far apart: most cells empty
        a = torch.where(r(B, P, 1) < 0.5, r(B, P, 3) * 1e-3, r(B, P, 3) * 1e-3 + 10.0)
        b = torch.where(r(B, Q, 1) < 0.1, r(B, Q, 3) * 1e-3, r(B, Q, 3) * 1e-3 + 10.0)
        return a, b
    raise ValueError(kind)


@pytest.mark.parametrize("kind,B,P,Q,k", [
    ("cube", 2, 3000, 2500, 10), ("sphere", 2, 10000, 10000, 10), ("far", 1, 500, 700, 4), ("plane", 2, 900, 1100, 10),
    ("point", 1, 300, 200, 16), ("clusters", 2, 2000, 2000, 10), ("cube", 3, 17, 16, 16), ("sphere", 1, 4000, 9000, 1),
    ("cube", 1, 1, 1, 1), ("cube", 2, 2000, 3000, 0)])
def test_knn_grid_equals_tiled_scan(lib, kind, B, P, Q, k):
    """The cell-grid search and the tiled brute-force scan must agree bit for bit (distances, nearest index, and the
    ordered k-NN lists incl. (distance, index) tie-breaking); the tiled scan is itself checked against the oracle."""
    from meshrcnn_b200 import functional as F_
    p, q = _knn_clouds(kind, B, P, Q, seed=P + Q + k)
    want = F_.knn_search(p.cuda(), q.cuda(), k, algo="tiled")
    for algo in ("grid", "auto"):
        got = F_.knn_search(p.cuda(), q.cuda(), k, algo=algo)
        for name, a, b in zip(("d_p", "i_p", "knn_p", "d_q", "i_q", "knn_q"), got, want):
            if a is None:
                assert b is None
                continue
            assert torch.equal(a, b), "%s (%s) differs on %s: %d of %d" % (name, algo, kind, int((a != b).sum()), a.numel())
    # and against exact fp64 distances (ties broken by index, like torch.min on the oracle's matrix)
    d = mesh_ops.p2p_distance(p.double(), q.double())
    dd = torch.gather(d, 2, got[1].long().cpu().unsqueeze(2)).squeeze(2)
    assert torch.allclose(dd, d.min(dim=2).values, rtol=1e-5, atol=1e-12)


def test_mesh_loss_matches_reference(lib, golden):
    """Full stage loss with injected randomness vs the unmodified reference (golden, fp64 run)."""
    from meshrcnn_b200 import loss_functions as LF
    g, t = _load(golden)
    v_index, f_index = g["v_index"].tolist(), g["f_index"].tolist()
    pos = cuda(g["pos"], grad=True)
    faces, adj = cuda(g["faces"]).long(), cuda(g["adj"]).long()
    batch = FakeBatch((cuda(g["gt_pos"]), cuda(g["gt_faces"]).long()), g["gt_v_index"].tolist(), g["gt_f_index"].tolist())
    rnd = (dict(face_idx=cuda(g["fi_p"]).long(), xi2=cuda(g["xi2_p"]), xi1=cuda(g["xi1_p"])),
           dict(face_idx=cuda(g["fi_g"]).long(), xi2=cuda(g["xi2_g"]), xi1=cuda(g["xi1_g"])))
    ch, nl, ed = LF.mesh_loss(pos, faces, adj, v_index, f_index, batch, float(g["n_points"]), int(g["k"]), randomness=rnd)
    close(ch, g["f64__chamfer"], what="chamfer")
    close(ed, g["f64__edge"], what="edge")
    gch, = torch.autograd.grad(ch, pos, retain_graph=True)
    close(gch, g["f64__chamfer_gpos"], what="chamfer grad")
    ged, = torch.autograd.grad(ed, pos, retain_graph=True)
    close(ged, g["f64__edge_gpos"], what="edge grad")
    # normal loss: against the oracle evaluated with the kernel's eigenvector sign convention
    close(nl, g["f64__normal_canonical"], what="normal (canonical signs)")
    gnl, = torch.autograd.grad(nl, pos)
    want = torch.as_tensor(g["f64__normal_canonical_gpos"])
    err = (gnl.cpu().double() - want).abs()
    tol = 1e-4 * want.abs() + 1e-4 * float(want.abs().max())
    frac_bad = float((err > tol).double().mean())
    assert frac_bad < 5e-3, frac_bad      # ill-conditioned rows (near-degenerate eigen-gaps) excepted, SURVEY section 7
    # Distance to the RAW reference value (LAPACK's own, unspecified eigenvector signs): bounded by twice the reference's
    # own |fp32 - fp64| gap on this fixture (SURVEY 7c; measured: ours 0.9 %, the reference's 1.0 %).
    ref64, ref32 = float(g["f64__normal"]), float(g["f32__normal"])
    own_gap = abs(ref32 - ref64)
    assert own_gap > 0
    assert abs(float(nl) - ref64) <= 2.0 * own_gap, (float(nl), ref64, ref32)


def test_losses_at_bench_shape_vs_oracle(lib):
    """Chamfer / normal / edge at the bench shape (10 000-point clouds, k = 10, two 24^3 meshes) against the fp64 oracle with
    injected draws -- the check `python bench.py --check` runs (rtol 1e-4; normal also within 2 % of LAPACK's signs)."""
    import bench
    out = bench.check_bench_shape_losses(meshes=2, verbose=False)
    assert out["points"] == 10000 and out["k"] == 10


def test_normals_eigenvectors_vs_oracle(lib):
    """compute_normals with injected k-NN sets: row 0 of the canonically signed eigenvector matrix."""
    from meshrcnn_b200 import functional as F_
    gen = torch.Generator().manual_seed(3)
    B, P, k = 2, 500, 10
    pt = torch.rand(B, P, 3, generator=gen)
    nn = torch.stack([torch.stack([torch.randperm(P, generator=gen)[:k] for _ in range(P)]) for _ in range(B)])
    got = F_.compute_normals(pt.cuda(), nn.cuda())
    want = mesh_ops.normals_from_neighbours(pt.double(), nn, canonical_signs=True)
    close(got, want, rtol=1e-5, atol=1e-5, what="normals")
    assert torch.allclose(got.norm(dim=2).cpu(), torch.ones(B, P), atol=1e-5)


def test_padded_gradient_rows_equal_packed_rows(lib):
    """C ABI: mrb_normals_bwd_ld / mrb_sample_points_bwd_ld with 4-float rows (vector reductions) against the 3-float
    entry points (scalar atomics); only the summation order differs."""
    from meshrcnn_b200 import _lib
    gen = torch.Generator().manual_seed(9)
    B, P, k = 3, 700, 10
    pt = torch.rand(B, P, 3, generator=gen).cuda()
    nn = torch.randint(0, P, (B, P, k), generator=gen, dtype=torch.int32).cuda()
    gn = torch.randn(B, P, 3, generator=gen).cuda()
    g3 = torch.zeros(B, P, 3, device="cuda")
    g4 = torch.zeros(B, P, 4, device="cuda")
    _lib.call("mrb_normals_bwd", _lib.ptr(pt), _lib.ptr(nn), B, P, k, _lib.ptr(gn), _lib.ptr(g3))
    _lib.call("mrb_normals_bwd_ld", _lib.ptr(pt), _lib.ptr(nn), B, P, k, _lib.ptr(gn), _lib.ptr(g4), 4, None)
    assert float(g4[..., 3].abs().max()) == 0.0
    scale = float(g3.abs().max())
    assert scale > 0 and float((g4[..., :3] - g3).abs().max()) <= 2e-5 * scale
    with pytest.raises(RuntimeError):
        _lib.call("mrb_normals_bwd_ld", _lib.ptr(pt), _lib.ptr(nn), B, P, k, _lib.ptr(gn), _lib.ptr(g4), 5, None)
    # the eigen-decomposition saved by the forward pass gives the same gradient as recomputing it
    n0, n1 = torch.empty(B, P, 3, device="cuda"), torch.empty(B, P, 3, device="cuda")
    eig = torch.empty(12, B * P, dtype=torch.float64, device="cuda")
    _lib.call("mrb_normals_fwd", _lib.ptr(pt), _lib.ptr(nn), B, P, k, _lib.ptr(n0))
    _lib.call("mrb_normals_fwd_eig", _lib.ptr(pt), _lib.ptr(nn), B, P, k, _lib.ptr(n1), _lib.ptr(eig))
    assert torch.equal(n0, n1) and torch.equal(eig[3:6].t().float().reshape(B, P, 3), n1)     # normal = row 0 of V
    g4e = torch.zeros(B, P, 4, device="cuda")
    _lib.call("mrb_normals_bwd_ld", _lib.ptr(pt), _lib.ptr(nn), B, P, k, _lib.ptr(gn), _lib.ptr(g4e), 4, _lib.ptr(eig))
    assert float((g4e - g4).abs().max()) <= 2e-5 * scale
    # sampling backward: two tetrahedra, 300 points each
    verts = torch.rand(8, 3, generator=gen).cuda()
    faces = torch.tensor([[0, 1, 2], [0, 1, 3], [0, 2, 3], [1, 2, 3]] * 2).cuda()
    v_off = torch.tensor([0, 4, 8], dtype=torch.int32).cuda()
    n = 300
    cloud = torch.rand(2, n, 3, generator=gen).cuda()
    gcloud = torch.randn(2, n, 3, generator=gen).cuda()
    stats = torch.zeros(2, 8, dtype=torch.float64).cuda()
    stats[:, 3] = 1.5
    stats[:, 4] = torch.tensor([7.0, -1.0], dtype=torch.float64).cuda()
    fidx = torch.cat([torch.randint(0, 4, (1, n), generator=gen), torch.randint(4, 8, (1, n), generator=gen)]).int().cuda()
    w = torch.rand(2, n, 3, generator=gen).cuda()
    out3, out4 = torch.zeros(8, 3, device="cuda"), torch.zeros(8, 4, device="cuda")
    scr = torch.empty(8, dtype=torch.float64, device="cuda")
    args = (_lib.ptr(gcloud), _lib.ptr(cloud), _lib.ptr(stats), _lib.ptr(fidx), _lib.ptr(w), _lib.ptr(faces), _lib.ptr(v_off), 2, n)
    _lib.call("mrb_sample_points_bwd", *args, _lib.ptr(out3), _lib.ptr(scr))
    _lib.call("mrb_sample_points_bwd_ld", *args, _lib.ptr(out4), 4, _lib.ptr(scr))
    assert float(out4[:, 3].abs().max()) == 0.0
    assert float((out4[:, :3] - out3).abs().max()) <= 2e-5 * float(out3.abs().max())


def test_batched_mesh_loss_runs_and_is_finite(lib):
    """Three stages, own RNG, gradient reaches the positions (shape/finite check at 10k points)."""
    from meshrcnn_b200 import loss_functions as LF, synthetic
    from meshrcnn_b200.layers import Cubify
    from meshrcnn_b200.mesh_sampling import normalize_mesh
    B = 2
    verts, vi, faces, fi, adj = Cubify(0.2)(synthetic.blob_voxels(B, 16, 0).cuda())
    gv, gvi, gfaces, gfi, _ = Cubify(0.5)(synthetic.blob_voxels(B, 16, 1000).cuda())
    gt = torch.cat([normalize_mesh(v) for v in gv.split(gvi)])
    batch = FakeBatch((gt, gfaces), gvi, gfi)
    pos = [(verts * 0.05 + 0.01 * i).requires_grad_() for i in range(3)]
    ch, nl, ed = LF.batched_mesh_loss(pos, faces, adj, vi, fi, batch)
    (ch + 0.1 * nl + 0.5 * ed).backward()
    for t in (ch, nl, ed):
        assert t.dim() == 0 and bool(torch.isfinite(t))
    for p in pos:
        assert bool(torch.isfinite(p.grad).all()) and float(p.grad.abs().sum()) > 0


def test_gt_sampling_cdf_cache(lib):
    """SURVEY 8 f-2: the area CDF of the static GT meshes is computed once per batch object; sampling through the cache is
    bit-identical to sampling without it, and an in-place edit of the vertices invalidates the cache."""
    from meshrcnn_b200 import _lib, functional as F_, synthetic
    from meshrcnn_b200.layers import Cubify
    B = 3
    verts, vi, faces, fi, _ = Cubify(0.5)(synthetic.blob_voxels(B, 12, 1000).cuda())
    verts = verts * 0.05
    owner = FakeBatch((verts, faces), vi, fi)
    plain, f0 = F_.sample_points(verts, faces, vi, fi, 500, seed=7)
    n0 = _lib.launch_count
    c1, f1 = F_.sample_points(verts, faces, vi, fi, 500, seed=7, cdf_owner=owner)
    first = _lib.launch_count - n0
    n0 = _lib.launch_count
    c2, f2 = F_.sample_points(verts, faces, vi, fi, 500, seed=7, cdf_owner=owner)
    second = _lib.launch_count - n0
    assert torch.equal(plain, c1) and torch.equal(c1, c2) and torch.equal(f0, f1) and torch.equal(f1, f2)
    assert second == first - _lib.LAUNCHES["mrb_face_area_cdf"]            # the CDF kernels ran only once
    key = owner._mrb_face_cdf[0]
    verts[: vi[0]] *= 2.0                                                   # in-place edit -> new version -> recomputed
    c3, _ = F_.sample_points(verts, faces, vi, fi, 500, seed=7, cdf_owner=owner)
    assert owner._mrb_face_cdf[0] != key
    want, _ = F_.sample_points(verts, faces, vi, fi, 500, seed=7)
    assert torch.equal(c3, want)


def test_validate_batch_on_eval_dict_vs_oracle(lib):
    """SURVEY 8 f-3: the device path of reference ``validate`` (eval_utils.py:160-164): batched_mesh_loss over ALL FOUR
    position sets of an eval-mode output dict (injected draws, vs the fp64 oracle) + F1@tau from the NN distances (vs dense
    fp64 distances on the same clouds)."""
    from oracle import cubify_np
    from meshrcnn_b200 import functional as F_, synthetic
    from meshrcnn_b200.eval_utils import validate_batch
    from meshrcnn_b200.mesh_sampling import normalize_mesh
    from meshrcnn_b200.pipeline import MeshTargets, RefinementHead
    B, V, n, k = 2, 12, 1500, 10
    vox = synthetic.blob_voxels(B, V, 2)
    fmap = synthetic.feature_maps(B, [synthetic.PIX3D_MAP], 2)[0] * 0.02
    torch.manual_seed(3)
    head = RefinementHead("pix3d", cubify_threshold=0.2).cuda().eval()
    with torch.no_grad():
        for prm in head.parameters():
            prm.mul_(0.2)
        out = head(vox.cuda(), fmap.cuda(), [(224, 224)] * B)
    out["voxels"] = vox.cuda()
    gverts, gvi, gfaces, gfi, _ = cubify_np.cubify(synthetic.blob_voxels(B, V, 1002).numpy(), 0.5)
    gt_pos = torch.cat([mesh_ops.normalize_cloud(v) for v in torch.from_numpy(gverts).double().split(gvi)])
    batch = MeshTargets(gt_pos.float().cuda(), torch.from_numpy(gfaces).cuda(), gvi, gfi)
    batch.voxels = (synthetic.blob_voxels(B, V, 1002) > 0.5).float().cuda()
    vi, fi = out["vertice_index"], out["face_index"]
    faces, adj = out["faces"].cpu(), out["edge_index"].cpu()
    rnd, want = [], [0.0, 0.0, 0.0]
    for s, pos in enumerate(out["vertex_positions"]):
        p64 = pos.cpu().double()
        u, x2, x1 = synthetic.sampling_randomness(B, n, 30 + s)
        ug, x2g, x1g = synthetic.sampling_randomness(B, n, 40 + s)
        fp = torch.stack([mesh_ops.face_cdf_draw(v, f, u[b]) for b, (v, f) in enumerate(zip(p64.split(vi), faces.split(fi)))])
        fg = torch.stack([mesh_ops.face_cdf_draw(v, f, ug[b]) for b, (v, f) in
                          enumerate(zip(gt_pos.split(gvi), torch.from_numpy(gfaces).split(gfi)))])
        rnd.append((dict(face_idx=fp, xi2=x2, xi1=x1), dict(face_idx=fg, xi2=x2g, xi1=x1g)))
        c, nl, e, _ = mesh_ops.mesh_loss_with(p64, faces, adj, vi, fi, gt_pos, torch.from_numpy(gfaces), gvi, gfi,
                                              (fp, x2.double(), x1.double()), (fg, x2g.double(), x1g.double()), float(n), k,
                                              canonical_signs=True)
        want = [want[0] + float(c), want[1] + float(nl), want[2] + float(e)]
    res = validate_batch(out, batch, float(n), k, randomness=rnd, f1_seed=11)
    assert len(out["vertex_positions"]) == 4
    for name, w in zip(("chamfer_loss", "normal_loss", "edge_loss"), want):
        assert abs(float(res[name]) - w) <= 1e-4 * abs(w) + 1e-7, (name, float(res[name]), w)
    bce = torch.nn.functional.binary_cross_entropy(vox.double(), batch.voxels.cpu().double())
    assert abs(float(res["voxel_loss"]) - float(bce)) <= 1e-5 * float(bce)
    # F1@tau: same clouds (same seeds), dense fp64 distances
    cp, _ = F_.sample_points(out["vertex_positions"][-1], out["faces"], vi, fi, n, seed=11)
    cg, _ = F_.sample_points(batch.meshes[0], batch.meshes[1], gvi, gfi, n, seed=12)
    d = mesh_ops.p2p_distance(cp.cpu().double(), cg.cpu().double()).clamp_min(0).sqrt()
    for tau in (0.1, 0.3, 0.5):
        pr, rc = (d.min(2).values < tau).double().mean(1), (d.min(1).values < tau).double().mean(1)
        f1 = float((100 * 2 * pr * rc / (pr + rc).clamp_min(1e-8)).mean())
        assert abs(float(res["f1@%g" % tau]) - f1) <= 0.2, (tau, float(res["f1@%g" % tau]), f1)     # points within 1e-6 of tau may flip
