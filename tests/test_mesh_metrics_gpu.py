"""The paper's mesh metrics on the device (eval_utils.compare_meshes, functional.sample_surface / mesh_gt_scale / mesh_metrics)
against the fp64 oracle (oracle/mesh_metrics.compare_meshes_with) and on known answers.

Tolerances: Chamfer-L2 rtol 1e-4; normal consistency 1e-5 with the oracle evaluated at the kernel's nearest-neighbour indices
(after checking that each lies in the oracle's tie set); every precision / recall count between the dense fp64 counts at
tau (1 -+ 1e-6) on the same samples."""
import math

import numpy as np
import pytest
import torch

from oracle import mesh_metrics as om

pytestmark = pytest.mark.gpu
TAUS = (0.1, 0.2, 0.3, 0.4, 0.5)


def _cubify(vox, thr=0.2):
    from meshrcnn_b200.functional import cubify
    v, vi, f, fi, _, _ = cubify(vox.cuda(), thr)
    return v, f, vi, fi


def _draws(f_index, B, n, seed):
    """Injected randomness: local face ids (any value for meshes without faces), xi2, xi1 -- B x n each."""
    g = torch.Generator().manual_seed(seed)
    fl = list(f_index) + [0] * (B - len(f_index))
    fi = torch.stack([torch.randint(0, max(int(c), 1), (n,), generator=g) for c in fl])
    return fi, torch.rand(B, n, generator=g), torch.rand(B, n, generator=g)


def _rnd(d):
    return dict(face_idx=d[0].cuda(), xi2=d[1].cuda(), xi1=d[2].cuda())


def _rnd64(d):
    return d[0], d[1].double(), d[2].double()


def _subset(verts, faces, vi, fi, keep):
    vs, fs = verts.split(list(vi)), faces.split(list(fi))
    return (torch.cat([vs[b] for b in keep]), torch.cat([fs[b] for b in keep]), [vi[b] for b in keep], [fi[b] for b in keep])


def _ragged(B=4, V=12, seed=7):
    from meshrcnn_b200 import synthetic
    pv, pf, pvi, pfi = _cubify(synthetic.blob_voxels(B, V, seed))
    gv, gf, gvi, gfi = _cubify(synthetic.blob_voxels(B, V, seed + 1000))
    assert len(set(pfi)) > 1 and len(pfi) == len(gfi) == B          # ragged, no empty mesh
    return pv, pf, pvi, pfi, gv, gf, gvi, gfi


def _check_against_oracle(res, pv, pf, pvi, pfi, gv, gf, gvi, gfi, dp, dg, n, rows):
    """res: compare_meshes(..., reduce=False) of the whole batch; rows: the meshes checked against the oracle."""
    from meshrcnn_b200 import functional as F_
    rnd_p, rnd_g = _rnd(dp), _rnd(dg)
    s = F_.mesh_gt_scale(gv, gvi)
    p, n_p, _ = F_.sample_surface(pv, pf, pvi, pfi, n, scale=s, **rnd_p)       # the samples compare_meshes draws
    q, n_q, _ = F_.sample_surface(gv, gf, gvi, gfi, n, scale=s, **rnd_g)
    _, i_p, _, _, i_q, _ = F_.knn_search(p, q, 0)
    sub = lambda d: tuple(t[rows] for t in _rnd64(d))
    P, G = _subset(pv, pf, pvi, pfi, rows), _subset(gv, gf, gvi, gfi, rows)
    want = om.compare_meshes_with(P[0].cpu().double(), P[1].cpu(), P[2], P[3], G[0].cpu().double(), G[1].cpu(), G[2],
                                        G[3], sub(dp), sub(dg), thresholds=TAUS)
    for w, b in zip(want, rows):
        got = lambda k: float(res[k][b])
        assert abs(got("Chamfer-L2") - float(w["Chamfer-L2"])) <= 1e-4 * float(w["Chamfer-L2"]), (b, got("Chamfer-L2"))
        ip, iq = i_p[b].cpu(), i_q[b].cpu()
        assert bool(om.in_tie_set(w["_p"], w["_q"], ip, w["_d_p"]).all())
        assert bool(om.in_tie_set(w["_q"], w["_p"], iq, w["_d_q"]).all())
        at = om.mesh_metrics_one(w["_p"], w["_n_p"], w["_q"], w["_n_q"], (), idx_p=ip, idx_q=iq)
        for k in ("NormalConsistency", "AbsNormalConsistency"):
            assert abs(got(k) - float(at[k])) <= 1e-5, (b, k, got(k), float(at[k]))
        # counts: dense fp64 distances of the device samples, thresholds widened / narrowed by 1e-6
        d_p, _ = om.nearest(p[b].cpu().double(), q[b].cpu().double())
        d_q, _ = om.nearest(q[b].cpu().double(), p[b].cpu().double())
        for tau in TAUS:
            for key, d in (("Precision", d_p), ("Recall", d_q)):
                cnt = round(got("%s@%g" % (key, tau)) * n / 100)
                lo = int((d.sqrt() < tau * (1 - 1e-6)).sum())
                hi = int((d.sqrt() < tau * (1 + 1e-6)).sum())
                assert lo <= cnt <= hi, (b, key, tau, lo, cnt, hi)
            pr, rc = got("Precision@%g" % tau), got("Recall@%g" % tau)
            assert abs(got("F1@%g" % tau) - 2 * pr * rc / (pr + rc + 1e-8)) <= 1e-4


# ---------------------------------------------------------------------------------------------------------------------
# sampling with normals
# ---------------------------------------------------------------------------------------------------------------------
def test_sample_surface_matches_oracle_with_injected_draws(lib):
    from meshrcnn_b200 import functional as F_
    pv, pf, pvi, pfi, *_ = _ragged()
    B, n = len(pfi), 3000
    d = _draws(pfi, B, n, 1)
    s = F_.mesh_gt_scale(pv, pvi)
    pts, nrm, gid = F_.sample_surface(pv, pf, pvi, pfi, n, **_rnd(d), scale=s)
    assert pts.shape == nrm.shape == (B, n, 3) and gid.shape == (B, n) and gid.dtype == torch.int32
    v64, f = pv.cpu().double(), pf.cpu()
    f_start = np.concatenate([[0], np.cumsum(pfi)[:-1]])
    for b, (vb, fb) in enumerate(zip(v64.split(pvi), f.split(pfi))):
        sb = om.gt_scale(vb)
        assert abs(float(s[b]) - float(sb)) <= 1e-6 * float(sb)
        p64, n64 = om.sample_surface_with(vb, fb, d[0][b], d[1][b].double(), d[2][b].double(), sb)
        assert float((pts[b].cpu().double() - p64).abs().max()) <= 1e-5 * float(p64.abs().max())
        assert float((nrm[b].cpu().double() - n64).abs().max()) <= 1e-5
        assert torch.equal(gid[b].cpu().long(), d[0][b] + int(f_start[b]))
    assert float((nrm.double().norm(dim=2) - 1).abs().max()) <= 1e-5


def test_sample_surface_philox_face_ids_and_unscaled_points_are_sample_points_bits(lib):
    from meshrcnn_b200 import _lib, functional as F_
    pv, pf, pvi, pfi, *_ = _ragged()
    B, n, seed = len(pfi), 4000, 12345
    _, fid_sp = F_.sample_points(pv, pf, pvi, pfi, n, seed=seed)
    pts, _, fid = F_.sample_surface(pv, pf, pvi, pfi, n, seed=seed)
    assert torch.equal(fid, fid_sp)
    # raw (pre-normalisation) points of mrb_sample_points_fwd for the same seed / the same injected draws
    dev = pv.device
    v_off, f_off = F_.offsets_table(pvi, dev), F_.offsets_table(pfi, dev)
    cdf = F_._face_cdf(pv, pf, v_off, f_off, B, max(pfi))
    d = _draws(pfi, B, n, 2)
    for rnd in (None, _rnd(d)):
        raw, cloud = torch.empty(B, n, 3, device=dev), torch.empty(B, n, 3, device=dev)
        fidx, w = torch.empty(B, n, dtype=torch.int32, device=dev), torch.empty(B, n, 3, device=dev)
        stats = torch.empty(B, 8, dtype=torch.float64, device=dev)
        r = rnd or {}
        _lib.call("mrb_sample_points_fwd", _lib.ptr(pv), _lib.ptr(pf), _lib.ptr(v_off), _lib.ptr(f_off), _lib.ptr(cdf), B, n,
                  None, _lib.ptr(r.get("face_idx")), _lib.ptr(r.get("xi2")), _lib.ptr(r.get("xi1")), seed, _lib.ptr(raw),
                  _lib.ptr(fidx), _lib.ptr(w), _lib.ptr(cloud), _lib.ptr(stats))
        pts, _, fid = F_.sample_surface(pv, pf, pvi, pfi, n, seed=seed, **r)
        assert torch.equal(pts, raw) and torch.equal(fid, fidx)


# ---------------------------------------------------------------------------------------------------------------------
# metrics
# ---------------------------------------------------------------------------------------------------------------------
def test_compare_meshes_matches_oracle_on_ragged_cubify_batch(lib):
    from meshrcnn_b200.eval_utils import compare_meshes
    pv, pf, pvi, pfi, gv, gf, gvi, gfi = _ragged()
    B, n = len(gfi), 2000
    dp, dg = _draws(pfi, B, n, 3), _draws(gfi, B, n, 4)
    res = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=n, randomness=(_rnd(dp), _rnd(dg)), reduce=False)
    assert all(res[k].shape == (B,) and res[k].dtype == torch.float32 for k in res if k != "valid")
    assert bool(res["valid"].all())
    _check_against_oracle(res, pv, pf, pvi, pfi, gv, gf, gvi, gfi, dp, dg, n, list(range(B)))
    # unscaled: the same kernels without the GT-10 multiply
    res1 = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=n, scale=None, randomness=(_rnd(dp), _rnd(dg)),
                          reduce=False)
    want = om.compare_meshes_with(pv.cpu().double(), pf.cpu(), pvi, pfi, gv.cpu().double(), gf.cpu(), gvi, gfi,
                                        _rnd64(dp), _rnd64(dg), scale=None, thresholds=TAUS)
    for b, w in enumerate(want):
        assert abs(float(res1["Chamfer-L2"][b]) - float(w["Chamfer-L2"])) <= 1e-4 * float(w["Chamfer-L2"])


def test_parallel_squares_on_device(lib):
    from meshrcnn_b200.eval_utils import compare_meshes
    h, n = 0.25, 10000
    sq = lambda z: torch.tensor([[0, 0, z], [10, 0, z], [10, 10, z], [0, 10, z]], dtype=torch.float32).cuda()
    f = torch.tensor([[0, 1, 2], [0, 2, 3]]).cuda()
    d = _rnd(_draws([2], 1, n, 5))
    res = compare_meshes(sq(0.0), f, [4], [2], sq(h), f, [4], [2], num_samples=n, randomness=(d, d), reduce=False)
    assert abs(float(res["Chamfer-L2"][0]) - 2 * h * h) <= 1e-6 * 2 * h * h
    assert abs(float(res["NormalConsistency"][0]) - 1) <= 1e-6 and abs(float(res["AbsNormalConsistency"][0]) - 1) <= 1e-6
    for tau in TAUS:
        assert float(res["F1@%g" % tau][0]) == pytest.approx(100.0 if tau > h else 0.0, abs=1e-4)


def test_same_seed_is_bitwise_reproducible(lib):
    from meshrcnn_b200.eval_utils import compare_meshes
    args = _ragged()
    a = compare_meshes(*args, num_samples=5000, seed=77, reduce=False)
    b = compare_meshes(*args, num_samples=5000, seed=77, reduce=False)
    assert all(torch.equal(a[k], b[k]) for k in a)
    c = compare_meshes(*args, num_samples=5000, seed=78, reduce=False)
    assert not torch.equal(a["Chamfer-L2"], c["Chamfer-L2"])


def test_gt10_scale_invariance(lib):
    from meshrcnn_b200.eval_utils import compare_meshes
    pv, pf, pvi, pfi, gv, gf, gvi, gfi = _ragged()
    B, n = len(gfi), 4000
    fp, fg = _draws(pfi, B, n, 6)[0].cuda(), _draws(gfi, B, n, 7)[0].cuda()
    rnd = (dict(face_idx=fp), dict(face_idx=fg))
    a = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=n, seed=3, randomness=rnd, reduce=False)
    b = compare_meshes(2.5 * pv, pf, pvi, pfi, 2.5 * gv, gf, gvi, gfi, num_samples=n, seed=3, randomness=rnd, reduce=False)
    for k in ("Chamfer-L2", "NormalConsistency", "AbsNormalConsistency"):
        assert torch.allclose(a[k], b[k], rtol=1e-5, atol=0), (k, a[k], b[k])
    # a sample whose distance lies within rounding of tau may change sides: at most one sample per count
    for tau in TAUS:
        for k in ("Precision", "Recall"):
            assert float((a["%s@%g" % (k, tau)] - b["%s@%g" % (k, tau)]).abs().max()) <= 100.0 / n + 1e-4
        assert float((a["F1@%g" % tau] - b["F1@%g" % tau]).abs().max()) <= 2 * 100.0 / n + 1e-4


def test_empty_predicted_meshes_interior_and_trailing(lib):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.eval_utils import compare_meshes, mesh_metric_names
    vox = synthetic.blob_voxels(5, 12, 8)
    vox[1] = 0.0
    vox[4] = 0.0
    gvox = synthetic.blob_voxels(5, 12, 1008)
    pv, pf, pvi, pfi = _cubify(vox)
    gv, gf, gvi, gfi = _cubify(gvox)
    assert len(pfi) == 4 and pfi[1] == 0 and len(gfi) == 5      # Cubify drops the trailing empty mesh
    res = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=3000, seed=9, reduce=False)
    assert res["valid"].tolist() == [True, False, True, True, False]
    names = mesh_metric_names(TAUS)
    for b in (1, 4):
        assert all(math.isnan(float(res[k][b])) for k in names[:3])
        assert all(float(res[k][b]) == 0.0 for k in names[3:])
    keep = [0, 2, 3]
    pv2, pf2, pvi2, pfi2 = _cubify(vox[keep])
    gv2, gf2, gvi2, gfi2 = _cubify(gvox[keep])
    res2 = compare_meshes(pv2, pf2, pvi2, pfi2, gv2, gf2, gvi2, gfi2, num_samples=3000, seed=9, reduce=False)
    for k in names:
        assert torch.equal(res[k][keep], res2[k]), k
    red = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=3000, seed=9, reduce=True)
    assert red["num_valid"] == 3
    for k in names:
        assert abs(float(red[k]) - float(res2[k].double().mean())) <= 1e-6 * max(1.0, abs(float(red[k]))), k


def test_bad_inputs_raise(lib):
    from meshrcnn_b200.eval_utils import compare_meshes
    pv, pf, pvi, pfi, gv, gf, gvi, gfi = _ragged()
    with pytest.raises(ValueError):                      # a GT mesh without faces
        compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi + [0], gfi + [0], num_samples=100)
    with pytest.raises(ValueError):                      # more predicted meshes than GT meshes
        compare_meshes(pv, pf, pvi + [0], pfi + [0], gv, gf, gvi, gfi, num_samples=100)
    with pytest.raises(ValueError):                      # more than 8 thresholds
        compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=100, thresholds=[0.1 * i for i in range(1, 10)])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        compare_meshes(pv.cpu(), pf.cpu(), pvi, pfi, gv.cpu(), gf.cpu(), gvi, gfi, num_samples=100)


def test_configuration_size_b32_10k_against_oracle_subset(lib):
    """Config-1 Pix3D meshes (24^3 blobs through Cubify, GT from seed + 1000), B = 32, 10 000 samples per mesh."""
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.eval_utils import compare_meshes
    pv, pf, pvi, pfi = _cubify(synthetic.blob_voxels(32, 24, 0))
    gv, gf, gvi, gfi = _cubify(synthetic.blob_voxels(32, 24, 1000))
    B, n = 32, 10000
    dp, dg = _draws(pfi, B, n, 10), _draws(gfi, B, n, 11)
    res = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=n, randomness=(_rnd(dp), _rnd(dg)), reduce=False)
    assert bool(torch.isfinite(torch.stack([res[k] for k in res if k != "valid"])).all())
    _check_against_oracle(res, pv, pf, pvi, pfi, gv, gf, gvi, gfi, dp, dg, n, [0, 9, 20, 31])


# ---------------------------------------------------------------------------------------------------------------------
# validate_batch / validate
# ---------------------------------------------------------------------------------------------------------------------
def _eval_setup():
    from oracle import cubify_np
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.pipeline import MeshTargets, RefinementHead
    B, V = 2, 12
    vox = synthetic.blob_voxels(B, V, 2)
    fmap = synthetic.feature_maps(B, [synthetic.PIX3D_MAP], 2)[0] * 0.02
    torch.manual_seed(3)
    head = RefinementHead("pix3d", cubify_threshold=0.2).cuda().eval()
    with torch.no_grad():
        for prm in head.parameters():
            prm.mul_(0.2)
        out = head(vox.cuda(), fmap.cuda(), [(224, 224)] * B)
    gverts, gvi, gfaces, gfi, _ = cubify_np.cubify(synthetic.blob_voxels(B, V, 1002).numpy(), 0.5)
    batch = MeshTargets(torch.from_numpy(gverts).cuda(), torch.from_numpy(gfaces).cuda(), gvi, gfi)
    return head, vox, fmap, out, batch


def test_validate_batch_defaults_unchanged(lib):
    from meshrcnn_b200.eval_utils import compare_meshes, mesh_metric_names, validate_batch
    _, _, _, out, batch = _eval_setup()
    torch.manual_seed(0)
    base = validate_batch(out, batch, 1500.0, 10, f1_seed=11)
    assert set(base) == {"chamfer_loss", "normal_loss", "edge_loss", "f1@0.1", "f1@0.3", "f1@0.5"}
    torch.manual_seed(0)
    more = validate_batch(out, batch, 1500.0, 10, f1_seed=11, mesh_metrics=True)
    assert set(more) == set(base) | set(mesh_metric_names(TAUS)) | {"num_valid"}
    for k in base:
        assert torch.equal(base[k], more[k]), k
    gt_pos, gt_faces = batch.meshes
    want = compare_meshes(out["vertex_positions"][-1], out["faces"], out["vertice_index"], out["face_index"], gt_pos, gt_faces,
                          batch.vertice_index, batch.face_index, seed=13)
    assert more["num_valid"] == want["num_valid"] == len(batch.face_index)
    for k in mesh_metric_names(TAUS):
        assert torch.equal(more[k], want[k]), k


def test_validate_weights_mesh_metrics_by_valid_meshes(lib):
    from meshrcnn_b200.eval_utils import validate, validate_batch
    head, vox, fmap, out, batch = _eval_setup()
    batch.images = None

    class Model:
        def eval(self):
            return self

        def __call__(self, images):
            return out

    meters = validate(Model(), [batch, batch], point_cloud_size=1500.0, mesh_metrics=True)
    assert "Chamfer-L2" in meters and "F1@0.3" in meters and "num_valid" not in meters
    assert meters["Chamfer-L2"].count == 2 * len(batch.face_index)
    one = validate_batch(out, batch, 1500.0, 10, mesh_metrics=True)
    assert abs(meters["Chamfer-L2"].avg - float(one["Chamfer-L2"])) <= 1e-6 * abs(float(one["Chamfer-L2"]))
