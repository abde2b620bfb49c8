"""Watertight Cubify topology (opt-in, DESIGN.md §2 item 8) on the device: bit-exact against the oracle, closed-surface
invariants at BASELINE config 4, the untouched default path, a refinement-head training step on the watertight graph, and the
mesh metrics on watertight meshes."""
import numpy as np
import pytest
import torch

from oracle import cubify_np, cubify_watertight as cw, mesh_metrics as om, mesh_ops

pytestmark = pytest.mark.gpu
CASES = ["rand10", "ragged", "empty_mid_tail", "single_voxel", "solid3", "at_threshold", "blob16", "dense24"]
WT = "watertight"


def _run(t, th, **kw):
    from meshrcnn_b200.layers import Cubify
    vs, vi, f, fi, adj = Cubify(th, topology=WT)(torch.from_numpy(np.ascontiguousarray(t)).cuda(), **kw)
    return vs.cpu().numpy(), vi, f.cpu().numpy(), fi, adj.cpu().numpy()


def _assert_same(got, want):
    assert got[1] == list(want[1]) and got[3] == list(want[3])
    assert got[0].dtype == np.float32 and np.array_equal(got[0], want[0])
    assert got[2].dtype == np.int64 and np.array_equal(got[2], want[2])
    assert got[4].dtype == np.int64 and np.array_equal(got[4], want[4])


def _recording_calls():
    """Context manager that records the names of the C-ABI entry points called through _lib.call."""
    from meshrcnn_b200 import _lib

    class Rec:
        def __enter__(self):
            self.calls, self.orig = [], _lib.call
            _lib.call = lambda name, *a: (self.calls.append(name), self.orig(name, *a))[1]
            return self

        def __exit__(self, *exc):
            _lib.call = self.orig
            return False

    return Rec()


# ---------------------------------------------------------------------------------------------------------------
# bit-exact against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASES)
def test_golden_inputs_vs_oracle(lib, golden, name):
    g = golden("cubify_cases")
    t, th = g[name + "__in"], float(g[name + "__th"])
    if not (t > np.float32(th)).any():
        with pytest.raises(ValueError, match="empty grid"):
            _run(t, th)
        return
    _assert_same(_run(t, th), cw.cubify(t, th, topology=WT))


@pytest.mark.parametrize("B,V,kind,th", [(4, 32, "blob", 0.2), (32, 24, "blob", 0.2), (3, 48, "blob", 0.2),
                                         (2, 48, "dense", 0.5), (5, 13, "dense", 0.8)])
def test_vs_oracle_at_config_sizes(lib, B, V, kind, th):
    from meshrcnn_b200 import synthetic
    t = (synthetic.blob_voxels(B, V, 0) if kind == "blob" else synthetic.dense_voxels(B, V, 0)).numpy()
    _assert_same(_run(t, th), cw.cubify(t, th, topology=WT))


def test_from_logits_vs_oracle(lib):
    g = torch.Generator().manual_seed(5)
    B, V, th = 3, 16, 0.2
    logits = torch.randn(B, V, V, V, generator=g) * 3.0
    near = (torch.sigmoid(logits) - th).abs() < 1e-5     # keep clear of the threshold: CPU / GPU expf may differ in the last ulp
    logits[near] += 0.01
    _assert_same(_run(logits.numpy(), th, from_logits=True), cw.cubify(torch.sigmoid(logits).numpy(), th, topology=WT))


# ---------------------------------------------------------------------------------------------------------------
# BASELINE config 4: 64 dense 48^3 grids
# ---------------------------------------------------------------------------------------------------------------
def test_config4_device_invariants_and_oracle_slice(lib):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.layers import Cubify
    t = synthetic.dense_voxels(64, 48, 0)
    td = t.cuda()
    vs, vi, f, fi, adj = Cubify(0.5, topology=WT)(td)
    ref = Cubify(0.5)(td)
    assert fi == ref[3] and len(vi) == 64 and sum(vi) == vs.shape[0] and sum(fi) == f.shape[0]
    assert vs.shape[0] < ref[0].shape[0] and adj.shape[1] < ref[4].shape[1]
    SV = vs.shape[0]
    # adjacency strictly increasing in (row, col), symmetric, no self loops
    key = adj[0] * SV + adj[1]
    assert bool((key[1:] > key[:-1]).all()) and bool((adj[0] != adj[1]).all())
    assert torch.equal((adj[1] * SV + adj[0]).sort().values, key)
    # faces in range of their own mesh
    counts = torch.tensor(fi, device="cuda")
    vcnt = torch.tensor(vi, device="cuda")
    assert bool((f >= 0).all()) and bool((f < vcnt.repeat_interleave(counts)[:, None]).all())
    g = f + (vcnt.cumsum(0) - vcnt).repeat_interleave(counts)[:, None]
    # fp64 signed volume per mesh == its occupied-voxel count (half-integer coordinates: every partial sum is exact)
    tri = vs.double()[g]
    six_vol = (tri[:, 0] * torch.linalg.cross(tri[:, 1], tri[:, 2])).sum(1)
    mesh_of_face = torch.arange(64, device="cuda").repeat_interleave(counts)
    per_mesh = torch.zeros(64, dtype=torch.float64, device="cuda").index_add_(0, mesh_of_face, six_vol)
    nvox = (td > 0.5).flatten(1).sum(1).double()
    assert torch.equal(per_mesh, 6 * nvox)
    # half-edge balance: the multiset of directed half-edges equals that of their reverses
    u, w = g.reshape(-1), g[:, [1, 2, 0]].reshape(-1)
    assert torch.equal((u * SV + w).sort().values, (w * SV + u).sort().values)
    del tri, six_vol, u, w, g
    # the oracle on the first two meshes (mesh-local outputs do not depend on the rest of the batch)
    o = cw.cubify(t[:2].numpy(), 0.5, topology=WT)
    nv, nf, ne = sum(o[1]), sum(o[3]), o[4].shape[1]
    assert vi[:2] == o[1] and fi[:2] == o[3]
    assert np.array_equal(vs[:nv].cpu().numpy(), o[0]) and np.array_equal(f[:nf].cpu().numpy(), o[2])
    assert np.array_equal(adj[:, :ne].cpu().numpy(), o[4])


# ---------------------------------------------------------------------------------------------------------------
# the default path is unchanged
# ---------------------------------------------------------------------------------------------------------------
def test_default_is_the_reference_topology_and_calls_no_topo_entry_point(lib):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.layers import Cubify
    t = synthetic.blob_voxels(4, 16, 3).cuda()
    outs, calls = {}, {}
    for name, kw in (("default", {}), ("reference", {"topology": "reference"}), (WT, {"topology": WT})):
        with _recording_calls() as rec:
            outs[name] = Cubify(0.2, **kw)(t)
        calls[name] = rec.calls
    assert calls["default"] == calls["reference"] == ["mrb_cubify_count", "mrb_cubify_emit"]
    assert calls[WT] == ["mrb_cubify_count_topo", "mrb_cubify_emit_topo"]
    d, r = outs["default"], outs["reference"]
    assert d[1] == r[1] and d[3] == r[3]
    assert all(torch.equal(d[i], r[i]) for i in (0, 2, 4))
    assert not torch.equal(d[2], outs[WT][2])


def test_invalid_topology_raises(lib):
    from meshrcnn_b200 import _lib, functional as F_
    from meshrcnn_b200.layers import Cubify
    from meshrcnn_b200.pipeline import RefinementHead
    t = torch.ones(1, 3, 3, 3, device="cuda")
    with pytest.raises(ValueError, match="topology"):
        Cubify(0.5, topology="closed")
    with pytest.raises(ValueError, match="topology"):
        F_.cubify(t, 0.5, topology="closed")
    with pytest.raises(ValueError, match="topology"):
        RefinementHead("pix3d", cubify_topology="closed")
    m = Cubify(0.5)
    m.topology = "closed"
    with pytest.raises(ValueError, match="topology"):
        m(t)
    # the C ABI rejects it before any launch
    ws = torch.empty(int(_lib.load().mrb_cubify_workspace_bytes(1, 3, 3, 3)), dtype=torch.uint8, device="cuda")
    meta = torch.empty(8, dtype=torch.int64, device="cuda")
    with pytest.raises(RuntimeError, match="bad topology"):
        _lib.call("mrb_cubify_count_topo", _lib.ptr(t), 1, 3, 3, 3, 0.5, 0, 2, _lib.ptr(ws), _lib.ptr(meta))


def test_state_dict_keys_and_attribute_on_a_loaded_model(lib):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.layers import Cubify
    from meshrcnn_b200.pipeline import RefinementHead
    a, b = Cubify(0.2), Cubify(0.2, topology=WT)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) == ["kernel", "deltas"]
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    ha, hb = RefinementHead("pix3d"), RefinementHead("pix3d", cubify_topology=WT)
    assert list(ha.state_dict()) == list(hb.state_dict())
    ha.load_state_dict(hb.state_dict())
    ha = ha.cuda()
    t = synthetic.blob_voxels(2, 12, 1)
    ha.cubify.topology = WT
    got = ha.cubify(t.cuda())
    _assert_same(tuple(x.cpu().numpy() if torch.is_tensor(x) else x for x in got), cw.cubify(t.numpy(), 0.2, topology=WT))


# ---------------------------------------------------------------------------------------------------------------
# the refinement head on the watertight graph (BASELINE configs[1] input)
# ---------------------------------------------------------------------------------------------------------------
def test_training_step_on_the_watertight_graph(lib):
    """One configs[1] training step of RefinementHead("pix3d", cubify_topology="watertight") with GT meshes cubified in
    the same mode: finite losses and gradients."""
    import meshrcnn_b200.layers as L
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.mesh_sampling import normalize_mesh
    from meshrcnn_b200.pipeline import MeshTargets, RefinementHead, weighted_loss
    B, V = 32, 24
    vox = synthetic.blob_voxels(B, V, 0)
    fmap_h = synthetic.feature_maps(B, [synthetic.PIX3D_MAP], 0)[0]
    sizes = [(224, 224)] * B
    torch.manual_seed(1)
    head = RefinementHead("pix3d", cubify_threshold=0.2, cubify_topology=WT).cuda().train()
    gv, gvi, gf, gfi, _ = L.Cubify(0.5, topology=WT)(synthetic.blob_voxels(B, V, 1000).cuda())
    targets = MeshTargets(torch.cat([normalize_mesh(v) for v in gv.split(gvi)]), gf, gvi, gfi)
    fm = fmap_h.cuda().requires_grad_()
    losses = head(vox.cuda(), fm, sizes, targets)
    weighted_loss(losses).backward()
    for k in ("chamfer_loss", "normal_loss", "edge_loss"):
        assert bool(torch.isfinite(losses[k]).all()), k
    grads = [p.grad for p in head.parameters()]
    assert all(gr is not None and bool(torch.isfinite(gr).all()) for gr in grads)
    assert any(float(gr.abs().max()) > 0 for gr in grads) and bool(torch.isfinite(fm.grad).all())


def test_stage_chain_on_the_watertight_graph_vs_oracle(lib):
    """Cubify(topology="watertight") -> 3 Pix3D stages at production width, fwd + bwd vs the oracle in fp64: the check of
    test_layers_gpu.py::test_stage_chain_on_cubified_batch_vs_oracle on the watertight graph (in-frustum positions)."""
    import meshrcnn_b200.layers as L
    from meshrcnn_b200 import synthetic
    B, V = 3, 12
    vox = synthetic.blob_voxels(B, V, 0)
    verts, v_index, faces, f_index, adj = L.Cubify(0.2, topology=WT)(vox.cuda())
    o = cw.cubify(vox.numpy(), 0.2, topology=WT)
    assert np.array_equal(adj.cpu().numpy(), o[4])
    SV = verts.shape[0]
    torch.manual_seed(1)
    stages = [L.VertixRefinePix3D(use_input_features=bool(i)).cuda() for i in range(3)]
    with torch.no_grad():                          # default init + neighbour sums grow ~20x per layer and saturate the tanh
        for st in stages:
            for prm in st.parameters():
                prm.mul_(0.2)
    fmap = synthetic.feature_maps(B, [synthetic.PIX3D_MAP], 0)[0] * 0.02
    pos0 = synthetic.in_frustum_positions(SV, 224, 5)
    sizes = [(224, 224)] * B
    fm_c = fmap.cuda().requires_grad_()
    p = pos0.cuda().requires_grad_()
    cur, feats = p, None
    for st in stages:
        cur, feats = st(v_index, fm_c, adj, cur, sizes, vertex_features=feats)
    go_p = torch.randn(SV, 3, generator=torch.Generator().manual_seed(2))
    (cur * go_p.cuda()).sum().backward()

    def oracle(dt):
        fmo = fmap.to(dt).requires_grad_()
        po = pos0.to(dt).requires_grad_()
        params = [{k: v.detach().cpu().to(dt).requires_grad_() for k, v in st.named_parameters()} for st in stages]
        c, f_ = po, None
        for sd in params:
            c, f_ = mesh_ops.stage_pix3d(sd, v_index, fmo, adj.cpu(), c, sizes, feats=f_)
        (c * go_p.to(dt)).sum().backward()
        out = {"pos3": c.detach(), "feat3": f_.detach(), "grad pos0": po.grad, "grad fmap": fmo.grad}
        for i, sd in enumerate(params):
            for k, v in sd.items():
                out["grad %d.%s" % (i, k)] = v.grad
        return out

    o64, o32 = oracle(torch.float64), oracle(torch.float32)
    got = {"pos3": cur, "feat3": feats, "grad pos0": p.grad, "grad fmap": fm_c.grad}
    for i, st in enumerate(stages):
        for k, prm in st.named_parameters():
            got["grad %d.%s" % (i, k)] = prm.grad
    assert got.keys() == o64.keys()
    for name, want in o64.items():
        w = want.double()
        assert float(w.norm()) > 0, name
        err = float((got[name].detach().cpu().double() - w).norm() / w.norm())
        ref = float((o32[name].double() - w).norm() / w.norm())
        bound = max(1e-4, 3 * ref)
        if name.startswith("grad"):                # ReLU masks within an ulp of zero, as in test_layers_gpu
            bound = max(bound, 1e-3)
        assert err <= bound, (name, err, ref)


# ---------------------------------------------------------------------------------------------------------------
# metrics on watertight meshes
# ---------------------------------------------------------------------------------------------------------------
def test_sample_surface_on_a_watertight_cube_returns_the_outward_axis_normals(lib):
    from meshrcnn_b200 import functional as F_
    t = torch.zeros(1, 3, 3, 3)
    t[0, 1, 1, 1] = 1
    v, vi, f, fi, _, _ = F_.cubify(t.cuda(), 0.5, topology=WT)
    pts, nrm, gid = F_.sample_surface(v, f, vi, fi, 4000, seed=3)
    nb = torch.tensor(cubify_np.NEIGHBOUR, dtype=torch.float32)
    axis = torch.stack([nb[:, 0], nb[:, 2], -nb[:, 1]], 1).cuda()      # (z, y, x) -> (z, x, -y), faces in direction order
    assert torch.equal(nrm[0], axis[gid[0].long() // 2])
    assert len(set(gid[0].tolist())) == 12
    # every sample lies on the plane of its face, half a voxel outward from the cube's centre
    off = ((pts[0] - v.mean(0)) * nrm[0]).sum(1)
    assert float((off - 0.5).abs().max()) <= 1e-6


def _draws(f_index, n, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.stack([torch.randint(0, int(c), (n,), generator=g) for c in f_index]),
            torch.rand(len(f_index), n, generator=g), torch.rand(len(f_index), n, generator=g))


def test_compare_meshes_on_watertight_blob_pairs_vs_oracle(lib):
    from meshrcnn_b200 import functional as F_, synthetic
    from meshrcnn_b200.eval_utils import compare_meshes
    B, n, taus = 4, 3000, (0.1, 0.2, 0.3, 0.4, 0.5)
    pv, pvi, pf, pfi, _, _ = F_.cubify(synthetic.blob_voxels(B, 16, 11).cuda(), 0.2, topology=WT)
    gv, gvi, gf, gfi, _, _ = F_.cubify(synthetic.blob_voxels(B, 16, 1011).cuda(), 0.2, topology=WT)
    assert len(pfi) == len(gfi) == B
    dp, dg = _draws(pfi, n, 3), _draws(gfi, n, 4)
    rnd = lambda d: dict(face_idx=d[0].cuda(), xi2=d[1].cuda(), xi1=d[2].cuda())
    res = compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=n, thresholds=taus,
                         randomness=(rnd(dp), rnd(dg)), reduce=False)
    # the nearest-neighbour indices the kernel used, to evaluate the normal terms where distances tie
    s = F_.mesh_gt_scale(gv, gvi)
    p, _, _ = F_.sample_surface(pv, pf, pvi, pfi, n, scale=s, **rnd(dp))
    q, _, _ = F_.sample_surface(gv, gf, gvi, gfi, n, scale=s, **rnd(dg))
    _, i_p, _, _, i_q, _ = F_.knn_search(p, q, 0)
    d64 = lambda d: (d[0], d[1].double(), d[2].double())
    want = om.compare_meshes_with(pv.cpu().double(), pf.cpu(), pvi, pfi, gv.cpu().double(), gf.cpu(), gvi, gfi,
                                  d64(dp), d64(dg), thresholds=taus)
    for b, w in enumerate(want):
        got = lambda k: float(res[k][b])
        assert abs(got("Chamfer-L2") - float(w["Chamfer-L2"])) <= 1e-4 * float(w["Chamfer-L2"]), b
        ip, iq = i_p[b].cpu(), i_q[b].cpu()
        assert bool(om.in_tie_set(w["_p"], w["_q"], ip, w["_d_p"]).all())
        assert bool(om.in_tie_set(w["_q"], w["_p"], iq, w["_d_q"]).all())
        at = om.mesh_metrics_one(w["_p"], w["_n_p"], w["_q"], w["_n_q"], (), idx_p=ip, idx_q=iq)
        for k in ("NormalConsistency", "AbsNormalConsistency"):
            assert abs(got(k) - float(at[k])) <= 1e-5, (b, k, got(k), float(at[k]))
        # outward winding everywhere: the signed normal consistency is meaningful (no winding flip to hide)
        assert got("NormalConsistency") > 0.3
        assert abs(got("NormalConsistency") - got("AbsNormalConsistency")) <= 0.01, b
