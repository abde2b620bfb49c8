"""Bilinear VertexAlign (layers.VertexAlign(mode="bilinear"), functional.vert_align_bilinear, vert_align_linear(bilinear=True),
align_mode="bilinear" on the stage classes and the refinement head) against the fp64 oracle
(oracle/bilinear_align.vert_align_bilinear): values and the gradients of the maps, the weights and the vertex positions at fp32
rtol 1e-4 unless a test says otherwise.  Positions are resampled to lie at least 1e-3 texel from every knot of every map, so
that fp32 and fp64 pick the same cell."""
import numpy as np
import pytest
import torch

from oracle import bilinear_align as bil, mesh_ops

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def close(got, want, rtol=RTOL, what=""):
    want = torch.as_tensor(want).detach().cpu().double()
    got = got.detach().cpu().double()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    atol = rtol * float(want.abs().max()) * 1e-1 + 1e-30          # gradients span decades: scale atol to the tensor
    err = (got - want).abs()
    tol = atol + rtol * want.abs()
    assert bool((err <= tol).all()), "%s: max err %.3e, max|want| %.3e" % (what, float(err.max()), float(want.abs().max()))


def rel_l2(got, want):
    w = want.detach().cpu().double()
    return float((got.detach().cpu().double() - w).norm() / max(float(w.norm()), 1e-300))


def off_knot_positions(n, img, map_sizes, seed, margin=1e-3):
    """n in-frustum positions (synthetic.in_frustum_positions) whose sampling coordinates x, y are >= margin texel from
    every integer for every map size (the knots, including the S-1 clamp)."""
    from meshrcnn_b200 import synthetic
    out, s = [], seed
    while sum(len(o) for o in out) < n:
        p = synthetic.in_frustum_positions(4 * n + 64, img, s).double()
        h = 248 * (p[:, 1] / p[:, 2]) + 111.5
        w = 248 * (p[:, 0] / -p[:, 2]) + 111.5
        ok = (h >= 0) & (h <= img - 1) & (w >= 0) & (w <= img - 1)
        for S in map_sizes:
            for c in (w / (img / S), h / (img / S)):
                ok &= (c - c.round()).abs() >= margin
        out.append(p[ok].float())
        s += 1000
    return torch.cat(out)[:n].contiguous()


def run_align(fn, maps, pos, vpm, sizes, mi, go, dtype):
    f = [m.to(dtype).requires_grad_() for m in maps]
    p = pos.to(dtype).requires_grad_()
    out = fn(f, p, vpm, sizes, mi)
    (out * go.to(out.dtype)).sum().backward()
    gp = p.grad if p.grad is not None else torch.zeros_like(p)
    return out.detach(), gp, [x.grad for x in f]


def cuda_align(maps, pos, vpm, sizes, mi, go):
    from meshrcnn_b200.layers import VertexAlign
    mod = VertexAlign(mode="bilinear").eval()
    f = [m.cuda().requires_grad_() for m in maps]
    p = pos.cuda().requires_grad_()
    out = mod(f, p, vpm, sizes, mi)
    (out * go.cuda()).sum().backward()
    return out, p.grad, [x.grad for x in f]


# ---------------------------------------------------------------------------------------------------------------
# 1. the module
# ---------------------------------------------------------------------------------------------------------------
CASES = {
    "shapenet": (lambda syn: syn.SHAPENET_MAPS, 137),
    "pix3d": (lambda syn: [syn.PIX3D_MAP], 224),
    "odd_channels": (lambda syn: [(3, 9, 9), (257, 6, 6)], 224),      # the scalar path
    "single_texel": (lambda syn: [(8, 1, 1), (12, 4, 4)], 224),        # S = 1
}


@pytest.mark.parametrize("case", list(CASES))
def test_module_vs_oracle(lib, case):
    """Ragged meshes, several meshes per image (eval mode): values, map gradients and position gradients."""
    from meshrcnn_b200 import synthetic
    shapes_of, img = CASES[case]
    shapes = shapes_of(synthetic)
    B = 3
    maps = synthetic.feature_maps(B, shapes, 5)
    vpm, mi = [37, 120, 5, 211, 64], [2, 1, 2]
    sizes = [(img, img)] * B
    pos = off_knot_positions(sum(vpm), img, [s for _, s, _ in shapes], 6)
    go = torch.randn(sum(vpm), sum(c for c, _, _ in shapes), generator=torch.Generator().manual_seed(7))
    want, want_gp, want_gf = run_align(bil.vert_align_bilinear, maps, pos, vpm, sizes, mi, go, torch.float64)
    got, gp, gf = cuda_align(maps, pos, vpm, sizes, mi, go)
    assert got.dtype == torch.float32 and gp.dtype == torch.float32
    close(got, want, what="values")
    close(gp, want_gp, what="position gradient")
    for i in range(len(maps)):
        close(gf[i], want_gf[i], what="map %d gradient" % i)
    if case == "single_texel":
        assert float(want_gp.abs().max()) > 0          # the 4 x 4 map moves the positions, the 1 x 1 map does not
    else:
        assert float((want_gp.abs() > 0).double().mean()) > 0.9


def test_module_bf16_maps(lib):
    """bf16 maps (converted by feature_rows): values and gradients at rtol 2e-2, map gradients returned in bf16."""
    from meshrcnn_b200 import synthetic
    shapes = [(256, 12, 12), (64, 18, 18)]
    B = 2
    maps = [m.bfloat16() for m in synthetic.feature_maps(B, shapes, 8)]
    vpm, mi, sizes = [300, 200], [1, 1], [(224, 224)] * B
    pos = off_knot_positions(sum(vpm), 224, [12, 18], 9)
    go = torch.randn(sum(vpm), 320, generator=torch.Generator().manual_seed(10))
    want, want_gp, want_gf = run_align(bil.vert_align_bilinear, [m.double() for m in maps], pos, vpm, sizes, mi, go,
                                       torch.float64)
    got, gp, gf = cuda_align(maps, pos, vpm, sizes, mi, go)
    close(got, want, rtol=2e-2, what="bf16 values")
    close(gp, want_gp, rtol=2e-2, what="bf16 position gradient")
    for i in range(2):
        assert gf[i].dtype == torch.bfloat16
        close(gf[i].float(), want_gf[i], rtol=2e-2, what="bf16 map %d gradient" % i)


# ---------------------------------------------------------------------------------------------------------------
# 2. edge cases
# ---------------------------------------------------------------------------------------------------------------
def test_far_outside_p2_zero_and_nan_positions(lib):
    """Far outside the frustum: the border sample and an exactly zero position gradient.  p2 = 0 and NaN positions: finite
    outputs (the clamped sample) and a zero gradient."""
    from meshrcnn_b200 import synthetic
    fm = synthetic.feature_maps(1, [(20, 12, 12)], 11)[0]
    g = torch.Generator().manual_seed(12)
    n = 64
    far = torch.stack([10 + 10 * torch.rand(n, generator=g), 10 + 10 * torch.rand(n, generator=g),
                       -(1 + torch.rand(n, generator=g))], 1)
    bad = torch.tensor([[0.3, 0.2, 0.0], [0.0, 0.0, 0.0], [float("nan"), 0.1, -1.0], [0.1, float("nan"), -1.0],
                        [float("nan")] * 3, [0.2, -0.1, float("inf")]])
    pos = torch.cat([far, bad])
    go = torch.randn(pos.shape[0], 20, generator=g)
    want, want_gp, want_gf = run_align(bil.vert_align_bilinear, [fm], pos, [pos.shape[0]], [(224, 224)], [1], go,
                                       torch.float64)
    got, gp, gf = cuda_align([fm], pos, [pos.shape[0]], [(224, 224)], [1], go)
    assert bool(torch.isfinite(got).all()) and bool(torch.isfinite(gp).all()) and bool(torch.isfinite(gf[0]).all())
    assert torch.equal(got[:n].cpu(), fm[0][:, 11, 0].expand(n, 20))          # w -> W-1 (x -> S-1), h -> 0
    assert float(gp.abs().max()) == 0.0
    close(got, want, what="clamped values")
    close(gf[0], want_gf[0], what="clamped map gradient")


def test_empty_non_square_and_deterministic_position_gradient(lib):
    from meshrcnn_b200 import functional as F_, synthetic
    from meshrcnn_b200.layers import VertexAlign
    fm = synthetic.feature_maps(2, [(16, 12, 12)], 13)[0].cuda().requires_grad_()
    empty = torch.zeros(0, 3, device="cuda", requires_grad=True)
    out = F_.vert_align_bilinear([fm], empty, [0, 0], [(224, 224)] * 2, [1, 1])
    assert out.shape == (0, 16)
    out.sum().backward()
    assert empty.grad.shape == (0, 3) and float(fm.grad.abs().sum()) == 0.0
    with pytest.raises(RuntimeError):
        F_.vert_align_bilinear([torch.randn(2, 4, 12, 10, device="cuda")], torch.randn(5, 3, device="cuda"), [2, 3],
                               [(224, 224)] * 2, [1, 1])
    with pytest.raises(RuntimeError):                                            # image 2 has a mesh, the map has 2 images
        F_.vert_align_bilinear([fm], torch.randn(5, 3, device="cuda"), [2, 2, 1], [(224, 224)] * 3, [1, 1, 1])
    with pytest.raises(ValueError):
        VertexAlign(mode="nearest")
    # the position gradient is written by the warp that owns the vertex: two identical backward calls agree bitwise
    maps = synthetic.feature_maps(2, synthetic.SHAPENET_MAPS, 14)
    pos = off_knot_positions(3000, 137, [35, 18, 9, 5], 15)
    go = torch.randn(3000, 3840, generator=torch.Generator().manual_seed(16))
    grads = []
    for _ in range(2):
        _, gp, _ = cuda_align(maps, pos, [1000, 2000], [(137, 137)] * 2, [1, 1], go)
        grads.append(gp)
    assert torch.equal(grads[0], grads[1])


# ---------------------------------------------------------------------------------------------------------------
# 3. the fused ShapeNet bottleneck
# ---------------------------------------------------------------------------------------------------------------
def test_fused_bottleneck_vs_oracle_and_unfused(lib):
    """vert_align_linear(bilinear=True) against the oracle's vert_align_bilinear(...) @ W^T and against the unfused CUDA
    composition linear(VertexAlign(mode="bilinear")(...)): values and the gradients of W, the maps and the positions."""
    from meshrcnn_b200 import functional as F_, synthetic
    from meshrcnn_b200.layers import VertexAlign
    shapes = [(c // 8, h, w) for (c, h, w) in synthetic.SHAPENET_MAPS]      # 480 channels
    B, n = 3, 700
    maps = [m * 0.25 for m in synthetic.feature_maps(B, shapes, 17)]
    pos = off_knot_positions(n, 137, [35, 18, 9, 5], 18)
    vpm, sizes, mi = [200, 260, 240], [(137, 137)] * B, [1] * B
    g = torch.Generator().manual_seed(19)
    w = (torch.rand(128, 480, generator=g) - 0.5) * 0.2
    go = torch.randn(n, 128, generator=g)

    f64 = [m.double().requires_grad_() for m in maps]
    p64, w64 = pos.double().requires_grad_(), w.double().requires_grad_()
    want = bil.vert_align_bilinear(f64, p64, vpm, sizes, mi) @ w64.t()
    (want * go.double()).sum().backward()

    def run(fused):
        f = [m.cuda().requires_grad_() for m in maps]
        p, wc = pos.cuda().requires_grad_(), w.cuda().requires_grad_()
        if fused:
            out = F_.vert_align_linear(f, p, vpm, sizes, mi, wc, bilinear=True)
        else:
            out = F_.linear(VertexAlign(mode="bilinear").eval()(f, p, vpm, sizes, mi), wc)
        (out * go.cuda()).sum().backward()
        return out, p.grad, wc.grad, [x.grad for x in f]

    out, gp, gw, gf = run(True)
    close(out, want, what="fused out")
    close(gp, p64.grad, what="fused position gradient")
    close(gw, w64.grad, what="fused gW")
    for i in range(4):
        close(gf[i], f64[i].grad, what="fused map %d gradient" % i)
    out_u, gp_u, gw_u, gf_u = run(False)
    close(out, out_u, what="fused vs unfused out")
    close(gp, gp_u, what="fused vs unfused position gradient")
    close(gw, gw_u, what="fused vs unfused gW")
    for i in range(4):
        close(gf[i], gf_u[i], what="fused vs unfused map %d gradient" % i)


# ---------------------------------------------------------------------------------------------------------------
# 4. the stage classes
# ---------------------------------------------------------------------------------------------------------------
def _stage_case(model, B=2, V=10):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.layers import Cubify
    vox = synthetic.blob_voxels(B, V, 3)
    verts, v_index, faces, f_index, adj = Cubify(0.2)(vox.cuda())
    img = 224 if model == "pix3d" else 137
    shapes = [synthetic.PIX3D_MAP] if model == "pix3d" else synthetic.SHAPENET_MAPS
    maps = [m * 0.05 for m in synthetic.feature_maps(B, shapes, 1)]
    pos0 = off_knot_positions(verts.shape[0], img, [s for _, s, _ in shapes], 9)     # the cubified graph, moved in-frustum
    return dict(v_index=v_index, faces=faces, f_index=f_index, adj=adj, maps=maps, pos0=pos0, sizes=[(img, img)] * B)


STAGE_CLASSES = {"pix3d": ("VertixRefinePix3D", 256), "shapenet": ("VertixRefineShapeNet", 3840),
                 "shapenet_residual": ("ResVertixRefineShapenet", 3840)}


@pytest.mark.parametrize("model", list(STAGE_CLASSES))
@pytest.mark.parametrize("use_feat", [False, True])
def test_stage_class_bilinear_vs_oracle_and_literal(lib, model, use_feat):
    """One stage with align_mode="bilinear": new positions, features and every weight, map and input-position gradient
    against the stages of oracle/bilinear_align.py in fp64, and the fused evaluation against the literal one
    (FUSE_STAGE_INPUTS = FUSE_ALIGN_BOTTLENECK = False).  A stage is a chain of ReLU layers, so the bound is relative L2
    per tensor: 1e-4, or 3x the oracle's own fp32-vs-fp64 deviation where that is larger (a ReLU input within an ulp of 0
    flips between any two fp32 evaluations)."""
    import meshrcnn_b200.layers as L
    cls_name, align_size = STAGE_CLASSES[model]
    c = _stage_case(model)
    torch.manual_seed(4)
    st = getattr(L, cls_name)(use_input_features=use_feat, alignment_size=align_size, align_mode="bilinear").cuda().eval()
    assert st.vertAlign.mode == "bilinear"
    with torch.no_grad():
        for prm in st.parameters():
            prm.mul_(0.2)
    SV = c["pos0"].shape[0]
    g = torch.Generator().manual_seed(21)
    feats0 = torch.randn(SV, 128, generator=g) * 0.1 if use_feat else None
    go_p, go_f = torch.randn(SV, 3, generator=g), torch.randn(SV, 128, generator=g) * 0.1

    def run_cuda(fused):
        L.FUSE_STAGE_INPUTS = L.FUSE_ALIGN_BOTTLENECK = fused
        try:
            st.zero_grad(set_to_none=True)
            fm = [m.cuda().requires_grad_() for m in c["maps"]]
            p = c["pos0"].cuda().requires_grad_()
            ft = feats0.cuda().requires_grad_() if use_feat else None
            arg = fm[0] if model == "pix3d" else fm
            new_pos, x = st(c["v_index"], arg, c["adj"], p, c["sizes"], vertex_features=ft)
            ((new_pos * go_p.cuda()).sum() + (x * go_f.cuda()).sum()).backward()
            out = {"pos": new_pos, "feat": x, "g pos": p.grad}
            if use_feat:
                out["g feats"] = ft.grad
            for i, m in enumerate(fm):
                out["g map%d" % i] = m.grad
            for k, prm in st.named_parameters():
                out["g " + k] = prm.grad.clone()
            return out
        finally:
            L.FUSE_STAGE_INPUTS = L.FUSE_ALIGN_BOTTLENECK = True

    def run_oracle(dt):
        fm = [m.to(dt).requires_grad_() for m in c["maps"]]
        p = c["pos0"].to(dt).requires_grad_()
        ft = feats0.to(dt).requires_grad_() if use_feat else None
        sd = {k: v.detach().cpu().to(dt).requires_grad_() for k, v in st.named_parameters()}
        arg = fm[0] if model == "pix3d" else fm
        new_pos, x = bil.STAGES[cls_name](sd, c["v_index"], arg, c["adj"].cpu(), p, c["sizes"], feats=ft)
        ((new_pos * go_p.to(dt)).sum() + (x * go_f.to(dt)).sum()).backward()
        out = {"pos": new_pos.detach(), "feat": x.detach(), "g pos": p.grad}
        if use_feat:
            out["g feats"] = ft.grad
        for i, m in enumerate(fm):
            out["g map%d" % i] = m.grad
        for k, v in sd.items():
            out["g " + k] = v.grad
        return out

    fused, literal = run_cuda(True), run_cuda(False)
    o64, o32 = run_oracle(torch.float64), run_oracle(torch.float32)
    assert fused.keys() == o64.keys() == literal.keys()
    for k in o64:
        if float(o64[k].norm()) == 0:               # e.g. the residual stage's 3-wide last GraphConv with every ReLU off
            assert float(fused[k].norm()) == 0 and float(literal[k].norm()) == 0, k
            continue
        err, ref = rel_l2(fused[k], o64[k]), rel_l2(o32[k], o64[k])
        assert err <= max(1e-4, 3 * ref), (k, err, ref)
        assert rel_l2(fused[k], literal[k]) <= 1e-4, (k, "fused vs literal")
    for k in ["pos", "feat", "g pos"] + ["g map%d" % i for i in range(len(c["maps"]))]:
        assert float(o64[k].abs().max()) > 0, k      # the aligned features and the position gradient are exercised


# ---------------------------------------------------------------------------------------------------------------
# 5. a chain of two stages through the positions, in training mode with the losses
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["pix3d", "shapenet"])
def test_two_stage_chain_with_losses_vs_oracle(lib, model):
    """RefinementHead(align_mode="bilinear") with two stages, in training mode: chamfer + 0.5 * edge loss of both stages
    (sampling draws injected) back to every weight, map and the input positions.  Stage 0's weights now also reach the loss
    through stage 1's sampling positions.  Bound: relative L2 per tensor, 1e-4 or 3x the oracle's own fp32-vs-fp64
    deviation where that is larger -- the chamfer term's nearest neighbours and the ReLU masks are discrete choices that any
    two fp32 evaluations may make differently for near-ties.  (The normal term is left out: its gradient is conditioned by
    eigen-gaps, which tests/test_loss_grads_gpu.py treats on its own.)"""
    from meshrcnn_b200 import loss_functions as LF, synthetic
    from meshrcnn_b200.pipeline import MeshTargets, RefinementHead
    c = _stage_case(model)
    B, n = 2, 1500
    torch.manual_seed(6)
    head = RefinementHead(model, cubify_threshold=0.2, num_refinement_stages=2, align_mode="bilinear").cuda().train()
    with torch.no_grad():
        for prm in head.parameters():
            prm.mul_(0.2)
    gvox = synthetic.blob_voxels(B, 8, 7)
    gverts, gvi, gfaces, gfi, _ = head.cubify(gvox.cuda())
    gverts = gverts * 0.1
    targets = MeshTargets(gverts, gfaces, gvi, gfi)
    g = torch.Generator().manual_seed(22)

    def draws(f_index):
        fi = torch.stack([torch.randint(0, int(f), (n,), generator=g) for f in f_index])
        return fi, torch.rand(B, n, generator=g), torch.rand(B, n, generator=g)

    rnd = [(draws(c["f_index"]), draws(gfi)) for _ in range(2)]
    as_kw = lambda r: dict(face_idx=r[0].cuda(), xi2=r[1].cuda(), xi1=r[2].cuda())

    fm = [m.cuda().requires_grad_() for m in c["maps"]]
    p = c["pos0"].cuda().requires_grad_()
    arg = fm[0] if model == "pix3d" else fm
    cur, feats, total = p, None, 0
    for s, st in enumerate(head.refineStages):
        kw = {} if feats is None else {"vertex_features": feats}
        cur, feats = st(c["v_index"], arg, c["adj"], cur, c["sizes"], **kw)
        ch, _, ed = LF.mesh_loss(cur, c["faces"], c["adj"], c["v_index"], c["f_index"], targets, float(n), 10,
                                 randomness=(as_kw(rnd[s][0]), as_kw(rnd[s][1])))
        total = total + ch + 0.5 * ed
    total.backward()
    got = {"loss": total, "g pos0": p.grad}
    for i, m in enumerate(fm):
        got["g map%d" % i] = m.grad
    for k, prm in head.refineStages.named_parameters():
        got["g " + k] = prm.grad

    cls_name = type(head.refineStages[0]).__name__

    def oracle(dt):
        fmo = [m.to(dt).requires_grad_() for m in c["maps"]]
        po = c["pos0"].to(dt).requires_grad_()
        sds = [{k: v.detach().cpu().to(dt).requires_grad_() for k, v in st.named_parameters()} for st in head.refineStages]
        a = fmo[0] if model == "pix3d" else fmo
        cur_o, f_o, tot = po, None, 0
        for s, sd in enumerate(sds):
            cur_o, f_o = bil.STAGES[cls_name](sd, c["v_index"], a, c["adj"].cpu(), cur_o, c["sizes"], feats=f_o)
            ch, _, ed, _ = mesh_ops.mesh_loss_with(cur_o, c["faces"].cpu(), c["adj"].cpu(), c["v_index"], c["f_index"],
                                                   gverts.cpu().to(dt), gfaces.cpu(), gvi, gfi, rnd[s][0], rnd[s][1],
                                                   float(n), 10)
            tot = tot + ch + 0.5 * ed
        tot.backward()
        out = {"loss": tot.detach(), "g pos0": po.grad}
        for i, m in enumerate(fmo):
            out["g map%d" % i] = m.grad
        for s, sd in enumerate(sds):
            for k, v in sd.items():
                out["g %d.%s" % (s, k)] = v.grad
        return out

    o64, o32 = oracle(torch.float64), oracle(torch.float32)
    assert got.keys() == o64.keys()
    for k in o64:
        assert float(o64[k].norm()) > 0, k
        err, ref = rel_l2(got[k], o64[k]), rel_l2(o32[k], o64[k])
        assert err <= max(1e-4, 3 * ref), (k, err, ref)


# ---------------------------------------------------------------------------------------------------------------
# 6. the default is unchanged
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", list(STAGE_CLASSES))
def test_default_construction_never_calls_the_bilinear_kernels(lib, model):
    """A default-constructed head issues no mrb_vert_align_bilinear_* call, and its outputs equal those of
    align_mode="reference" passed explicitly, bit for bit."""
    from meshrcnn_b200 import _lib
    from meshrcnn_b200.pipeline import RefinementHead
    c = _stage_case(model)

    def run(**kw):
        torch.manual_seed(8)
        head = RefinementHead(model, cubify_threshold=0.2, **kw).cuda().eval()
        calls = []
        orig = _lib.call
        _lib.call = lambda name, *a: (calls.append(name), orig(name, *a))[1]
        try:
            fm = [m.cuda().requires_grad_() for m in c["maps"]]
            p = c["pos0"].cuda().requires_grad_()
            cur, feats = p, None
            for st in head.refineStages:
                kw2 = {} if feats is None else {"vertex_features": feats}
                cur, feats = st(c["v_index"], fm[0] if model == "pix3d" else fm, c["adj"], cur, c["sizes"], **kw2)
            (cur.sum() + feats.sum()).backward()
        finally:
            _lib.call = orig
        return cur.detach(), feats.detach(), calls

    pos_d, feat_d, calls_d = run()
    pos_r, feat_r, calls_r = run(align_mode="reference")
    assert not [n for n in calls_d if "bilinear" in n]
    assert calls_d == calls_r
    assert torch.equal(pos_d, pos_r) and torch.equal(feat_d, feat_r)
    _, _, calls_b = run(align_mode="bilinear")
    assert "mrb_vert_align_bilinear_fwd" in calls_b and "mrb_vert_align_bilinear_bwd" in calls_b


def test_mode_set_on_a_loaded_model(lib):
    """stage.vertAlign.mode = "bilinear" on a model built (and loaded) with the default switches the stage over; the state
    dict keys do not depend on the mode."""
    from meshrcnn_b200.pipeline import RefinementHead
    a = RefinementHead("pix3d", num_refinement_stages=1)
    b = RefinementHead("pix3d", num_refinement_stages=1, align_mode="bilinear")
    assert list(a.state_dict()) == list(b.state_dict())
    b.load_state_dict(a.state_dict())
    c = _stage_case("pix3d")
    a, b = a.cuda().eval(), b.cuda().eval()
    args = lambda: (c["v_index"], c["maps"][0].cuda(), c["adj"], c["pos0"].cuda(), c["sizes"])
    want, _ = b.refineStages[0](*args())
    before, _ = a.refineStages[0](*args())
    a.refineStages[0].vertAlign.mode = "bilinear"
    got, _ = a.refineStages[0](*args())
    assert torch.equal(got, want) and not torch.equal(before, want)
