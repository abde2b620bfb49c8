"""The bilinear VertexAlign oracle (oracle/bilinear_align.vert_align_bilinear) against torch's grid_sample in fp64, plus known
answers: exact texels at integer coordinates, a 1 x 1 map, clamped and non-finite projections.  CPU only."""
import pytest
import torch
import torch.nn.functional as F

from oracle import bilinear_align as bil, mesh_ops


def _xy(pos, size, S):
    """The oracle's sampling coordinates (x on the H axis, y on the W axis), before the [0, S-1] clamp."""
    H, W = size
    h = (248 * (pos[:, 1] / pos[:, 2]) + 111.5).clamp(0, H - 1)
    w = (248 * (pos[:, 0] / -pos[:, 2]) + 111.5).clamp(0, W - 1)
    return w / (float(W) / S), h / (float(H) / S)


def _grid_sample_align(fmaps, pos, vpm, sizes, mi):
    """The same quantity through grid_sample(align_corners=True, padding_mode="border"): the grid is (y, x) in that
    order, because grid_sample's first coordinate indexes the last (W) axis."""
    chunks = pos.split(vpm)
    rows, k = [], 0
    for img, (n_mesh, size) in enumerate(zip(mi, sizes)):
        for p in chunks[k:k + n_mesh]:
            parts = []
            for f in fmaps:
                S = f.shape[-1]
                x, y = _xy(p, size, S)
                grid = torch.stack([2 * y / (S - 1) - 1, 2 * x / (S - 1) - 1], 1).view(1, 1, -1, 2)
                s = F.grid_sample(f[img:img + 1], grid, mode="bilinear", padding_mode="border", align_corners=True)
                parts.append(s[0, :, 0, :].t())
            rows.append(torch.cat(parts, 1))
        k += n_mesh
    return torch.cat(rows, 0)


def test_oracle_matches_grid_sample_values_and_gradients():
    from meshrcnn_b200 import synthetic
    shapes = [(6, 12, 12), (5, 35, 35), (4, 5, 5)]
    fm = [f.double() for f in synthetic.feature_maps(3, shapes, 1)]
    vpm, mi, sizes = [40, 25, 35, 50], [2, 1, 1], [(224, 224), (137, 137), (224, 224)]
    pos = synthetic.in_frustum_positions(sum(vpm), 224, 2).double()
    go = torch.randn(sum(vpm), sum(c for c, _, _ in shapes), generator=torch.Generator().manual_seed(3), dtype=torch.float64)

    def run(fn):
        f = [x.clone().requires_grad_() for x in fm]
        p = pos.clone().requires_grad_()
        out = fn(f, p, vpm, sizes, mi)
        (out * go).sum().backward()
        return out.detach(), p.grad, [x.grad for x in f]

    got, gp, gf = run(bil.vert_align_bilinear)
    want, wp, wf = run(_grid_sample_align)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-12)
    assert torch.allclose(gp, wp, rtol=1e-10, atol=1e-10)
    assert float(gp.abs().max()) > 0
    for a, b in zip(gf, wf):
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12)


def test_integer_coordinates_hit_texels_exactly_where_the_reference_gives_zero():
    """At integer (x, y) the sample is f[x, y], last row and column included; the reference mode's mask
    (x2 > x1 and y2 > y1) is 0 there."""
    S, size = 7, (224, 224)
    fm = torch.randn(1, 3, S, S, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    ij = torch.tensor([[0, 0], [3, 5], [6, 6], [6, 0], [0, 6], [2, 6]], dtype=torch.float64)
    s = 224.0 / S
    # x = w / s, y = h / s with w = 248 p0 / (-p2) + 111.5, h = 248 p1 / p2 + 111.5 and p2 = -1
    w, h = ij[:, 0] * s, ij[:, 1] * s
    pos = torch.stack([(w - 111.5) / 248, -(h - 111.5) / 248, -torch.ones(len(ij), dtype=torch.float64)], 1)
    x, y = _xy(pos, size, S)
    assert torch.allclose(x, ij[:, 0], atol=1e-12) and torch.allclose(y, ij[:, 1], atol=1e-12)
    got = bil.vert_align_bilinear([fm], pos, [len(ij)], [size], [1])
    want = fm[0][:, ij[:, 0].long(), ij[:, 1].long()].t()
    assert torch.allclose(got, want, rtol=0, atol=1e-12)
    ref = mesh_ops.vert_align([fm], pos, [len(ij)], [size], [1])
    assert float(ref.abs().max()) == 0.0


def test_single_texel_map():
    from meshrcnn_b200 import synthetic
    fm = torch.randn(2, 4, 1, 1, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    pos = synthetic.in_frustum_positions(30, 224, 1).double().requires_grad_()
    out = bil.vert_align_bilinear([fm], pos, [10, 20], [(224, 224)] * 2, [1, 1])
    want = torch.cat([fm[0, :, 0, 0].expand(10, 4), fm[1, :, 0, 0].expand(20, 4)])
    assert torch.equal(out, want)
    assert not out.requires_grad or pos.grad is None


def test_clamped_and_non_finite_positions_have_zero_position_gradient():
    S, size = 12, (224, 224)
    fm = torch.randn(1, 5, S, S, generator=torch.Generator().manual_seed(2), dtype=torch.float64).requires_grad_()
    pos = torch.tensor([[20.0, 15.0, -1.0],          # far outside: w, h clamp to the image
                        [-20.0, -15.0, -1.5],
                        [0.3, 0.2, 0.0],             # p2 == 0: h, w are +-inf
                        [0.0, 0.0, 0.0],             # 0 / 0: NaN
                        [float("nan"), 0.1, -1.0],
                        [0.0, 0.0, -1.0]], dtype=torch.float64).requires_grad_()   # the last one is inside
    out = bil.vert_align_bilinear([fm], pos, [6], [size], [1])
    assert bool(torch.isfinite(out).all())
    f = fm.detach()[0]
    assert torch.equal(out[0].detach(), f[:, S - 1, 0])        # w -> W-1 (x -> S-1), h -> 0
    assert torch.equal(out[1].detach(), f[:, 0, S - 1])        # w -> 0, h -> H-1
    assert torch.equal(out[2].detach(), f[:, 0, S - 1])        # w = -inf -> 0, h = +inf -> H-1
    assert torch.equal(out[3].detach(), f[:, 0, 0])            # NaN -> 0
    out.sum().backward()
    assert torch.equal(pos.grad[:5], torch.zeros(5, 3, dtype=torch.float64))
    assert float(pos.grad[5].abs().max()) > 0
    assert bool(torch.isfinite(fm.grad).all())


@pytest.mark.parametrize("name", list(bil.STAGES))
def test_bilinear_oracle_stages_restate_the_reference_stages(name):
    """The stage functions of oracle/bilinear_align.py with ``align=mesh_ops.vert_align`` are mesh_ops' reference stages:
    only the aligned features differ between the two oracles."""
    from meshrcnn_b200 import synthetic
    g = torch.Generator().manual_seed(4)
    n, D = 40, 16
    img, shapes = (224, [synthetic.PIX3D_MAP]) if name == "VertixRefinePix3D" else (137, list(synthetic.SHAPENET_MAPS))
    C = sum(c for c, _, _ in shapes)
    fm = [f.double() for f in synthetic.feature_maps(2, shapes, 3)]
    pos = synthetic.in_frustum_positions(n, img, 5).double()
    adj = torch.stack([torch.arange(n), torch.roll(torch.arange(n), 1)])
    adj = torch.cat([adj, adj.flip(0)], 1)
    w = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64) * 0.1
    if name == "VertixRefinePix3D":
        sd = {"graphConv0.w0": w(C + 3, D), "graphConv0.w1": w(C + 3, D), "linear.weight": w(3, D + 3)}
    elif name == "VertixRefineShapeNet":
        sd = {"linear0.weight": w(D, C), "graphConv0.w0": w(D + 3, D), "graphConv0.w1": w(D + 3, D), "linear1.weight": w(3, D)}
    else:
        sd = {"linear.weight": w(D, C), "resGraphConv0.projection.weight": w(D, D + 3), "graphConv.w0": w(D, 3),
              "graphConv.w1": w(D, 3)}
        for i in range(3):
            k = D + 3 if i == 0 else D
            sd.update({"resGraphConv%d.conv0.w0" % i: w(k, D), "resGraphConv%d.conv0.w1" % i: w(k, D),
                       "resGraphConv%d.conv1.w0" % i: w(D, D), "resGraphConv%d.conv1.w1" % i: w(D, D)})
    if name != "ResVertixRefineShapenet":
        for i in (1, 2):
            sd.update({"graphConv%d.w0" % i: w(D + 3, D), "graphConv%d.w1" % i: w(D + 3, D)})
    arg = fm[0] if name == "VertixRefinePix3D" else fm
    want = mesh_ops.STAGES[name](sd, [15, 25], arg, adj, pos, [(img, img)] * 2)
    got = bil.STAGES[name](sd, [15, 25], arg, adj, pos, [(img, img)] * 2, align=mesh_ops.vert_align)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    other = bil.STAGES[name](sd, [15, 25], arg, adj, pos, [(img, img)] * 2)
    assert not torch.equal(other[0], want[0])
