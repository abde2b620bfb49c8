"""Loss-path values and gradients against fp64 autograd of the oracle on the same fp32 inputs, at the trained shape and on
every size- and argument-dependent branch of the kernels: sampling + unit-ball normalisation (cluster and single-CTA
paths, scaled and unscaled backward, 3- and 4-float gradient rows), chamfer backward with P != Q and one upstream gradient
absent, PCA normals (k = 10 template and generic k, saved eigen-decomposition, degenerate spectra), normal consistency with
exact-zero dot products, grid-stride loops of the edge loss and the voxel BCE, saturated logits, and the composed stage loss.

The discrete choices (face draws, nearest indices, k-NN sets) are pinned to the kernel's, and the oracle differentiates the
continuous part (``oracle/mesh_ops.py``, ``*_given``).  Tolerance: rtol 1e-4 elementwise (``close``); normals are compared
on the rows ``normals_conditioning`` classes as well-conditioned, with no fraction allowance."""
import numpy as np
import pytest
import torch

from oracle import mesh_ops
from tests.test_layers_gpu import close

pytestmark = pytest.mark.gpu

COND = 1e-3        # relative eigen-gap and sign-rule margins below which a normals row is not compared elementwise


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _i32(t):
    return t.to(torch.int32).contiguous()


# ---------------------------------------------------------------------------------------------------------------------
# (a) sampling + normalisation
# ---------------------------------------------------------------------------------------------------------------------
def _spiked_meshes(B, n, scaled, seed):
    """Ragged batch (mesh 0 a single thin triangle) whose sample has a unique farthest point by construction: point m_b
    of mesh b is injected exactly onto a far 'spike' vertex (face corner 1, xi1 = 1, xi2 = 0); every other draw keeps
    away from it.  Coordinates are x4 (normalisation divides by the largest norm) or x0.5 (centred cloud inside
    [-1, 1]^3: no division).  Returns fp32 verts, int64 local faces, v_index, f_index, (face_idx, xi2, xi1) B x n."""
    g = _gen(seed)
    vs, fs, vi, fi = [], [], [], []
    fidx, xi2, xi1 = torch.empty(B, n, dtype=torch.int64), torch.rand(B, n, generator=g), torch.rand(B, n, generator=g)
    for b in range(B):
        if b == 0:
            v = torch.tensor([[0.0, 0.0, 0.0], [0.9, 0.5, 0.3], [0.06, 0.02, 0.04]])
            f = torch.tensor([[0, 1, 2]])
            fidx[b] = 0
            xi1[b] *= 0.25                                      # sqrt(xi1) <= 0.5: away from the spike corner
        else:
            nv = 8 + 13 * b
            v = torch.cat([(torch.rand(nv, 3, generator=g) - 0.5) * 0.3, torch.tensor([[0.8, -0.7, 0.75]])])
            body = torch.stack([torch.randperm(nv, generator=g)[:3] for _ in range(2 * nv)])
            f = torch.cat([body, torch.tensor([[0, nv, 1]])])    # the spike face is the last one
            fidx[b] = torch.randint(0, 2 * nv, (n,), generator=g)
            xi1[b] *= 0.9
        m = int(torch.randint(0, n, (1,), generator=g))
        fidx[b, m], xi1[b, m], xi2[b, m] = f.shape[0] - 1, 1.0, 0.0
        vs.append(v * (4.0 if scaled else 0.5) + 0.25 * b)
        fs.append(f)
        vi.append(v.shape[0])
        fi.append(f.shape[0])
    return torch.cat(vs), torch.cat(fs), vi, fi, (fidx, xi2, xi1)


def _sample_abi(verts, faces, vi, fi, n, draws):
    """mrb_sample_points_fwd with injected draws: (cloud, stats, fidx, w, v_off)."""
    from meshrcnn_b200 import _lib, functional as F_
    dev = verts.device
    B = len(fi)
    v_off, f_off = F_.offsets_table(vi, dev), F_.offsets_table(fi, dev)
    raw, cloud, w = (torch.empty(B, n, 3, device=dev) for _ in range(3))
    fidx = torch.empty(B, n, dtype=torch.int32, device=dev)
    stats = torch.empty(B, 8, dtype=torch.float64, device=dev)
    fi_d, x2, x1 = draws[0].cuda(), draws[1].cuda(), draws[2].cuda()
    _lib.call("mrb_sample_points_fwd", _lib.ptr(verts), _lib.ptr(faces), _lib.ptr(v_off), _lib.ptr(f_off), None, B, n, None,
              _lib.ptr(fi_d), _lib.ptr(x2), _lib.ptr(x1), 0, _lib.ptr(raw), _lib.ptr(fidx), _lib.ptr(w), _lib.ptr(cloud),
              _lib.ptr(stats))
    return cloud, stats, fidx, w, v_off


def _check_sampling(B, n, scaled, seed):
    from meshrcnn_b200 import _lib, functional as F_
    verts, faces, vi, fi, draws = _spiked_meshes(B, n, scaled, seed)
    vc, fc = verts.cuda(), faces.cuda()
    cloud, stats, fidx, w, v_off = _sample_abi(vc, fc, vi, fi, n, draws)

    # forward: cloud and stats (mean, factor, argmax row exactly)
    v64 = verts.double().requires_grad_()
    want = mesh_ops.batched_sample_with(v64, faces, vi, fi, draws[0], draws[1].double(), draws[2].double())
    close(cloud, want.detach(), what="cloud n=%d" % n)
    st = stats.cpu()
    for b, (v, f) in enumerate(zip(verts.double().split(vi), faces.split(fi))):
        raw = mesh_ops.sample_raw_with(v, f, draws[0][b], draws[1][b].double(), draws[2][b].double())
        mean = raw.mean(0)
        c = raw - mean
        r2 = (c * c).sum(1)
        do_scale = bool(c.abs().max() > 1)
        assert torch.allclose(st[b, :3], mean, rtol=0, atol=1e-6 * max(1.0, float(raw.abs().max()))), (b, st[b], mean)
        if n >= 5:
            assert do_scale == scaled, (b, n, scaled)
        if do_scale:
            top = r2.topk(2)
            assert float(top.values[1]) < (1 - 1e-4) * float(top.values[0])          # unique farthest point (no tie)
            assert int(st[b, 4]) == int(top.indices[0]), (b, st[b, 4], top.indices)
            assert abs(float(st[b, 3]) - float(top.values[0].sqrt())) <= 1e-6 * float(top.values[0].sqrt())
        else:
            assert float(st[b, 4]) == -1.0 and float(st[b, 3]) == 1.0

    # backward: fp64 autograd through sampling + normalisation
    gcloud = torch.randn(B, n, 3, generator=_gen(seed + 1))
    gw, = torch.autograd.grad((want * gcloud.double()).sum(), v64)
    g3 = torch.zeros(verts.shape[0], 3, device="cuda")
    g4 = torch.zeros(verts.shape[0], 4, device="cuda")
    scr = torch.empty(4 * B, dtype=torch.float64, device="cuda")
    gc = gcloud.cuda()
    args = (_lib.ptr(gc), _lib.ptr(cloud), _lib.ptr(stats), _lib.ptr(fidx), _lib.ptr(w), _lib.ptr(fc), _lib.ptr(v_off), B, n)
    _lib.call("mrb_sample_points_bwd", *args, _lib.ptr(g3), _lib.ptr(scr))
    _lib.call("mrb_sample_points_bwd_ld", *args, _lib.ptr(g4), 4, _lib.ptr(scr))
    close(g3, gw, what="gverts, 3-float rows, n=%d" % n)
    close(g4[:, :3], gw, what="gverts, 4-float rows, n=%d" % n)
    assert float(g4[:, 3].abs().max()) == 0.0
    # and through the autograd Function the losses use
    va = vc.clone().requires_grad_()
    c2, _ = F_.sample_points(va, fc, vi, fi, n, face_idx=draws[0].cuda(), xi2=draws[1].cuda(), xi1=draws[2].cuda())
    assert torch.equal(c2, cloud)
    (c2 * gc).sum().backward()
    close(va.grad, gw, what="sample_points backward, n=%d" % n)


@pytest.mark.parametrize("scaled", [True, False])
@pytest.mark.parametrize("n", [1, 5, 8, 9, 2047, 2048, 2049, 10000, 16384, 16385, 40000])
def test_sampling_normalisation_vs_fp64(lib, n, scaled):
    """n <= 16 384: cluster kernel (n < 8 leaves cluster ranks without points); n > 16 384: one CTA per cloud."""
    _check_sampling(3, n, scaled, seed=n)


@pytest.mark.parametrize("scaled", [True, False])
def test_sampling_normalisation_b32_vs_fp64(lib, scaled):
    _check_sampling(32, 10000, scaled, seed=32)


@pytest.mark.parametrize("V", [16384, 16385, 40000])
@pytest.mark.parametrize("spread", [0.3, 3.0])
def test_normalize_mesh_vs_fp64(lib, V, spread):
    """normalize_mesh of one GT mesh: the cluster kernel up to 16 384 vertices, the single-CTA kernel above."""
    from meshrcnn_b200.mesh_sampling import normalize_mesh
    v = (torch.rand(V, 3, generator=_gen(V)) - 0.5) * spread + 0.7
    v[V // 3] = torch.tensor([0.7, 0.7 + 1.2 * spread, 0.7])         # unique farthest vertex
    got = normalize_mesh(v.cuda())
    close(got, mesh_ops.normalize_cloud(v.double()), what="normalize_mesh V=%d" % V)


# ---------------------------------------------------------------------------------------------------------------------
# (b) chamfer backward
# ---------------------------------------------------------------------------------------------------------------------
def _assert_nearest(p, q, ip, iq, batches):
    """The kernel's nearest indices are optimal in fp64 up to fp32 ties, in both directions."""
    for a, b, idx in ((p[:batches], q[:batches], ip[:batches]), (q[:batches], p[:batches], iq[:batches])):
        a64, b64 = a.detach().cpu().double(), b.detach().cpu().double()
        ar = torch.arange(a64.shape[0]).view(-1, 1)
        chosen = ((a64 - b64[ar, idx.cpu().long()]) ** 2).sum(2)
        best = mesh_ops.nearest_chunked(a64, b64)
        assert bool((chosen <= best * (1 + 1e-5) + 1e-12).all()), float((chosen - best).max())


@pytest.mark.parametrize("B,P,Q", [(3, 777, 1301), (2, 10000, 6000), (32, 10000, 10000)])
@pytest.mark.parametrize("used", ["both", "l1", "l2"])
def test_chamfer_grads_vs_fp64(lib, B, P, Q, used):
    """chamfer_knn with both sums or one of them (the other upstream gradient is then None), and chamfer_total."""
    from meshrcnn_b200 import functional as F_
    g = _gen(B + P + Q)
    p = (torch.rand(B, P, 3, generator=g) - 0.5).cuda().requires_grad_()
    q = (torch.randn(B, Q, 3, generator=g) * torch.tensor([0.3, 0.2, 0.1])).cuda().requires_grad_()
    l1, l2, ip, iq, _, _ = F_.chamfer_knn(p, q, 0)
    _assert_nearest(p, q, ip, iq, min(B, 2))
    a, b = {"both": (0.7, 1.3), "l1": (0.7, 0.0), "l2": (0.0, 1.3)}[used]
    loss = a * l1 if not b else (b * l2 if not a else a * l1 + b * l2)
    gp, gq = torch.autograd.grad(loss, [p, q])
    p64, q64 = p.detach().cpu().double().requires_grad_(), q.detach().cpu().double().requires_grad_()
    w1, w2 = mesh_ops.chamfer_given(p64, q64, ip.cpu(), iq.cpu())
    close(l1, w1.detach(), what="loss_1")
    close(l2, w2.detach(), what="loss_2")
    hp, hq = torch.autograd.grad(a * w1 + b * w2, [p64, q64], retain_graph=True)
    close(gp, hp, what="grad p (%s)" % used)
    close(gq, hq, what="grad q (%s)" % used)
    if used == "both":
        tot, ip2, iq2, _, _ = F_.chamfer_total(p, q, 0, 1e-4)
        assert torch.equal(ip2, ip) and torch.equal(iq2, iq)
        close(tot, 1e-4 * (w1 + w2).detach(), what="chamfer_total")
        gp, gq = torch.autograd.grad(2.5 * tot, [p, q])
        hp, hq = torch.autograd.grad(2.5e-4 * (w1 + w2), [p64, q64])
        close(gp, hp, what="chamfer_total grad p")
        close(gq, hq, what="chamfer_total grad q")


# ---------------------------------------------------------------------------------------------------------------------
# (c) normals
# ---------------------------------------------------------------------------------------------------------------------
def _groups(B, G, k, seed, planar=0, long_axis=1, spectrum=(1.0, 0.3, 0.05), size=0.05):
    """B clouds of G * k points in G groups of k; every row of a group uses the group as its k-NN set (shuffled order) and
    the points are permuted over the cloud.  Groups are randomly rotated anisotropic Gaussians with variances ~ spectrum;
    the first ``planar`` groups are instead exact 2 x 5 lattices in a z = const plane, 5 points long along x (long_axis = 0)
    or y (1): dyadic coordinates, so the scatter matrix is exactly diagonal with distinct eigenvalues and the normal (row 0
    of V) is exactly +-e_z (long_axis = 0) or +-e_y (1)."""
    g = _gen(seed)
    P = G * k
    pts = torch.empty(B, P, 3)
    nn = torch.empty(B, P, k, dtype=torch.int64)
    h = 2.0 ** -5
    lat = torch.tensor([[u * h, v * h / 2] for u in (-0.5, 0.5) for v in (-2, -1, 0, 1, 2)])
    inplane = (1, 0) if long_axis == 0 else (0, 1)
    for b in range(B):
        rot = torch.linalg.qr(torch.randn(G, 3, 3, generator=g)).Q
        loc = torch.randn(G, k, 3, generator=g) * torch.tensor(spectrum).sqrt() * size
        grp = torch.einsum("gij,gkj->gki", rot, loc) + torch.rand(G, 1, 3, generator=g)
        for i in range(planar):
            c = torch.randint(0, 16, (3,), generator=g).float() / 16
            grp[i] = c
            grp[i, :, inplane[0]] += lat[:, 0]
            grp[i, :, inplane[1]] += lat[:, 1]
        perm = torch.randperm(P, generator=g)
        pts[b, perm] = grp.reshape(P, 3)
        ids = perm.view(G, k)
        order = torch.argsort(torch.rand(G, k, k, generator=g), -1)
        nn[b, perm] = torch.gather(ids.unsqueeze(1).expand(G, k, k), 2, order).reshape(P, k)
    return pts, nn


def _well_conditioned(pts, nn):
    gap, m20, m1, mdet = mesh_ops.normals_conditioning(pts, nn)
    return (gap > COND) & (m20 > COND) & (m1 > COND) & (mdet > 0.5)


def _normals_abi(pts, nn, k, gn, ld, saved_eig):
    """(normals, gradient rows) from mrb_normals_fwd[_eig] + mrb_normals_bwd[_ld]."""
    from meshrcnn_b200 import _lib
    B, P, _ = pts.shape
    pc, nc, gc = pts.cuda().contiguous(), _i32(nn).cuda(), gn.cuda().contiguous()
    out = torch.empty(B, P, 3, device="cuda")
    eig = torch.empty(12, B * P, dtype=torch.float64, device="cuda") if saved_eig else None
    if saved_eig:
        _lib.call("mrb_normals_fwd_eig", _lib.ptr(pc), _lib.ptr(nc), B, P, k, _lib.ptr(out), _lib.ptr(eig))
    else:
        _lib.call("mrb_normals_fwd", _lib.ptr(pc), _lib.ptr(nc), B, P, k, _lib.ptr(out))
    gpt = torch.zeros(B, P, ld, device="cuda")
    if ld == 3 and not saved_eig:
        _lib.call("mrb_normals_bwd", _lib.ptr(pc), _lib.ptr(nc), B, P, k, _lib.ptr(gc), _lib.ptr(gpt))
    else:
        _lib.call("mrb_normals_bwd_ld", _lib.ptr(pc), _lib.ptr(nc), B, P, k, _lib.ptr(gc), _lib.ptr(gpt), ld, _lib.ptr(eig))
    if ld == 4:
        assert float(gpt[..., 3].abs().max()) == 0.0
    return out, gpt[..., :3]


@pytest.mark.parametrize("saved_eig", [False, True])
@pytest.mark.parametrize("ld", [3, 4])
@pytest.mark.parametrize("k", [3, 4, 9, 10, 11, 16])
def test_normals_fwd_bwd_vs_fp64(lib, k, ld, saved_eig):
    """k = 10 runs the unrolled template, every other k the generic one.  Every well-conditioned row: rtol 1e-4
    elementwise forward; the upstream gradient is zero on the other rows, and then the whole backward is compared."""
    B, G = 2, 1200 // k
    pts, nn = _groups(B, G, k, seed=100 + k)
    good = _well_conditioned(pts, nn)
    assert float(good.double().mean()) > 0.9
    gn = torch.randn(pts.shape, generator=_gen(k)) * good.unsqueeze(-1)
    got, gpt = _normals_abi(pts, nn, k, gn, ld, saved_eig)
    p64 = pts.double().requires_grad_()
    want = mesh_ops.normals_from_neighbours(p64, nn, canonical_signs=True)
    close(got[good.cuda()], want.detach()[good], what="normals k=%d" % k)
    assert torch.allclose(got.norm(dim=2), torch.ones(B, pts.shape[1], device="cuda"), atol=1e-6)
    gw, = torch.autograd.grad((want * gn.double()).sum(), p64)
    close(gpt, gw, what="normals backward k=%d ld=%d eig=%s" % (k, ld, saved_eig))


def test_normals_degenerate_neighbourhoods(lib):
    """k = 1, k = 2, duplicated points, isotropic and square axis-aligned planar neighbourhoods: finite unit normals and a
    finite gradient; exactly zero where all three eigenvalues coincide (the cut-off drops every pair's term)."""
    g = _gen(5)
    P = 60
    base = torch.rand(1, P, 3, generator=g)
    ar = torch.arange(P)
    s = 0.125
    octa = torch.tensor([[s, 0, 0], [-s, 0, 0], [0, s, 0], [0, -s, 0], [0, 0, s], [0, 0, -s]])
    square = torch.tensor([[x * s, y * s, 0.0] for x in (-1, 0, 1) for y in (-1, 0, 1)])          # 3 x 3 lattice, z = const
    c = torch.tensor([0.5, 0.25, 0.625])

    def cloud_of(block):        # one block of points at c, replicated over the cloud (10 blocks of 6 / 9 points max)
        pts = base.clone()
        m = block.shape[0]
        for r in range(P // m):
            pts[0, r * m:(r + 1) * m] = block + c + r
        return pts

    cases = [  # (name, points, knn, exact zero gradient)
        ("k=1", base, ar.view(1, P, 1), True),
        ("k=2", base, torch.stack([ar, (ar + 1) % P], -1).unsqueeze(0), False),
        ("duplicated k=4", base, ar.view(1, P, 1).expand(1, P, 4), True),
        ("duplicated k=10", base, ar.view(1, P, 1).expand(1, P, 10), True),
        ("isotropic k=6", cloud_of(octa), (ar // 6 * 6).view(1, P, 1) + torch.arange(6).view(1, 1, 6), True),
        ("isotropic k=10", cloud_of(torch.cat([octa, torch.zeros(4, 3)])),
         (ar // 10 * 10).view(1, P, 1) + torch.arange(10).view(1, 1, 10), True),
        ("planar square k=9", cloud_of(square), (ar // 9 * 9).clamp(max=P - 9).view(1, P, 1) + torch.arange(9).view(1, 1, 9),
         False),
    ]
    for name, pts, nn, zero in cases:
        k = nn.shape[2]
        gn = torch.randn(1, P, 3, generator=g)
        for ld in (3, 4):
            for saved in (False, True):
                n, gpt = _normals_abi(pts, nn.contiguous(), k, gn, ld, saved)
                assert bool(torch.isfinite(n).all()) and bool(torch.isfinite(gpt).all()), name
                assert torch.allclose(n.norm(dim=2), torch.ones(1, P, device="cuda"), atol=1e-6), name
                if zero:
                    assert float(gpt.abs().max()) == 0.0, (name, ld, saved, float(gpt.abs().max()))
                else:
                    assert float(gpt.abs().max()) > 0.0, name


# ---------------------------------------------------------------------------------------------------------------------
# (d) normal consistency
# ---------------------------------------------------------------------------------------------------------------------
def test_normal_consistency_grads_with_exact_zero_dots(lib):
    """normal_total and normal_distance (both sums, and one of them) with pinned index sets.  The first groups of p and q
    are axis-aligned planar lattices (Cubify-like) whose normals are +-e_y in p and +-e_z in q; half of their rows are
    paired with each other, so those dot products are exactly 0 on both sides and sign(0) = 0 must hold in the kernel as
    in the oracle."""
    from meshrcnn_b200 import functional as F_
    B, G, k, Z = 2, 200, 10, 20
    P = G * k
    p, kp = _groups(B, G, k, seed=8, planar=Z, long_axis=1)
    q, kq = _groups(B, G, k, seed=14, planar=Z, long_axis=0)
    assert bool(_well_conditioned(p, kp).all()) and bool(_well_conditioned(q, kq).all())
    g = _gen(9)
    ip, iq = torch.randint(0, P, (B, P), generator=g), torch.randint(0, P, (B, P), generator=g)
    n_p = mesh_ops.normals_from_neighbours(p.double(), kp, canonical_signs=True)
    n_q = mesh_ops.normals_from_neighbours(q.double(), kq, canonical_signs=True)
    flat_p = (n_p.abs() == 1).any(-1)                       # exactly axis-aligned normals = the lattice rows
    flat_q = (n_q.abs() == 1).any(-1)
    assert int(flat_p.sum()) == B * Z * k and int(flat_q.sum()) == B * Z * k
    for b in range(B):                                       # pair lattice rows with lattice rows (half of them)
        rp, rq = flat_p[b].nonzero().squeeze(1), flat_q[b].nonzero().squeeze(1)
        h = rp.shape[0] // 2
        ip[b, rp[:h]] = rq[torch.randint(0, rq.shape[0], (h,), generator=g)]
        iq[b, rq[:h]] = rp[torch.randint(0, rp.shape[0], (h,), generator=g)]
    ar = torch.arange(B).view(-1, 1)
    d0, d1 = (n_p * n_q[ar, ip]).sum(2), (n_q * n_p[ar, iq]).sum(2)
    zero0, zero1 = d0 == 0, d1 == 0
    assert int(zero0.sum()) >= B * Z * k // 2 and int(zero1.sum()) >= B * Z * k // 2
    assert float(torch.cat([d0[~zero0], d1[~zero1]]).abs().min()) > 1e-5          # no sign near a tie elsewhere
    nk_p, nk_q = F_.compute_normals(p.cuda(), kp.cuda()), F_.compute_normals(q.cuda(), kq.cuda())
    kd0 = (nk_p.cpu().double() * nk_q.cpu().double()[ar, ip]).sum(2)
    assert bool((kd0[zero0] == 0).all())                                          # the kernel's normals are exact too

    pc, qc = p.cuda().requires_grad_(), q.cuda().requires_grad_()
    args = (kp.cuda(), kq.cuda(), ip.cuda(), iq.cuda())
    p64, q64 = p.double().requires_grad_(), q.double().requires_grad_()
    tot = F_.normal_total(pc, qc, *args, -1e-4)
    want = mesh_ops.normal_total_given(p64, q64, kp, kq, ip, iq, -1e-4)
    close(tot, want.detach(), what="normal_total")
    gp, gq = torch.autograd.grad(tot, [pc, qc])
    hp, hq = torch.autograd.grad(want, [p64, q64])
    close(gp, hp, what="normal_total grad p")
    close(gq, hq, what="normal_total grad q")
    l0, l1 = F_.normal_distance(pc, qc, *args)
    w0, w1 = mesh_ops.normal_sums_given(p64, q64, kp, kq, ip, iq)
    close(l0, w0.detach(), what="normal_distance l0")
    close(l1, w1.detach(), what="normal_distance l1")
    for a, b in ((0.6, -1.7), (0.6, 0.0), (0.0, -1.7)):
        loss = a * l0 if not b else (b * l1 if not a else a * l0 + b * l1)
        gp, gq = torch.autograd.grad(loss, [pc, qc], retain_graph=True)
        hp, hq = torch.autograd.grad(a * w0 + b * w1, [p64, q64], retain_graph=True)
        close(gp, hp, what="normal_distance grad p (%g, %g)" % (a, b))
        close(gq, hq, what="normal_distance grad q (%g, %g)" % (a, b))


# ---------------------------------------------------------------------------------------------------------------------
# (e) edge loss
# ---------------------------------------------------------------------------------------------------------------------
def test_edge_loss_grid_stride_vs_fp64(lib):
    """Dense 48^3 grids: E > 10^6 directed edges, several grid-stride iterations of the forward kernel."""
    from meshrcnn_b200 import functional as F_, synthetic
    verts, vi, faces, fi, adj, _ = F_.cubify(synthetic.dense_voxels(4, 48, 3).cuda(), 0.5)
    E = adj.shape[1]
    assert E >= 1_000_000, E
    pos = (verts.cpu() * 0.05 + 0.01 * torch.randn(verts.shape, generator=_gen(4))).cuda().requires_grad_()
    loss = F_.edge_length(pos, adj)
    g, = torch.autograd.grad(loss, pos)
    p64 = pos.detach().cpu().double().requires_grad_()
    want = mesh_ops.edge_loss(p64, adj.cpu())
    close(loss, want.detach(), what="edge loss E=%d" % E)
    gw, = torch.autograd.grad(want, p64)
    close(g, gw, what="edge grad")


def test_edge_loss_without_edges(lib):
    from meshrcnn_b200 import functional as F_
    pos = torch.randn(5, 3, generator=_gen(1)).cuda().requires_grad_()
    loss = F_.edge_length(pos, torch.empty(2, 0, dtype=torch.int64, device="cuda"))
    assert float(loss.detach()) == 0.0
    loss.backward()
    torch.cuda.synchronize()
    assert float(pos.grad.abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# (f) voxel BCE
# ---------------------------------------------------------------------------------------------------------------------
SATURATED = torch.tensor([20.0, 30.0, 90.0, 17.5, -20.0, -30.0, -104.0, -120.0])


@pytest.mark.parametrize("from_logits", [True, False])
@pytest.mark.parametrize("n", [64 * 48 ** 3, 1_000_003])
def test_voxel_bce_vs_fp64(lib, n, from_logits):
    """Grid-stride loops (n >> 8 * SMs * 256), a tail that is not a multiple of 256, and saturated inputs at both ends.
    Logits: the gradient is (sigmoid(x) - t) / n, compared with fp64 BCE-with-logits -- it stays (1 - t) / n or -t / n
    where the fp32 sigmoid has saturated, whereas the reference's fp32 BCE(sigmoid(x)) gives 0 there (DESIGN.md section 2).
    Probabilities: torch's BCE backward (p - t) / max(p (1 - p), 1e-12)."""
    from meshrcnn_b200 import functional as F_
    g = _gen(n % 1000 + from_logits)
    x = torch.randn(n, generator=g) * 4
    t = (torch.rand(n, generator=g) < 0.3).float()
    s = SATURATED.shape[0]
    x[:s], x[-s:] = SATURATED, SATURATED
    t[:s], t[-s:] = 0.0, 1.0
    sat = torch.zeros(n, dtype=torch.bool)
    sat[:s], sat[-s:] = True, True
    if not from_logits:
        x = 1.0 / (1.0 + torch.exp(-x))                     # probabilities, exact 0 and 1 among them
    shape = (64, 48, 48, 48) if n == 64 * 48 ** 3 else (n,)
    xc = x.view(shape).cuda().requires_grad_()
    loss, _ = F_.voxel_bce(xc, t.view(shape).cuda(), from_logits=from_logits)
    gx, = torch.autograd.grad(loss, xc)
    gx = gx.reshape(-1).cpu()
    t64 = t.double()
    p32 = 1.0 / (1.0 + torch.exp(-x)) if from_logits else x          # the kernel's fp32 sigmoid formula
    want = torch.nn.functional.binary_cross_entropy(p32.double(), t64)
    close(loss, want, what="bce n=%d logits=%s" % (n, from_logits))
    if from_logits:
        gw = (torch.sigmoid(x.double()) - t64) / n
    else:
        x64 = x.double().requires_grad_()
        gw, = torch.autograd.grad(torch.nn.functional.binary_cross_entropy(x64, t64), x64)
    close(gx[~sat], gw[~sat], what="bce grad")
    close(gx[sat], gw[sat], what="bce grad, saturated")
    if from_logits:
        inv_n = np.float32(1.0 / n)
        pos_sat = sat & (x >= 20) & (t == 0)
        assert bool((gx[pos_sat] == float(inv_n)).all())                # (1 - 0) / n exactly
        assert bool((gx[sat & (x < -100) & (t == 1)] == -float(inv_n)).all())
        xr = x[pos_sat].clone().requires_grad_()                      # the reference's fp32 composition: zero gradient
        gr, = torch.autograd.grad(torch.nn.functional.binary_cross_entropy(torch.sigmoid(xr), t[pos_sat]), xr)
        assert float(gr.abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# (g) composed stage loss at the training shape
# ---------------------------------------------------------------------------------------------------------------------
def _rel_l2(a, b):
    return float((a - b).norm() / b.norm())


def test_mesh_loss_grads_at_training_shape_vs_fp64(lib):
    """LF.mesh_loss on B = 8 cubified and perturbed 24^3 blobs, 10 000 points, k = 10, injected draws, against the fp64
    oracle with the kernel's index sets (nearest indices verified optimal first).  Chamfer and edge vertex gradients:
    rtol 1e-4 elementwise.  Normal term: the per-point gradient (w.r.t. the predicted cloud) elementwise on the rows that no
    ill-conditioned neighbourhood and no near-zero dot product touches; the per-vertex gradient in relative L2 within
    max(1e-4, twice the oracle's own fp32-vs-fp64 gap)."""
    from oracle import cubify_np
    from meshrcnn_b200 import functional as F_, loss_functions as LF, synthetic
    from meshrcnn_b200.pipeline import MeshTargets
    B, n, k = 8, 10000, 10
    verts, vi, faces, fi, adj = cubify_np.cubify(synthetic.blob_voxels(B, 24, 0).numpy(), 0.2)
    gverts, gvi, gfaces, gfi, _ = cubify_np.cubify(synthetic.blob_voxels(B, 24, 1000).numpy(), 0.5)
    pos32 = ((torch.from_numpy(verts).double() + 0.3 * torch.randn(verts.shape, generator=_gen(5), dtype=torch.float64))
             * 0.06).float()
    gt32 = torch.cat([mesh_ops.normalize_cloud(v) for v in torch.from_numpy(gverts).double().split(gvi)]).float()
    faces_t, adj_t, gfaces_t = torch.from_numpy(faces), torch.from_numpy(adj), torch.from_numpy(gfaces)
    u, x2, x1 = synthetic.sampling_randomness(B, n, 10)
    ug, x2g, x1g = synthetic.sampling_randomness(B, n, 20)
    fp = torch.stack([mesh_ops.face_cdf_draw(v, f, u[b]) for b, (v, f) in enumerate(zip(pos32.double().split(vi), faces_t.split(fi)))])
    fg = torch.stack([mesh_ops.face_cdf_draw(v, f, ug[b]) for b, (v, f) in
                      enumerate(zip(gt32.double().split(gvi), gfaces_t.split(gfi)))])

    # CUDA: the loss API, then the same composition with the predicted cloud kept for its per-point gradient
    pos = pos32.cuda().requires_grad_()
    batch = MeshTargets(gt32.cuda(), gfaces_t.cuda(), gvi, gfi)
    rnd = (dict(face_idx=fp.cuda(), xi2=x2.cuda(), xi1=x1.cuda()), dict(face_idx=fg.cuda(), xi2=x2g.cuda(), xi1=x1g.cuda()))
    ch, nl, ed = LF.mesh_loss(pos, faces_t.cuda(), adj_t.cuda(), vi, fi, batch, float(n), k, randomness=rnd)
    g_ch, = torch.autograd.grad(ch, pos, retain_graph=True)
    g_nl, = torch.autograd.grad(nl, pos, retain_graph=True)
    g_ed, = torch.autograd.grad(ed, pos)
    cloud, _ = F_.sample_points(pos, faces_t.cuda(), vi, fi, n, **rnd[0])
    cloud.retain_grad()
    cloud_gt = LF.sample_gt_cloud(batch, n, **rnd[1])
    ch2, ip, iq, kp, kq = F_.chamfer_total(cloud, cloud_gt, k, 1.0 / n)
    nl2 = F_.normal_total(cloud, cloud_gt, kp, kq, ip, iq, -1.0 / n)
    assert abs(float(ch2) / float(ch) - 1) <= 1e-6 and abs(float(nl2) / float(nl) - 1) <= 1e-6     # fp64 atomics: order only
    nl2.backward()
    _assert_nearest(cloud, cloud_gt, ip, iq, B)
    ip, iq, kp, kq = ip.cpu().long(), iq.cpu().long(), kp.cpu().long(), kq.cpu().long()

    # fp64 oracle from the same fp32 inputs, index sets pinned to the kernel's
    def oracle(dtype):
        p_ = pos32.to(dtype).requires_grad_()
        cp = mesh_ops.batched_sample_with(p_, faces_t, vi, fi, fp, x2.to(dtype), x1.to(dtype))
        cq = mesh_ops.batched_sample_with(gt32.to(dtype), gfaces_t, gvi, gfi, fg, x2g.to(dtype), x1g.to(dtype))
        c = sum(mesh_ops.chamfer_given(cp, cq, ip, iq)) / n
        m = mesh_ops.normal_total_given(cp, cq, kp, kq, ip, iq, -1.0 / n)
        e = mesh_ops.edge_loss(p_, adj_t)
        grads = [torch.autograd.grad(t_, p_, retain_graph=True)[0] for t_ in (c, m, e)]
        return (float(c), float(m), float(e)), grads

    (c64, m64, e64), (h_ch, h_nl, h_ed) = oracle(torch.float64)
    _, (_, h_nl32, _) = oracle(torch.float32)
    rel = lambda a, b: abs(float(a) - b) / abs(b)
    assert rel(ch, c64) <= 1e-4 and rel(ed, e64) <= 1e-4 and rel(nl, m64) <= 1e-4, (float(ch), c64, float(ed), e64, float(nl), m64)
    close(g_ch, h_ch, what="chamfer vertex gradient")
    close(g_ed, h_ed, what="edge vertex gradient")
    own_gap = _rel_l2(h_nl32.double(), h_nl)
    assert _rel_l2(g_nl.cpu().double(), h_nl) <= max(1e-4, 2 * own_gap), (_rel_l2(g_nl.cpu().double(), h_nl), own_gap)

    # per-point normal term on the kernel's own cloud
    c64p = cloud.detach().cpu().double().requires_grad_()
    q64 = cloud_gt.cpu().double()
    want, = torch.autograd.grad(mesh_ops.normal_total_given(c64p, q64, kp, kq, ip, iq, -1.0 / n), c64p)
    ar = torch.arange(B).view(-1, 1)
    n_p = mesh_ops.normals_from_neighbours(c64p.detach(), kp, canonical_signs=True)
    n_q = mesh_ops.normals_from_neighbours(q64, kq, canonical_signs=True)
    ok_p, ok_q = _well_conditioned(c64p.detach(), kp), _well_conditioned(q64, kq)
    bad0 = ((n_p * n_q[ar, ip]).sum(2).abs() < 1e-5) | ~ok_p | ~ok_q[ar, ip]      # pair (i, ip[i])
    bad1 = ((n_q * n_p[ar, iq]).sum(2).abs() < 1e-5) | ~ok_q | ~ok_p[ar, iq]      # pair (iq[j], j)
    bad = bad0 | ~ok_p
    for b in range(B):
        bad[b].index_fill_(0, iq[b][bad1[b]], True)
    taint = bad.clone()
    for b in range(B):
        taint[b].index_fill_(0, kp[b][bad[b]].reshape(-1), True)
    keep = ~taint
    assert float(keep.double().mean()) > 0.9, float(keep.double().mean())
    close(cloud.grad.cpu()[keep], want[keep], what="normal term, per-point gradient")
