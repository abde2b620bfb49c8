"""The index-given fp64 loss helpers of ``oracle/mesh_ops.py`` (``chamfer_given``, ``normal_total_given``,
``normals_conditioning``, ``nearest_chunked``) against the dense oracle they stand in for at small sizes, so the O(n) oracle
the GPU gradient tests use at the trained shape is itself pinned to the one ``oracle/make_golden.py`` checks against the
reference.  CPU only."""
import torch

from oracle import mesh_ops


def _clouds(B, P, Q, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(B, P, 3, generator=g, dtype=torch.float64) - 0.5,
            torch.rand(B, Q, 3, generator=g, dtype=torch.float64) * 0.8 - 0.3)


def test_chamfer_given_equals_dense_chamfer_values_and_grads():
    p, q = _clouds(3, 41, 67, 0)
    p.requires_grad_()
    q.requires_grad_()
    l1, i1, l2, i2 = mesh_ops.chamfer(mesh_ops.p2p_distance(p, q))
    gp, gq = torch.autograd.grad(0.7 * l1 + 1.3 * l2, [p, q])
    w1, w2 = mesh_ops.chamfer_given(p, q, i1, i2)
    hp, hq = torch.autograd.grad(0.7 * w1 + 1.3 * w2, [p, q])
    assert torch.allclose(w1, l1, rtol=1e-12) and torch.allclose(w2, l2, rtol=1e-12)
    assert torch.allclose(hp, gp, rtol=1e-9, atol=1e-12) and torch.allclose(hq, gq, rtol=1e-9, atol=1e-12)


def test_normal_total_given_equals_dense_normal_distance():
    B, P, k = 2, 60, 6
    p, q = _clouds(B, P, P, 1)
    p.requires_grad_()
    d = mesh_ops.p2p_distance(p, q)
    _, i1, _, i2 = mesh_ops.chamfer(d)
    kp, kq = mesh_ops.knn_indices(d, k), mesh_ops.knn_indices(d.transpose(1, 2), k)
    for canon in (True, False):
        l0, l1 = mesh_ops.normal_distance(p, q, d, i1, i2, k, canonical_signs=canon)
        want = -(l0 + l1) / 100.0
        got = mesh_ops.normal_total_given(p, q, kp, kq, i1, i2, -1.0 / 100.0, canonical_signs=canon)
        assert torch.allclose(got, want, rtol=1e-12)
        gw, = torch.autograd.grad(want, p)
        gg, = torch.autograd.grad(got, p)
        assert torch.allclose(gg, gw, rtol=1e-9, atol=1e-12)
        s0, s1 = mesh_ops.normal_sums_given(p, q, kp, kq, i1, i2, canon)
        assert torch.allclose(s0, l0, rtol=1e-12) and torch.allclose(s1, l1, rtol=1e-12)


def test_given_helpers_reproduce_mesh_loss_with():
    """chamfer / normal terms of the dense ``mesh_loss_with`` from the given-index helpers on its own clouds and indices."""
    g = torch.Generator().manual_seed(2)
    verts = torch.rand(12, 3, generator=g, dtype=torch.float64) * 3
    faces = torch.tensor([[0, 1, 2], [2, 3, 4], [4, 5, 0], [1, 3, 5], [6, 7, 8], [8, 9, 10], [10, 11, 6]])
    adj = torch.tensor([[0, 1, 2, 6, 7], [1, 2, 0, 7, 8]])
    vi, fi, n, k = [6, 6], [4, 3], 80, 5
    faces = torch.cat([faces[:4], faces[4:] - 6])
    draws = lambda s: (torch.stack([torch.randint(0, c, (n,), generator=g) for c in fi]),
                       torch.rand(2, n, generator=g, dtype=torch.float64), torch.rand(2, n, generator=g, dtype=torch.float64))
    rp, rg = draws(0), draws(1)
    ch, nl, e, aux = mesh_ops.mesh_loss_with(verts, faces, adj, vi, fi, verts, faces, vi, fi, rp, rg, float(n), k,
                                             canonical_signs=True)
    cp, cq, ip, iq = aux["cloud_pred"], aux["cloud_gt"], aux["idx_p"], aux["idx_gt"]
    d = mesh_ops.p2p_distance(cp, cq)
    kp, kq = mesh_ops.knn_indices(d, k), mesh_ops.knn_indices(d.transpose(1, 2), k)
    w1, w2 = mesh_ops.chamfer_given(cp, cq, ip, iq)
    assert torch.allclose((w1 + w2) / n, ch, rtol=1e-12)
    assert torch.allclose(mesh_ops.normal_total_given(cp, cq, kp, kq, ip, iq, -1.0 / n), nl, rtol=1e-12)


def test_nearest_chunked_equals_dense_min():
    p, q = _clouds(2, 300, 170, 3)
    want = mesh_ops.p2p_distance(p, q).min(2).values.clamp_min(0)
    for rows in (7, 64, 1024):
        got = mesh_ops.nearest_chunked(p.float(), q.float(), rows=rows)
        ref = mesh_ops.p2p_distance(p.float().double(), q.float().double()).min(2).values
        assert torch.allclose(got, ref, rtol=1e-10, atol=1e-14)
    assert torch.allclose(mesh_ops.nearest_chunked(p, q), want, rtol=1e-10, atol=1e-14)


def test_normals_conditioning_known_spectra():
    """Axis-aligned neighbourhoods with known scatter matrices: the relative gap and the sign-rule margins."""
    e = torch.eye(3, dtype=torch.float64)
    aniso = torch.cat([e * torch.tensor([1.0, 0.5, 0.25], dtype=torch.float64).view(3, 1),
                       -e * torch.tensor([1.0, 0.5, 0.25], dtype=torch.float64).view(3, 1)])     # S = diag(2, 0.5, 0.125)
    iso = torch.cat([e * 0.5, -e * 0.5])                                                              # S = 0.5 I
    flat = torch.tensor([[1.0, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 0], [0, 0, 0]], dtype=torch.float64)
    pt = torch.cat([aniso, iso + 3.0, flat - 2.0]).unsqueeze(0)                                       # 18 points
    nn = torch.stack([torch.arange(6), torch.arange(6, 12), torch.arange(12, 18)]).unsqueeze(0)      # 3 rows, k = 6
    gap, m20, m1, mdet = mesh_ops.normals_conditioning(pt, nn)
    assert abs(float(gap[0, 0]) - (0.5 - 0.125) / 2.0) < 1e-12          # min(1.5, 0.375) / 2
    assert float(gap[0, 1]) < 1e-12                                      # isotropic: fully degenerate
    assert float(gap[0, 2]) < 1e-12                                      # square planar patch: degenerate in-plane pair
    assert torch.allclose(mdet, torch.ones_like(mdet))
    # row 0: V = permutation of the axes (w ascending: z, y, x), so V[2,0] = 1 and column 1 (= +-e_y) has margin 1
    assert abs(float(m20[0, 0]) - 1.0) < 1e-12 and abs(float(m1[0, 0]) - 1.0) < 1e-12
