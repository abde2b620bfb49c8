"""Watertight Cubify topology (opt-in, DESIGN.md §2 item 8): the oracle's known answers and closed-surface invariants, and
the lattice-mask / corner tables of csrc/cubify.cu derived from the oracle's tables.  CPU only."""
import os
import re

import numpy as np
import pytest

from oracle import cubify_np, cubify_watertight as cw

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUBIFY_CU = os.path.join(ROOT, "mesh_r-cnn_computer_vision_project_b200", "csrc", "cubify.cu")
CASES = ["rand10", "ragged", "empty_mid_tail", "single_voxel", "solid3", "at_threshold", "blob16", "dense24"]


def _grid(shape, cells):
    t = np.zeros(shape, np.float32)
    for c in cells:
        t[c] = 1.0
    return t


def _quad_dirs(probs, th):
    """Direction of every face, in the oracle's (b, dir, z, y, x) face order (two triangles per quad)."""
    flags = cubify_np.face_flags(cubify_np.occupancy(probs, th))
    return np.repeat(np.nonzero(flags)[1], 2)


def _outward_normals(dirs):
    """Axis normal of each face's direction in the output frame: (dz, dy, dx) rotated (z, y, x) -> (z, x, -y)."""
    n = cubify_np.NEIGHBOUR[dirs]
    return np.stack([n[:, 0], n[:, 2], -n[:, 1]], 1).astype(np.float64)


def mesh_report(verts, faces):
    """Closed-surface figures of one mesh (local face ids): fp64 signed volume, unbalanced directed half-edges (a
    half-edge u->w whose reverse w->u has a different multiplicity), duplicate faces (as vertex sets), total area,
    undirected edge count and the per-face cross products (v1 - v0) x (v2 - v0)."""
    v = verts.astype(np.float64)
    tri = v[faces]
    cross = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    volume = float(np.einsum("ij,ij->i", tri[:, 0], np.cross(tri[:, 1], tri[:, 2])).sum() / 6.0)
    n = max(int(verts.shape[0]), 1)
    u = faces.reshape(-1)
    w = faces[:, [1, 2, 0]].reshape(-1)
    keys, cnt = np.unique(u * n + w, return_counts=True)
    rev = (keys % n) * n + keys // n
    pos = np.searchsorted(keys, rev)
    found = (pos < keys.shape[0]) & (keys[np.minimum(pos, keys.shape[0] - 1)] == rev)
    rcnt = np.where(found, cnt[np.minimum(pos, keys.shape[0] - 1)], 0)
    und = np.unique(np.minimum(u, w) * n + np.maximum(u, w))
    return {"volume": volume, "unbalanced": int((rcnt != cnt).sum()),
            "duplicates": int(faces.shape[0] - np.unique(np.sort(faces, 1), axis=0).shape[0]),
            "area": float(0.5 * np.linalg.norm(cross, axis=1).sum()), "edges": int(und.shape[0]), "cross": cross}


def check_watertight(probs, th):
    """Every invariant of the watertight mode, per mesh, against the reference mode's face counts."""
    probs = np.asarray(probs, np.float32)
    verts, vi, faces, fi, adj = cw.cubify(probs, th, topology="watertight")
    ref = cubify_np.cubify(probs, th)
    assert fi == ref[3]                                   # same face flags => same face counts and truncation
    assert faces.shape == ref[2].shape
    occ = cubify_np.occupancy(probs, th)
    exposed = cubify_np.face_flags(occ).sum(axis=(1, 2, 3, 4))
    normals = _outward_normals(_quad_dirs(probs, th))
    vo, fo = 0, 0
    for b, (nv, nf) in enumerate(zip(vi, fi)):
        f = faces[fo:fo + nf]
        assert nf == 0 or (f.min() >= 0 and f.max() < nv)
        r = mesh_report(verts[vo:vo + nv], f)
        assert r["volume"] == float(occ[b].sum()), (b, r["volume"], int(occ[b].sum()))
        assert r["unbalanced"] == 0 and r["duplicates"] == 0, b
        assert r["area"] == float(exposed[b])
        assert np.array_equal(r["cross"], normals[fo:fo + nf])
        vo, fo = vo + nv, fo + nf
    assert vo == verts.shape[0] and fo == faces.shape[0]
    # adjacency: sorted, symmetric, no self loops, at most 18 neighbours per vertex (csrc/cubify.cu ADJ_CAP)
    key = adj[0] * verts.shape[0] + adj[1]
    assert (key[1:] > key[:-1]).all() and (adj[0] != adj[1]).all()
    assert np.array_equal(np.sort(adj[1] * verts.shape[0] + adj[0]), key)
    assert np.bincount(adj[0]).max() <= 18
    return verts, vi, faces, fi, adj


# ---------------------------------------------------------------------------------------------------------------
def test_one_voxel():
    t = _grid((1, 3, 3, 3), [(0, 1, 1, 1)])
    verts, vi, faces, fi, adj = check_watertight(t, 0.5)
    r = mesh_report(verts, faces)
    assert (vi, fi, r["edges"], adj.shape[1], r["volume"]) == ([8], [12], 18, 36, 1.0)


def test_two_voxels_stacked_in_y():
    t = _grid((1, 3, 4, 3), [(0, 1, 1, 1), (0, 1, 2, 1)])
    verts, vi, faces, fi, adj = check_watertight(t, 0.5)
    r = mesh_report(verts, faces)
    assert (vi, fi, r["edges"], r["volume"], r["duplicates"]) == ([12], [20], 30, 2.0, 0)
    ref = cubify_np.cubify(t, 0.5)
    assert mesh_report(ref[0], ref[2])["duplicates"] == 2         # what the reference placement does here


def test_two_voxels_sharing_only_an_edge():
    t = _grid((1, 4, 4, 4), [(0, 1, 1, 1), (0, 2, 2, 1)])
    verts, vi, faces, fi, adj = check_watertight(t, 0.5)
    r = mesh_report(verts, faces)
    assert (vi, fi, r["edges"], r["volume"]) == ([14], [24], 35, 2.0)


def test_triangle_normals_are_the_outward_axis_normals():
    t = _grid((1, 3, 3, 3), [(0, 1, 1, 1)])
    verts, _, faces, _, _ = cw.cubify(t, 0.5, topology="watertight")
    cross = mesh_report(verts, faces)["cross"]
    centre = verts.astype(np.float64).mean(0)
    tri_c = verts[faces].astype(np.float64).mean(1)
    assert np.array_equal(np.abs(cross).sum(1), np.ones(12))             # unit axis vectors
    assert ((tri_c - centre) * cross).sum(1).min() > 0                    # pointing away from the cube's centre
    assert np.array_equal(cross, _outward_normals(np.repeat(np.arange(6), 2)))


@pytest.mark.parametrize("kind,B,V,th,seed", [("blob", 4, 24, 0.2, 0), ("blob", 3, 16, 0.5, 7), ("dense", 2, 16, 0.5, 0),
                                              ("dense", 3, 9, 0.8, 4), ("dense", 2, 12, 0.2, 9)])
def test_invariants_on_seeded_grids(kind, B, V, th, seed):
    from meshrcnn_b200 import synthetic
    t = (synthetic.blob_voxels(B, V, seed) if kind == "blob" else synthetic.dense_voxels(B, V, seed)).numpy()
    check_watertight(t, th)


@pytest.mark.parametrize("name", CASES)
def test_invariants_on_golden_inputs(golden, name):
    """Empty middle / tail meshes (truncated lists), voxels on the grid border, p == threshold (empty: strict >)."""
    g = golden("cubify_cases")
    check_watertight(g[name + "__in"], float(g[name + "__th"]))


def test_ragged_batch_meshes_equal_their_single_mesh_runs():
    from meshrcnn_b200 import synthetic
    t = synthetic.dense_voxels(4, 10, 2).numpy()
    t[1] = 0.0                                                           # an empty mesh in the middle
    verts, vi, faces, fi, adj = check_watertight(t, 0.6)
    vo = fo = 0
    for b in range(len(vi)):
        if fi[b] == 0:
            assert vi[b] == 0
            continue
        one = cw.cubify(t[b:b + 1], 0.6, topology="watertight")
        assert np.array_equal(verts[vo:vo + vi[b]], one[0]) and np.array_equal(faces[fo:fo + fi[b]], one[2])
        sel = (adj[0] >= vo) & (adj[0] < vo + vi[b])
        assert np.array_equal(adj[:, sel] - vo, one[4])
        vo, fo = vo + vi[b], fo + fi[b]


@pytest.mark.parametrize("name", CASES)
def test_reference_corners_reproduce_the_pinned_oracle(golden, name):
    """cubify_with(..., CORNERS) is cubify_np.cubify (pinned to the reference's outputs), so the two topologies differ in
    the corner table only."""
    g = golden("cubify_cases")
    t, th = g[name + "__in"], float(g[name + "__th"])
    if not cubify_np.occupancy(t, th).any():
        return
    got, want = cw.cubify_with(t, th, cubify_np.CORNERS), cubify_np.cubify(t, th)
    assert got[1] == want[1] and got[3] == want[3]
    for i in (0, 2, 4):
        assert got[i].dtype == want[i].dtype and np.array_equal(got[i], want[i])


def test_empty_grid_and_bad_topology():
    with pytest.raises(ValueError, match="empty grid"):
        cw.cubify(np.zeros((2, 3, 3, 3), np.float32), 0.5, topology="watertight")
    with pytest.raises(ValueError, match="topology"):
        cw.cubify(np.ones((1, 2, 2, 2), np.float32), 0.5, topology="closed")


# ---------------------------------------------------------------------------------------------------------------
# csrc/cubify.cu tables vs the oracle
def lattice_mask_table(corners):
    """kLatMask rule: for corner s = cz<<2|cy<<1|cx of a direction-d quad, OR bit (dz+1)*9+(dy+1)*3+(dx+1) for every
    triangle edge leaving that corner (both orientations of each edge of TRIANGLES)."""
    edges = set()
    for tri in cubify_np.TRIANGLES:
        for i in range(3):
            a, b = tri[i], tri[(i + 1) % 3]
            edges |= {(a, b), (b, a)}
    T = np.zeros((8, 6), np.int64)
    for d in range(6):
        for a, b in edges:
            ca, cb = corners[d][a], corners[d][b]
            dz, dy, dx = cb - ca
            T[ca[0] * 4 + ca[1] * 2 + ca[2], d] |= 1 << int((dz + 1) * 9 + (dy + 1) * 3 + (dx + 1))
    return T


def _cu_table(src, decl, rows, cols):
    block = src[src.index(decl):]
    block = block[block.index("=") + 1:block.index(";")]
    vals = [int(v, 0) for v in re.findall(r"0x[0-9a-fA-F]+|\d+", block.replace("u}", "}").replace("u,", ","))]
    assert len(vals) == rows * cols, decl
    return np.array(vals, np.int64).reshape(rows, cols)


@pytest.mark.parametrize("decl,topology", [("kLatMask[8][6]", "reference"), ("kLatMaskWT[8][6]", "watertight")])
def test_cuda_lattice_masks_derive_from_the_oracle_tables(decl, topology):
    src = open(CUBIFY_CU).read()
    assert np.array_equal(_cu_table(src, decl, 8, 6), lattice_mask_table(cw.TOPOLOGIES[topology]))


@pytest.mark.parametrize("decl,topology", [("constexpr int T[6][4]", "reference"), ("constexpr int W[6][4]", "watertight")])
def test_cuda_corner_ids_match_the_oracle_tables(decl, topology):
    src = open(CUBIFY_CU).read()
    c = cw.TOPOLOGIES[topology]
    assert np.array_equal(_cu_table(src, decl, 6, 4), c[:, :, 0] * 4 + c[:, :, 1] * 2 + c[:, :, 2])


def test_watertight_corner_table_follows_the_spec():
    """Quad on the empty neighbour's side, c0 the lowest corner, cyclic (unit sides), (c1-c0) x (c2-c0) outward."""
    for d, n in enumerate(cubify_np.NEIGHBOUR):
        c = cw.WATERTIGHT_CORNERS[d]
        ax = int(np.nonzero(n)[0][0])
        assert (c[:, ax] == (1 if n[ax] > 0 else 0)).all()
        assert tuple(c[0]) == min(map(tuple, c))
        assert all(np.abs(c[(i + 1) % 4] - c[i]).sum() == 1 for i in range(4))
        assert np.array_equal(np.cross(c[1] - c[0], c[2] - c[0]), n)
