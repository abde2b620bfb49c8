"""TEST INFRASTRUCTURE ONLY -- CPU oracle for Cubify's opt-in watertight topology (numpy, bit-exact).

``cubify_with(probs, threshold, corners)`` is the algorithm of ``oracle/cubify_np.py`` (same occupancy test, face flags,
orders, coordinates and adjacency rule) with the quad-corner table as an argument.  With ``cubify_np.CORNERS`` it equals
``cubify_np.cubify``, which is pinned to the reference (``tests/test_cubify_watertight_cpu.py`` checks that equality);
with ``WATERTIGHT_CORNERS`` it is the executable specification of ``Cubify(topology="watertight")`` (DESIGN.md §2 item 8).

Only ``tests/`` may import this module.  The product path (``meshrcnn_b200``) never does.
"""
import numpy as np

from .cubify_np import CORNERS, TRIANGLES, EmptyGrid, face_flags, occupancy

# Watertight topology: every quad lies on the side of the empty neighbour, its corners are in cyclic order starting at the
# quad's lowest lattice corner, and (c1-c0) x (c2-c0) points toward the empty neighbour.  With the same TRIANGLES the quad is
# split along its c0-c2 diagonal, both triangles wound outward, so the triangles of a mesh form a closed, consistently
# oriented surface (voxels that touch only along an edge or at a vertex stay non-manifold there).
WATERTIGHT_CORNERS = np.array([
    [(0, 0, 0), (0, 0, 1), (0, 1, 1), (0, 1, 0)],   # 0 (z-1 empty) plane z-1/2
    [(1, 0, 0), (1, 1, 0), (1, 1, 1), (1, 0, 1)],   # 1 (z+1 empty) plane z+1/2
    [(0, 1, 0), (0, 1, 1), (1, 1, 1), (1, 1, 0)],   # 2 (y+1 empty) plane y+1/2
    [(0, 0, 0), (1, 0, 0), (1, 0, 1), (0, 0, 1)],   # 3 (y-1 empty) plane y-1/2
    [(0, 0, 0), (0, 1, 0), (1, 1, 0), (1, 0, 0)],   # 4 (x-1 empty) plane x-1/2
    [(0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)],   # 5 (x+1 empty) plane x+1/2
], dtype=np.int64)

TOPOLOGIES = {"reference": CORNERS, "watertight": WATERTIGHT_CORNERS}


def cubify(probs: np.ndarray, threshold: float = 0.5, topology: str = "reference"):
    """``Cubify(threshold, topology=topology).forward`` -> (verts, v_index, faces, f_index, adj), see ``cubify_with``."""
    if topology not in TOPOLOGIES:
        raise ValueError("cubify: topology must be one of %s, got %r" % (tuple(TOPOLOGIES), topology))
    return cubify_with(probs, threshold, TOPOLOGIES[topology])


def cubify_with(probs: np.ndarray, threshold: float, corners: np.ndarray):
    """Returns (verts float32 [SV,3], v_index list, faces int64 [SF,3] per-mesh-local, f_index list, adj int64 [2,E]
    global) for the quad corners ``corners`` (6 x 4 x 3 lattice offsets in (z, y, x)).  Orders: vertices by (b,z,y,x);
    faces by (b,dir,z,y,x), two per quad; adjacency by (row,col); lists truncated after the last non-empty mesh."""
    occ = occupancy(probs, threshold)
    B, Z, Y, X = occ.shape
    b_i, d_i, z_i, y_i, x_i = np.nonzero(face_flags(occ))          # C order == (b, dir, z, y, x)
    if b_i.shape[0] == 0:
        raise EmptyGrid("empty grid")

    LZ, LY, LX = Z + 1, Y + 1, X + 1
    corner = np.asarray(corners, dtype=np.int64)[d_i]               # (N,4,3)
    cz = z_i[:, None] + corner[:, :, 0]
    cy = y_i[:, None] + corner[:, :, 1]
    cx = x_i[:, None] + corner[:, :, 2]
    lin = ((b_i[:, None] * LZ + cz) * LY + cy) * LX + cx             # (N,4) lattice linear ids

    used = np.zeros(B * LZ * LY * LX, dtype=bool)
    used[lin.ravel()] = True
    rank = np.cumsum(used, dtype=np.int64) - 1                       # vertex id = lexicographic rank of the lattice point
    ids = np.nonzero(used)[0]
    vb = ids // (LZ * LY * LX)
    rem = ids % (LZ * LY * LX)
    fz = (rem // (LY * LX)).astype(np.float32) - np.float32(0.5)
    fy = ((rem // LX) % LY).astype(np.float32) - np.float32(0.5)
    fx = (rem % LX).astype(np.float32) - np.float32(0.5)
    verts = np.stack([fz, fx, -fy], axis=1).astype(np.float32)      # (z,y,x) -> (z,x,-y)

    v_counts = np.bincount(vb)
    f_counts = np.bincount(b_i) * 2
    g = rank[lin]                                                    # (N,4) global vertex ids
    tri = np.stack([g[:, TRIANGLES[0]], g[:, TRIANGLES[1]]], axis=1).reshape(-1, 3)
    v_off = np.zeros(B, dtype=np.int64)
    v_off[:len(v_counts)] = np.concatenate([[0], np.cumsum(v_counts)])[:-1]
    faces = tri - v_off[np.repeat(b_i, 2)][:, None]                  # per-mesh local ids

    rows = np.concatenate([tri[:, 0], tri[:, 1], tri[:, 0], tri[:, 1], tri[:, 2], tri[:, 2]])
    cols = np.concatenate([tri[:, 1], tri[:, 2], tri[:, 2], tri[:, 0], tri[:, 1], tri[:, 0]])
    nv = ids.shape[0]
    key = np.unique(rows * nv + cols)
    adj = np.stack([key // nv, key % nv]).astype(np.int64)
    return verts, [int(c) for c in v_counts], faces.astype(np.int64), [int(c) for c in f_counts], adj
