"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the floating-point half of the hot path (torch on CPU).

A restatement of the reference's *arithmetic* for VertexAlign, GraphConv / ResGraphConv, the three
refinement-stage classes, surface sampling, and the chamfer / normal / edge losses.  Every function cites the
reference lines it follows.  All functions are dtype-agnostic: run them with float64 inputs to obtain the
arbiter the fp32 CUDA kernels are compared with (the reference disagrees with itself fp32-vs-fp64 by more
than the kernels do, SURVEY.md section 7), and with float32 inputs to time the reference's CPU algorithm
(dense P x Q distance matrices, ``topk``, LAPACK ``eigh``) for ``bench.py``'s cpu_baseline.

Gradients come from torch autograd over this restatement (same graph as the reference's).

Parity pin: ``oracle/make_golden.py`` runs the *unmodified* reference (``oracle/ref_import.py``) and this file on
the same seeded inputs in the dev container and asserts agreement; its outputs are committed as
``tests/golden/*.npz`` and re-checked on every CPU test run (``tests/test_oracle_golden.py``).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs may
import this module.
"""
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor


# ----------------------------------------------------------------------------------------------------------
# VertexAlign  (meshRCNN/layers.py:509-613)
# ----------------------------------------------------------------------------------------------------------
def _project_one_map(fmap: Tensor, h: Tensor, w: Tensor, size: Tuple[int, int]) -> Tensor:
    """layers.py:572-613.  ``fmap`` is C x size_y x size_x; h, w are clamped pixel coordinates."""
    size_y, size_x = fmap.shape[-2:]
    H, W = size
    x = w / (float(W) / size_x)                      # :577  (python-double divisor applied to the tensor)
    y = h / (float(H) / size_y)                      # :578
    x_lo, x_hi = torch.floor(x).long(), torch.ceil(x).long()
    y_lo, y_hi = torch.floor(y).long(), torch.ceil(y).long()
    x_hi = x_hi.clamp(max=size_x - 1)                # :583
    y_hi = y_hi.clamp(max=size_y - 1)                # :584
    xi, yi = x.long(), y.long()                      # :592 -- integer cast kills the fractional weights
    corners = ((x_lo, y_lo, (x_hi - xi) * (y_hi - yi)),     # :594
               (x_lo, y_hi, (x_hi - xi) * (yi - y_lo)),     # :598
               (x_hi, y_lo, (xi - x_lo) * (y_hi - yi)),     # :602
               (x_hi, y_hi, (xi - x_lo) * (yi - y_lo)))     # :606
    out = None
    for a, b, wt in corners:
        # NB: the x-derived index addresses the H axis and the y-derived one the W axis (:587-590)
        term = fmap[:, a, b].t() * wt.to(fmap.dtype).unsqueeze(1)
        out = term if out is None else out + term
    return out


def vert_align(img_features: Sequence[Tensor], vertex_positions: Tensor, vertices_per_mesh: List[int],
               image_sizes: Sequence[Tuple[int, int]], mesh_index: List[int]) -> Tensor:
    """layers.py:521-570.  Returns SV x sum(C_m)."""
    chunks = vertex_positions.split(list(vertices_per_mesh))
    rows = []
    k = 0
    for img, (n_mesh, size) in enumerate(zip(mesh_index, image_sizes)):
        for pos in chunks[k:k + n_mesh]:
            h = 248 * (pos[:, 1] / pos[:, 2]) + 111.5           # :557
            w = 248 * (pos[:, 0] / -pos[:, 2]) + 111.5          # :558
            H, W = size
            h = h.clamp(min=0, max=H - 1)                       # :561
            w = w.clamp(min=0, max=W - 1)                       # :562
            rows.append(torch.cat([_project_one_map(f[img], h, w, size) for f in img_features], dim=1))
        k += n_mesh
    return torch.cat(rows, dim=0)


# ----------------------------------------------------------------------------------------------------------
# GraphConv  (meshRCNN/layers.py:25-100, meshRCNN/utils.py:52-57)
# ----------------------------------------------------------------------------------------------------------
def aggregate_neighbours(index: Tensor, matrix: Tensor) -> Tensor:
    """utils.py:52-57: out[row] += matrix[col] over the COO edge list."""
    row, col = index[0], index[1]
    out = torch.zeros_like(matrix)
    return out.index_add(0, row, matrix[col])


def graph_conv(x: Tensor, adj: Tensor, w0: Tensor, w1: Tensor) -> Tensor:
    """layers.py:47-68: relu(x W0 + A (x W1)); weights are stored in x out; ReLU always applied."""
    return torch.relu(x @ w0 + aggregate_neighbours(adj, x @ w1))


def res_graph_conv(x: Tensor, adj: Tensor, sd: Dict[str, Tensor], prefix: str) -> Tensor:
    """layers.py:88-100.  ``projection.weight`` (out x in, nn.Linear) exists iff in != out."""
    key = prefix + "projection.weight"
    skip = x @ sd[key].t() if key in sd else x
    y = graph_conv(x, adj, sd[prefix + "conv0.w0"], sd[prefix + "conv0.w1"])
    y = graph_conv(y, adj, sd[prefix + "conv1.w0"], sd[prefix + "conv1.w1"])
    return skip + y


def _stage_input(pos: Tensor, projected: Tensor, feats: Optional[Tensor]) -> Tensor:
    parts = [pos, projected]
    if feats is not None:
        parts = [feats] + parts
    return torch.cat(parts, dim=1)


def stage_res_shapenet(sd, v_index, fmaps, adj, pos, sizes, feats=None, mesh_index=None):
    """ResVertixRefineShapenet.forward, layers.py:130-178."""
    mesh_index = mesh_index or [1] * len(sizes)
    aligned = vert_align(fmaps, pos, v_index, sizes, mesh_index)
    x = _stage_input(pos, aligned @ sd["linear.weight"].t(), feats)
    x = res_graph_conv(x, adj, sd, "resGraphConv0.")
    x = res_graph_conv(x, adj, sd, "resGraphConv1.")
    x = res_graph_conv(x, adj, sd, "resGraphConv2.")
    delta = torch.tanh(graph_conv(x, adj, sd["graphConv.w0"], sd["graphConv.w1"]))   # tanh(relu(.)), :174-175
    return pos + delta, x


def stage_shapenet(sd, v_index, fmaps, adj, pos, sizes, feats=None, mesh_index=None):
    """VertixRefineShapeNet.forward, layers.py:207-259."""
    mesh_index = mesh_index or [1] * len(sizes)
    aligned = vert_align(fmaps, pos, v_index, sizes, mesh_index)
    x = _stage_input(pos, aligned @ sd["linear0.weight"].t(), feats)
    x = graph_conv(x, adj, sd["graphConv0.w0"], sd["graphConv0.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv1.w0"], sd["graphConv1.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv2.w0"], sd["graphConv2.w1"])
    delta = torch.tanh(x @ sd["linear1.weight"].t())
    return pos + delta, x


def stage_pix3d(sd, v_index, fmap, adj, pos, sizes, feats=None, mesh_index=None):
    """VertixRefinePix3D.forward, layers.py:289-339."""
    mesh_index = mesh_index or [1] * len(sizes)
    aligned = vert_align([fmap], pos, v_index, sizes, mesh_index)
    x = _stage_input(pos, aligned, feats)
    x = graph_conv(x, adj, sd["graphConv0.w0"], sd["graphConv0.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv1.w0"], sd["graphConv1.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv2.w0"], sd["graphConv2.w1"])
    delta = torch.tanh(torch.cat([pos, x], 1) @ sd["linear.weight"].t())
    return pos + delta, x


STAGES = {"ResVertixRefineShapenet": stage_res_shapenet, "VertixRefineShapeNet": stage_shapenet,
          "VertixRefinePix3D": stage_pix3d}


# ----------------------------------------------------------------------------------------------------------
# surface sampling  (utils/mesh_sampling.py:6-57, utils/process.py:7-20)
# ----------------------------------------------------------------------------------------------------------
def surface_areas(verts: Tensor, faces: Tensor) -> Tensor:
    """mesh_sampling.py:39-57: |AB x AC| / 2."""
    tri = verts[faces]
    n = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0], dim=1)
    return n.norm(p=2, dim=1) / 2


def normalize_cloud(pts: Tensor) -> Tensor:
    """process.py:11-20: centre; if any |coord| > 1, divide by the largest row L2 norm."""
    c = pts - pts.mean(0)
    if c.abs().max() <= 1:
        return c
    return c / torch.sqrt((c * c).sum(1).max())


def sample_raw_with(verts: Tensor, faces: Tensor, face_idx: Tensor, xi2: Tensor, xi1: Tensor) -> Tensor:
    """mesh_sampling.py:18-35 with the three random draws injected: ``face_idx`` (= multinomial, :16),
    ``xi2`` (= first rand, :20), ``xi1`` (= second rand, before the sqrt, :21); the points before normalisation."""
    tri = verts[faces[face_idx]]                       # n x 3 x 3
    r = xi1.sqrt()
    w = torch.stack([1.0 - r, (1 - xi2) * r, xi2 * r], dim=1).to(verts.dtype)
    return (tri * w.unsqueeze(2)).sum(1)


def sample_with(verts: Tensor, faces: Tensor, face_idx: Tensor, xi2: Tensor, xi1: Tensor) -> Tensor:
    """``sample_raw_with`` normalised into the unit ball (mesh_sampling.py:6-35)."""
    return normalize_cloud(sample_raw_with(verts, faces, face_idx, xi2, xi1))


def face_cdf_draw(verts: Tensor, faces: Tensor, u: Tensor) -> Tensor:
    """Inverse-CDF draw of faces proportional to area (the distribution mesh_sampling.py:13-16 samples from):
    index of the first face whose inclusive cumulative area exceeds u * total."""
    cdf = torch.cumsum(surface_areas(verts, faces).double(), 0)
    return torch.searchsorted(cdf, u.double() * cdf[-1], right=True).clamp(max=faces.shape[0] - 1)


def batched_sample_with(verts, faces, v_index, f_index, face_idx, xi2, xi1) -> Tensor:
    """loss_functions.py:80-89; face_idx/xi2/xi1 are B x n."""
    clouds = [sample_with(v, f, face_idx[b], xi2[b], xi1[b])
              for b, (v, f) in enumerate(zip(verts.split(list(v_index)), faces.split(list(f_index))))]
    return torch.stack(clouds)


# ----------------------------------------------------------------------------------------------------------
# losses  (meshRCNN/loss_functions.py)
# ----------------------------------------------------------------------------------------------------------
def p2p_distance(a: Tensor, b: Optional[Tensor] = None) -> Tensor:
    """loss_functions.py:192-220: |a_i|^2 + |b_j|^2 - 2 a_i.b_j, batched (dense B x P x Q)."""
    if a.ndim == 2:
        a = a.unsqueeze(0)
    if b is None:
        b = a
    elif b.ndim == 2:
        b = b.unsqueeze(0)
    ra = (a * a).sum(2)
    rb = (b * b).sum(2)
    return ra.unsqueeze(2) + rb.unsqueeze(1) - 2 * torch.bmm(a, b.transpose(1, 2))


def chamfer(d: Tensor):
    """loss_functions.py:93-102."""
    m1, i1 = d.min(2)
    m2, i2 = d.min(1)
    return m1.sum(), i1, m2.sum(), i2


def edge_loss(pos: Tensor, adj: Tensor) -> Tensor:
    """loss_functions.py:47-48,175-189: mean over the directed edge list of |v_r - v_c|^2, taken from the dense
    SV x SV matrix in the reference; evaluated per edge here with the same |x|^2+|y|^2-2xy expression."""
    r, c = adj[0], adj[1]
    sq = (pos * pos).sum(1)
    d = sq[r] + sq[c] - 2 * (pos[r] * pos[c]).sum(1)
    return d.sum() / d.shape[0]


def knn_indices(d: Tensor, k: int) -> Tensor:
    """loss_functions.py:141."""
    return d.topk(k, dim=2, largest=False, sorted=False).indices


def canonical_eigvec_signs(v: Tensor) -> Tensor:
    """Sign convention of the CUDA kernel (DESIGN.md, 'normal loss'): returns a +-1 tensor (... x 1 x 3) to
    multiply the eigenvector *columns* with, such that (i) V[2,0] >= 0, (ii) the largest-|.| component of
    column 1 is > 0 (first such component on ties), (iii) det V = +1.  LAPACK's own choice is unspecified
    (MKL satisfies (i) and (iii); its column-1 sign follows no closed rule), and the reference's 'normal'
    -- a *row* of V, see below -- is not invariant under it."""
    vd = v.detach()
    s0 = torch.where(vd[..., 2, 0] < 0, -1.0, 1.0)
    c1 = vd[..., :, 1]
    big = c1.gather(-1, c1.abs().argmax(-1, keepdim=True)).squeeze(-1)
    s1 = torch.where(big < 0, -1.0, 1.0)
    signs = torch.stack([s0, s1, torch.ones_like(s0)], dim=-1).to(v.dtype)
    det = torch.linalg.det(vd * signs.unsqueeze(-2))
    signs[..., 2] = torch.where(det < 0, -1.0, 1.0).to(v.dtype)
    return signs.unsqueeze(-2)


def normals_from_neighbours(pt: Tensor, nn_idx: Tensor, canonical_signs: bool = False) -> Tensor:
    """loss_functions.py:146-170: gather ``pt`` rows at ``nn_idx`` (B x P x k), centre, 3x3 scatter matrix
    S = Y^T Y, ``symeig`` (upper == eigh UPLO='U', eigenvalues ascending, eigenvectors in columns).

    NB (reference quirk, :165-168): ``eigen_vectors[b, p, argmin]`` indexes the *row* dimension of V, so the
    'normal' is row ``argmin(eigenvalues)`` (= row 0) of V, i.e. (v0[0], v1[0], v2[0]) -- the first
    component of each eigenvector -- not the eigenvector of the smallest eigenvalue.  It is a unit vector,
    but each component inherits the arbitrary sign of a different eigenvector, so |n_p . n_q| depends on the
    eigensolver's sign choices.  ``canonical_signs=True`` re-signs the columns with
    :func:`canonical_eigvec_signs` (the convention the CUDA kernel implements) before the row is taken."""
    B, P, _ = pt.shape
    nb = pt[torch.arange(B).view(-1, 1, 1), nn_idx]           # B x P x k x 3
    y = nb - nb.mean(2, keepdim=True)
    s = y.transpose(-2, -1) @ y
    w, v = torch.linalg.eigh(s, UPLO="U")
    if canonical_signs:
        v = v * canonical_eigvec_signs(v)
    pick = w.argmin(2)
    return v[torch.arange(B).view(B, 1), torch.arange(P).view(1, P).expand(B, P), pick]


def normal_distance(p: Tensor, q: Tensor, d: Tensor, idx_p: Tensor, idx_q: Tensor, k: int,
                    nn_p: Optional[Tensor] = None, nn_q: Optional[Tensor] = None,
                    canonical_signs: bool = False):
    """loss_functions.py:107-126.  NB (reference quirk): the k-NN of p_i are searched in the *other* cloud
    (columns of d) and the resulting column indices are then used to gather rows of p itself."""
    B = p.shape[0]
    if nn_p is None:
        nn_p = knn_indices(d, k)
    if nn_q is None:
        nn_q = knn_indices(d.transpose(2, 1), k)
    n_p = normals_from_neighbours(p, nn_p, canonical_signs)
    n_q = normals_from_neighbours(q, nn_q, canonical_signs)
    ar = torch.arange(B).view(-1, 1)
    l0 = (n_p * n_q[ar, idx_p]).sum(2).abs().sum()
    l1 = (n_q * n_p[ar, idx_q]).sum(2).abs().sum()
    return l0, l1


# ----------------------------------------------------------------------------------------------------------
# the same losses with the discrete choices given (face draws, nearest indices, k-NN sets): O(n) memory, so the
# continuous part can be differentiated in fp64 at the trained shape (B = 32, 10 000 points) where the dense
# B x P x Q matrices above would not fit
# ----------------------------------------------------------------------------------------------------------
def chamfer_given(p: Tensor, q: Tensor, idx_p: Tensor, idx_q: Tensor):
    """(sum_i |p_i - q_{idx_p[i]}|^2, sum_j |q_j - p_{idx_q[j]}|^2) for B x P x 3 / B x Q x 3 clouds: ``chamfer`` of the
    dense matrix when idx_* are its argmins (loss_functions.py:93-102)."""
    ar = torch.arange(p.shape[0]).view(-1, 1)
    return ((p - q[ar, idx_p.long()]) ** 2).sum(), ((q - p[ar, idx_q.long()]) ** 2).sum()


def normal_sums_given(p: Tensor, q: Tensor, knn_p: Tensor, knn_q: Tensor, idx_p: Tensor, idx_q: Tensor,
                      canonical_signs: bool = True):
    """``normal_distance`` (loss_functions.py:107-126) with the k-NN sets and nearest indices given."""
    n_p = normals_from_neighbours(p, knn_p.long(), canonical_signs)
    n_q = normals_from_neighbours(q, knn_q.long(), canonical_signs)
    ar = torch.arange(p.shape[0]).view(-1, 1)
    return (n_p * n_q[ar, idx_p.long()]).sum(2).abs().sum(), (n_q * n_p[ar, idx_q.long()]).sum(2).abs().sum()


def normal_total_given(p: Tensor, q: Tensor, knn_p: Tensor, knn_q: Tensor, idx_p: Tensor, idx_q: Tensor, scale: float,
                       canonical_signs: bool = True) -> Tensor:
    """scale * (sum of both normal-consistency sums) -- loss_functions.py:69-72 with scale = -1 / point_cloud_size."""
    l0, l1 = normal_sums_given(p, q, knn_p, knn_q, idx_p, idx_q, canonical_signs)
    return scale * (l0 + l1)


def normals_conditioning(pt: Tensor, nn_idx: Tensor):
    """How far each row of ``normals_from_neighbours`` is from a discontinuity, in fp64, as four B x P tensors:
    (gap, m_v20, m_col1, m_det).  gap = min_{i != j} |w_i - w_j| / w_2 is the smallest relative eigen-gap (the
    eigenvector derivative divides by it; 0 for a degenerate spectrum).  The other three are the margins of the
    canonical sign rules (``canonical_eigvec_signs``): |V[2,0]|, the difference of the two largest |.| of column 1, and
    |det V|.  A row whose gap or margin is at the level of the rounding of its inputs may legitimately differ between
    two correct implementations."""
    pt = pt.detach().double()
    B, P, _ = pt.shape
    nb = pt[torch.arange(B).view(-1, 1, 1), nn_idx.long()]
    y = nb - nb.mean(2, keepdim=True)
    w, v = torch.linalg.eigh(y.transpose(-2, -1) @ y, UPLO="U")
    top = w[..., 2].abs().clamp_min(1e-300)
    gap = torch.stack([w[..., 1] - w[..., 0], w[..., 2] - w[..., 1]], -1).abs().min(-1).values / top
    c1 = v[..., :, 1].abs().sort(-1, descending=True).values
    return gap, v[..., 2, 0].abs(), c1[..., 0] - c1[..., 1], torch.linalg.det(v).abs()


def nearest_chunked(p: Tensor, q: Tensor, rows: int = 1024) -> Tensor:
    """B x P fp64 squared distance from every p_i to its nearest q_j, in row chunks of ``rows`` (memory rows x Q per
    cloud instead of P x Q for the whole batch).  |p|^2 + |q|^2 - 2 p.q in fp64: for fp32 clouds of unit scale the
    cancellation error (~1e-15) is far below the fp32 resolution the callers compare at."""
    p, q = p.detach().double(), q.detach().double()
    out = torch.empty(p.shape[:2], dtype=torch.float64)
    rq = (q * q).sum(2)
    for b in range(p.shape[0]):
        for s in range(0, p.shape[1], rows):
            a = p[b, s:s + rows]
            d = (a * a).sum(1, keepdim=True) + rq[b].unsqueeze(0) - 2.0 * (a @ q[b].t())
            out[b, s:s + rows] = d.min(1).values.clamp_min(0.0)
    return out


def mesh_loss_with(pos, faces, adj, v_index, f_index, gt_pos, gt_faces, gt_v_index, gt_f_index,
                   rnd_pred, rnd_gt, n_points: float = 10e3, k: int = 10, nn_override=None,
                   canonical_signs: bool = False):
    """loss_functions.py:40-74 with sampling randomness injected: rnd_* = (face_idx, xi2, xi1), each B x n.
    Returns (chamfer, normal, edge) and the intermediates the kernel tests look at."""
    e = edge_loss(pos, adj)
    cp = batched_sample_with(pos, faces, v_index, f_index, *rnd_pred)
    cq = batched_sample_with(gt_pos, gt_faces, gt_v_index, gt_f_index, *rnd_gt)
    d = p2p_distance(cp, cq)
    l1, i1, l2, i2 = chamfer(d)
    ch = (l1 + l2) / n_points
    nn_p, nn_q = nn_override if nn_override is not None else (None, None)
    n0, n1 = normal_distance(cp, cq, d, i1, i2, k, nn_p, nn_q, canonical_signs)
    nl = -(n0 + n1) / n_points
    return ch, nl, e, dict(cloud_pred=cp, cloud_gt=cq, idx_p=i1, idx_gt=i2)
