"""TEST INFRASTRUCTURE ONLY -- fp64 CPU restatement of the Mesh R-CNN paper's mesh metrics (``eval_utils.compare_meshes``):
GT-10 scale, surface samples with injected draws and their face normals, dense nearest neighbours, and the per-mesh
Chamfer-L2 / normal consistency / precision-recall-F1@tau.  Only ``tests/`` import it."""
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor


# ----------------------------------------------------------------------------------------------------------
# mesh metrics of the Mesh R-CNN paper (eval_utils.compare_meshes): GT-10 scale, surface samples with face normals,
# dense nearest neighbours, Chamfer-L2 / normal consistency / precision-recall-F1@tau per mesh
# ----------------------------------------------------------------------------------------------------------
def face_normals(verts: Tensor, faces: Tensor) -> Tensor:
    """Unit normals (B-A)x(C-A)/|.| of every face; a degenerate face gets the zero vector."""
    tri = verts[faces]
    n = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0], dim=1)
    length = n.norm(dim=1, keepdim=True)
    return torch.where(length > 0, n / torch.where(length > 0, length, torch.ones_like(length)), torch.zeros_like(n))


def gt_scale(verts: Tensor, target: float = 10.0) -> Tensor:
    """target / longest side of the bounding box of one mesh."""
    return target / (verts.max(0).values - verts.min(0).values).max()


def sample_surface_with(verts: Tensor, faces: Tensor, face_idx: Tensor, xi2: Tensor, xi1: Tensor, scale=1.0):
    """Unnormalised surface points (mesh_sampling.py:18-35 with injected draws, times ``scale``) and their face normals."""
    tri = verts[faces[face_idx]]
    r = xi1.sqrt()
    w = torch.stack([1.0 - r, (1 - xi2) * r, xi2 * r], dim=1).to(verts.dtype)
    return scale * (tri * w.unsqueeze(2)).sum(1), face_normals(verts, faces)[face_idx]


def nearest(a: Tensor, b: Tensor, chunk: int = 512) -> Tuple[Tensor, Tensor]:
    """Squared distance and index of the nearest point of b for every point of a (dense, direct (a-b)^2, row chunks)."""
    ds, ids = [], []
    for lo in range(0, a.shape[0], chunk):
        d = ((a[lo:lo + chunk].unsqueeze(1) - b.unsqueeze(0)) ** 2).sum(2)
        m, i = d.min(1)
        ds.append(m)
        ids.append(i)
    return torch.cat(ds), torch.cat(ids)


def in_tie_set(a: Tensor, b: Tensor, idx: Tensor, d_min: Tensor, atol: float = 1e-5) -> Tensor:
    """bool per point of a: b[idx] is a nearest neighbour up to atol * (1 + d_min) in squared distance."""
    d_sel = ((a - b[idx.long()]) ** 2).sum(1)
    return d_sel <= d_min + atol * (1 + d_min)


def mesh_metrics_one(p: Tensor, n_p: Tensor, q: Tensor, n_q: Tensor, thresholds: Sequence[float],
                     idx_p: Optional[Tensor] = None, idx_q: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """Metrics of one pair of samples from dense distances.  ``idx_p`` / ``idx_q`` (optional) evaluate the normal terms at
    given nearest-neighbour indices (e.g. a kernel's, after checking them with ``in_tie_set``) instead of the argmin."""
    d_p, a_p = nearest(p, q)
    d_q, a_q = nearest(q, p)
    idx_p = a_p if idx_p is None else idx_p.long()
    idx_q = a_q if idx_q is None else idx_q.long()
    dot_p = (n_p * n_q[idx_p]).sum(1)
    dot_q = (n_q * n_p[idx_q]).sum(1)
    out = {"Chamfer-L2": d_p.mean() + d_q.mean(),
           "NormalConsistency": 0.5 * (dot_p.mean() + dot_q.mean()),
           "AbsNormalConsistency": 0.5 * (dot_p.abs().mean() + dot_q.abs().mean())}
    r_p, r_q = d_p.sqrt(), d_q.sqrt()
    for tau in thresholds:
        prec = 100.0 * (r_p < tau).double().mean()
        rec = 100.0 * (r_q < tau).double().mean()
        out["Precision@%g" % tau] = prec
        out["Recall@%g" % tau] = rec
        out["F1@%g" % tau] = 2 * prec * rec / (prec + rec + 1e-8)
    out["_d_p"], out["_d_q"] = d_p, d_q
    return out


def compare_meshes_with(pred_verts, pred_faces, pred_v_index, pred_f_index, gt_verts, gt_faces, gt_v_index, gt_f_index,
                        rnd_pred, rnd_gt, scale: Optional[str] = "gt-10",
                        thresholds: Sequence[float] = (0.1, 0.2, 0.3, 0.4, 0.5)) -> List[Dict[str, Tensor]]:
    """Per-mesh metric dicts (one per GT mesh) with injected draws rnd_* = (face_idx, xi2, xi1), each B x n.  A predicted mesh
    without faces gets NaN Chamfer / NC / AbsNC and 0 precision / recall / F1.  Each dict also holds the samples
    (``_p``, ``_q``, ``_n_p``, ``_n_q``), the scale (``_s``) and the nearest-neighbour distances (``_d_p``, ``_d_q``)."""
    B = len(gt_f_index)
    pv = list(pred_v_index) + [0] * (B - len(pred_v_index))
    pf = list(pred_f_index) + [0] * (B - len(pred_f_index))
    pvs, pfs = pred_verts.split(pv), pred_faces.split(pf)
    gvs, gfs = gt_verts.split(list(gt_v_index)), gt_faces.split(list(gt_f_index))
    res = []
    for b in range(B):
        if pf[b] == 0:
            row = {"Chamfer-L2": torch.tensor(float("nan")), "NormalConsistency": torch.tensor(float("nan")),
                   "AbsNormalConsistency": torch.tensor(float("nan"))}
            for tau in thresholds:
                for k in ("Precision", "Recall", "F1"):
                    row["%s@%g" % (k, tau)] = torch.tensor(0.0)
            res.append(row)
            continue
        s = gt_scale(gvs[b]) if scale == "gt-10" else 1.0
        p, n_p = sample_surface_with(pvs[b], pfs[b], rnd_pred[0][b], rnd_pred[1][b], rnd_pred[2][b], s)
        q, n_q = sample_surface_with(gvs[b], gfs[b], rnd_gt[0][b], rnd_gt[1][b], rnd_gt[2][b], s)
        row = mesh_metrics_one(p, n_p, q, n_q, thresholds)
        row.update(_p=p, _q=q, _n_p=n_p, _n_q=n_q, _s=s)
        res.append(row)
    return res
