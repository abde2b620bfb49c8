"""Eval-side helpers next to the hot path (SURVEY.md 8 f-3): the metrics of the reference ``utils/metrics.py``, the
detection-selection + adjacency rebuild of ``utils/eval_utils.py:12-90``, and the device path of ``validate``
(``utils/eval_utils.py:93-194``): ``validate_batch`` evaluates the voxel / chamfer / normal / edge losses of an eval-mode
output dict over all its position sets through the CUDA kernels and adds the geometric F1@tau of the final meshes from
the nearest-neighbour distances the k-NN kernel already returns; ``validate`` averages it over a loader with the
reference's metric names.  The metric helpers are device-agnostic tensor code; the rebuilt adjacency is handed to the CSR
path through ``topology.from_coo`` like any foreign COO tensor.

Reference semantics kept: ``f_score`` works on a confusion matrix c[i, j] = #(predicted i, ground truth j) and returns
percentages with the 1e-8 guards of :20-26; ``mesh_precision_recall`` zeroes ALL true positives through the scalar-mask
assignment ``tp[f1 <= 0.5] = 0`` when the running F0.3 is <= 0.5 (:53-60) and integrates precision over recall with
the trapezoid rule (sklearn ``auc``: the recall values must be monotonic)."""
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor


def f_score(confusion: Tensor, beta: float = 1.0) -> Tensor:
    tp = confusion.diagonal()
    precision = 100 * (tp / (1e-8 + confusion.sum(1)))
    recall = 100 * (tp / (1e-8 + confusion.sum(0)))
    return (1 + beta ** 2) * precision * recall / (1e-8 + recall + (beta ** 2) * precision)


def _auc(x: Tensor, y: Tensor) -> float:
    """Trapezoid area under y(x) for monotonic x (what ``sklearn.metrics.auc`` computes; decreasing x flips the sign)."""
    if x.numel() < 2:
        raise ValueError("At least 2 points are needed to compute area under curve, but x.shape = %d" % x.numel())
    dx = x[1:] - x[:-1]
    if bool((dx < 0).any()):
        if bool((dx <= 0).all()):
            sign = -1.0
        else:
            raise ValueError("x is neither increasing nor decreasing : {}.".format(x.tolist()))
    else:
        sign = 1.0
    return sign * float((dx.double() * (y[1:] + y[:-1]).double() / 2).sum())


def mesh_precision_recall(confusion: Tensor, f1_score: float) -> float:
    tp = confusion.diagonal().clone()
    if f1_score <= 0.5:                     # reference: tp[f1_score <= 0.5] = 0 with a Python scalar -> all or nothing
        tp = torch.zeros_like(tp)
    precision = 100 * (tp / (1e-8 + confusion.sum(1)))
    recall = 100 * (tp / (1e-8 + confusion.sum(0)))
    return _auc(recall, precision)


def box_iou(a: Tensor, b: Tensor) -> Tensor:
    """Pairwise IoU of (x1, y1, x2, y2) boxes, N x 4 and M x 4 -> N x M."""
    area_a = (a[:, 2] - a[:, 0]) * (a[:, 3] - a[:, 1])
    area_b = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    lt = torch.max(a[:, None, :2], b[None, :, :2])
    rb = torch.min(a[:, None, 2:], b[None, :, 2:])
    wh = (rb - lt).clamp(min=0)
    inter = wh[..., 0] * wh[..., 1]
    return inter / (area_a[:, None] + area_b[None, :] - inter)


def calc_precision_box(boxes: Sequence[Tensor], gt_boxes: Sequence[Tensor]) -> float:
    hits = sum(1 for g, p in zip(gt_boxes, boxes) if box_iou(g, p.unsqueeze(0))[0][0] > 0.5)
    return hits / len(boxes)


def calc_precision_mask(masks: Sequence[Tensor], gt_masks: Sequence[Tensor]) -> float:
    hits = 0
    for mask, gt in zip(masks, gt_masks):
        m, g = (mask > 0.5).to(torch.int32), gt.to(torch.int32)
        if torch.sum(m & g) / torch.sum(m | g) > 0.5:
            hits += 1
    return hits / len(masks)


def get_max_box(boxes: Tensor, gt_box: Tensor) -> Tuple[Tensor, Tensor]:
    idx = torch.argmax(box_iou(boxes, gt_box), dim=0)[0]
    return boxes[idx], idx


def faces_to_adjacency(faces_global: Tensor) -> Tensor:
    """2 x E symmetric COO adjacency (sorted by (row, col), duplicates removed) from SF x 3 faces with GLOBAL vertex ids:
    the three edges of every triangle in both directions (reference eval_utils.py:77-88 == layers.py:469-478)."""
    ft = faces_global.t()
    i, j = torch.cat([ft[:2], ft[1:], ft[::2]], dim=1)
    i, j = torch.cat([i, j], dim=0), torch.cat([j, i], dim=0)
    return torch.stack([i, j], dim=0).unique(dim=1)


def get_only_max(max_indexes: Sequence[int], voxels: Tensor, vertex_positions: List[Tensor], faces: Tensor,
                 vertice_index: List[int], face_index: List[int], mesh_index: List[int]):
    """Keeps, per image, the detection ``max_indexes[img]`` of its ``mesh_index[img]`` meshes and rebuilds the packed batch:
    (voxels, per-stage positions, faces (local ids), adjacency (global ids), vertice_index, face_index)."""
    vxls = torch.stack([g[idx] for g, idx in zip(voxels.split(mesh_index), max_indexes)])
    fs = faces.split(face_index)
    res_fs, i = [], 0
    for n, idx in zip(mesh_index, max_indexes):
        res_fs.append(fs[i:i + n][idx])
        i += n
    res_f_index = [f.size(0) for f in res_fs]
    res_vs, res_v_index = [], []
    for j, stage in enumerate(vertex_positions):
        vs, picked, i = stage.split(vertice_index), [], 0
        for n, idx in zip(mesh_index, max_indexes):
            picked.append(vs[i:i + n][idx])
            i += n
        if j == 0:
            res_v_index = [v.size(0) for v in picked]
        res_vs.append(torch.cat(picked))
    offsets, run = [], 0
    for n in res_v_index:
        offsets.append(run)
        run += n
    adj = faces_to_adjacency(torch.cat([f + off for f, off in zip(res_fs, offsets)]))
    return vxls, res_vs, torch.cat(res_fs), adj, res_v_index, res_f_index


# ---------------------------------------------------------------------------------------------------------------
# mesh metrics of the Mesh R-CNN paper (Chamfer-L2, normal consistency, F1@tau on GT-10 scaled surface samples)
# ---------------------------------------------------------------------------------------------------------------
def mesh_metric_names(thresholds: Sequence[float]) -> List[str]:
    """Keys of ``compare_meshes`` in the column order of its per-mesh table."""
    names = ["Chamfer-L2", "NormalConsistency", "AbsNormalConsistency"]
    for tau in thresholds:
        names += ["Precision@%g" % tau, "Recall@%g" % tau, "F1@%g" % tau]
    return names


MESH_METRIC_THRESHOLDS = (0.1, 0.2, 0.3, 0.4, 0.5)
_PAPER_KEYS = frozenset(mesh_metric_names(MESH_METRIC_THRESHOLDS))


def mesh_metric_sums(per_mesh: dict) -> Tuple[List[str], Tensor]:
    """(metric keys, fp64 [len(keys) + 1]): the sums of every per-mesh metric over the valid meshes, then their count."""
    valid = per_mesh["valid"]
    keys = [k for k in per_mesh if k != "valid"]
    vals = torch.stack([per_mesh[k].double() for k in keys])
    sums = torch.where(valid.unsqueeze(0), vals, torch.zeros_like(vals)).sum(1)
    return keys, torch.cat([sums, valid.double().sum().reshape(1)])


@torch.no_grad()
def compare_meshes(pred_verts: Tensor, pred_faces: Tensor, pred_v_index: Sequence[int], pred_f_index: Sequence[int],
                   gt_verts: Tensor, gt_faces: Tensor, gt_v_index: Sequence[int], gt_f_index: Sequence[int],
                   num_samples: int = 10000, scale: Optional[str] = "gt-10",
                   thresholds: Sequence[float] = MESH_METRIC_THRESHOLDS, seed: Optional[int] = None, randomness=None,
                   reduce: bool = True) -> dict:
    """The mesh metrics of the Mesh R-CNN paper for packed predicted / ground-truth batches (faces hold per-mesh local ids).

    Both meshes of pair b are sampled at ``num_samples`` area-weighted surface points with the normal of the face each
    point lies on; with ``scale="gt-10"`` both samples are multiplied by ``10 / longest side of the GT bounding box``
    (``scale=None``: no scaling).  With d_p / d_q the squared distances to the nearest sample of the other mesh:

    - ``Chamfer-L2`` = mean d_p + mean d_q;
    - ``NormalConsistency`` = 0.5 (mean n_i . m_nn(i) + mean m_j . n_nn(j)), ``AbsNormalConsistency`` the same with |.|;
    - ``Precision@tau`` / ``Recall@tau`` = 100 x share of predicted / GT samples with sqrt(d) < tau, ``F1@tau`` =
      2PR / (P + R + 1e-8) for every threshold (at most 8).

    Cubify's reference topology emits the two triangles of a quad with opposite winding, so the signed ``NormalConsistency``
    of such meshes is dominated by that flip; ``AbsNormalConsistency`` is the meaningful one for them.  Meshes of
    ``Cubify(topology="watertight")`` are wound outward throughout, and their signed ``NormalConsistency`` is meaningful.

    B is ``len(gt_f_index)``; shorter prediction lists (Cubify drops trailing empty meshes) are padded with empty meshes.  A
    predicted mesh without faces is invalid: NaN Chamfer / NC / AbsNC, 0 for P / R / F1.  Randomness: ``seed`` (predicted
    samples; the GT samples use ``seed + 1``; default: drawn from torch's generator) or ``randomness = (rnd_pred, rnd_gt)``
    with ``rnd_* = dict(u=|face_idx=, xi2=, xi1=)`` (B x num_samples tensors, rows of invalid meshes ignored).

    Returns ``{key: fp32 tensor [B]}`` plus ``valid`` (bool [B]) with ``reduce=False``; with ``reduce=True`` the 0-dim means
    over the valid meshes plus ``num_valid`` (int).  No device -> host read."""
    from . import functional as F_
    F_._require_cuda(pred_verts, "compare_meshes")
    F_._require_cuda(gt_verts, "compare_meshes")
    thresholds = [float(t) for t in thresholds]
    if len(thresholds) > F_.MAX_THRESHOLDS:
        raise ValueError("compare_meshes: at most %d thresholds, got %d" % (F_.MAX_THRESHOLDS, len(thresholds)))
    if scale not in (None, "gt-10"):
        raise ValueError("compare_meshes: scale must be 'gt-10' or None, got %r" % (scale,))
    B = len(gt_f_index)
    if len(gt_v_index) != B:
        raise ValueError("compare_meshes: gt_v_index and gt_f_index differ in length")
    if B == 0 or min(gt_f_index) <= 0:
        raise ValueError("compare_meshes: every ground-truth mesh needs at least one face")
    if len(pred_v_index) > B or len(pred_f_index) > B:
        raise ValueError("compare_meshes: %d / %d predicted meshes for %d ground-truth meshes"
                         % (len(pred_v_index), len(pred_f_index), B))
    pv = list(pred_v_index) + [0] * (B - len(pred_v_index))
    pf = list(pred_f_index) + [0] * (B - len(pred_f_index))
    if sum(pv) != pred_verts.shape[0] or sum(pf) != pred_faces.shape[0]:
        raise ValueError("compare_meshes: predicted index lists do not match the packed tensors")
    n = int(num_samples)
    rnd_pred, rnd_gt = randomness if randomness is not None else ({}, {})
    if seed is None:
        seed = 0 if ("xi2" in rnd_pred and "xi2" in rnd_gt) else F_._next_seed()

    valid = [b for b in range(B) if pf[b] > 0]
    cols = mesh_metric_names(thresholds)
    dev = pred_verts.device
    met = rows = None
    if valid:
        starts = [0]
        for c in pv:
            starts.append(starts[-1] + c)
        gv, gf, gvi, gfi = gt_verts, gt_faces, list(gt_v_index), list(gt_f_index)
        if len(valid) < B:
            # empty predicted meshes occupy no rows: only their offsets drop out; the GT meshes of the pairs are gathered
            gv = torch.cat([v for b, v in enumerate(gt_verts.split(gvi)) if pf[b] > 0])
            gf = torch.cat([f for b, f in enumerate(gt_faces.split(gfi)) if pf[b] > 0])
            gvi, gfi = [gvi[b] for b in valid], [gfi[b] for b in valid]
            rows = torch.tensor(valid, dtype=torch.int64).to(dev)
            pick = lambda r: {k: (t.to(dev)[rows] if isinstance(t, Tensor) else t) for k, t in r.items()}
            rnd_pred, rnd_gt = pick(rnd_pred), pick(rnd_gt)
        s = F_.mesh_gt_scale(gv, gvi, 10.0) if scale == "gt-10" else None
        p, n_p, _ = F_.sample_surface(pred_verts, pred_faces, [pv[b] for b in valid], [pf[b] for b in valid], n,
                                      seed=int(seed), scale=s, v_starts=[starts[b] for b in valid], **rnd_pred)
        q, n_q, _ = F_.sample_surface(gv, gf, gvi, gfi, n, seed=int(seed) + 1, scale=s, **rnd_gt)
        d_p, i_p, _, d_q, i_q, _ = F_.knn_search(p, q, 0)
        met = F_.mesh_metrics(d_p, i_p, d_q, i_q, n_p, n_q, thresholds)
    if len(valid) == B:
        table = met
    else:
        table = torch.empty(B, len(cols), dtype=torch.float32, device=dev)
        table[:, :3] = float("nan")
        table[:, 3:] = 0.0
        if met is not None:
            table[rows] = met
    per_mesh = {k: table[:, i] for i, k in enumerate(cols)}
    per_mesh["valid"] = torch.tensor([pf[b] > 0 for b in range(B)]).to(dev)
    if not reduce:
        return per_mesh
    keys, sums = mesh_metric_sums(per_mesh)
    means = (sums[:-1] / len(valid)).float() if valid else torch.full((len(keys),), float("nan"), device=dev)
    out = {k: means[i] for i, k in enumerate(keys)}
    out["num_valid"] = len(valid)
    return out


# ---------------------------------------------------------------------------------------------------------------
# validate on the device path (reference utils/eval_utils.py:93-194)
# ---------------------------------------------------------------------------------------------------------------
@torch.no_grad()
def validate_batch(model_output: dict, batch, point_cloud_size: float = 10e3, num_neighbours_for_normal_loss: int = 10,
                   f1_thresholds: Sequence[float] = (0.1, 0.3, 0.5), randomness=None, f1_seed: int = 0,
                   mesh_metrics: bool = False) -> dict:
    """Losses of one eval-mode output dict (keys ``vertex_positions`` (list, incl. the cubified stage-0 set), ``faces``,
    ``edge_index``, ``vertice_index``, ``face_index``; optional ``voxels``) against ``batch`` (``.meshes``,
    ``.vertice_index``, ``.face_index``, optional ``.voxels``) -- what reference ``validate`` computes per batch
    (eval_utils.py:160-164: ``voxel_loss`` + ``batched_mesh_loss`` over ALL position sets), on the CUDA kernels.

    Added (SURVEY 8 f-3): ``f1@tau`` of the final meshes -- precision = share of predicted surface samples within ``tau`` of
    the ground-truth samples, recall the converse, F1 = 2PR / (P + R) in percent, averaged over the meshes; it costs one
    extra nearest-neighbour call (k = 0) on 10 000-point clouds of the normalised meshes.

    ``mesh_metrics=True`` adds the ``compare_meshes`` keys of the final meshes (GT-10 scale, default thresholds, seed
    ``f1_seed + 2``) and ``num_valid``; the default leaves the output as it was."""
    from . import functional as F_
    from .loss_functions import batched_mesh_loss, voxel_loss
    vs, fs, e_index = model_output["vertex_positions"], model_output["faces"], model_output["edge_index"]
    v_index, f_index = model_output["vertice_index"], model_output["face_index"]
    out = {}
    if model_output.get("voxels") is not None and getattr(batch, "voxels", None) is not None:
        out["voxel_loss"] = voxel_loss(model_output["voxels"], batch.voxels)
    chamfer, normal, edge = batched_mesh_loss(list(vs), fs, e_index, v_index, f_index, batch, point_cloud_size,
                                              num_neighbours_for_normal_loss, randomness=randomness)
    out.update({"chamfer_loss": chamfer, "normal_loss": normal, "edge_loss": edge})
    n = int(point_cloud_size)
    gt_pos, gt_faces = batch.meshes
    cloud_p, _ = F_.sample_points(vs[-1], fs, v_index, f_index, n, seed=f1_seed)
    cloud_g, _ = F_.sample_points(gt_pos, gt_faces, batch.vertice_index, batch.face_index, n, seed=f1_seed + 1, cdf_owner=batch)
    d_p, _, _, d_g, _, _ = F_.knn_search(cloud_p, cloud_g, 0)
    d_p, d_g = d_p.sqrt(), d_g.sqrt()
    for tau in f1_thresholds:
        prec = (d_p < tau).float().mean(dim=1)
        rec = (d_g < tau).float().mean(dim=1)
        out["f1@%g" % tau] = (100.0 * 2 * prec * rec / (prec + rec).clamp_min(1e-8)).mean()
    if mesh_metrics:
        out.update(compare_meshes(vs[-1], fs, v_index, f_index, gt_pos, gt_faces, batch.vertice_index, batch.face_index,
                                  seed=f1_seed + 2))
    return out


class AverageMeter:
    """Running average with the reference's interface (utils/train_utils.py AverageMeter: ``update(val, n)``, ``.avg``)."""

    def __init__(self, name: str):
        self.name, self.sum, self.count, self.val = name, 0.0, 0, 0.0

    def update(self, val: float, n: int = 1) -> None:
        self.val = float(val)
        self.sum += float(val) * n
        self.count += n

    @property
    def avg(self) -> float:
        return self.sum / max(self.count, 1)


def validate(model, val_loader, device=None, point_cloud_size: float = 10e3, num_neighbours_for_normal_loss: int = 10,
             mesh_metrics: bool = False) -> dict:
    """Mesh-side validation loop (reference ``validate``, eval_utils.py:93-194, without the backbone / classification
    metrics that are outside the hot path): ``model(images)`` must return the eval-mode output dict; returns AverageMeters
    named like the reference's (``voxel_loss``, ``chamfer_loss``, ``normal_loss``, ``edge_loss``) plus ``f1@tau``.
    ``mesh_metrics=True`` adds the ``compare_meshes`` metrics of the final meshes, each batch weighted by its number of
    valid (non-empty) predicted meshes."""
    model.eval()
    meters = {}
    for batch in val_loader:
        if device is not None:
            batch = batch.to(device, non_blocking=True)
        res = validate_batch(model(batch.images), batch, point_cloud_size, num_neighbours_for_normal_loss,
                             mesh_metrics=mesh_metrics)
        n = len(batch.vertice_index)
        n_valid = res.pop("num_valid", None)
        for k, v in res.items():
            if k not in _PAPER_KEYS:
                meters.setdefault(k, AverageMeter(k)).update(float(v), n)
            elif n_valid:                        # a batch without a valid predicted mesh adds nothing to these means
                meters.setdefault(k, AverageMeter(k)).update(float(v), n_valid)
    return meters
