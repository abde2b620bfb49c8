"""TEST INFRASTRUCTURE ONLY -- CPU oracle of the opt-in bilinear VertexAlign (csrc/vert_align_bilinear.cu, DESIGN.md §2
item 7) and of the three refinement stages with it.

A literal torch statement of the semantics, dtype-agnostic and differentiable in the maps and the vertex positions: run it
in float64 to obtain the arbiter the fp32 kernels are compared with.  The stage functions are those of ``mesh_ops`` with the
aligned features taken from ``align`` (``mesh_ops.vert_align`` gives the reference stages back).

Only ``tests/`` may import this module.
"""
from typing import List, Sequence, Tuple

import torch
from torch import Tensor

from .mesh_ops import _stage_input, graph_conv, res_graph_conv


def _bilinear_one_map(fmap: Tensor, h: Tensor, w: Tensor, size: Tuple[int, int]) -> Tensor:
    """One square C x S x S map sampled bilinearly at clamped pixel coordinates (h, w): x = w / sx indexes the H axis and
    y = h / sy the W axis (the reference's axes, layers.py:577-590), both clamped to [0, S-1]; then x0 = clamp(floor(x), 0,
    S-2), fx = x - x0 (y alike) and the four-corner blend.  The cell indices are discrete (no gradient); the weights carry
    the gradient, so at a knot it is the one-sided derivative of the chosen cell."""
    S = fmap.shape[-1]
    H, W = size
    if S == 1:
        return fmap[:, 0, 0].unsqueeze(0).expand(h.shape[0], -1)
    x = (w / (float(W) / S)).clamp(min=0, max=S - 1)
    y = (h / (float(H) / S)).clamp(min=0, max=S - 1)
    x0 = torch.floor(x.detach()).clamp(min=0, max=S - 2)
    y0 = torch.floor(y.detach()).clamp(min=0, max=S - 2)
    fx, fy = (x - x0).unsqueeze(1), (y - y0).unsqueeze(1)
    xi, yi = x0.long(), y0.long()
    f = lambda a, b: fmap[:, a, b].t()
    return ((1 - fx) * (1 - fy) * f(xi, yi) + (1 - fx) * fy * f(xi, yi + 1) + fx * (1 - fy) * f(xi + 1, yi)
            + fx * fy * f(xi + 1, yi + 1))


def vert_align_bilinear(img_features: Sequence[Tensor], vertex_positions: Tensor, vertices_per_mesh: List[int],
                        image_sizes: Sequence[Tuple[int, int]], mesh_index: List[int]) -> Tensor:
    """Bilinear VertexAlign: the projection of ``mesh_ops.vert_align`` (layers.py:557-562), then ``_bilinear_one_map`` per
    map.  Where h or w is not finite (p2 == 0, NaN positions) the coordinate takes the value fminf / fmaxf give it
    (NaN -> 0, +-inf -> the bound) and the position gradient is exactly 0.  Returns SV x sum(C_m)."""
    chunks = vertex_positions.split(list(vertices_per_mesh))
    rows = []
    k = 0
    for img, (n_mesh, size) in enumerate(zip(mesh_index, image_sizes)):
        H, W = size
        for pos in chunks[k:k + n_mesh]:
            with torch.no_grad():
                h_raw = 248 * (pos[:, 1] / pos[:, 2]) + 111.5
                w_raw = 248 * (pos[:, 0] / -pos[:, 2]) + 111.5
                ok = torch.isfinite(h_raw) & torch.isfinite(w_raw)
                h_bad = torch.nan_to_num(h_raw, nan=0.0).clamp(min=0, max=H - 1)
                w_bad = torch.nan_to_num(w_raw, nan=0.0).clamp(min=0, max=W - 1)
            safe = torch.where(ok.unsqueeze(1), pos, torch.tensor([0.0, 0.0, -1.0], dtype=pos.dtype))   # no NaN in backward
            h = (248 * (safe[:, 1] / safe[:, 2]) + 111.5).clamp(min=0, max=H - 1)
            w = (248 * (safe[:, 0] / -safe[:, 2]) + 111.5).clamp(min=0, max=W - 1)
            h = torch.where(ok, h, h_bad)
            w = torch.where(ok, w, w_bad)
            rows.append(torch.cat([_bilinear_one_map(f[img], h, w, size) for f in img_features], dim=1))
        k += n_mesh
    return torch.cat(rows, dim=0)


def stage_res_shapenet(sd, v_index, fmaps, adj, pos, sizes, feats=None, mesh_index=None, align=vert_align_bilinear):
    """ResVertixRefineShapenet.forward (layers.py:130-178) with the aligned features from ``align``."""
    mesh_index = mesh_index or [1] * len(sizes)
    aligned = align(fmaps, pos, v_index, sizes, mesh_index)
    x = _stage_input(pos, aligned @ sd["linear.weight"].t(), feats)
    x = res_graph_conv(x, adj, sd, "resGraphConv0.")
    x = res_graph_conv(x, adj, sd, "resGraphConv1.")
    x = res_graph_conv(x, adj, sd, "resGraphConv2.")
    delta = torch.tanh(graph_conv(x, adj, sd["graphConv.w0"], sd["graphConv.w1"]))   # tanh(relu(.)), :174-175
    return pos + delta, x


def stage_shapenet(sd, v_index, fmaps, adj, pos, sizes, feats=None, mesh_index=None, align=vert_align_bilinear):
    """VertixRefineShapeNet.forward (layers.py:207-259) with the aligned features from ``align``."""
    mesh_index = mesh_index or [1] * len(sizes)
    aligned = align(fmaps, pos, v_index, sizes, mesh_index)
    x = _stage_input(pos, aligned @ sd["linear0.weight"].t(), feats)
    x = graph_conv(x, adj, sd["graphConv0.w0"], sd["graphConv0.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv1.w0"], sd["graphConv1.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv2.w0"], sd["graphConv2.w1"])
    delta = torch.tanh(x @ sd["linear1.weight"].t())
    return pos + delta, x


def stage_pix3d(sd, v_index, fmap, adj, pos, sizes, feats=None, mesh_index=None, align=vert_align_bilinear):
    """VertixRefinePix3D.forward (layers.py:289-339) with the aligned features from ``align``."""
    mesh_index = mesh_index or [1] * len(sizes)
    aligned = align([fmap], pos, v_index, sizes, mesh_index)
    x = _stage_input(pos, aligned, feats)
    x = graph_conv(x, adj, sd["graphConv0.w0"], sd["graphConv0.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv1.w0"], sd["graphConv1.w1"])
    x = graph_conv(torch.cat([pos, x], 1), adj, sd["graphConv2.w0"], sd["graphConv2.w1"])
    delta = torch.tanh(torch.cat([pos, x], 1) @ sd["linear.weight"].t())
    return pos + delta, x


STAGES = {"ResVertixRefineShapenet": stage_res_shapenet, "VertixRefineShapeNet": stage_shapenet,
          "VertixRefinePix3D": stage_pix3d}
