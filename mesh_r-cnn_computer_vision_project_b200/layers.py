"""Drop-in mirror of the reference ``meshRCNN/layers.py`` module API for the hot path: ``Cubify``,
``VertexAlign``, ``GraphConv``, ``ResGraphConv`` and the three refinement-stage classes -- same class names,
constructor arguments, ``forward`` argument orders, return tuples and ``state_dict`` keys, so that
``meshRCNN/shapenet_model.py:11-13,27-41,72-90`` and ``meshRCNN/pix3d_model.py:16-17,32-44,87-106`` work
unchanged after ``from meshrcnn_b200.layers import ...``.

Every numerical op runs in hand-written sm_100a CUDA behind the C ABI (``include/meshrcnn_b200.h``); there is
no CPU path: CPU tensors raise ``RuntimeError``.
"""
import math
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _lib, functional as F_, topology


class Cubify(nn.Module):
    """Voxel occupancy probabilities -> packed cuboid triangle meshes.

    Mirrors reference ``Cubify`` (meshRCNN/layers.py:342-484): ``forward(t)`` with ``t`` of shape B x Z x Y x X
    returns ``(vs, v_index, faces, f_index, adj_index)``: ``vs`` SV x 3 fp32 in voxel units rotated to
    (z, x, -y); ``v_index`` / ``f_index`` Python lists of per-mesh counts (truncated after the last non-empty
    mesh, like ``bincount``); ``faces`` SF x 3 int64 with per-mesh local vertex ids; ``adj_index`` 2 x E int64 with
    global ids sorted by (row, col).  Vertex / face / edge order equals the reference's (bit-exact).
    Raises ``ValueError("empty grid")`` when no voxel of the whole batch is occupied (layers.py:434-435).
    """

    def __init__(self, threshold: float = 0.5):
        super().__init__()
        self.threshold = threshold
        # state-dict compatibility with the reference ("cubify.kernel", "cubify.deltas", layers.py:365,401);
        # the CUDA path does not read them (the same tables live in csrc/cubify.cu as constants).
        nbr = [(-1, 0, 0), (1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, -1), (0, 0, 1)]
        kernel = torch.zeros(6, 1, 3, 3, 3)
        for d, (dz, dy, dx) in enumerate(nbr):
            kernel[d, 0, 1, 1, 1] = 1
            kernel[d, 0, 1 + dz, 1 + dy, 1 + dx] = -1
        corners = F_.CUBIFY_CORNERS
        deltas = torch.zeros(6, 4, 5)
        for d in range(6):
            for c in range(4):
                for a in range(3):
                    deltas[d, c, 2 + a] = corners[d][c][a] - 0.5
        self.register_buffer("kernel", kernel)
        self.register_buffer("deltas", deltas)

    def forward(self, t: Tensor, from_logits: bool = False):
        """``from_logits=True`` (extension, SURVEY 8 f-1): ``t`` holds the voxel head's logits; ``sigmoid(t) > threshold`` is
        evaluated inside the first kernel, so the probability grid is never written."""
        verts, v_index, faces, f_index, adj, _ = F_.cubify(t, float(self.threshold), from_logits)
        return verts, v_index, faces, f_index, adj


class VoxelBranch(nn.Sequential):
    """Voxel occupancy head -- reference meshRCNN/layers.py:487-506, same modules and state-dict keys (``0.weight`` ...
    ``3.bias``; the convolutions are library calls and outside the hot path).  ``forward`` returns probabilities like the
    reference; ``forward_logits`` stops before the final ``nn.Sigmoid`` so that its two consumers -- ``voxel_loss_with_logits``
    and ``Cubify(..)(logits, from_logits=True)`` -- evaluate the sigmoid inside their own first pass."""

    def __init__(self, in_channels: int, out_channels: int, hidden_channels: int = 256):
        super().__init__(
            nn.Conv2d(in_channels, hidden_channels, kernel_size=3, padding=1),
            nn.Conv2d(hidden_channels, hidden_channels, kernel_size=3, padding=1),
            nn.ConvTranspose2d(hidden_channels, hidden_channels, kernel_size=2, stride=2),
            nn.Conv2d(hidden_channels, out_channels, kernel_size=1),
            nn.Sigmoid())

    def forward_logits(self, x: Tensor) -> Tensor:
        for m in list(self)[:-1]:
            x = m(x)
        return x


ALIGN_MODES = ("reference", "bilinear")


class VertexAlign(nn.Module):
    """Projects mesh vertices into the image plane and pools feature-map texels.

    Mirrors reference ``VertexAlign.forward(img_features, vertex_positions, vertices_per_mesh, image_sizes,
    mesh_index)`` (meshRCNN/layers.py:521-546) including its actual arithmetic (:557-611): fixed intrinsics
    (248, 111.5), clamp to the image, nearest-floor texel with the H/W axes swapped, 0/1 mask, no gradient to the
    positions.  Output: SV x sum(C_m).

    ``mode="bilinear"`` (opt-in, a plain attribute that may also be set on a loaded model): the same projection, then a
    bilinear sample of each map (``functional.vert_align_bilinear``), differentiable in the maps and in the vertex
    positions.  No parameters or buffers either way, so state dicts do not depend on the mode."""

    def __init__(self, mode: str = "reference"):
        super().__init__()
        if mode not in ALIGN_MODES:
            raise ValueError("VertexAlign: mode must be one of %s, got %r" % (ALIGN_MODES, mode))
        self.mode = mode

    def forward(self, img_features: List[Tensor], vertex_positions: Tensor, vertices_per_mesh: List[int],
                image_sizes: List[Tuple[int, int]], mesh_index: List[int]) -> Tensor:
        if self.training:                                       # layers.py:528-530
            assert len(vertices_per_mesh) == len(image_sizes)
            assert list(mesh_index) == [1 for _ in image_sizes]
        assert len(mesh_index) == len(image_sizes)              # layers.py:532
        if _bilinear(self):
            return F_.vert_align_bilinear(img_features, vertex_positions, vertices_per_mesh, image_sizes, mesh_index)
        return F_.vert_align(img_features, vertex_positions, vertices_per_mesh, image_sizes, mesh_index)


def _bilinear(align: VertexAlign) -> bool:
    mode = getattr(align, "mode", "reference")
    if mode not in ALIGN_MODES:
        raise ValueError("VertexAlign: mode must be one of %s, got %r" % (ALIGN_MODES, mode))
    return mode == "bilinear"


# Stage inputs are column concatenations [features | position | aligned features] (reference layers.py:160-165,241-252,
# 321-334).  True: the layers consume them as parts (split-input GraphConv, csrc/graphconv2.cu: dense blocks on the tensor
# cores, the 3 position columns in the gather epilogue, VertexAlign as a texel-row gather, fused tanh head) and nothing is
# concatenated.  False: the literal evaluation (concatenate, then the generic kernels) -- kept for the parity tests.
FUSE_STAGE_INPUTS = True


class GraphConv(nn.Module):
    """f'_i = ReLU(W0 f_i + sum_{j in N(i)} W1 f_j)  -- reference meshRCNN/layers.py:25-68.
    Parameters ``w0`` / ``w1`` are stored in x out and initialised U(+-1/sqrt(in)) (:42-45); no bias; the ReLU
    is always applied (:68)."""

    def __init__(self, in_features: int, out_features: int):
        super().__init__()
        self.w0 = nn.Parameter(torch.empty(in_features, out_features))
        self.w1 = nn.Parameter(torch.empty(in_features, out_features))
        self.reset_parameters()

    def reset_parameters(self):
        bound = 1.0 / math.sqrt(self.w0.size(0))
        self.w0.data.uniform_(-bound, bound)
        self.w1.data.uniform_(-bound, bound)

    def forward(self, vertex_features, vertex_adjacency: Tensor, residual: Optional[Tensor] = None) -> Tensor:
        """``vertex_features``: SV x in_features (the reference signature), or -- an extension used by the stage classes -- a
        list of parts ``[("x", dense block) | ("pos", SV x 3) | ("tex", functional.TexelTerm), ...]`` standing for their
        column concatenation, which is then never materialised (functional.graph_conv_parts)."""
        if isinstance(vertex_features, (list, tuple)):
            return F_.graph_conv_parts(vertex_features, vertex_adjacency, self.w0, self.w1, residual)
        if FUSE_STAGE_INPUTS and self.w0.shape[1] % 4 == 0:
            return F_.graph_conv_parts([("x", vertex_features)], vertex_adjacency, self.w0, self.w1, residual)
        out = F_.graph_conv(vertex_features, vertex_adjacency, self.w0, self.w1)
        return out if residual is None else out + residual


class _BiasFreeLinear(nn.Linear):
    """``nn.Linear(bias=False)`` whose product runs on the library GEMM (same ``weight`` state-dict key)."""

    def __init__(self, in_features: int, out_features: int):
        super().__init__(in_features, out_features, bias=False)

    def forward(self, x: Tensor) -> Tensor:
        return F_.linear(x, self.weight)


class ResGraphConv(nn.Module):
    """Two GraphConvs plus an additive skip, linearly projected when the widths differ -- reference
    meshRCNN/layers.py:71-100 (submodules ``conv0``, ``conv1``, ``projection``)."""

    def __init__(self, in_features: int, out_features: int):
        super().__init__()
        self.conv0 = GraphConv(in_features, out_features)
        self.conv1 = GraphConv(out_features, out_features)
        self.projection = _BiasFreeLinear(in_features, out_features) if in_features != out_features else nn.Identity()

    def forward(self, vertex_features, vertex_adjacency: Tensor) -> Tensor:
        """``vertex_features``: SV x in_features or a list of parts (see ``GraphConv.forward``)."""
        if isinstance(vertex_features, (list, tuple)):
            dense = [t for _, t in vertex_features]
            skip = self.projection(dense[0] if len(dense) == 1 else F_.concat_cols(dense))
        else:
            skip = self.projection(vertex_features)
        # the skip connection is added in the epilogue of conv1's gather kernel
        return self.conv1(self.conv0(vertex_features, vertex_adjacency), vertex_adjacency, residual=skip)


def _default_mesh_index(mesh_index, image_sizes):
    return [1 for _ in image_sizes] if mesh_index is None else mesh_index


# ShapeNet stages: evaluate linear(VertexAlign(maps)) as per-texel projections + a 128-wide row gather
# (functional.vert_align_linear, csrc/align_proj.cu) instead of materialising the SV x 3840 VertexAlign output.
# Same values up to fp32 summation order; False restores the literal two-step evaluation (used by the parity tests).
FUSE_ALIGN_BOTTLENECK = True


def _align_and_project(align: "VertexAlign", linear: nn.Linear, img_feature_maps, vertex_positions, vertice_index,
                       image_sizes, mesh_index) -> Tensor:
    """``linear(align(maps, positions, ...))`` of reference meshRCNN/layers.py:151-155 / :226-230."""
    if not FUSE_ALIGN_BOTTLENECK or linear.bias is not None:
        return linear(align(img_feature_maps, vertex_positions, vertice_index, image_sizes, mesh_index))
    if align.training:                                          # the checks of VertexAlign.forward (layers.py:528-532)
        assert len(vertice_index) == len(image_sizes)
        assert list(mesh_index) == [1 for _ in image_sizes]
    assert len(mesh_index) == len(image_sizes)
    return F_.vert_align_linear(img_feature_maps, vertex_positions, vertice_index, image_sizes, mesh_index, linear.weight,
                                bilinear=_bilinear(align))


def _stage_input(vertex_positions, pooled, vertex_features, use_input_features):
    """[features? | positions | pooled] (reference layers.py:160-165) -- as parts, or concatenated (literal mode)."""
    if vertex_features is not None:
        assert use_input_features
    else:
        assert not use_input_features
    if FUSE_STAGE_INPUTS:
        parts = [("pos", vertex_positions), ("tex", pooled) if isinstance(pooled, F_.TexelTerm) else ("x", pooled)]
        return ([("x", vertex_features)] if vertex_features is not None else []) + parts
    parts = [vertex_positions, pooled]
    if vertex_features is not None:
        parts = [vertex_features] + parts
    return F_.concat_cols(parts)


def _with_pos(vertex_positions, x):
    """[positions | x] (reference layers.py:245,250,327,332)."""
    if FUSE_STAGE_INPUTS:
        return [("pos", vertex_positions), ("x", x)]
    return F_.concat_cols([vertex_positions, x])


class ResVertixRefineShapenet(nn.Module):
    """Residual ShapeNet refinement stage -- reference meshRCNN/layers.py:103-178.
    NB the argument order of ``forward`` differs from the other two stage classes (:130-133)."""

    def __init__(self, use_input_features: bool = True, num_features: int = 128, alignment_size: int = 3840,
                 ndims: int = 3, align_mode: str = "reference"):
        super().__init__()
        self.vertAlign = VertexAlign(align_mode)
        self.linear = _BiasFreeLinear(alignment_size, num_features)
        in_channels = num_features + ndims + (num_features if use_input_features else 0)
        self.resGraphConv0 = ResGraphConv(in_channels, num_features)
        self.use_input_features = use_input_features
        self.resGraphConv1 = ResGraphConv(num_features, num_features)
        self.resGraphConv2 = ResGraphConv(num_features, num_features)
        self.graphConv = GraphConv(num_features, ndims)
        self.tanh = nn.Tanh()

    def forward(self, vertice_index: List[int], img_feature_maps: List[Tensor], vertex_adjacency: Tensor,
                vertex_positions: Tensor, image_sizes: List, vertex_features: Optional[Tensor] = None,
                mesh_index: List[int] = None) -> Tuple[Tensor, Tensor]:
        mesh_index = _default_mesh_index(mesh_index, image_sizes)
        projected = _align_and_project(self.vertAlign, self.linear, img_feature_maps, vertex_positions, vertice_index,
                                       image_sizes, mesh_index)
        x = _stage_input(vertex_positions, projected, vertex_features, self.use_input_features)
        x = self.resGraphConv0(x, vertex_adjacency)
        x = self.resGraphConv1(x, vertex_adjacency)
        x = self.resGraphConv2(x, vertex_adjacency)
        delta = self.tanh(self.graphConv(x, vertex_adjacency))      # tanh(relu(.)): offsets >= 0 (:174-175)
        return vertex_positions + delta, x


class VertixRefineShapeNet(nn.Module):
    """Plain ShapeNet refinement stage -- reference meshRCNN/layers.py:181-259."""

    def __init__(self, use_input_features: bool = True, num_features: int = 128, alignment_size: int = 3840,
                 ndims: int = 3, align_mode: str = "reference"):
        super().__init__()
        self.vertAlign = VertexAlign(align_mode)
        self.linear0 = _BiasFreeLinear(alignment_size, num_features)
        in_channels = num_features + ndims + (num_features if use_input_features else 0)
        self.graphConv0 = GraphConv(in_channels, num_features)
        self.use_input_features = use_input_features
        self.graphConv1 = GraphConv(num_features + ndims, num_features)
        self.graphConv2 = GraphConv(num_features + ndims, num_features)
        self.linear1 = _BiasFreeLinear(num_features, ndims)
        self.tanh = nn.Tanh()

    def forward(self, vertice_index: List[int], img_feature_maps: List[Tensor], vertex_adjacency: Tensor,
                vertex_positions: Tensor, image_sizes: List, mesh_index: List[int] = None,
                vertex_features: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
        mesh_index = _default_mesh_index(mesh_index, image_sizes)
        projected = _align_and_project(self.vertAlign, self.linear0, img_feature_maps, vertex_positions, vertice_index,
                                       image_sizes, mesh_index)
        x = _stage_input(vertex_positions, projected, vertex_features, self.use_input_features)
        x = self.graphConv0(x, vertex_adjacency)
        x = self.graphConv1(_with_pos(vertex_positions, x), vertex_adjacency)
        x = self.graphConv2(_with_pos(vertex_positions, x), vertex_adjacency)
        if FUSE_STAGE_INPUTS:
            return F_.position_head(x, vertex_positions, self.linear1.weight, pos_first=None), x
        delta = self.tanh(self.linear1(x))
        return vertex_positions + delta, x


class VertixRefinePix3D(nn.Module):
    """Pix3D refinement stage (single RoI feature map, no bottleneck) -- reference meshRCNN/layers.py:262-339."""

    def __init__(self, use_input_features: bool = True, num_features: int = 128, alignment_size: int = 256,
                 ndims: int = 3, align_mode: str = "reference"):
        super().__init__()
        self.vertAlign = VertexAlign(align_mode)
        in_channels = alignment_size + ndims + (num_features if use_input_features else 0)
        self.graphConv0 = GraphConv(in_channels, num_features)
        self.use_input_features = use_input_features
        self.graphConv1 = GraphConv(num_features + ndims, num_features)
        self.graphConv2 = GraphConv(num_features + ndims, num_features)
        self.linear = _BiasFreeLinear(num_features + ndims, ndims)
        self.tanh = nn.Tanh()

    def forward(self, vertice_index: List[int], back_bone_features: Tensor, vertex_adjacency: Tensor,
                vertex_positions: Tensor, image_sizes: List, mesh_index: List[int] = None,
                vertex_features: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
        mesh_index = _default_mesh_index(mesh_index, image_sizes)
        if FUSE_STAGE_INPUTS and self.graphConv0.w0.shape[1] % 4 == 0 and not _bilinear(self.vertAlign):
            # VertexAlign stays factored: graphConv0 projects the texels and gathers rows (functional.TexelTerm)
            if self.vertAlign.training:                             # the checks of VertexAlign.forward (layers.py:528-532)
                assert len(vertice_index) == len(image_sizes)
                assert list(mesh_index) == [1 for _ in image_sizes]
            assert len(mesh_index) == len(image_sizes)
            # (the registered topology of a Cubify adjacency already holds the per-vertex mesh ids)
            aligned = F_.TexelTerm(back_bone_features, vertex_positions, vertice_index, image_sizes, mesh_index,
                                   topo=topology.lookup(vertex_adjacency, vertex_positions.shape[0]))
        else:
            # literal mode, and bilinear mode: the SV x C aligned features are materialised and enter as a dense part
            aligned = self.vertAlign([back_bone_features], vertex_positions, vertice_index, image_sizes, mesh_index)
        x = _stage_input(vertex_positions, aligned, vertex_features, self.use_input_features)
        x = self.graphConv0(x, vertex_adjacency)
        x = self.graphConv1(_with_pos(vertex_positions, x), vertex_adjacency)
        x = self.graphConv2(_with_pos(vertex_positions, x), vertex_adjacency)
        if FUSE_STAGE_INPUTS:
            return F_.position_head(x, vertex_positions, self.linear.weight, pos_first=True), x
        delta = self.tanh(self.linear(F_.concat_cols([vertex_positions, x])))
        return vertex_positions + delta, x
