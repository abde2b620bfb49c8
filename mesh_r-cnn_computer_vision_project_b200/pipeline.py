"""The refinement-stage loop (SURVEY.md 8a-8): Cubify -> stage 0 (no input features) -> stages 1.. (with features)
-> training losses or the eval output dict.  Mirrors the hot-path section of ``ShapeNetModel.forward``
(reference meshRCNN/shapenet_model.py:71-99) and ``Pix3DModel.forward`` (meshRCNN/pix3d_model.py:87-115); the
backbone / voxel branch upstream of it are out of scope and are replaced by the ``voxel_probs`` /
``feature_maps`` arguments.
"""
import os
from typing import List, Optional, Sequence, Tuple, Union

import torch
import torch.nn as nn
from torch import Tensor

from .layers import Cubify, ResVertixRefineShapenet, VertixRefinePix3D, VertixRefineShapeNet
from .loss_functions import batched_mesh_loss, mesh_loss, sample_gt_cloud


class MeshTargets:
    """Ground-truth side of a packed batch; same fields as reference ``data.dataloader.Batch`` (:21-36) that the
    losses read: ``meshes = (vertices SVgt x 3, faces SFgt x 3 local ids)``, ``vertice_index``, ``face_index``."""

    def __init__(self, vertices: Tensor, faces: Tensor, vertice_index: Sequence[int], face_index: Sequence[int]):
        self.meshes = (vertices, faces)
        self.vertice_index = list(vertice_index)
        self.face_index = list(face_index)

    def to(self, *args, **kwargs):
        v, f = self.meshes
        return MeshTargets(v.to(*args, **kwargs), f.to(*args, **kwargs), self.vertice_index, self.face_index)

    def slice(self, lo: int, hi: int) -> "MeshTargets":
        v, f = self.meshes
        vo, fo = sum(self.vertice_index[:lo]), sum(self.face_index[:lo])
        vn, fn = sum(self.vertice_index[lo:hi]), sum(self.face_index[lo:hi])
        return MeshTargets(v[vo:vo + vn], f[fo:fo + fn], self.vertice_index[lo:hi], self.face_index[lo:hi])


class RefinementHead(nn.Module):
    """``cubify`` + ``refineStages`` with the reference's attribute names (state-dict keys ``cubify.*``,
    ``refineStages.{i}.*`` as in shapenet_model.py:27-41 / pix3d_model.py:32-44).

    ``model``: "pix3d" (VertixRefinePix3D, 256-channel RoI map), "shapenet" (VertixRefineShapeNet) or
    "shapenet_residual" (ResVertixRefineShapenet).  ``align_mode``: "reference" (the reference's VertexAlign arithmetic) or
    "bilinear" (bilinear sampling with gradients to the vertex positions, ``layers.VertexAlign``)."""

    def __init__(self, model: str = "pix3d", cubify_threshold: float = 0.2, alignment_channels: Optional[int] = None,
                 vertex_feature_dim: int = 128, num_refinement_stages: int = 3, align_mode: str = "reference"):
        super().__init__()
        cls = {"pix3d": VertixRefinePix3D, "shapenet": VertixRefineShapeNet,
               "shapenet_residual": ResVertixRefineShapenet}[model]
        if alignment_channels is None:
            alignment_channels = 256 if model == "pix3d" else 3840
        self.model = model
        self.cubify = Cubify(cubify_threshold)
        stages = [cls(alignment_size=alignment_channels, use_input_features=False, num_features=vertex_feature_dim,
                      align_mode=align_mode)]
        for _ in range(num_refinement_stages - 1):
            stages.append(cls(alignment_size=alignment_channels, use_input_features=True,
                              num_features=vertex_feature_dim, align_mode=align_mode))
        self.refineStages = nn.ModuleList(stages)
        self.overlap_losses = True          # training: per-stage losses on a second CUDA stream (see forward)
        self._loss_stream = None
        self._pack_plan = None              # functional.PackPlan: the blocks' weight images of a pass in one launch
        self.sample_gt_early = os.environ.get("MRB_EARLY_GT", "1") != "0"   # training: GT clouds of all stages drawn during Cubify's read-back stall

    def forward(self, voxel_probs: Tensor, feature_maps: Union[Tensor, List[Tensor]], image_sizes,
                targets: Optional[MeshTargets] = None, mesh_index: Optional[List[int]] = None,
                loss_randomness=None, voxel_logits: bool = False) -> dict:
        """``voxel_logits=True``: ``voxel_probs`` holds the voxel head's logits (``VoxelBranch.forward_logits``); the sigmoid
        is evaluated inside Cubify's first kernel (SURVEY 8 f-1)."""
        if self.training and targets is None:
            raise ValueError("In training mode, targets should be passed")
        mesh_index = [1 for _ in image_sizes] if mesh_index is None else mesh_index
        from . import functional as F_
        if self._pack_plan is None:
            self._pack_plan = F_.PackPlan()
        single_map = feature_maps if torch.is_tensor(feature_maps) else None
        with F_.pack_plan(self._pack_plan if voxel_probs.is_cuda else None, single_map):   # one weight-packing launch per pass
            return self._forward(voxel_probs, feature_maps, image_sizes, targets, mesh_index, loss_randomness, voxel_logits)

    def _forward(self, voxel_probs, feature_maps, image_sizes, targets, mesh_index, loss_randomness, voxel_logits) -> dict:
        from . import functional as F_
        gt_clouds = None
        if self.training and voxel_probs.is_cuda and loss_randomness is None and self.sample_gt_early:
            # The ground-truth samples of the stages do not depend on the predicted mesh: they are drawn while the launching
            # thread waits for Cubify's counters (functional.defer_until_stall).  The Philox seeds are taken from torch's
            # generator here, in the order the lazy path would take them (stage by stage: predicted cloud, GT cloud), so the
            # draws are the ones batched_mesh_loss(positions, ...) would make after the same torch.manual_seed.
            n_stage = len(self.refineStages)
            seeds = F_._next_seeds(2 * n_stage)
            loss_randomness = [({"seed": seeds[2 * s]}, {"seed": seeds[2 * s + 1]}) for s in range(n_stage)]
            gt_clouds = []
            F_.defer_until_stall(lambda: gt_clouds.extend(sample_gt_cloud(targets, **loss_randomness[s][1])
                                                          for s in range(n_stage)))
        pos0, vertice_index, faces, face_index, adj_index = self.cubify(voxel_probs, from_logits=voxel_logits)
        if gt_clouds is not None and len(gt_clouds) != len(self.refineStages):
            gt_clouds = None                            # the hook did not run (a Cubify path without the stall): lazy sampling
        positions = [pos0]
        feats = None
        overlap = self.training and self.overlap_losses and voxel_probs.is_cuda
        if overlap:
            main = torch.cuda.current_stream()
            if self._loss_stream is None or self._loss_stream.device != voxel_probs.device:
                self._loss_stream = torch.cuda.Stream(device=voxel_probs.device)
            side = self._loss_stream
        terms = []
        for s, stage in enumerate(self.refineStages):
            kw = {} if feats is None else {"vertex_features": feats}
            new_pos, feats = stage(vertice_index, feature_maps, adj_index, positions[-1], image_sizes,
                                   mesh_index=mesh_index, **kw)
            positions.append(new_pos)
            if overlap:
                # The loss of stage s depends only on its positions.  It is issued on a second stream right away, so that its
                # long, issue-bound nearest-neighbour kernels share the SMs with the tensor-core / gather kernels of stage
                # s + 1 (those leave ~75 % of the issue slots idle) and the GPU never waits for launches -- same terms, same
                # order of sampler draws as batched_mesh_loss(positions[1:], ...) after the loop (reference
                # shapenet_model.py:92-95).  Autograd runs each backward node on the stream of its forward, so the backward
                # passes overlap the same way.  (Stream priorities -- stages high, losses low -- were measured: no gain.)
                side.wait_stream(main)
                new_pos.record_stream(side)
                if gt_clouds is not None:
                    gt_clouds[s].record_stream(side)
                with torch.cuda.stream(side):
                    terms.append(mesh_loss(new_pos, faces, adj_index, vertice_index, face_index, targets,
                                           randomness=None if loss_randomness is None else loss_randomness[s],
                                           gt_cloud=None if gt_clouds is None else gt_clouds[s]))
        out = {}
        if self.training:
            if overlap:
                main.wait_stream(side)
                for t in terms:
                    for x in t:
                        x.record_stream(main)
                from . import functional as F_
                chamfer, normal, edge = (F_.weighted_scalar_sum([t[i] for t in terms]) for i in range(3))
            else:
                chamfer, normal, edge = batched_mesh_loss(positions[1:], faces, adj_index, vertice_index, face_index,
                                                          targets, randomness=loss_randomness, gt_clouds=gt_clouds)
            out.update({"chamfer_loss": chamfer, "edge_loss": edge, "normal_loss": normal})
        else:
            out.update({"vertex_positions": positions, "edge_index": adj_index, "face_index": face_index,
                        "vertice_index": vertice_index, "faces": faces, "mesh_index": mesh_index})
        return out


# default loss weights of the reference CLI (train.py:19-74): chamfer 1, normal 0.1, edge 0.5
LOSS_WEIGHTS = {"chamfer_loss": 1.0, "normal_loss": 0.1, "edge_loss": 0.5}


def weighted_loss(losses: dict, weights: dict = LOSS_WEIGHTS) -> Tensor:
    """Weighted sum of the loss dict (reference utils/train_utils.py:208-225)."""
    from . import functional as F_
    keys = [k for k in weights if k in losses]
    if not keys:
        return None
    return F_.weighted_scalar_sum([losses[k] for k in keys], [weights[k] for k in keys])
