"""Drop-in boundary (SURVEY 8b / INTEGRATION.md): the reference's OWN ``meshRCNN/shapenet_model.py`` is executed unmodified
(byte-for-byte copy under oracle/_ref, see oracle/build_ref.py) with its ``.layers`` / ``.loss_functions`` imports bound to
this repo's modules -- exactly the edit INTEGRATION.md describes -- and run on the GPU in training and eval mode."""
import importlib.util
import os
import sys
import types

import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_MODEL = os.path.join(ROOT, "oracle", "_ref", "meshRCNN", "shapenet_model.py")


class TinyBackbone(nn.Module):
    """Stands in for ShapeNetResNet50 (out of scope): returns (class output | loss, four maps of the ResNet50 shapes for a
    137 x 137 input) like reference shapenet_model.py:112-136."""

    SHAPES = ((256, 35), (512, 18), (1024, 9), (2048, 5))

    def __init__(self):
        super().__init__()
        self.proj = nn.ModuleList([nn.Conv2d(3, c, 1) for c, _ in self.SHAPES])

    def forward(self, x, targets=None):
        maps = [p(nn.functional.adaptive_avg_pool2d(x, s)) for p, (_, s) in zip(self.proj, self.SHAPES)]
        out = x.mean(dim=(1, 2, 3))
        return (out.sum() * 0.0 if self.training else out), maps


def _load_reference_model_module():
    import meshrcnn_b200.layers as our_layers
    import meshrcnn_b200.loss_functions as our_losses
    from meshrcnn_b200.batch import Batch
    import torchvision.models.resnet as tv_resnet
    if not hasattr(tv_resnet, "model_urls"):
        tv_resnet.model_urls = {"resnet50": ""}                    # removed in torchvision >= 0.13 (SURVEY 8c shim)
    saved = {k: sys.modules.get(k) for k in ("meshRCNN", "meshRCNN.layers", "meshRCNN.loss_functions", "data", "data.dataloader")}
    try:
        pkg = types.ModuleType("meshRCNN"); pkg.__path__ = [os.path.dirname(REF_MODEL)]
        data = types.ModuleType("data"); data.__path__ = []
        dl = types.ModuleType("data.dataloader"); dl.Batch = Batch
        sys.modules.update({"meshRCNN": pkg, "meshRCNN.layers": our_layers, "meshRCNN.loss_functions": our_losses,
                            "data": data, "data.dataloader": dl})
        spec = importlib.util.spec_from_file_location("meshRCNN.shapenet_model", REF_MODEL)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


@pytest.mark.skipif(not os.path.exists(REF_MODEL), reason="oracle/_ref not populated (run oracle/build_ref.py in the dev container)")
@pytest.mark.parametrize("residual", [True, False])
def test_reference_shapenet_model_runs_on_our_layers(lib, residual):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.batch import Batch
    from meshrcnn_b200.layers import Cubify
    from meshrcnn_b200.mesh_sampling import normalize_mesh
    from meshrcnn_b200.serialization import Mesh
    mod = _load_reference_model_module()
    assert mod.Cubify.__module__.startswith("mesh") and "b200" in mod.Cubify.__module__        # our classes were bound
    torch.manual_seed(0)
    model = mod.ShapeNetModel(TinyBackbone(), residual=residual).cuda()
    keys = set(model.state_dict())
    assert {"cubify.kernel", "cubify.deltas", "voxelBranch.0.weight", "voxelBranch.3.bias",
            "refineStages.2." + ("graphConv.w0" if residual else "linear1.weight"),
            "refineStages.0." + ("resGraphConv0.projection.weight" if residual else "graphConv0.w1")} <= keys
    B = 2
    images = torch.rand(B, 3, 137, 137).cuda()
    gv, gvi, gf, gfi, _ = Cubify(0.5)(synthetic.blob_voxels(B, 24, 1000).cuda())
    meshes = [Mesh(normalize_mesh(v), f) for v, f in zip(gv.split(gvi), gf.split(gfi))]
    gt_vox = (synthetic.blob_voxels(B, 48, 1000) > 0.5).float().cuda()
    batch = Batch(images, gt_vox, 48, meshes, torch.zeros(B, dtype=torch.long).cuda())
    # training mode: the reference forward (shapenet_model.py:43-99) on our Cubify / stages / losses
    model.train()
    out = model(images, batch)
    assert {"voxel_loss", "chamfer_loss", "edge_loss", "normal_loss", "backbone_loss"} <= set(out)
    total = out["voxel_loss"] + out["chamfer_loss"] + 0.1 * out["normal_loss"] + 0.5 * out["edge_loss"]
    assert bool(torch.isfinite(total))
    total.backward()
    g = [p.grad for n, p in model.named_parameters() if n.startswith("refineStages") or n.startswith("voxelBranch")]
    assert all(x is not None and bool(torch.isfinite(x).all()) for x in g)
    assert float(model.voxelBranch[0].weight.grad.abs().sum()) > 0            # voxel_loss gradient reached the voxel head
    # eval mode: the output dict of shapenet_model.py:92-99
    model.eval()
    with torch.no_grad():
        res = model(images)
    assert {"voxels", "vertex_positions", "edge_index", "face_index", "vertice_index", "faces", "mesh_index", "backbone"} <= set(res)
    assert len(res["vertex_positions"]) == 4 and res["voxels"].shape == (B, 48, 48, 48)
    assert sum(res["vertice_index"]) == res["vertex_positions"][-1].shape[0]
    assert bool(torch.isfinite(res["vertex_positions"][-1]).all())


class ShapeNetCallSites(nn.Module):
    """The hot-path half of a ShapeNet model written only against the module API that INTEGRATION.md section 2 documents: the
    six names imported there and the call shapes of the stage loop (Cubify -> stages with ``mesh_index`` / ``vertex_features``
    -> ``batched_mesh_loss(positions[1:], ...)`` on a ``Batch``, ``voxel_loss`` on the VoxelBranch output).  It runs on every
    checkout; the test above additionally runs the original project's own file where a copy of that project is present."""

    def __init__(self, backbone, residual, cubify_threshold=0.2):
        super().__init__()
        from meshrcnn_b200.layers import Cubify, ResVertixRefineShapenet, VertixRefineShapeNet, VoxelBranch
        self.backbone = backbone
        self.voxelBranch = VoxelBranch(2048, 48)
        self.cubify = Cubify(cubify_threshold)
        stage = ResVertixRefineShapenet if residual else VertixRefineShapeNet
        self.refineStages = nn.ModuleList([stage(use_input_features=i > 0) for i in range(3)])

    def forward(self, images, targets=None):
        from meshrcnn_b200.loss_functions import batched_mesh_loss, voxel_loss
        backbone_out, maps = self.backbone(images, targets)
        voxel_grid = self.voxelBranch(nn.functional.interpolate(maps[-1], scale_factor=4.8, mode="bilinear",
                                                                align_corners=True))
        sizes = [tuple(images.shape[-2:])] * images.shape[0]
        mesh_index = [1] * images.shape[0]
        vs, vertice_index, faces, face_index, adj_index = self.cubify(voxel_grid)
        positions, feats = [vs], None
        for stage in self.refineStages:
            kw = {} if feats is None else {"vertex_features": feats}
            new_pos, feats = stage(vertice_index, maps, adj_index, positions[-1], sizes, mesh_index=mesh_index, **kw)
            positions.append(new_pos)
        if self.training:
            chamfer, normal, edge = batched_mesh_loss(positions[1:], faces, adj_index, vertice_index, face_index, targets)
            return {"voxel_loss": voxel_loss(voxel_grid, targets.voxels), "chamfer_loss": chamfer, "normal_loss": normal,
                    "edge_loss": edge, "backbone_loss": backbone_out}
        return {"voxels": voxel_grid, "vertex_positions": positions, "edge_index": adj_index, "face_index": face_index,
                "vertice_index": vertice_index, "faces": faces, "mesh_index": mesh_index, "backbone": backbone_out}


@pytest.mark.parametrize("residual", [True, False])
def test_documented_call_sites_run_on_our_layers(lib, residual):
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.batch import Batch
    from meshrcnn_b200.layers import Cubify
    from meshrcnn_b200.mesh_sampling import normalize_mesh
    from meshrcnn_b200.serialization import Mesh
    torch.manual_seed(0)
    model = ShapeNetCallSites(TinyBackbone(), residual).cuda()
    with torch.no_grad():             # occupancy ~0.9 everywhere: one closed 48^3 cube per image, whatever the random weights
        model.voxelBranch[3].weight.mul_(1e-3)
        model.voxelBranch[3].bias.fill_(2.0)
    keys = set(model.state_dict())    # checkpoint keys of the original project (INTEGRATION.md section 2)
    assert {"cubify.kernel", "cubify.deltas", "voxelBranch.0.weight", "voxelBranch.3.bias",
            "refineStages.2." + ("graphConv.w0" if residual else "linear1.weight"),
            "refineStages.0." + ("resGraphConv0.projection.weight" if residual else "graphConv0.w1")} <= keys
    B = 2
    images = torch.rand(B, 3, 137, 137).cuda()
    gv, gvi, gf, gfi, _ = Cubify(0.5)(synthetic.blob_voxels(B, 24, 1000).cuda())
    meshes = [Mesh(normalize_mesh(v), f) for v, f in zip(gv.split(gvi), gf.split(gfi))]
    gt_vox = (synthetic.blob_voxels(B, 48, 1000) > 0.5).float().cuda()
    batch = Batch(images, gt_vox, 48, meshes, torch.zeros(B, dtype=torch.long).cuda())
    model.train()
    out = model(images, batch)
    total = out["voxel_loss"] + out["chamfer_loss"] + 0.1 * out["normal_loss"] + 0.5 * out["edge_loss"]
    assert all(bool(torch.isfinite(out[k])) for k in ("voxel_loss", "chamfer_loss", "normal_loss", "edge_loss"))
    total.backward()
    g = [p.grad for n, p in model.named_parameters() if n.startswith("refineStages") or n.startswith("voxelBranch")]
    assert all(x is not None and bool(torch.isfinite(x).all()) for x in g)
    assert float(model.voxelBranch[0].weight.grad.abs().sum()) > 0
    model.eval()
    with torch.no_grad():
        res = model(images)
    assert len(res["vertex_positions"]) == 4 and res["voxels"].shape == (B, 48, 48, 48)
    assert res["vertice_index"] == [6 * 48 * 48 + 2] * B              # a closed 48^3 cube surface: 6 n^2 + 2 corners
    assert sum(res["vertice_index"]) == res["vertex_positions"][-1].shape[0]
    assert bool(torch.isfinite(res["vertex_positions"][-1]).all())
