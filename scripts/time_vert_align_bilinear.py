"""Times the opt-in bilinear VertexAlign against the reference mode, forward + backward, with CUDA events:

  * the configs[1] Pix3D head: B = 32 blobs on a 24^3 grid through Cubify (threshold 0.2), 256 x 12 x 12 RoI maps, 224-px
    images, three VertixRefinePix3D stages;
  * one ResVertixRefineShapenet stage at the configs[2] shard size: B = 32 blobs on a 48^3 grid, the four ResNet50 maps
    (3840 channels) of 137-px images;
  * the bilinear VertexAlign call alone at both sizes (functional.vert_align_bilinear / vert_align_linear(bilinear=True)).

Positions are the cubified vertex count moved in-frustum (synthetic.in_frustum_positions), so both modes sample real
texels.  The two modes use the same weights and alternate repetition by repetition; the loss is a fixed random linear
functional of the stage outputs.  Working sets stay in L2 between repetitions where they fit.  Prints one JSON record with
the device name and power limit.

    python scripts/time_vert_align_bilinear.py [--reps 30]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import meshrcnn_b200.layers as L  # noqa: E402
from meshrcnn_b200 import functional as F_, synthetic  # noqa: E402
from meshrcnn_b200.pipeline import RefinementHead  # noqa: E402


def device_record():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        power, clock = [x.strip() for x in out.strip().split(",")]
    except Exception:                                 # no nvidia-smi: record that instead of guessing
        power = clock = "unknown"
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def time_pair(fns, reps):
    """{name: stats} for callables timed alternately (one repetition of each per round), after warm-up."""
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    out = {}
    for k, v in ms.items():
        v.sort()
        out[k] = {"median_ms": v[len(v) // 2], "min_ms": v[0], "max_ms": v[-1]}
    return out


def case(model, B, grid, dev):
    head = RefinementHead(model, cubify_threshold=0.2).to(dev).train()
    with torch.no_grad():
        for p in head.parameters():
            p.mul_(0.2)
    vox = synthetic.blob_voxels(B, grid, 0).to(dev)
    verts, v_index, faces, f_index, adj = head.cubify(vox)
    img = 224 if model == "pix3d" else 137
    maps = [synthetic.PIX3D_MAP] if model == "pix3d" else synthetic.SHAPENET_MAPS
    fmaps = [m.to(dev) * 0.05 for m in synthetic.feature_maps(B, maps, 1)]
    pos = synthetic.in_frustum_positions(verts.shape[0], img, 9).to(dev)
    return head, v_index, adj, fmaps, pos, [(img, img)] * B


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_vert_align_bilinear: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {**device_record(), "reps": args.reps}

    # configs[1]: the Pix3D head, three stages
    head, v_index, adj, fmaps, pos, sizes = case("pix3d", 32, 24, dev)
    SV = pos.shape[0]
    g = torch.Generator().manual_seed(3)
    go_p, go_f = torch.randn(SV, 3, generator=g).to(dev), torch.randn(SV, 128, generator=g).to(dev)
    fm = fmaps[0].requires_grad_()
    p0 = pos.clone().requires_grad_()

    def head_step(mode):
        def run():
            for st in head.refineStages:
                st.vertAlign.mode = mode
            cur, feats = p0, None
            for st in head.refineStages:
                kw = {} if feats is None else {"vertex_features": feats}
                cur, feats = st(v_index, fm, adj, cur, sizes, **kw)
            ((cur * go_p).sum() + (feats * go_f).sum()).backward()
            head.zero_grad(set_to_none=True)
            fm.grad = p0.grad = None
        return run

    go_a = torch.randn(SV, 256, generator=g).to(dev)

    def align_only():
        out = F_.vert_align_bilinear([fm], p0, v_index, sizes, [1] * len(sizes))
        (out * go_a).sum().backward()
        fm.grad = p0.grad = None

    res["pix3d_head"] = {
        "workload": "configs[1] Pix3D head: B=32, 24^3 blobs th=0.2, 256x12x12 maps, 224px, 3 x VertixRefinePix3D, fwd+bwd "
                    "of the stages (no losses), in-frustum positions",
        "vertices": SV,
        "timing": time_pair({"reference": head_step("reference"), "bilinear": head_step("bilinear")}, args.reps),
        "vert_align_bilinear_fwd_bwd_alone": time_pair({"bilinear": align_only}, args.reps)["bilinear"],
        "aligned_matrix_bytes": SV * 256 * 4}
    t = res["pix3d_head"]["timing"]
    res["pix3d_head"]["bilinear_minus_reference_ms"] = t["bilinear"]["median_ms"] - t["reference"]["median_ms"]
    del head, fm, p0

    # configs[2] shard: one residual ShapeNet stage
    head, v_index, adj, fmaps, pos, sizes = case("shapenet_residual", 32, 48, dev)
    st = head.refineStages[0]
    SV = pos.shape[0]
    go_p, go_f = torch.randn(SV, 3, generator=g).to(dev), torch.randn(SV, 128, generator=g).to(dev)
    fms = [m.requires_grad_() for m in fmaps]
    p0 = pos.clone().requires_grad_()

    def stage_step(mode):
        def run():
            st.vertAlign.mode = mode
            cur, feats = st(v_index, fms, adj, p0, sizes)
            ((cur * go_p).sum() + (feats * go_f).sum()).backward()
            st.zero_grad(set_to_none=True)
            for m in fms:
                m.grad = None
            p0.grad = None
        return run

    go_l = torch.randn(SV, 128, generator=g).to(dev)

    def bottleneck(bilinear):
        def run():
            out = F_.vert_align_linear(fms, p0, v_index, sizes, [1] * len(sizes), st.linear.weight, bilinear=bilinear)
            (out * go_l).sum().backward()
            st.zero_grad(set_to_none=True)
            for m in fms:
                m.grad = None
            p0.grad = None
        return run

    res["shapenet_residual_stage"] = {
        "workload": "configs[2] shard: B=32, 48^3 blobs th=0.2, four ResNet50 maps (3840 ch) of 137px images, one "
                    "ResVertixRefineShapenet stage (no input features), fwd+bwd, in-frustum positions",
        "vertices": SV,
        "timing": time_pair({"reference": stage_step("reference"), "bilinear": stage_step("bilinear")}, args.reps),
        "align_bottleneck_fwd_bwd": time_pair({"reference": bottleneck(False), "bilinear": bottleneck(True)}, args.reps)}
    t = res["shapenet_residual_stage"]["timing"]
    res["shapenet_residual_stage"]["bilinear_minus_reference_ms"] = t["bilinear"]["median_ms"] - t["reference"]["median_ms"]
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
