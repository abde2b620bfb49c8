"""Times the reference-mode ``VertexAlign()`` module, forward and forward + backward, through the module API only (so the
same script times any tree that has the module), with CUDA events:

  * the configs[2]-shard shape: B = 32 blobs on a 48^3 grid through Cubify (threshold 0.2), about 206 k vertices, the four
    ResNet50 maps (3840 channels) of 137-px images;
  * Pix3D: B = 32 blobs on a 24^3 grid, about 50 k vertices, one 256 x 12 x 12 RoI map, 224-px images.

Maps are fp32 and bf16.  Positions are the cubified vertex count moved in-frustum (synthetic.in_frustum_positions), so the
gather reads real texels.  The backward takes a fixed random upstream gradient.  The SV x C output is written to HBM (it
exceeds L2 at the ShapeNet shape); the maps stay L2 resident between repetitions.  Prints one JSON record with the device
name and power limit.

    python scripts/time_vert_align_module.py [--reps 30]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from meshrcnn_b200 import synthetic  # noqa: E402
from meshrcnn_b200.layers import Cubify, VertexAlign  # noqa: E402


def device_record():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        power, clock = [x.strip() for x in out.strip().split(",")]
    except Exception:                                 # no nvidia-smi: record that instead of guessing
        power = clock = "unknown"
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def time_alternating(fns, reps):
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


def case(grid, maps, img, dev, reps):
    verts, v_index, _, _, _ = Cubify(0.2)(synthetic.blob_voxels(32, grid, 0).to(dev))
    SV = verts.shape[0]
    pos = synthetic.in_frustum_positions(SV, img, 9).to(dev)
    sizes, mi = [(img, img)] * len(v_index), [1] * len(v_index)
    align = VertexAlign().eval()
    fmaps = [m.to(dev) * 0.05 for m in synthetic.feature_maps(32, maps, 1)]
    gout = torch.randn(SV, sum(c for c, _, _ in maps), generator=torch.Generator().manual_seed(2)).to(dev)
    res = {"vertices": SV, "channels": sum(c for c, _, _ in maps)}
    for dtype in (torch.float32, torch.bfloat16):
        fm = [m.to(dtype).requires_grad_() for m in fmaps]

        def fwd():
            with torch.no_grad():
                align(fm, pos, v_index, sizes, mi)

        def fwd_bwd():
            out = align(fm, pos, v_index, sizes, mi)
            out.backward(gout)
            for m in fm:
                m.grad = None

        res["fp32" if dtype == torch.float32 else "bf16"] = time_alternating({"fwd": fwd, "fwd_bwd": fwd_bwd}, reps)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_vert_align_module: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {**device_record(), "reps": args.reps}
    res["shapenet_configs2_shard"] = case(48, synthetic.SHAPENET_MAPS, 137, dev, args.reps)
    res["pix3d"] = case(24, [synthetic.PIX3D_MAP], 224, dev, args.reps)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
