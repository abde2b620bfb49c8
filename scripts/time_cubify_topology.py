"""Times Cubify's watertight topology against the reference topology, with CUDA events, the two modes alternating repetition
by repetition in one process:

  * the whole ``Cubify.forward`` (count kernels, the counter read-back, output allocation, emit kernels) at
    BASELINE configs[3] (64 dense 48^3 grids, threshold 0.5) and at the configs[1] input (32 blobs on a 24^3 grid,
    threshold 0.2);
  * one configs[1] Pix3D training step per mode: ``RefinementHead("pix3d", cubify_topology=mode)`` on 32 blobs of 24^3 at
    0.2, 256 x 12 x 12 RoI maps, 224-px images, losses and backward, with the ground truth the normalised
    ``Cubify(0.5, topology=mode)`` of a second blob set -- built as bench.py's ``HeadWorkload`` builds it (same seeds, same
    weights), without the gradient all-reduce buckets.  The L2 is overwritten before every timed step, as bench.py does.

Also records the vertex / face / directed-edge counts of each mode and the device name and power limit.  Prints one JSON
record.

    python scripts/time_cubify_topology.py [--reps 30] [--step-reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from meshrcnn_b200 import synthetic  # noqa: E402
from meshrcnn_b200.layers import Cubify  # noqa: E402
from meshrcnn_b200.mesh_sampling import normalize_mesh  # noqa: E402
from meshrcnn_b200.pipeline import MeshTargets, RefinementHead, weighted_loss  # noqa: E402

MODES = ("reference", "watertight")


def device_record():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        power, clock = [x.strip() for x in out.strip().split(",")]
    except Exception:                                 # no nvidia-smi: record that instead of guessing
        power = clock = "unknown"
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def time_alternating(fns, reps, before=None, warmup=3):
    """{name: stats} for callables timed alternately (one repetition of each per round), after warm-up.  ``before`` runs
    outside the event bracket ahead of every timed call."""
    for fn in fns.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            if before is not None:
                before()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    out = {}
    for k, v in ms.items():
        v.sort()
        out[k] = {"median_ms": round(v[len(v) // 2], 4), "min_ms": round(v[0], 4), "max_ms": round(v[-1], 4)}
    return out


def cubify_case(label, vox, th, reps):
    mods = {m: Cubify(th, topology=m) for m in MODES}
    counts = {}
    for m, mod in mods.items():
        v, vi, f, fi, adj = mod(vox)
        counts[m] = {"vertices": int(v.shape[0]), "faces": int(f.shape[0]), "directed_edges": int(adj.shape[1])}
    timing = time_alternating({m: (lambda mod=mod: mod(vox)) for m, mod in mods.items()}, reps)
    return {"workload": label, "counts": counts, "timing": timing,
            "watertight_over_reference": round(timing["watertight"]["median_ms"] / timing["reference"]["median_ms"], 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--step-reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_cubify_topology: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {**device_record(), "reps": args.reps, "step_reps": args.step_reps}

    res["cubify_configs3"] = cubify_case("configs[3]: 64 dense 48^3 grids, th=0.5, whole Cubify.forward",
                                         synthetic.dense_voxels(64, 48, 0).to(dev), 0.5, args.reps)
    res["cubify_configs1"] = cubify_case("configs[1] input: 32 blobs on 24^3, th=0.2, whole Cubify.forward",
                                         synthetic.blob_voxels(32, 24, 0).to(dev), 0.2, args.reps)

    # configs[1] training step, bench.HeadWorkload's inputs and weights (seed-0 batch, GT seed 1000, torch.manual_seed(1))
    B, grid, img = 32, 24, 224
    vox = synthetic.blob_voxels(B, grid, 0).to(dev)
    fmap = synthetic.feature_maps(B, [synthetic.PIX3D_MAP], 0)[0].to(dev).requires_grad_()
    gt_vox = synthetic.blob_voxels(B, grid, 1000).to(dev)
    sizes = [(img, img)] * B
    heads, targets, counts = {}, {}, {}
    for m in MODES:
        torch.manual_seed(1)
        heads[m] = RefinementHead("pix3d", cubify_threshold=0.2, cubify_topology=m).to(dev).train()
        gv, gvi, gf, gfi, _ = Cubify(0.5, topology=m)(gt_vox)
        targets[m] = MeshTargets(torch.cat([normalize_mesh(v) for v in gv.split(gvi)]), gf, gvi, gfi)
        v, _, f, _, adj = heads[m].cubify(vox)
        counts[m] = {"vertices": int(v.shape[0]), "faces": int(f.shape[0]), "directed_edges": int(adj.shape[1]),
                     "gt_vertices": int(gv.shape[0])}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)       # larger than the 126 MB L2
    losses = {}

    def step(m):
        def run():
            heads[m].zero_grad(set_to_none=True)
            fmap.grad = None
            out = heads[m](vox, fmap, sizes, targets[m])
            weighted_loss(out).backward()
            losses[m] = {k: float(v.detach()) for k, v in out.items()}
        return run

    timing = time_alternating({m: step(m) for m in MODES}, args.step_reps, before=flush.zero_)
    res["pix3d_step_configs1"] = {
        "workload": "configs[1] Pix3D training step: B=32, 24^3 blobs th=0.2, 256x12x12 maps, 224px, 3 x VertixRefinePix3D, "
                    "10k-point chamfer+normal(k=10)+edge losses, fwd+bwd; predicted and GT meshes from the same topology; "
                    "L2 overwritten before each step",
        "counts": counts, "timing": timing, "last_losses": losses,
        "watertight_over_reference": round(timing["watertight"]["median_ms"] / timing["reference"]["median_ms"], 4)}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
