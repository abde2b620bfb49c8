"""Times eval_utils.compare_meshes (GT-10 scale, 5 thresholds) at B = 32 and 10 000 samples per mesh on the config-1 Pix3D
meshes (24^3 blobs through Cubify at 0.2, ground truth from seed + 1000), stage by stage, and in the same run a chunked
torch.cdist composition of the same metrics on the same samples (what a user without the kernels would write).  CUDA events,
warm-up first; the working set (a few MB) stays in L2 between repetitions.  Prints the device name and power limit.

    python scripts/time_mesh_metrics.py [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from meshrcnn_b200 import functional as F_, synthetic  # noqa: E402
from meshrcnn_b200.eval_utils import compare_meshes, mesh_metric_names  # noqa: E402

B, N, TAUS, SEED = 32, 10000, (0.1, 0.2, 0.3, 0.4, 0.5), 5


def device_record():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        power, clock = [x.strip() for x in out.strip().split(",")]
    except Exception:                                 # no nvidia-smi: record that instead of guessing
        power = clock = "unknown"
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def timeit(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    return {"median_ms": ms[len(ms) // 2], "min_ms": ms[0], "max_ms": ms[-1]}


def cdist_metrics(p, n_p, q, n_q, chunk=2048):
    """The same per-mesh metrics from dense fp32 distance blocks (torch.cdist, chunk x Q at a time)."""
    rows = []
    for b in range(p.shape[0]):
        def nn(a, c):
            d, i = [], []
            for lo in range(0, a.shape[0], chunk):
                m, j = (torch.cdist(a[lo:lo + chunk], c) ** 2).min(1)
                d.append(m)
                i.append(j)
            return torch.cat(d), torch.cat(i)
        d_p, i_p = nn(p[b], q[b])
        d_q, i_q = nn(q[b], p[b])
        dot_p, dot_q = (n_p[b] * n_q[b][i_p]).sum(1), (n_q[b] * n_p[b][i_q]).sum(1)
        row = [d_p.double().mean() + d_q.double().mean(), 0.5 * (dot_p.double().mean() + dot_q.double().mean()),
               0.5 * (dot_p.abs().double().mean() + dot_q.abs().double().mean())]
        r_p, r_q = d_p.sqrt(), d_q.sqrt()
        for tau in TAUS:
            pr, rc = 100 * (r_p < tau).double().mean(), 100 * (r_q < tau).double().mean()
            row += [pr, rc, 2 * pr * rc / (pr + rc + 1e-8)]
        rows.append(torch.stack(row))
    return torch.stack(rows).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_mesh_metrics: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    pv, pvi, pf, pfi, _, _ = F_.cubify(synthetic.blob_voxels(B, 24, 0).to(dev), 0.2)
    gv, gvi, gf, gfi, _, _ = F_.cubify(synthetic.blob_voxels(B, 24, 1000).to(dev), 0.2)
    call = lambda: compare_meshes(pv, pf, pvi, pfi, gv, gf, gvi, gfi, num_samples=N, thresholds=TAUS, seed=SEED, reduce=False)

    # the stages of one call, each timed on its own
    s = F_.mesh_gt_scale(gv, gvi)
    p, n_p, _ = F_.sample_surface(pv, pf, pvi, pfi, N, seed=SEED, scale=s)
    q, n_q, _ = F_.sample_surface(gv, gf, gvi, gfi, N, seed=SEED + 1, scale=s)
    d_p, i_p, _, d_q, i_q, _ = F_.knn_search(p, q, 0)
    res = {"workload": "compare_meshes, B=%d, %d samples per mesh, GT-10, %d thresholds, config-1 Pix3D meshes" % (B, N, len(TAUS)),
           **device_record(),
           "compare_meshes": timeit(call, args.reps),
           "stages": {
               "mesh_gt_scale": timeit(lambda: F_.mesh_gt_scale(gv, gvi), args.reps),
               "sample_surface_pred_and_gt": timeit(lambda: (F_.sample_surface(pv, pf, pvi, pfi, N, seed=SEED, scale=s),
                                                             F_.sample_surface(gv, gf, gvi, gfi, N, seed=SEED + 1, scale=s)),
                                                    args.reps),
               "knn_search_k0": timeit(lambda: F_.knn_search(p, q, 0), args.reps),
               "mesh_metrics": timeit(lambda: F_.mesh_metrics(d_p, i_p, d_q, i_q, n_p, n_q, TAUS), args.reps)},
           "cdist_composition_same_samples": timeit(lambda: cdist_metrics(p, n_p, q, n_q), max(3, args.reps // 4))}

    # agreement of the two compositions on the same samples
    got = call()
    ref = cdist_metrics(p, n_p, q, n_q)
    names = mesh_metric_names(TAUS)
    table = torch.stack([got[k] for k in names], 1)
    res["agreement_vs_cdist"] = {
        "chamfer_max_rel": float(((table[:, 0] - ref[:, 0]).abs() / ref[:, 0]).max()),
        "abs_nc_max_abs": float((table[:, 2] - ref[:, 2]).abs().max()),
        "pr_max_abs_percent": float((table[:, 3:] - ref[:, 3:]).abs().max())}
    res["means"] = {k: float(got[k].double().mean()) for k in names}
    res["speedup_vs_cdist"] = res["cdist_composition_same_samples"]["median_ms"] / res["compare_meshes"]["median_ms"]
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
