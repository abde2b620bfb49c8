#!/usr/bin/env python
"""Benchmark of the voxel-to-mesh refinement hot path (BASELINE.json metric: meshes/s, fwd+bwd, 3 refine stages).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's own CPU implementation (oracle/_ref)
    python bench.py --check                                        # bench-shape loss parity: CUDA arm vs the fp64 oracle
    python bench.py --steps K --dump-outputs DIR                   # + the last timed step's losses and gradients as .npy

The library is the one build() left in the tree: bench.py compiles nothing, and refuses a library that was not built from
the sources as they are now.  The inputs, the weights and the sampling seeds of the timed steps depend only on the
arguments, so two builds run with the same arguments can be compared output for output.

Headline workload (BASELINE.json configs[1], the configuration the metric is quoted on for one GPU): Pix3D head,
random-init, batch 32 of synthetic 24^3 blob voxel probabilities (threshold 0.2) + 32 x 256 x 12 x 12 RoI feature maps for
224 x 224 images, 3 x VertixRefinePix3D, chamfer / normal / edge losses on 10 000-point clouds (k = 10) against
ground-truth meshes = normalised Cubify(0.5) of a second blob set, weighted sum, backward to the GCN weights and the
feature maps.  A "step" = Cubify + 3 stages + losses + backward over one batch.  With N GPUs every rank runs 32 meshes
(weak scaling; the 32 N meshes of the job are dealt to the ranks by occupied-voxel count) and the weight gradients are
all-reduced (SUM) with NCCL inside the timed region, one bucket per stage, issued from backward hooks.

One JSON line on stdout (rank 0).  `value` = steps with inputs resident in HBM; `e2e` = the same through the public module
API with inputs in pinned host memory, H2D + D2H inside the timed region.  `extra_configs` carries the other BASELINE
configs measured in the same run: configs[2] (ShapeNet residual head, 48^3, 3840 channels, per-rank shard of the
batch-256 job, with the all-reduce when N > 1), configs[3] (Cubify stress) and configs[4] (chamfer sweep, Gpairs/s).
"""
import argparse
import gc
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B_PER_GPU = 32
THRESH = 0.2
N_POINTS = 10000
KNN = 10
STARTUP_SECONDS = 2.0                   # untimed start-up phase of the CUDA arm (see run_cuda)
E2E_WARMUP_MIN = 12                     # untimed e2e steps before the timed e2e region (first uses of the copy path)
# ncu dram__bytes_read.sum + dram__bytes_write.sum of one k_nn_grid<10> launch at the bench shape (profiles/); one
# mrb_knn_fwd call = k_grid_build + 2 such launches (one per direction)
KNN_DRAM_BYTES_PER_LAUNCH = 11.74e6
KNN_ISSUE_SLOTS_BUSY_NCU = 0.79

WORKLOADS = {
    # BASELINE configs[1]
    "pix3d": dict(model="pix3d", grid=24, img=224, maps="PIX3D",
                  label="pix3d head: batch %d/GPU, 24^3 blob voxels th=0.2, 256x12x12 RoI features, 224px images, "
                        "3 x VertixRefinePix3D, 10k-point chamfer+normal(k=10)+edge losses, fwd+bwd (BASELINE configs[1])"),
    # BASELINE configs[2]: one rank's shard of the batch-256 job
    "shapenet_residual": dict(model="shapenet_residual", grid=48, img=137, maps="SHAPENET",
                              label="shapenet residual head: batch %d/GPU (per-rank shard of the batch-256 job), 48^3 blob voxels "
                                    "th=0.2, four ResNet50 maps (3840 channels) of 137px images, 3 x ResVertixRefineShapenet, "
                                    "10k-point chamfer+normal(k=10)+edge losses, fwd+bwd (BASELINE configs[2])"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + throttle reasons with a background `nvidia-smi -lms 200` process while the timed regions run
    (a separate process: NVML calls made from inside the benchmark process were seen to stall kernel launches)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, "/tmp/mrb_clocks_%d.csv" % os.getpid()

    def start(self):
        import shutil
        import subprocess
        exe = shutil.which("nvidia-smi")
        if exe is None:
            log("[bench] nvidia-smi not found: no clock samples")
            return
        self.out = open(self.path, "w")
        self.proc = subprocess.Popen([exe, "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                      "-lms", "200"], stdout=self.out, stderr=subprocess.DEVNULL)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:      # noqa: BLE001
            self.proc.kill()
        self.out.close()
        mhz, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6 or not f[0].isdigit():
                continue
            mhz.append(int(f[0]))
            mx = int(f[1]) if f[1].isdigit() else mx
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.remove(self.path)
        except OSError:
            pass
        mhz.sort()
        # median of the samples taken under load (the sampler also runs through idle phases between regions)
        loaded = [m for m in mhz if mx is None or m >= 0.5 * mx] or mhz
        return {"sm_mhz": loaded[len(loaded) // 2] if loaded else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(mhz)}


# ---------------------------------------------------------------------------------------------------------------
# timing-event pool
# ---------------------------------------------------------------------------------------------------------------
class EventPool:
    """Every CUDA timing event the benchmark uses is created AND recorded once here, before anything is timed, and then
    reused.  Round 1 found that the ~11th step of every loop bracketed by *freshly created* timing events stalled the
    launching thread for 20 - 130 ms (the driver grows its event storage in chunks at first record); creating a throw-away
    pool and deleting it did not remove the stall on every box, keeping the very same event objects does."""

    def __init__(self, n_pairs):
        self.pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_pairs)]
        for a, b in self.pairs:
            a.record()
            b.record()
        torch.cuda.synchronize()
        self.next = 0

    def take(self, n):
        if self.next + n > len(self.pairs):
            self.next = 0
        out = self.pairs[self.next:self.next + n]
        assert len(out) == n, "event pool too small"
        self.next += n
        return out


def _stats(ms):
    s = sorted(ms)
    return {"mean_ms": round(sum(s) / len(s), 3), "median_ms": round(s[len(s) // 2], 3), "max_ms": round(s[-1], 3),
            "min_ms": round(s[0], 3)}


# ---------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------
def _maps(kind):
    from meshrcnn_b200 import synthetic
    return [synthetic.PIX3D_MAP] if kind == "PIX3D" else list(synthetic.SHAPENET_MAPS)


def make_host_inputs(name, B, rank, world, balance=True):
    """Host tensors of this rank's shard: voxel probabilities, feature maps, GT voxel probabilities.

    The job's 32 * world meshes are the per-rank seeded sets concatenated (seed r -> meshes 32 r .. 32 r + 31); in
    throughput mode they are dealt to the ranks by occupied-voxel count in snake order (sharding.balanced_split,
    equal_counts) so that no rank waits for a rank that drew larger meshes.  world == 1 keeps the seed-0 batch unchanged."""
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.sharding import balanced_split
    w = WORKLOADS[name]
    if world > 1 and balance:
        vox_all = torch.cat([synthetic.blob_voxels(B, w["grid"], r) for r in range(world)])
        costs = (vox_all > THRESH).flatten(1).sum(1).tolist()
        mine = balanced_split(costs, world, equal_counts=True)[rank]
        vox = vox_all[mine].contiguous()
        del vox_all
    else:
        vox = synthetic.blob_voxels(B, w["grid"], rank)
    fmaps = synthetic.feature_maps(vox.shape[0], _maps(w["maps"]), rank)
    gt_vox = synthetic.blob_voxels(vox.shape[0], w["grid"], rank + 1000)
    return vox, fmaps, gt_vox


class HeadWorkload:
    """Cubify + 3 refinement stages + losses + backward (+ the per-stage gradient all-reduce) on this rank's shard."""

    def __init__(self, name, dev, rank, world, map_dtype=torch.float32):
        from meshrcnn_b200.layers import Cubify
        from meshrcnn_b200.mesh_sampling import normalize_mesh
        from meshrcnn_b200.pipeline import MeshTargets, RefinementHead
        from meshrcnn_b200.sharding import StagedGradBuckets
        self.name, self.dev, self.w = name, dev, WORKLOADS[name]
        self.vox_h, self.fmaps_h, gt_vox_h = make_host_inputs(name, B_PER_GPU, rank, world)
        self.B = self.vox_h.shape[0]
        self.sizes = [(self.w["img"], self.w["img"])] * self.B
        self.single_map = self.w["maps"] == "PIX3D"
        torch.manual_seed(1)                                         # identical weights on every rank
        self.head = RefinementHead(self.w["model"], cubify_threshold=THRESH).to(dev).train()
        self.buckets = StagedGradBuckets.per_stage(self.head)
        # ground truth: normalised Cubify(0.5) of a second blob set (the reference's GT recipe, download_dataset.py:88-114)
        gv, gvi, gfaces, gfi, _ = Cubify(0.5)(gt_vox_h.to(dev))
        self.gt = MeshTargets(torch.cat([normalize_mesh(v) for v in gv.split(gvi)]), gfaces, gvi, gfi)
        self.vox_d = self.vox_h.to(dev)
        if map_dtype != torch.float32:                               # bf16 feature-map mode (north star: rtol 2e-2)
            self.fmaps_h = [f.to(map_dtype) for f in self.fmaps_h]
        self.fmaps_d = [f.to(dev).requires_grad_() for f in self.fmaps_h]

    def step(self, vox_d=None, fmaps_d=None, exchange=True):
        vox_d = self.vox_d if vox_d is None else vox_d
        fmaps_d = self.fmaps_d if fmaps_d is None else fmaps_d
        from meshrcnn_b200.pipeline import weighted_loss
        self.buckets.enabled = exchange
        self.buckets.zero()
        for f in fmaps_d:
            f.grad = None
        losses = self.head(vox_d, fmaps_d[0] if self.single_map else fmaps_d, self.sizes, self.gt)
        weighted_loss(losses).backward()
        # the step's collective: one NCCL all-reduce(SUM) per stage bucket, issued from backward hooks as soon as that
        # stage's weight gradients are final; here the stream waits for them
        self.buckets.finish(exchange)
        return losses

    def stats(self):
        verts, vi, faces, fi, adj = self.head.cubify(self.vox_d)
        return {"B": self.B, "SV": int(verts.shape[0]), "SF": int(faces.shape[0]), "E": int(adj.shape[1])}

    def h2d_bytes(self):
        return int(self.vox_h.numel() * 4 + sum(f.numel() * 4 for f in self.fmaps_h))


def timed_resident(wl, pool, steps, flush, sync_all):
    from meshrcnn_b200 import _lib
    ev = pool.take(steps)
    sync_all()
    l0 = _lib.launch_count
    for i, (a, b) in enumerate(ev):
        flush.zero_()                      # L2 flush between timed iterations (outside the event bracket)
        a.record()
        losses = wl.step()
        if i == steps - 1:
            last = {k: v.detach() for k, v in losses.items()}
        # the graph keeps tensors of the step alive: freed inside the bracket, so the next step does not allocate around it
        del losses
        b.record()
    sync_all()
    launches = (_lib.launch_count - l0) // steps
    return [a.elapsed_time(b) for a, b in ev], launches, last


def step_outputs(wl, losses):
    """What the last step handed its caller, as host float32 arrays: the three losses and, from backward, the gradient of
    every refinement weight and of the feature maps (this rank's shard)."""
    out = {k: v.float().cpu().numpy() for k, v in losses.items()}
    for i, f in enumerate(wl.fmaps_d):
        out["feature_map%d.grad" % i] = f.grad.float().cpu().numpy()
    for name, p in wl.head.named_parameters():
        if p.grad is not None:
            out[name + ".grad"] = p.grad.float().cpu().numpy()
    return out


def dump_outputs(arrays, path, limit=64 << 20):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        raise SystemExit("bench.py: %d bytes of outputs exceed the %d-byte dump limit" % (total, limit))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    log("[bench] wrote %d arrays (%d bytes) to %s" % (len(arrays), total, path))


def timed_e2e(wl, pool, steps, warmup, flush, sync_all):
    """The same step through the public module API with the inputs in pinned host memory: per step the H2D copy of one
    batch (voxel grid + feature maps) into pre-allocated device buffers, the step, and a D2H read of the three losses.

    The copies run on a copy stream into two alternating sets of device buffers, like a prefetching loader: the bracket of
    step i issues the copy of step i + 1's inputs (step 0's bracket issues its own copy and step 1's, the last bracket
    none), so K copies fall inside the K timed brackets, the step waits on its buffers' event, and a buffer set is
    overwritten only after the step that read it has finished."""
    dev = wl.dev
    vox_pin = wl.vox_h.pin_memory()
    fmaps_pin = [f.pin_memory() for f in wl.fmaps_h]
    slots = [(torch.empty_like(wl.vox_d), [torch.empty_like(f).requires_grad_() for f in wl.fmaps_d]) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    host_out = torch.empty(3, dtype=torch.float32).pin_memory()
    main = torch.cuda.current_stream(dev)
    copy_stream = torch.cuda.Stream(dev)
    for e in consumed:
        e.record(main)

    def issue_copy(slot):
        vox_s, fmap_s = slots[slot]
        with torch.cuda.stream(copy_stream), torch.no_grad():
            copy_stream.wait_event(consumed[slot])
            vox_s.copy_(vox_pin, non_blocking=True)
            for s_, p_ in zip(fmap_s, fmaps_pin):
                s_.copy_(p_, non_blocking=True)
            ready[slot].record(copy_stream)

    def one(i, last):
        t0 = time.perf_counter()
        if i == 0:
            issue_copy(0)
        if not last:
            issue_copy((i + 1) % 2)
        slot = i % 2
        main.wait_event(ready[slot])
        t1 = time.perf_counter()
        losses = wl.step(slots[slot][0], slots[slot][1])
        consumed[slot].record(main)
        t2 = time.perf_counter()
        host_out.copy_(torch.stack([losses["chamfer_loss"], losses["normal_loss"], losses["edge_loss"]]).detach(),
                       non_blocking=True)
        main.synchronize()                 # the step's result is on the host
        t3 = time.perf_counter()
        return (t1 - t0, t2 - t1, t3 - t2)

    for i in range(warmup):
        one(i, i == warmup - 1)
    sync_all()
    ev = pool.take(steps)
    phases = []
    for i, (a, b) in enumerate(ev):
        flush.zero_()
        a.record()
        phases.append(one(i, i == steps - 1))
        b.record()
    sync_all()
    ms = [a.elapsed_time(b) for a, b in ev]
    return ms, phases, host_out.clone()


def measure_fma_peak(dev):
    """FP32 FMA issue rate measured in this run (TFLOP/s, 2 flop per FMA): the peak of the FP32-issue-bound kernels."""
    from meshrcnn_b200 import _lib
    lib = _lib.load()
    out = torch.zeros(1, dtype=torch.float32, device=dev)
    blocks, iters = 148 * 16, 2000
    best = 0.0
    for i in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        flop = lib.mrb_fma_peak(_lib.ptr(out), iters, blocks, _lib.stream_ptr())
        b.record()
        torch.cuda.synchronize()
        if flop < 0:
            raise RuntimeError("mrb_fma_peak failed")
        if i:
            best = max(best, flop / (a.elapsed_time(b) * 1e-3) / 1e12)
    return best


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "src": "fallback (B200_PROFILING.md)"}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
        peaks["src"] = "MEASURED_PEAKS.json"
    return peaks


def kernel_rooflines(breakdown, stats, peaks, fma_peak, widths):
    """Per-kernel achieved rates from the instrumented steps (CUDA events around every C-ABI call, single stream)."""
    B, SV, SF, E = stats["B"], stats["SV"], stats["SF"], stats["E"]
    roof = {}

    def per_call(name):
        return breakdown[name]["ms_per_step"] / breakdown[name]["calls_per_step"] * 1e-3

    if "mrb_knn_fwd" in breakdown:
        t = per_call("mrb_knn_fwd")
        pairs = B * N_POINTS * N_POINTS                       # BASELINE.md section 3: B*P*Q per call (both directions)
        tflops = pairs * 8 / t / 1e12                         # SURVEY 8d: 8 flop per pair (3 sub, 3 mul, 2 add)
        roof["mrb_knn_fwd"] = {
            "kernel": "k_grid_build + 2 x k_nn_grid<10> (one mrb_knn_fwd call)", "bound": "fp32_issue",
            "achieved": round(tflops, 2), "peak": round(fma_peak, 2), "unit": "TFLOP/s", "frac": round(tflops / fma_peak, 4),
            "peak_src": "FP32 FMA microbenchmark of this run (mrb_fma_peak, 2 flop per FMA)",
            "pairs_per_call": pairs, "ms_per_call": round(t * 1e3, 4), "Gpairs_per_s": round(pairs / t / 1e9, 1),
            "issue_slots_busy_ncu": KNN_ISSUE_SLOTS_BUSY_NCU,
            "note": "algorithmic work of the brute-force problem; the exact cell-grid search visits ~0.8 % of the pairs, "
                    "so the kernel's own hardware bound is its issue-slot utilisation (ncu)"}
    if "mrb_csr_gather_fwd" in breakdown:
        t = per_call("mrb_csr_gather_fwd")
        byts = 2 * 4 * SV * 128 + 4 * (E + SV + 1)            # SURVEY 8d compulsory bytes
        roof["mrb_csr_gather_fwd"] = {"bound": "hbm", "achieved": round(byts / t / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                      "frac": round(byts / t / 1e9 / peaks["hbm_gbs"], 4)}
    if "mrb_gemm_tc_acc" in breakdown and "mrb_gemm_tc" in breakdown and widths:
        # split-input GraphConv: forward projections x @ [W0x | W1x] (mrb_gemm_tc_acc) and input gradients gy @ [W0x | W1x]^T
        # (mrb_gemm_tc); `widths` = (rows M, K, N) of every call of one step
        ms = (breakdown["mrb_gemm_tc_acc"]["ms_per_step"] + breakdown["mrb_gemm_tc"]["ms_per_step"]) * 1e-3
        flops = sum(2.0 * m * k * n for m, k, n in widths)
        byts = sum(4.0 * m * (k + n) for m, k, n in widths)
        tf32_peak = peaks.get("bf16_tflops", 2250.0) / 2.0
        roof["tcgen05 projections (mrb_gemm_tc_acc + mrb_gemm_tc)"] = {
            "bound": "tensor", "achieved": round(3 * flops / ms / 1e12, 1), "peak": round(tf32_peak, 1),
            "unit": "TFLOP/s (TF32 issued, 3xTF32; peak = measured bf16 peak / 2)",
            "frac": round(3 * flops / ms / 1e12 / tf32_peak, 4), "tensor_tflops_fp32_equiv": round(flops / ms / 1e12, 1),
            "hbm_gbs": round(byts / ms / 1e9, 1), "hbm_frac": round(byts / ms / 1e9 / peaks["hbm_gbs"], 4),
            "calls_per_step": len(widths)}
    if "mrb_gemm_tc_wgrad_split" in breakdown:
        ms = breakdown["mrb_gemm_tc_wgrad_split"]["ms_per_step"] * 1e-3
        calls = breakdown["mrb_gemm_tc_wgrad_split"]["calls_per_step"]
        flops = calls * 2.0 * SV * 128 * 256
        byts = calls * 4.0 * SV * (128 + 256)
        tf32_peak = peaks.get("bf16_tflops", 2250.0) / 2.0
        roof["mrb_gemm_tc_wgrad_split"] = {"bound": "tensor", "achieved": round(3 * flops / ms / 1e12, 1), "peak": round(tf32_peak, 1),
                                           "unit": "TFLOP/s (TF32 issued)", "frac": round(3 * flops / ms / 1e12 / tf32_peak, 4),
                                           "hbm_gbs": round(byts / ms / 1e9, 1), "hbm_frac": round(byts / ms / 1e9 / peaks["hbm_gbs"], 4)}
    if "mrb_gc_gather_fwd" in breakdown:
        t = per_call("mrb_gc_gather_fwd")
        byts = 3 * 4 * SV * 128 + 4 * (E + SV + 1)            # self + neighbour matrix read once + output (DESIGN.md section 4)
        roof["mrb_gc_gather_fwd"] = {"bound": "hbm", "achieved": round(byts / t / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                     "frac": round(byts / t / 1e9 / peaks["hbm_gbs"], 4),
                                     "note": "per-call average over the y-only, +position and +texel variants of one step"}
    if "mrb_cubify_emit" in breakdown:
        t = (breakdown["mrb_cubify_emit"]["ms_per_step"] + breakdown["mrb_cubify_count"]["ms_per_step"]) * 1e-3
        byts = 4 * B * stats["grid"] ** 3 + 12 * SV + 24 * SF + 16 * E + 16 * B
        roof["mrb_cubify"] = {"bound": "hbm", "achieved": round(byts / t / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                              "frac": round(byts / t / 1e9 / peaks["hbm_gbs"], 4)}
    return roof


def instrumented_breakdown(wl, reps=2):
    from meshrcnn_b200 import _lib
    wl.head.overlap_losses = False                      # single stream: per-call device times are not stretched by co-running kernels
    with _lib.timed_calls() as tc:
        for _ in range(reps):
            wl.step(exchange=False)                     # rank-local: the other ranks are not in this region
    wl.head.overlap_losses = True
    return {k: {"ms_per_step": round(v / reps, 4), "calls_per_step": tc.calls[k] // reps} for k, v in
            sorted(tc.ms.items(), key=lambda kv: -kv[1])}


# ---------------------------------------------------------------------------------------------------------------
# extra configs (BASELINE configs[2], [3], [4]) measured in the same run
# ---------------------------------------------------------------------------------------------------------------
def reduce_max_ms(ms, dev, world):
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def extra_shapenet_shard(dev, rank, world, pool, flush, sync_all, steps, peaks):
    wl = HeadWorkload("shapenet_residual", dev, rank, world)
    torch.cuda.reset_peak_memory_stats(dev)
    for _ in range(3):
        wl.step()
    sync_all()
    ms, launches, _ = timed_resident(wl, pool, steps, flush, sync_all)
    total = reduce_max_ms(sum(ms), dev, world)
    out = None
    if rank == 0:
        st = wl.stats()
        bd = instrumented_breakdown(wl, reps=1)
        out = {"workload": wl.w["label"] % wl.B, "metric": "meshes/sec (fwd+bwd, 3 refine stages)",
               "value": round(wl.B * world * steps / (total * 1e-3), 1), "unit": "meshes/s", "n_gpus": world, "steps": steps,
               "warmup": 3, "ms_per_step": round(total / steps, 3), "scaling": "weak", "per_gpu": st,
               "grad_bucket_bytes": 4 * wl.buckets.flat_numel, "gpu_launches": int(launches),
               "peak_mem_GB": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2),
               "collective": "NCCL all-reduce(SUM), one bucket per stage, issued from backward hooks" if world > 1 else "none (N = 1)",
               "breakdown_ms": {k: v for k, v in list(bd.items())[:14]}}
    del wl
    torch.cuda.empty_cache()
    return out


def extra_bf16_maps(dev, rank, world, pool, flush, sync_all, steps):
    """The headline workload with the feature maps held in bf16 (half the map bytes in HBM and over PCIe; positions,
    weights, accumulation and every loss stay fp32; parity: rtol 2e-2, tests/test_layers_gpu.py)."""
    wl = HeadWorkload("pix3d", dev, rank, world, map_dtype=torch.bfloat16)
    for _ in range(3):
        wl.step()
    sync_all()
    ms, launches, _ = timed_resident(wl, pool, steps, flush, sync_all)
    total = reduce_max_ms(sum(ms), dev, world)
    out = None
    if rank == 0:
        out = {"workload": (WORKLOADS["pix3d"]["label"] % wl.B) + " -- feature maps in bf16", "metric": "meshes/sec (fwd+bwd, 3 refine stages)",
               "value": round(wl.B * world * steps / (total * 1e-3), 1), "unit": "meshes/s", "n_gpus": world, "steps": steps, "warmup": 3,
               "ms_per_step": round(total / steps, 3), "dtype": "bf16 feature maps, f32 everything else",
               "map_bytes_per_step": int(sum(f.numel() * 2 for f in wl.fmaps_h)), "gpu_launches": int(launches)}
    del wl
    torch.cuda.empty_cache()
    return out


def extra_cubify_stress(dev, rank, world, pool, flush, sync_all, peaks, reps=5):
    """BASELINE configs[3]: 64 dense 48^3 grids (density 0.5, ~116k-vertex meshes); whole Cubify.forward per call."""
    from meshrcnn_b200 import _lib, synthetic
    from meshrcnn_b200.layers import Cubify
    vox = synthetic.dense_voxels(64, 48, rank).to(dev)
    cub = Cubify(0.5)
    for _ in range(3):
        v, vi, f, fi, adj = cub(vox)
    SV, SF, E = int(v.shape[0]), int(f.shape[0]), int(adj.shape[1])
    del v, f, adj
    sync_all()
    ev = pool.take(reps)
    for a, b in ev:
        flush.zero_()
        a.record()
        cub(vox)
        b.record()
    sync_all()
    ms = [a.elapsed_time(b) for a, b in ev]
    t = reduce_max_ms(sum(ms) / reps, dev, world) * 1e-3
    out = None
    if rank == 0:
        with _lib.timed_calls() as tc:
            for _ in range(reps):
                cub(vox)
        byts = 4 * vox.numel() + 12 * SV + 24 * SF + 16 * E + 16 * 64          # SURVEY 8d algorithmic bytes
        k_ms = (tc.ms["mrb_cubify_count"] + tc.ms["mrb_cubify_emit"]) / reps
        out = {"workload": "Cubify stress: 64 dense 48^3 grids/GPU, density 0.5, th=0.5 (BASELINE configs[3])",
               "SV": SV, "SF": SF, "E": E, "algorithmic_bytes": byts, "ms_per_call": round(t * 1e3, 4),
               "value": round(byts * world / t / 1e9, 1), "unit": "GB/s", "n_gpus": world,
               "roofline": {"bound": "hbm", "achieved": round(byts / t / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": round(byts / t / 1e9 / peaks["hbm_gbs"], 4),
                            "note": "whole Cubify.forward incl. the count read-back sync and output allocation"},
               "kernels_only": {"ms": round(k_ms, 4), "GBps": round(byts / (k_ms * 1e-3) / 1e9, 1),
                                "frac": round(byts / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                                "count_ms": round(tc.ms["mrb_cubify_count"] / reps, 4),
                                "emit_ms": round(tc.ms["mrb_cubify_emit"] / reps, 4)},
               "meshes_per_s": round(64 * world / t, 1)}
    del vox
    torch.cuda.empty_cache()
    return out


def extra_chamfer_sweep(dev, rank, world, pool, flush, sync_all, fma_peak, reps=10):
    """BASELINE configs[4]: B = 32 clouds of P = Q = 10 000 surface samples per GPU; Gpairs/s = B*P*Q / time of one call that
    produces both directions (BASELINE.md section 3); also the full chamfer + normal loss forward + backward."""
    from meshrcnn_b200 import functional as F_, synthetic
    from meshrcnn_b200.layers import Cubify
    B, P = 32, N_POINTS

    def cloud(seed):
        vv, vvi, ff, ffi, _ = Cubify(THRESH)(synthetic.blob_voxels(B, 24, seed).to(dev))
        c, _ = F_.sample_points(vv * 0.05, ff, vvi, ffi, P, seed=seed + 1)
        return c

    p, q = cloud(rank), cloud(rank + 1000)
    res = {}

    def timeit(fn, key):
        for _ in range(3):
            fn()
        sync_all()
        ev = pool.take(reps)
        for a, b in ev:
            a.record()
            fn()
            b.record()
        sync_all()
        res[key] = reduce_max_ms(sum(a.elapsed_time(b) for a, b in ev) / reps, dev, world) * 1e-3

    timeit(lambda: F_.chamfer_knn(p, q, KNN), "k10")
    timeit(lambda: F_.chamfer_knn(p, q, 0), "k0")
    pg = p.clone().requires_grad_()

    def loss_fwd_bwd():
        pg.grad = None
        l1, l2, ip, iq, kp, kq = F_.chamfer_knn(pg, q, KNN)
        n1, n2 = F_.normal_distance(pg, q, kp, kq, ip, iq)
        ((l1 + l2) / N_POINTS - 0.1 * (n1 + n2) / N_POINTS).backward()

    timeit(loss_fwd_bwd, "loss")
    if rank != 0:
        return None
    pairs = B * P * P
    tf = pairs * 8 / res["k10"] / 1e12
    return {"workload": "chamfer+normal sweep: B=32 clouds/GPU of P=Q=10000 surface samples (BASELINE configs[4])",
            "pairs_per_call": pairs, "n_gpus": world,
            "value": round(world * pairs / res["k10"] / 1e9, 1), "unit": "Gpairs/s (B*P*Q / time, one call = both directions + top-10 sets)",
            "ms_per_call": round(res["k10"] * 1e3, 4),
            "chamfer_only_k0": {"Gpairs_per_s": round(world * pairs / res["k0"] / 1e9, 1), "ms_per_call": round(res["k0"] * 1e3, 4)},
            "chamfer_normal_loss_fwd_bwd": {"ms": round(res["loss"] * 1e3, 4), "clouds_per_s": round(world * B / res["loss"], 1)},
            "roofline": {"bound": "fp32_issue", "achieved": round(tf, 2), "peak": round(fma_peak, 2), "unit": "TFLOP/s",
                         "frac": round(tf / fma_peak, 4), "flop_per_pair": 8,
                         "peak_src": "FP32 FMA microbenchmark of this run"},
            "l2": "inputs (7.7 MB) are L2-resident by construction; the kernel is issue-bound, no flush"}


# ---------------------------------------------------------------------------------------------------------------
# the CUDA arm
# ---------------------------------------------------------------------------------------------------------------
def load_built_library():
    """The library build() left in the tree.  Nothing is compiled here (the tree may be read-only); a library built from other
    sources than the tree's would be timed and dumped in their place, so it is refused."""
    from meshrcnn_b200 import _lib, build
    if build.needs_build():
        raise SystemExit("bench.py: %s is missing or was not built from the sources in this tree -- run build() "
                         "(python -m meshrcnn_b200.build) first" % build.LIB)
    return _lib.load()


def run_cuda(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    load_built_library()
    steps, warmup = args.steps, max(args.warmup, 3)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl = HeadWorkload("pix3d", dev, rank, world)

    # clock sampler: started before the warm-up so that the fork + NVML start-up of nvidia-smi (tens of ms during which
    # kernel launches stall) is not charged to the first timed step; it samples the same workload throughout.
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.5)
    # ---- process start-up (untimed) ---------------------------------------------------------------------------
    #  * every timing event is created and recorded once now and reused afterwards (EventPool);
    #  * the first ~12 steps of a fresh process ramp from 7.4 to 6.3 ms (clocks, allocator growth): the same step is run
    #    untimed for STARTUP_SECONDS before the W warm-up steps.  Both are start-up cost, not steady-state throughput.
    pool = EventPool(2 * steps + 72)
    t_start = time.perf_counter()
    startup_steps = 0
    while time.perf_counter() - t_start < STARTUP_SECONDS:
        wl.step(exchange=False)      # NO collective here: the loop is time-based, ranks run different counts
        startup_steps += 1
        if startup_steps % 8 == 0:
            torch.cuda.synchronize()
    # ---- warm-up -------------------------------------------------------------------------------------------
    for _ in range(warmup):
        wl.step()
    sync_all()
    stats = dict(wl.stats(), grid=wl.w["grid"])
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2
    flush.zero_()
    wl.step()               # one more untimed step with the flush buffer allocated (first-touch / allocator effects)
    sync_all()
    gc.collect()
    gc.disable()            # no cyclic-GC pause inside a timed step (autograd graphs are freed by refcount)
    # settle (untimed, collective-free, bounded): the timed region starts once 5 consecutive steps run within 5 % of the fastest
    # step seen so far -- a disturbed box (another tenant's burst, a slow NVML query) otherwise lands in the first timed steps
    settle_ev = pool.take(2)
    best, streak, settle_steps = float("inf"), 0, 0
    while settle_steps < 120 and streak < 5:
        settle_ev[0][0].record()
        wl.step(exchange=False)
        settle_ev[0][1].record()
        torch.cuda.synchronize()
        t_ms = settle_ev[0][0].elapsed_time(settle_ev[0][1])
        best = min(best, t_ms)
        streak = streak + 1 if t_ms <= 1.05 * best else 0
        settle_steps += 1
    for _ in range(2):
        wl.step()           # back to the pipelined, collective-carrying rhythm (every rank runs exactly these two)
    sync_all()

    # ---- timed region 1: inputs resident in HBM ----------------------------------------------------------------
    # Every step draws its surface-sampling seeds from torch's generator and the start-up loop runs a wall-clock-dependent
    # number of steps: reseeding here gives the timed steps the same draws on every run (--dump-outputs compares builds).
    torch.manual_seed(0)
    res_ms, launches, last_losses = timed_resident(wl, pool, steps, flush, sync_all)
    outputs = step_outputs(wl, last_losses) if args.dump_outputs and rank == 0 else None
    del last_losses
    log("[bench] per-step ms (resident):", " ".join("%.2f" % x for x in res_ms))
    # ---- timed region 2: end to end through the module API from pinned host memory --------------------------------
    e2e_ms, phases, host_losses = timed_e2e(wl, pool, steps, max(warmup, E2E_WARMUP_MIN), flush, sync_all)
    log("[bench] e2e host phases ms (h2d, step, d2h):", " ".join("%.1f/%.1f/%.1f" % (x * 1e3, y * 1e3, z * 1e3) for x, y, z in phases))
    log("[bench] per-step ms (e2e):", " ".join("%.2f" % x for x in e2e_ms))
    gc.enable()

    t = torch.tensor([sum(res_ms), sum(e2e_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                  # max over ranks
    dev_ms, e2e_total = float(t[0]), float(t[1])

    # ---- per-kernel breakdown + FP32 peak (instrumented extra steps, not part of the headline numbers) --------------
    peaks = load_peaks()
    breakdown = roof_all = roofline = None
    fma_peak = measure_fma_peak(dev)
    if rank == 0:
        breakdown = instrumented_breakdown(wl, reps=2)
        SVn, R = stats["SV"], stats["B"] * 144
        # one headline step: 8 GraphConvs with a dense 128-wide block (stage 0's graphConv0 has none) forward + input gradient,
        # 3 texel projections (4 608 texels x 256 channels -> 256) forward + their gradient
        widths = [(SVn, 128, 256)] * 8 + [(SVn, 256, 128)] * 8 + [(R, 256, 256)] * 6
        roof_all = kernel_rooflines(breakdown, stats, peaks, fma_peak, widths)
        top = next(iter(breakdown))
        if top == "mrb_knn_fwd":
            r = roof_all[top]
            roofline = {"kernel": r["kernel"], "bound": "fp32_issue", "achieved": r["achieved"], "peak": r["peak"], "unit": "TFLOP/s",
                        "frac": r["frac"], "traffic": 2 * KNN_DRAM_BYTES_PER_LAUNCH,
                        "traffic_src": "profiles/: ncu dram read+write of the two k_nn_grid<10> launches of one call",
                        "peak_src": r["peak_src"], "issue_slots_busy_ncu": KNN_ISSUE_SLOTS_BUSY_NCU,
                        "algorithmic": "B*P*Q = %d pairs x 8 flop per mrb_knn_fwd call (SURVEY 8d; both directions, BASELINE.md 3)" % r["pairs_per_call"],
                        "ms_per_call": r["ms_per_call"], "Gpairs_per_s": r["Gpairs_per_s"],
                        "share_of_step": round(breakdown[top]["ms_per_step"] / sum(v["ms_per_step"] for v in breakdown.values()), 3)}
        else:
            r = roof_all.get(top) or next(iter(roof_all.values()))
            roofline = dict(r, kernel=top, traffic=None, peak_src=peaks["src"])
    clocks = sampler.stop() if sampler else None

    # ---- the other BASELINE configs, same run ------------------------------------------------------------------------
    extras = {}
    if args.extras:
        if sampler:
            sampler2 = ClockSampler(local_rank)
            sampler2.start()
        del wl
        torch.cuda.empty_cache()
        ex_steps = max(3, min(steps, 10))
        extras["configs[1] with bf16 feature maps"] = extra_bf16_maps(dev, rank, world, pool, flush, sync_all, ex_steps)
        extras["configs[2]"] = extra_shapenet_shard(dev, rank, world, pool, flush, sync_all, ex_steps, peaks)
        extras["configs[3]"] = extra_cubify_stress(dev, rank, world, pool, flush, sync_all, peaks)
        extras["configs[4]"] = extra_chamfer_sweep(dev, rank, world, pool, flush, sync_all, fma_peak)
        if sampler:
            extras["clocks"] = sampler2.stop()

    result = None
    if rank == 0:
        B = stats["B"]
        total_meshes = B * world * steps
        e2e_stats = _stats(e2e_ms)
        result = {
            "metric": "meshes/sec (fwd+bwd, 3 refine stages)", "value": round(total_meshes / (dev_ms * 1e-3), 2),
            "unit": "meshes/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": round(dev_ms / steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS["pix3d"]["label"] % B,
                       "global_batch": B * world,
                       "parallelism": "mesh-sharded dp%d (meshes dealt by occupied-voxel count), NCCL grad all-reduce(SUM) per stage "
                                      "bucket from backward hooks" % world,
                       "per_gpu": stats, "l2": "256 MiB flush write between timed iterations",
                       "startup": "%d untimed steps (%.0f s) + pre-recorded timing-event pool, before the W warm-up steps; %d settle "
                                  "steps (until 5 in a row within 5 %% of the fastest); %d untimed e2e steps before the e2e region"
                                  % (startup_steps, STARTUP_SECONDS, settle_steps, max(warmup, E2E_WARMUP_MIN)),
                       "optimizer": "none (metric is fwd+bwd)"},
            "e2e": {"value": round(total_meshes / (e2e_total * 1e-3), 2), "unit": "meshes/s",
                    "h2d_bytes_per_step": wl_h2d_bytes(B), "d2h_bytes_per_step": 12,
                    "ms_per_step": round(e2e_total / steps, 3), "rank0_step_ms": e2e_stats,
                    "h2d": "pinned host -> device on a copy stream, one step ahead, into two alternating device buffer sets (a "
                           "prefetching loader); K copies inside the K timed brackets; D2H of the 3 losses + stream sync every step"},
            "resident_rank0_step_ms": _stats(res_ms),
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_kernels": roof_all,
            "fp32_fma_peak_tflops": round(fma_peak, 2),
            "breakdown_ms": breakdown,
            "losses": {k: float(v) for k, v in zip(("chamfer", "normal", "edge"), host_losses)},
            "extra_configs": extras,
        }
        if args.cpu_baseline and world == 1:          # the CPU arm is timed at N = 1 only (the other ranks would just wait)
            result["cpu_baseline"] = cpu_reference(steps=2, warmup=1, meshes=1)    # ~20 s of host work on the box
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    if result is not None:
        emit(result)


def wl_h2d_bytes(B):
    from meshrcnn_b200 import synthetic
    c, h, w = synthetic.PIX3D_MAP
    return int(4 * B * WORKLOADS["pix3d"]["grid"] ** 3 + 4 * B * c * h * w)


# ---------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref), or the oracle port when it is not available
# ---------------------------------------------------------------------------------------------------------------
def _reference_available():
    from oracle import ref_import
    return ref_import.available()


def cpu_reference(steps, warmup, meshes):
    """Times the reference's CPU path on `meshes` meshes of the headline workload (same grids, maps, 10k-point clouds,
    k = 10, fwd + bwd), all host threads.  `kind: "reference"`: the UNMODIFIED reference files (oracle/_ref: a byte-for-byte
    copy of meshRCNN/layers.py, loss_functions.py, utils.py, utils/mesh_sampling.py, process.py, rotation.py made by
    oracle/build_ref.py) behind the import shims of oracle/ref_import.py -- its dict-based Cubify, per-map Python
    VertexAlign, dense B x P x Q distance tensors, CPU symeig.  `kind: "port"` (fallback when oracle/_ref is absent): the
    oracle restatement, which executes the same torch-CPU ops but a faster numpy Cubify."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if _reference_available():
        one_step, kind = _reference_step(meshes), "reference"
    else:
        one_step, kind = _port_step(meshes), "port"
    for _ in range(warmup):
        one_step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one_step()
        times.append(time.perf_counter() - t0)
    sec = sum(times)
    return {"value": round(meshes * steps / sec, 4), "unit": "meshes/s", "cores": cores, "kind": kind,
            "sample": "%d timed step(s) after %d warm-up of %d mesh(es) of the headline workload (same grids, maps, default-init "
                      "weights, 10k-point clouds, k=10, fwd+bwd), torch threads=%d; the reference needs 1.6 GB of dense distance "
                      "tensors per mesh and stage, hence the bounded batch" % (steps, warmup, meshes, torch.get_num_threads()),
            "s_per_step": round(sec / steps, 3)}


def _reference_step(meshes):
    from oracle import ref_import
    from meshrcnn_b200 import synthetic
    R = ref_import.load_reference()
    w = WORKLOADS["pix3d"]
    vox = synthetic.blob_voxels(meshes, w["grid"], 0)
    fmap = synthetic.feature_maps(meshes, _maps("PIX3D"), 0)[0]
    gt_vox = synthetic.blob_voxels(meshes, w["grid"], 1000)
    torch.manual_seed(1)
    cub = R.layers.Cubify(THRESH)
    stages = [R.layers.VertixRefinePix3D(use_input_features=bool(i)) for i in range(3)]
    gv, gvi, gf, gfi, _ = R.layers.Cubify(0.5)(gt_vox)
    gt = R.Batch((torch.cat([R.process.normalize_mesh(v) for v in gv.split(gvi)]), gf), gvi, gfi)
    sizes = [(w["img"], w["img"])] * meshes

    def one_step():
        for st in stages:
            st.zero_grad()
        pos, vi, faces, fi, adj = cub(vox)
        fm = fmap.clone().requires_grad_()
        feats, cur, positions = None, pos, []
        for st in stages:
            cur, feats = st(vi, fm, adj, cur, sizes, vertex_features=feats)
            positions.append(cur)
        ch, nl, ed = R.loss_functions.batched_mesh_loss(positions, faces, adj, vi, fi, gt)     # 10e3 points, k = 10 (defaults)
        total = ch + 0.1 * nl + 0.5 * ed
        total.backward()
        return float(total.detach())

    return one_step


def _port_step(meshes):
    from oracle import cubify_np, mesh_ops
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200.layers import VertixRefinePix3D
    w = WORKLOADS["pix3d"]
    vox = synthetic.blob_voxels(meshes, w["grid"], 0)
    fmap = synthetic.feature_maps(meshes, _maps("PIX3D"), 0)[0]
    gt_vox = synthetic.blob_voxels(meshes, w["grid"], 1000)
    torch.manual_seed(1)
    stages = [VertixRefinePix3D(use_input_features=bool(i)) for i in range(3)]
    params = [{k: v.detach().clone().requires_grad_() for k, v in st.named_parameters()} for st in stages]
    sizes = [(w["img"], w["img"])] * meshes
    gv, gvi, gf, gfi, _ = cubify_np.cubify(gt_vox.numpy(), 0.5)
    gt_pos = torch.cat([mesh_ops.normalize_cloud(v) for v in torch.from_numpy(gv).split(gvi)])
    gt_faces = torch.from_numpy(gf)

    def one_step():
        verts, vi, faces, fi, adj = cubify_np.cubify(vox.numpy(), THRESH)
        pos, faces, adj = torch.from_numpy(verts), torch.from_numpy(faces), torch.from_numpy(adj)
        fm = fmap.clone().requires_grad_()
        feats, cur, positions = None, pos, []
        for sd in params:
            cur, feats = mesh_ops.stage_pix3d(sd, vi, fm, adj, cur, sizes, feats=feats)
            positions.append(cur)
        total = 0
        for s, p in enumerate(positions):
            u, x2, x1 = synthetic.sampling_randomness(meshes, N_POINTS, 10 + s)
            ug, x2g, x1g = synthetic.sampling_randomness(meshes, N_POINTS, 20 + s)
            fi_p = torch.stack([mesh_ops.face_cdf_draw(v.detach(), f, u[b]) for b, (v, f) in
                                enumerate(zip(p.split(vi), faces.split(fi)))])
            fi_g = torch.stack([mesh_ops.face_cdf_draw(v, f, ug[b]) for b, (v, f) in
                                enumerate(zip(gt_pos.split(gvi), gt_faces.split(gfi)))])
            ch, nl, ed, _ = mesh_ops.mesh_loss_with(p, faces, adj, vi, fi, gt_pos, gt_faces, gvi, gfi, (fi_p, x2, x1),
                                                    (fi_g, x2g, x1g), float(N_POINTS), KNN)
            total = total + ch + 0.1 * nl + 0.5 * ed
        total.backward()
        return float(total)

    return one_step


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                       # rank 0 alone runs the CPU arm
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cb = cpu_reference(steps=args.steps, warmup=args.warmup, meshes=1)
    line = {
        "impl": "reference", "metric": "meshes/sec (fwd+bwd, 3 refine stages)", "value": cb["value"], "unit": "meshes/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(cb["s_per_step"] * 1e3, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the same workload string as the CUDA arm; what the CPU arm actually runs per step is in cpu_baseline.sample
        "config": {"workload": WORKLOADS["pix3d"]["label"] % B_PER_GPU},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "meshes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------------
# --check: loss parity at the bench shape (10 000-point clouds, k = 10) against the fp64 oracle
# ---------------------------------------------------------------------------------------------------------------
def check_bench_shape_losses(meshes=2, dev=None, verbose=True):
    """Runs `meshes` meshes of the headline workload (24^3 blobs, 10 000-point clouds, k = 10) with injected sampling
    draws through the CUDA arm and through the fp64 oracle: chamfer and edge must agree to rtol 1e-4, the normal term to
    rtol 1e-4 against the oracle evaluated under the kernel's eigenvector sign rule (DESIGN.md section 2, quirk 5) and to
    2 % against the oracle with LAPACK's signs (the reference's own fp32-vs-fp64 gap is 1 %).  Returns the dict of values;
    raises AssertionError on a mismatch."""
    from oracle import cubify_np, mesh_ops
    from meshrcnn_b200 import synthetic
    from meshrcnn_b200 import loss_functions as LF
    from meshrcnn_b200.pipeline import MeshTargets
    dev = dev or torch.device("cuda", torch.cuda.current_device())
    n, k = N_POINTS, KNN
    vox = synthetic.blob_voxels(meshes, 24, 0)
    verts, vi, faces, fi, adj = cubify_np.cubify(vox.numpy(), THRESH)
    gverts, gvi, gfaces, gfi, _ = cubify_np.cubify(synthetic.blob_voxels(meshes, 24, 1000).numpy(), 0.5)
    g = torch.Generator().manual_seed(5)
    pos = torch.from_numpy(verts).double()
    pos = (pos + 0.3 * torch.randn(pos.shape, generator=g, dtype=torch.float64)) * 0.06          # refined-looking, unit-ish scale
    gt_pos = torch.cat([mesh_ops.normalize_cloud(v) for v in torch.from_numpy(gverts).double().split(gvi)])
    faces_t, adj_t, gfaces_t = torch.from_numpy(faces), torch.from_numpy(adj), torch.from_numpy(gfaces)
    u, x2, x1 = synthetic.sampling_randomness(meshes, n, 10)
    ug, x2g, x1g = synthetic.sampling_randomness(meshes, n, 20)
    fi_p = torch.stack([mesh_ops.face_cdf_draw(v, f, u[b]) for b, (v, f) in enumerate(zip(pos.split(vi), faces_t.split(fi)))])
    fi_g = torch.stack([mesh_ops.face_cdf_draw(v, f, ug[b]) for b, (v, f) in enumerate(zip(gt_pos.split(gvi), gfaces_t.split(gfi)))])
    want = {}
    for canon in (True, False):
        ch, nl, ed, _ = mesh_ops.mesh_loss_with(pos, faces_t, adj_t, vi, fi, gt_pos, gfaces_t, gvi, gfi,
                                                (fi_p, x2.double(), x1.double()), (fi_g, x2g.double(), x1g.double()),
                                                float(n), k, canonical_signs=canon)
        want["canonical" if canon else "lapack"] = (float(ch), float(nl), float(ed))
    gt = MeshTargets(gt_pos.float().to(dev), gfaces_t.to(dev), gvi, gfi)
    rnd = (dict(face_idx=fi_p, xi2=x2, xi1=x1), dict(face_idx=fi_g, xi2=x2g, xi1=x1g))
    ch, nl, ed = LF.mesh_loss(pos.float().to(dev), faces_t.to(dev), adj_t.to(dev), vi, fi, gt, float(n), k, randomness=rnd)
    got = (float(ch), float(nl), float(ed))
    out = {"cuda": got, "oracle_fp64_canonical_signs": want["canonical"], "oracle_fp64_lapack_signs": want["lapack"],
           "meshes": meshes, "points": n, "k": k}
    if verbose:
        log("[check]", json.dumps(out))
    rel = lambda a, b: abs(a - b) / max(abs(b), 1e-30)
    assert rel(got[0], want["canonical"][0]) <= 1e-4, ("chamfer", got[0], want["canonical"][0])
    assert rel(got[2], want["canonical"][2]) <= 1e-4, ("edge", got[2], want["canonical"][2])
    assert rel(got[1], want["canonical"][1]) <= 1e-4, ("normal (canonical signs)", got[1], want["canonical"][1])
    assert rel(got[1], want["lapack"][1]) <= 2e-2, ("normal (LAPACK signs)", got[1], want["lapack"][1])
    return out


_REAL_STDOUT = None


def emit(line: dict) -> None:
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    global _REAL_STDOUT
    # Everything except the result line goes to stderr: libraries (NCCL prints its version banner) write to fd 1.
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-extras", dest="extras", action="store_false", help="skip BASELINE configs[2..4]")
    ap.add_argument("--check", action="store_true", help="bench-shape loss parity against the fp64 oracle, then exit")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the losses and gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.check or args.impl != "b200"):
        ap.error("--dump-outputs dumps the timed steps of the CUDA arm; it does not go with --check or --impl reference")
    if args.check:
        load_built_library()
        emit({"check": "bench-shape losses vs fp64 oracle", "ok": True, **check_bench_shape_losses()})
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
