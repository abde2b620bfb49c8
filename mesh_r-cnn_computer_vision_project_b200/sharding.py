"""Multi-GPU: one process per GPU, meshes sharded by index, one NCCL all-reduce(SUM) of the gradients.

Replaces the reference's single-process ``dataParallel.CustomDP`` (dataParallel/dataParallel.py:28-46): per-forward
parameter broadcast (replicate.py:26-43), Python-thread ``parallel_apply`` and ``reduce_add`` of the losses
(gather.py:13-28,109-112).  Here weights stay resident on every rank, every rank runs the hot path on its own packed
shard (meshes are independent units -- adjacency is block-diagonal per mesh), and the only exchange step is the
gradient all-reduce -- SUM, not mean, like the reference's reduce-add -- over NVLink/NVSwitch.
"""
from typing import Iterable, List, Tuple

import torch
import torch.distributed as dist
from torch import Tensor


def split_to_n(n_items: int, n_parts: int) -> List[Tuple[int, int]]:
    """Contiguous [lo, hi) chunks; the first ``n_items % n_parts`` chunks get one extra item -- the reference's
    ``split_to_n`` (dataParallel/scatter.py:5-13), kept so that results match the reference DP shard for shard."""
    base, extra = divmod(n_items, n_parts)
    out, lo = [], 0
    for r in range(n_parts):
        hi = lo + base + (1 if r < extra else 0)
        out.append((lo, hi))
        lo = hi
    return out


def balanced_split(costs: List[float], n_parts: int, equal_counts: bool = False) -> List[List[int]]:
    """Assignment of meshes to ranks by a per-mesh cost (e.g. the occupied-voxel count; mesh sizes vary ~1.4x) -- the
    throughput mode of SURVEY.md 8(e), not used for parity runs (those keep ``split_to_n``).

    ``equal_counts=False``: greedy longest-processing-time (each mesh to the least loaded rank).
    ``equal_counts=True``: meshes sorted by cost are dealt in snake order (0..n-1, n-1..0, ...), so every rank gets the
    same number of meshes (+-1) -- the per-mesh constant work (10k-point sampling, k-NN) stays balanced as well."""
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    parts: List[List[int]] = [[] for _ in range(n_parts)]
    if equal_counts:
        for pos, i in enumerate(order):
            rnd, k = divmod(pos, n_parts)
            parts[k if rnd % 2 == 0 else n_parts - 1 - k].append(i)
        return [sorted(p) for p in parts]
    loads = [0.0] * n_parts
    for i in order:
        r = min(range(n_parts), key=lambda j: loads[j])
        parts[r].append(i)
        loads[r] += costs[i]
    return [sorted(p) for p in parts]


def _dist_on() -> bool:
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


class FlatGradBucket:
    """All parameter gradients live in one contiguous fp32 buffer (``p.grad`` are views into it), so the step's
    exchange is a single all-reduce launch: 1.9 MB for the Pix3D head, 8.9 MB for the residual ShapeNet head.

    ``optimizer.zero_grad()`` / ``module.zero_grad()`` default to ``set_to_none=True`` (torch >= 2.0), which drops the
    views: the next backward then allocates fresh ``.grad`` tensors and an all-reduce of the flat buffer would silently
    exchange stale zeros.  ``zero()`` therefore re-binds the views and ``all_reduce()`` first calls ``sync_views()``,
    which copies any detached ``.grad`` back into the buffer and re-attaches it -- use ``bucket.zero()`` instead of
    ``zero_grad()``, but a training loop that calls ``zero_grad(set_to_none=True)`` still reduces the right values."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params = [p for p in params if p.requires_grad]
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.offsets = []
        off = 0
        for p in self.params:
            self.offsets.append(off)
            off += p.numel()
        self._bind()

    def _view(self, i: int) -> Tensor:
        p = self.params[i]
        return self.flat[self.offsets[i]:self.offsets[i] + p.numel()].view_as(p)

    def _bind(self) -> None:
        for i, p in enumerate(self.params):
            p.grad = self._view(i)

    def sync_views(self) -> int:
        """Makes every ``p.grad`` a view of the flat buffer again (copying detached gradients into it; a parameter whose
        ``.grad`` is None contributes zeros).  Returns the number of parameters that had to be re-attached."""
        esz = self.flat.element_size()
        base = self.flat.data_ptr()
        fixed = 0
        for i, p in enumerate(self.params):
            g = p.grad
            if g is not None and g.data_ptr() == base + esz * self.offsets[i] and g.is_contiguous():
                continue
            v = self._view(i)
            if g is None:
                v.zero_()
            else:
                v.copy_(g)
            p.grad = v
            fixed += 1
        return fixed

    def zero(self) -> None:
        self.flat.zero_()
        for i, p in enumerate(self.params):
            if p.grad is None or p.grad.data_ptr() != self.flat.data_ptr() + self.flat.element_size() * self.offsets[i]:
                p.grad = self._view(i)

    def all_reduce(self, async_op: bool = False):
        self.sync_views()
        if _dist_on():
            return dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, async_op=async_op)
        return None


class StagedGradBuckets:
    """Overlapped gradient exchange (SURVEY.md 8e: "launched as soon as the last stage's backward finishes its weight
    grads and overlapped with the remaining backward"): one flat bucket per group of parameters (here: per refinement
    stage).  A post-accumulate-grad hook counts the parameters of a group whose gradient of this backward pass is final;
    when the last one arrives the group's gradients are packed into its flat buffer (one multi-tensor copy) and the
    all-reduce(SUM) is issued asynchronously -- backward runs the stages in reverse, so stage 2's exchange overlaps the
    backward of stages 1 and 0.  ``finish()`` waits for the outstanding handles and makes every ``p.grad`` a view of the
    reduced buffer.

    ``zero()`` sets the gradients to ``None`` (like ``zero_grad(set_to_none=True)``): autograd then *assigns* each weight
    gradient instead of launching one ``grad += new`` kernel per parameter into a zero-filled buffer (27 adds + 3 fills per
    step for the Pix3D head), and a single-GPU run copies nothing at all.  Reduction is SUM like the reference's
    ``reduce_add`` (dataParallel/gather.py:13-28)."""

    def __init__(self, groups: Iterable[Iterable[torch.nn.Parameter]]):
        self.groups = [[p for p in g if p.requires_grad] for g in groups]
        self.groups = [g for g in self.groups if g]
        dev = self.groups[0][0].device
        self.flats = [torch.zeros(sum(p.numel() for p in g), dtype=torch.float32, device=dev) for g in self.groups]
        self.views = []
        for g, flat in zip(self.groups, self.flats):
            off, vs = 0, []
            for p in g:
                vs.append(flat[off:off + p.numel()].view_as(p))
                off += p.numel()
            self.views.append(vs)
        self.enabled = True
        self._pending = [0] * len(self.groups)
        self._issued = [False] * len(self.groups)
        self._handles = []
        self._hooks = []
        for gi, g in enumerate(self.groups):
            for p in g:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._make_hook(gi)))
        self.zero()

    @classmethod
    def per_stage(cls, head) -> "StagedGradBuckets":
        """One bucket per refinement stage of a ``pipeline.RefinementHead`` (plus one for any other parameters)."""
        groups = [list(st.parameters()) for st in head.refineStages]
        seen = {id(p) for g in groups for p in g}
        rest = [p for p in head.parameters() if id(p) not in seen]
        if rest:
            groups.append(rest)
        return cls([g for g in groups if g])

    def _make_hook(self, gi: int):
        def hook(_param):
            self._pending[gi] -= 1
            if self._pending[gi] == 0 and self.enabled:
                self._issue(gi)
        return hook

    def _pack(self, gi: int) -> None:
        """Copies the group's gradients into its flat buffer (parameters without a gradient contribute zeros)."""
        src, dst = [], []
        for p, v in zip(self.groups[gi], self.views[gi]):
            if p.grad is None:
                v.zero_()
            elif p.grad.data_ptr() != v.data_ptr():
                src.append(p.grad)
                dst.append(v)
        if src:
            torch._foreach_copy_(dst, src)

    def _issue(self, gi: int) -> None:
        if self._issued[gi]:
            return
        self._issued[gi] = True
        if _dist_on():
            self._pack(gi)
            self._handles.append((gi, dist.all_reduce(self.flats[gi], op=dist.ReduceOp.SUM, async_op=True)))

    def zero(self) -> None:
        for gi, g in enumerate(self.groups):
            for p in g:
                p.grad = None
            self._pending[gi] = len(g)
            self._issued[gi] = False
        self._handles = []

    def finish(self, exchange: bool = True) -> None:
        """Call after ``backward()``: issues what the hooks did not, blocks the current stream on every exchange and binds
        ``p.grad`` to the reduced values.  Without a process group (or with ``exchange=False``) the gradients stay where
        autograd put them."""
        if exchange:
            for gi in range(len(self.groups)):
                self._issue(gi)
        for gi, h in self._handles:
            h.wait()
            for p, v in zip(self.groups[gi], self.views[gi]):
                p.grad = v
        self._handles = []

    @property
    def flat_numel(self) -> int:
        return sum(f.numel() for f in self.flats)


def all_reduce_losses(losses: dict) -> dict:
    """Replica losses are summed (reference gather.py:109-112)."""
    if not _dist_on():
        return losses
    keys = sorted(losses)
    buf = torch.stack([losses[k].detach().float() for k in keys])
    dist.all_reduce(buf, op=dist.ReduceOp.SUM)
    return {k: buf[i] for i, k in enumerate(keys)}


def reduce_mesh_metrics(per_mesh: dict) -> dict:
    """Means of the per-mesh metrics of ``eval_utils.compare_meshes(..., reduce=False)`` over the valid meshes of ALL ranks,
    plus ``num_valid`` (int): one all-reduce(SUM) of the per-key sums and the count, so that evaluation with one process per
    GPU does not average per-rank means.  Without a process group (or at world size 1) the same means over the local
    meshes.  The input is not modified."""
    from .eval_utils import mesh_metric_sums
    keys, buf = mesh_metric_sums(per_mesh)
    if _dist_on():
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
    count = int(buf[-1])
    means = (buf[:-1] / count).float() if count else torch.full((len(keys),), float("nan"), device=buf.device)
    out = {k: means[i] for i, k in enumerate(keys)}
    out["num_valid"] = count
    return out


def _all_gather_ragged(t: Tensor, dim: int = 0) -> List[Tensor]:
    """all_gather of tensors whose size along ``dim`` differs per rank (sizes exchanged first, payload padded to the max)."""
    world = dist.get_world_size()
    t = t.contiguous()
    size = torch.tensor([t.shape[dim]], dtype=torch.int64, device=t.device)
    sizes = [torch.zeros_like(size) for _ in range(world)]
    dist.all_gather(sizes, size)
    sizes = [int(x) for x in sizes]
    mx = max(sizes)
    moved = t.movedim(dim, 0)
    pad = torch.zeros((mx,) + tuple(moved.shape[1:]), dtype=t.dtype, device=t.device)
    pad[:moved.shape[0]] = moved
    bufs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    return [b[:n].movedim(0, dim) for b, n in zip(bufs, sizes)]


def gather_eval_outputs(out: dict) -> dict:
    """Eval-mode output dicts of all ranks merged into one packed batch on every rank -- the reference's
    ``gather_GCN_outputs`` (dataParallel/gather.py:65-92): per-stage vertex positions and faces concatenated in rank
    order, ``edge_index`` re-offset by the number of vertices of the preceding shards (:80-83), the per-mesh count lists
    chained.  Keys: ``vertex_positions`` (list), ``edge_index``, ``faces``, ``vertice_index``, ``face_index``,
    ``mesh_index``.  Without an initialised process group (or world size 1) the input is returned unchanged."""
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return out
    world = dist.get_world_size()
    lists = [None] * world
    dist.all_gather_object(lists, {k: list(out[k]) for k in ("vertice_index", "face_index", "mesh_index")})
    res = {k: [x for d in lists for x in d[k]] for k in ("vertice_index", "face_index", "mesh_index")}
    res["vertex_positions"] = [torch.cat(_all_gather_ragged(p, 0), 0) for p in out["vertex_positions"]]
    res["faces"] = torch.cat(_all_gather_ragged(out["faces"], 0), 0)
    offsets, run = [], 0
    for d in lists:
        offsets.append(run)
        run += sum(d["vertice_index"])
    edges = _all_gather_ragged(out["edge_index"], 1)
    res["edge_index"] = torch.cat([e + off for e, off in zip(edges, offsets)], 1)
    return res
