"""Host-side operators: thin ``torch.autograd.Function`` wrappers around the C-ABI kernels.

Nothing here computes on the CPU and nothing falls back to PyTorch ops for the hot path: each function
allocates its outputs with torch (device memory only) and launches hand-written sm_100a kernels on the
caller's current stream through ``_lib.call``.
"""
import ctypes
import os
import threading
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from .topology import MeshTopology, from_coo, lookup, register

# quad corners per direction as lattice offsets in (z, y, x); same table as csrc/cubify.cu (layers.py:370-400)
CUBIFY_CORNERS = (
    ((0, 0, 0), (0, 0, 1), (0, 1, 0), (0, 1, 1)), ((1, 0, 0), (1, 0, 1), (1, 1, 0), (1, 1, 1)),
    ((1, 0, 0), (1, 0, 1), (0, 0, 0), (0, 0, 1)), ((0, 1, 0), (0, 1, 1), (1, 1, 0), (1, 1, 1)),
    ((1, 0, 0), (0, 0, 0), (1, 1, 0), (0, 1, 0)), ((0, 0, 1), (1, 0, 1), (0, 1, 1), (1, 1, 1)))


def _require_cuda(t: Tensor, what: str) -> None:
    """The kernels are launched on the *current* device's current stream (``_lib.stream_ptr``), so a tensor that lives on
    another GPU is rejected instead of being handed to a kernel running on the wrong device: multi-GPU callers (one
    thread per GPU like the reference's ``parallel_apply``, dataParallel/dataParallel.py:33) run each replica under
    ``torch.cuda.device(i)``."""
    if not isinstance(t, Tensor) or not t.is_cuda:
        raise RuntimeError("meshrcnn_b200.%s: expected a CUDA tensor -- the hot path has no CPU fallback" % what)
    if t.device.index != torch._C._cuda_getDevice():
        raise RuntimeError("meshrcnn_b200.%s: tensor lives on %s but the current CUDA device is cuda:%d -- call under "
                           "`with torch.cuda.device(tensor.device):`" % (what, t.device, torch._C._cuda_getDevice()))


# ----------------------------------------------------------------------------------------------------------
# Cubify
# ----------------------------------------------------------------------------------------------------------
_PINNED = {}


def _pinned_i64(n: int, device) -> Tensor:
    """A reusable pinned int64 staging buffer per (thread, device, size) -- cudaHostAlloc per call would cost more than the copy."""
    key = (threading.get_ident(), str(device), n)
    buf = _PINNED.get(key)
    if buf is None:
        if len(_PINNED) > 64:
            _PINNED.clear()
        buf = _PINNED[key] = torch.empty(n, dtype=torch.int64).pin_memory()
    return buf


@torch.no_grad()
def cubify(t: Tensor, threshold: float, from_logits: bool = False):
    """See ``layers.Cubify``.  Returns (verts, v_index, faces, f_index, adj, topology).  ``from_logits``: ``t`` holds the
    voxel head's logits and ``sigmoid(t) > threshold`` is tested inside the first kernel (SURVEY 8 f-1)."""
    _require_cuda(t, "Cubify")
    if t.dim() != 4:
        raise RuntimeError("Cubify expects B x Z x Y x X, got %s" % (tuple(t.shape),))
    B, Z, Y, X = t.shape
    probs = t.detach().to(torch.float32).contiguous()
    dev = probs.device
    with torch.cuda.device(dev):
        lib = _lib.load()
        ws_bytes = lib.mrb_cubify_workspace_bytes(B, Z, Y, X)
        if ws_bytes < 0:
            raise RuntimeError("Cubify: bad grid shape %s" % (tuple(t.shape),))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        meta = torch.empty(4 + 4 * B, dtype=torch.int64, device=dev)
        _lib.call("mrb_cubify_count", _lib.ptr(probs), B, Z, Y, X, float(threshold), int(bool(from_logits)), _lib.ptr(ws),
                  _lib.ptr(meta))
        # The one unavoidable sync: the API returns Python lists.  The counters are copied into pinned memory asynchronously;
        # work that does not depend on the mesh (the texel projections of the pass, functional.PackPlan) is launched behind
        # the copy, so the device has something to do while this thread waits, allocates and issues the emit kernels.
        meta_h = _pinned_i64(4 + 4 * B, dev)
        meta_h.copy_(meta, non_blocking=True)
        copied = torch.cuda.Event()
        copied.record()
        run_deferred()
        copied.synchronize()
        SV, SF, E = int(meta_h[0]), int(meta_h[1]), int(meta_h[2])
        if SF == 0:
            raise ValueError("empty grid")       # reference layers.py:434-435
        v_counts = meta_h[4:4 + B].tolist()
        f_counts = meta_h[4 + B:4 + 2 * B].tolist()
        last = max(i for i, c in enumerate(f_counts) if c > 0) + 1   # bincount truncation (layers.py:445,448)
        verts = torch.empty(SV, 3, dtype=torch.float32, device=dev)
        faces = torch.empty(SF, 3, dtype=torch.int64, device=dev)
        adj = torch.empty(2, E, dtype=torch.int64, device=dev)
        rowptr = torch.empty(SV + 1, dtype=torch.int32, device=dev)
        col32 = torch.empty(E, dtype=torch.int32, device=dev)
        vert_mesh = torch.empty(SV, dtype=torch.int32, device=dev)
        aux = torch.empty(2 * SV, dtype=torch.int32, device=dev)
        _lib.call("mrb_cubify_emit", B, Z, Y, X, _lib.ptr(ws), _lib.ptr(meta), SV, SF, E, _lib.ptr(verts),
                  _lib.ptr(faces), _lib.ptr(adj), _lib.ptr(rowptr), _lib.ptr(col32), _lib.ptr(vert_mesh),
                  _lib.ptr(aux))
    topo = MeshTopology(SV, E, rowptr, col32, symmetric=True, vert_mesh=vert_mesh)
    register(adj, topo)
    return verts, v_counts[:last], faces, f_counts[:last], adj, topo


class _VoxelBCE(torch.autograd.Function):
    """mean BCE on probabilities (reference voxel_loss, loss_functions.py:10-14) or on logits with the sigmoid fused."""

    @staticmethod
    def forward(ctx, x, target, from_logits, want_probs):
        _require_cuda(x, "voxel_loss")
        xc = _f32c(x)
        tc = _f32c(target)
        if xc.shape != tc.shape:
            raise RuntimeError("voxel_loss: prediction %s and target %s differ in shape" % (tuple(xc.shape), tuple(tc.shape)))
        dev = x.device
        probs = torch.empty_like(xc) if (from_logits and want_probs) else None
        acc = torch.empty(1, dtype=torch.float64, device=dev)
        out = torch.empty(1, dtype=torch.float32, device=dev)
        _lib.call("mrb_voxel_bce_fwd", _lib.ptr(xc), _lib.ptr(tc), xc.numel(), int(from_logits), _lib.ptr(probs), _lib.ptr(acc),
                  _lib.ptr(out))
        ctx.save_for_backward(xc, tc)
        ctx.from_logits = bool(from_logits)
        ctx.set_materialize_grads(False)        # no zero-filled "gradient" of the probabilities
        if probs is not None:
            ctx.mark_non_differentiable(probs)
        return out[0], probs

    @staticmethod
    def backward(ctx, g, _gprobs):
        if g is None:
            return None, None, None, None
        xc, tc = ctx.saved_tensors
        gx = torch.empty_like(xc)
        _lib.call("mrb_voxel_bce_bwd", _lib.ptr(xc), _lib.ptr(tc), xc.numel(), int(ctx.from_logits), _lib.ptr(_f32c(g).reshape(1)),
                  _lib.ptr(gx))
        return gx, None, None, None


def voxel_bce(x: Tensor, target: Tensor, from_logits: bool = False, want_probs: bool = False):
    """(loss, probs | None): mean binary cross entropy of the voxel head -- one pass over ``x`` (fp64 accumulation)."""
    return _VoxelBCE.apply(x, target, from_logits, want_probs)


# ----------------------------------------------------------------------------------------------------------
# small cached host -> device tables (mesh offsets, per-mesh image records)
# ----------------------------------------------------------------------------------------------------------
_TABLE_CACHE = {}


def _device_table(key, values, device) -> Tensor:
    k = (key, tuple(values), str(device))
    t = _TABLE_CACHE.get(k)
    if t is None:
        if len(_TABLE_CACHE) > 256:
            _TABLE_CACHE.clear()
        t = torch.tensor(list(values), dtype=torch.int32).to(device)
        _TABLE_CACHE[k] = t
    return t


def offsets_table(counts: Sequence[int], device) -> Tensor:
    """int32 [len+1] exclusive offsets of a list of per-mesh counts (``v_index`` / ``f_index``)."""
    off = [0]
    for c in counts:
        off.append(off[-1] + int(c))
    return _device_table("off", off, device)


def vertex_mesh_ids(v_index: Sequence[int], num_vertices: int, device, topo: Optional[MeshTopology] = None) -> Tensor:
    if topo is not None and topo.vert_mesh is not None and topo.num_vertices == num_vertices:
        return topo.vert_mesh
    off = offsets_table(v_index, device)
    ids = torch.empty(num_vertices, dtype=torch.int32, device=device)
    _lib.call("mrb_segment_ids", _lib.ptr(off), len(v_index), num_vertices, _lib.ptr(ids))
    return ids


def mesh_info_table(mesh_index: Sequence[int], image_sizes, device) -> Tensor:
    """int32 [n_meshes, 3] = (image index, image H, image W) per mesh (reference layers.py:538-543)."""
    rows = []
    for img, (n_mesh, size) in enumerate(zip(mesh_index, image_sizes)):
        H, W = int(size[0]), int(size[1])
        for _ in range(int(n_mesh)):
            rows += [img, H, W]
    return _device_table("info", rows, device)


def _f32c(t: Tensor) -> Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _rows(t: Tensor) -> Tensor:
    """fp32 matrix whose rows are dense (stride(1) == 1) but may have a row pitch > width (a column slice of a wider
    buffer, e.g. the 16-byte aligned rows ``concat_cols`` produces): the kernels take the pitch as ld, no copy is made."""
    if t.dtype == torch.float32 and t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]:
        return t
    return _f32c(t)


def _pitch(width: int) -> int:
    return (width + 3) // 4 * 4


def _padded_rows(n: int, width: int, device) -> Tensor:
    """n x width view of a buffer whose rows start on 16-byte boundaries."""
    return torch.empty(n, _pitch(width), dtype=torch.float32, device=device)[:, :width]


class _ConcatCols(torch.autograd.Function):
    """torch.cat(parts, dim=1) into rows padded to a multiple of 4 floats (one kernel); the backward hands out column
    slices of the upstream gradient (views, no copies)."""

    @staticmethod
    def forward(ctx, *parts):
        ps = [_rows(p) for p in parts]
        _require_cuda(ps[0], "concat_cols")
        n = ps[0].shape[0]
        widths = [p.shape[1] for p in ps]
        out = torch.empty(n, _pitch(sum(widths)), dtype=torch.float32, device=ps[0].device)
        a = [(p.data_ptr(), p.shape[1], p.stride(0)) for p in ps] + [(None, 0, 0)] * (3 - len(ps))
        _lib.call("mrb_concat_cols", a[0][0], a[0][1], a[0][2], a[1][0], a[1][1], a[1][2], a[2][0], a[2][1], a[2][2], n,
                  _lib.ptr(out), out.shape[1])
        ctx.widths = widths
        return out[:, :sum(widths)]

    @staticmethod
    def backward(ctx, g):
        outs, off = [], 0
        for i, w in enumerate(ctx.widths):
            outs.append(g[:, off:off + w] if ctx.needs_input_grad[i] else None)
            off += w
        return tuple(outs)


def concat_cols(parts: Sequence[Tensor]) -> Tensor:
    """``torch.cat(parts, dim=1)`` for 1-3 fp32 CUDA matrices with 16-byte aligned output rows (a strided view)."""
    if not 1 <= len(parts) <= 3:
        raise RuntimeError("concat_cols: 1 to 3 parts")
    return _ConcatCols.apply(*parts)


# ----------------------------------------------------------------------------------------------------------
# dense contraction on the library's GEMM
# ----------------------------------------------------------------------------------------------------------
def _gemm(ta: bool, tb: bool, M: int, N: int, K: int, a_ptr: int, lda: int, b_ptr: int, ldb: int, beta: float,
          c_ptr: int, ldc: int) -> None:
    _lib.call("mrb_sgemm", int(ta), int(tb), M, N, K, a_ptr, lda, b_ptr, ldb, float(beta), c_ptr, ldc)


def _use_tc(K: int, N: int) -> bool:
    """Products wide enough for a UMMA tile run on tcgen05; skinny heads (N = 3 / 6) stay on the CUDA-core kernel."""
    return N >= 16 and K >= 16


def _use_tc_wgrad(V: int, N: int) -> bool:
    return N % 32 == 0 and 32 <= N <= 256 and V >= 256


class _MatMul(torch.autograd.Function):
    """y = x @ (w^T if trans_w else w)."""

    @staticmethod
    def forward(ctx, x, w, trans_w):
        _require_cuda(x, "matmul")
        x, w = _rows(x), _f32c(w)
        M, K = x.shape
        ldx = x.stride(0)
        N = w.shape[0] if trans_w else w.shape[1]
        y = torch.empty(M, N, dtype=torch.float32, device=x.device)
        if _use_tc(K, N):
            img = tc_pack(w, None, 1 if trans_w else N, K if trans_w else 1, 0, 0, K, N)
            tc_gemm(x.data_ptr(), ldx, M, K, img, N, _lib.ptr(y), N)
        else:
            _gemm(False, trans_w, M, N, K, x.data_ptr(), ldx, _lib.ptr(w), w.shape[1], 0.0, _lib.ptr(y), N)
        ctx.save_for_backward(x, w)
        ctx.trans_w = trans_w
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        gy = _f32c(gy)
        M, K = x.shape
        ldx = x.stride(0)
        N = gy.shape[1]
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = _padded_rows(M, K, x.device)
            ldg = gx.stride(0)
            # gx = gy @ w (trans_w) or gy @ w^T :  logical B(k = out index, n = in index)
            if _use_tc(N, K):
                img = tc_pack(w, None, K if ctx.trans_w else 1, 1 if ctx.trans_w else N, 0, 0, N, K)
                tc_gemm(_lib.ptr(gy), N, M, N, img, K, gx.data_ptr(), ldg)
            else:
                _gemm(False, not ctx.trans_w, M, K, N, _lib.ptr(gy), N, _lib.ptr(w), w.shape[1], 0.0, gx.data_ptr(), ldg)
        if ctx.needs_input_grad[1]:
            if _use_tc_wgrad(M, N):       # x^T @ gy (K x N) on the tensor cores; nn.Linear stores the transpose
                gwt = torch.zeros(K, N, dtype=torch.float32, device=x.device)
                _lib.call("mrb_gemm_tc_wgrad", x.data_ptr(), ldx, _lib.ptr(gy), N, M, K, N, _lib.ptr(gwt), None, N, N)
                gw = gwt.t().contiguous() if ctx.trans_w else gwt
            else:
                gw = torch.empty_like(w)
                if ctx.trans_w:   # w: N x K ; gw = gy^T @ x
                    _gemm(True, False, N, K, M, _lib.ptr(gy), N, x.data_ptr(), ldx, 0.0, _lib.ptr(gw), K)
                else:             # w: K x N ; gw = x^T @ gy
                    _gemm(True, False, K, N, M, x.data_ptr(), ldx, _lib.ptr(gy), N, 0.0, _lib.ptr(gw), N)
        return gx, gw, None


def linear(x: Tensor, weight: Tensor) -> Tensor:
    """nn.Linear(bias=False): x @ weight^T with weight stored out x in."""
    return _MatMul.apply(x, weight, True)


def matmul(x: Tensor, w: Tensor) -> Tensor:
    return _MatMul.apply(x, w, False)


# ----------------------------------------------------------------------------------------------------------
# GraphConv
# ----------------------------------------------------------------------------------------------------------
def _gather(topo_rowptr, topo_col, n, self_ptr, ld_self, nbr_ptr, ld_nbr, D, relu, out_ptr, ld_out):
    _lib.call("mrb_csr_gather_fwd", _lib.ptr(topo_rowptr), _lib.ptr(topo_col), n, self_ptr, ld_self, nbr_ptr, ld_nbr, D,
              int(relu), out_ptr, ld_out)


class _Aggregate(torch.autograd.Function):
    """out[row] = sum over edges (row, col) of matrix[col]   (reference meshRCNN/utils.py:52-57)."""

    @staticmethod
    def forward(ctx, matrix, topo):
        _require_cuda(matrix, "aggregate_neighbours")
        m = _f32c(matrix)
        n, D = m.shape
        out = torch.empty_like(m)
        _gather(topo.rowptr, topo.col, n, None, 0, _lib.ptr(m), D, D, False, _lib.ptr(out), D)
        ctx.topo = topo
        return out

    @staticmethod
    def backward(ctx, g):
        g = _f32c(g)
        n, D = g.shape
        topo = ctx.topo
        out = torch.empty_like(g)
        _gather(topo.rowptr_t, topo.col_t, n, None, 0, _lib.ptr(g), D, D, False, _lib.ptr(out), D)
        return out, None


def aggregate_neighbours(index: Tensor, matrix: Tensor) -> Tensor:
    return _Aggregate.apply(matrix, from_coo(index, matrix.shape[0]))


class _GraphConv(torch.autograd.Function):
    """relu(x W0 + A (x W1))  (reference meshRCNN/layers.py:47-68) as: one [x W0 | x W1] projection into a
    n x 2D buffer, then one CSR gather with the add and the ReLU fused."""

    @staticmethod
    def forward(ctx, x, w0, w1, topo):
        _require_cuda(x, "GraphConv")
        x, w0, w1 = _rows(x), _f32c(w0), _f32c(w1)
        n, K = x.shape
        ldx, xp = x.stride(0), x.data_ptr()
        D = w0.shape[1]
        y = torch.empty(n, 2 * D, dtype=torch.float32, device=x.device)
        yp = _lib.ptr(y)
        ctx.img_bwd = None
        ctx.wcat = None
        if _use_tc(K, 2 * D):      # one tensor-core pass over x for [x W0 | x W1]
            if ctx.needs_input_grad[0] and _use_tc(2 * D, K):
                # the operand image of the input gradient is packed by the same launch (the weights cannot change between
                # this forward and its backward: autograd would raise on an in-place update of a saved tensor)
                lib = _lib.load()
                img = torch.empty(lib.mrb_gemm_tc_image_bytes(K, 2 * D), dtype=torch.uint8, device=x.device)
                ctx.img_bwd = torch.empty(lib.mrb_gemm_tc_image_bytes(2 * D, K), dtype=torch.uint8, device=x.device)
                _lib.call("mrb_gemm_tc_pack_graphconv", _lib.ptr(w0), _lib.ptr(w1), K, D, _lib.ptr(img), _lib.ptr(ctx.img_bwd))
            else:
                img = tc_pack(w0, w1, D, 1, 1, D, K, 2 * D)
            tc_gemm(xp, ldx, n, K, img, 2 * D, yp, 2 * D)
        else:                      # narrow layers (the 3-wide ShapeNet head): one CUDA-core pass over x for [x W0 | x W1]
            ctx.wcat = torch.cat([w0, w1], 1)
            _gemm(False, False, n, 2 * D, K, xp, ldx, _lib.ptr(ctx.wcat), 2 * D, 0.0, yp, 2 * D)
        out = torch.empty(n, D, dtype=torch.float32, device=x.device)
        _gather(topo.rowptr, topo.col, n, yp, 2 * D, yp + 4 * D, 2 * D, D, True, _lib.ptr(out), D)
        ctx.save_for_backward(x, w0, w1, out)
        ctx.topo = topo
        return out

    @staticmethod
    def backward(ctx, gout):
        x, w0, w1, out = ctx.saved_tensors
        topo = ctx.topo
        n, K = x.shape
        ldx, xp = x.stride(0), x.data_ptr()
        D = w0.shape[1]
        # upstream gradients are often column slices of a wider matrix (autograd of torch.cat): read them in place
        if gout.dtype != torch.float32 or gout.stride(1) != 1 or gout.stride(0) < D:
            gout = _f32c(gout)
        ld_g = gout.stride(0)
        gy = torch.empty(n, 2 * D, dtype=torch.float32, device=x.device)
        gp = _lib.ptr(gy)
        if D % 4 == 0:
            _lib.call("mrb_graphconv_bwd_gather", _lib.ptr(topo.rowptr_t), _lib.ptr(topo.col_t), n, gout.data_ptr(), ld_g,
                      _lib.ptr(out), D, D, gp)
        else:
            _lib.call("mrb_relu_mask", gout.data_ptr(), ld_g, _lib.ptr(out), D, n, D, gp, 2 * D)
            _gather(topo.rowptr_t, topo.col_t, n, None, 0, gp, 2 * D, D, False, gp + 4 * D, 2 * D)
        gx = gw0 = gw1 = None
        if ctx.needs_input_grad[0]:
            gx = _padded_rows(n, K, x.device)      # 16-byte aligned rows: coalesced epilogue of the tensor-core kernel
            ldgx, gxp = gx.stride(0), gx.data_ptr()
            if _use_tc(2 * D, K):  # gx = [gz | A^T gz] @ [W0 | W1]^T in one pass
                img = ctx.img_bwd if ctx.img_bwd is not None else tc_pack(w0, w1, 1, D, 2, D, 2 * D, K)
                tc_gemm(gp, 2 * D, n, 2 * D, img, K, gxp, ldgx)
            else:
                wcat = getattr(ctx, "wcat", None)
                if wcat is None:
                    wcat = torch.cat([w0, w1], 1)
                _gemm(False, True, n, K, 2 * D, gp, 2 * D, _lib.ptr(wcat), 2 * D, 0.0, gxp, ldgx)
        if (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]) and _use_tc_wgrad(n, 2 * D) and D % 32 == 0:
            # dW0 | dW1 = x^T @ [gz | A^T gz]: one tensor-core pass over x and gy, reduced over the vertices
            gw = torch.zeros(2, K, D, dtype=torch.float32, device=x.device)
            _lib.call("mrb_gemm_tc_wgrad", xp, ldx, gp, 2 * D, n, K, 2 * D, _lib.ptr(gw), _lib.ptr(gw) + 4 * K * D, D, D)
            gw0, gw1 = gw[0], gw[1]
        elif ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            gwcat = torch.empty(K, 2 * D, dtype=torch.float32, device=x.device)      # [dW0 | dW1] = x^T gy in one pass
            _gemm(True, False, K, 2 * D, n, xp, ldx, gp, 2 * D, 0.0, _lib.ptr(gwcat), 2 * D)
            gw0, gw1 = gwcat[:, :D], gwcat[:, D:]
        return gx, gw0, gw1, None


def graph_conv(x: Tensor, adj: Tensor, w0: Tensor, w1: Tensor) -> Tensor:
    return _GraphConv.apply(x, w0, w1, from_coo(adj, x.shape[0]))


# ----------------------------------------------------------------------------------------------------------
# split-input GraphConv (csrc/graphconv2.cu): GraphConv on a column concatenation that is never formed
# ----------------------------------------------------------------------------------------------------------
_ROWS_CACHE = {}


def feature_rows(fmap: Tensor) -> Tensor:
    """Channels-last fp32 rows (n_img * H * W x C) of an NCHW fp32 / bf16 feature map: the A operand of the per-texel
    projections.  The three stages of a forward pass read the same map, so the last conversion is cached by tensor identity
    and version."""
    key = (fmap.data_ptr(), fmap._version, tuple(fmap.shape), fmap.dtype, fmap.device.index)
    hit = _ROWS_CACHE.get("last")
    if hit is not None and hit[0] == key:
        return hit[1]
    m = _map_tensor(fmap.detach())
    n_img, C, H, W = m.shape
    rows = torch.empty(n_img * H * W, C, dtype=torch.float32, device=m.device)
    _lib.call("mrb_feature_map_to_rows", _lib.ptr(m), int(m.dtype == torch.bfloat16), n_img, C, H * W, _lib.ptr(rows))
    _ROWS_CACHE["last"] = (key, rows)
    return rows


class TexelTerm:
    """VertexAlign of ONE square feature map in factored form (reference meshRCNN/layers.py:548-613): the channels-last
    texel rows and, per vertex, the row it gathers (-1 = masked).  ``align(f) @ W_a = (rows @ W_a)[texrow]``, so a layer that
    multiplies the aligned features by a weight block projects the n_img * H * W texels instead of the SV vertices."""

    def __init__(self, fmap: Tensor, vertex_positions: Tensor, vertices_per_mesh: Sequence[int], image_sizes,
                 mesh_index: Sequence[int], topo: Optional[MeshTopology] = None):
        _require_cuda(fmap, "VertexAlign")
        _require_cuda(vertex_positions, "VertexAlign")
        if fmap.dim() != 4 or fmap.shape[2] != fmap.shape[3]:
            raise RuntimeError("VertexAlign: feature maps must be N x C x H x W with H == W (the reference indexes H with the "
                               "x coordinate)")
        if sum(int(m) for m in mesh_index) != len(vertices_per_mesh):
            raise RuntimeError("VertexAlign: sum(mesh_index) must equal the number of meshes")
        if sum(vertices_per_mesh) != vertex_positions.shape[0]:
            raise RuntimeError("VertexAlign: vertices_per_mesh does not sum to the number of vertex positions")
        dev = vertex_positions.device
        SV = vertex_positions.shape[0]
        self.fmap = fmap
        self.n_img, self.C, self.size = int(fmap.shape[0]), int(fmap.shape[1]), int(fmap.shape[2])
        self.rows = feature_rows(fmap)
        vert_mesh = vertex_mesh_ids(vertices_per_mesh, SV, dev, topo)
        info = mesh_info_table(mesh_index, image_sizes, dev)
        self.texrow = torch.empty(SV, dtype=torch.int32, device=dev)
        _lib.call("mrb_vert_align_texrows", _lib.ptr(_f32c(vertex_positions.detach())), _lib.ptr(vert_mesh), _lib.ptr(info), SV,
                  self.size, _lib.ptr(self.texrow))


EARLY_TEXEL_PROJECTION = os.environ.get("MRB_EARLY_TEXEL", "1") != "0"     # A/B switch of PackPlan.begin's early projections
_IMAGE_BYTES = {}       # (K, N) -> mrb_gemm_tc_image_bytes(K, N) rounded up to 256


def _image_bytes(K: int, N: int) -> int:
    v = _IMAGE_BYTES.get((K, N))
    if v is None:
        v = _IMAGE_BYTES[(K, N)] = (_lib.load().mrb_gemm_tc_image_bytes(K, N) + 255) & ~255
    return v


class _ImageRef:
    """A packed weight image inside a PackPlan buffer: address + a reference that keeps the buffer alive (what ``_lib.ptr``
    needs of a tensor, without the cost of a tensor view per image on the launching thread)."""
    __slots__ = ("addr", "owner")
    is_cuda = True

    def __init__(self, addr: int, owner: Tensor):
        self.addr, self.owner = addr, owner

    def data_ptr(self) -> int:
        return self.addr

    def is_contiguous(self) -> bool:
        return True


class PackPlan:
    """Weight images of all dense GraphConv blocks of ONE forward pass, packed by a single launch.

    Every block of a pass asks for its images through ``take``; what it asked for is remembered, and the next ``begin`` (the
    start of the next pass through the same modules) packs that whole list at once (``mrb_gemm_tc_pack_graphconv_batch``: one
    launch instead of one per block).  Nothing is carried over between passes -- the images are re-packed from the current
    weights at every ``begin`` -- and a block the list does not hold (first pass, changed structure, re-allocated weights)
    simply packs its own image as before."""

    def __init__(self):
        self._asked = {}       # key -> (w0, w1, row, K, D, want_bwd), insertion order = call order of the last pass
        self._images = {}      # key -> (img, img_bwd | None) of the current pass
        self._tex_asked = {}   # keys whose A operand is the texel-row matrix of the pass's feature map
        self._tex_out = {}     # key -> (rows data_ptr, T) projected by ``launch_early``
        self._pending = None   # (feature map, keys) of the projections ``launch_early`` will issue

    @staticmethod
    def _key(w0, w1, row, K, D):
        return (w0.data_ptr(), w1.data_ptr(), row, K, D)

    def begin(self, fmap: Optional[Tensor] = None):
        """``fmap``: the pass's single feature map (Pix3D head).  The projections of its texel rows (one per stage) do not
        depend on the mesh: they are queued here and launched by ``launch_early``."""
        reqs = [r for r in self._asked.values() if r[0].is_cuda]
        tex_keys = self._tex_asked
        self._asked, self._images, self._tex_asked, self._tex_out, self._pending = {}, {}, {}, {}, None
        if not reqs:
            return
        dev = reqs[0][0].device
        sizes, total = [], 0
        for (w0, w1, row, K, D, want_bwd) in reqs:
            nf = _image_bytes(K, 2 * D)
            nb = _image_bytes(2 * D, K) if want_bwd else 0
            sizes.append((total, nf, nb))
            total += nf + nb
        buf = torch.empty(total, dtype=torch.uint8, device=dev)
        base = buf.data_ptr()
        n = len(reqs)
        VP, IA = ctypes.c_void_p * n, ctypes.c_int * n
        w0a = VP(*[r[0].data_ptr() + 4 * r[2] * r[4] for r in reqs])
        w1a = VP(*[r[1].data_ptr() + 4 * r[2] * r[4] for r in reqs])
        fa = VP(*[base + o for (o, nf, nb) in sizes])
        ba = VP(*[(base + o + nf) if nb else None for (o, nf, nb) in sizes])
        Ka, Da = IA(*[r[3] for r in reqs]), IA(*[r[4] for r in reqs])
        _lib.call("mrb_gemm_tc_pack_graphconv_batch", n, *(ctypes.addressof(x) for x in (w0a, w1a, Ka, Da, fa, ba)))
        for r, (o, nf, nb) in zip(reqs, sizes):
            key = self._key(r[0], r[1], r[2], r[3], r[4])
            self._images[key] = (_ImageRef(base + o, buf), _ImageRef(base + o + nf, buf) if nb else None, r[0]._version,
                                 r[1]._version)
        if EARLY_TEXEL_PROJECTION and fmap is not None and fmap.is_cuda and fmap.dim() == 4 and tex_keys:
            self._pending = (fmap, list(tex_keys))      # launched by ``launch_early`` (behind Cubify's count kernels)

    def launch_early(self):
        """The projections of the feature map's texel rows (one per stage): they do not depend on the mesh, so Cubify calls
        this between its count kernels and the read-back of the counters -- the device works on them while the launching
        thread is stalled."""
        pending, self._pending = self._pending, None
        if pending is None:
            return
        fmap, tex_keys = pending
        rows = feature_rows(fmap)
        R, C = rows.shape
        for key in tex_keys:
            hit = self._images.get(key)
            if hit is None or key[3] != C:
                continue
            D = key[4]
            T = torch.empty(R, 2 * D, dtype=torch.float32, device=rows.device)
            _lib.call("mrb_gemm_tc_acc", _lib.ptr(rows), C, R, C, _lib.ptr(hit[0]), 2 * D, _lib.ptr(T), 2 * D, 0)
            self._tex_out[key] = (rows.data_ptr(), T)

    def take(self, w0, w1, row, K, D, want_bwd, a_ptr=None, texel_rows=False):
        """(img, img_bwd, T | None) packed at ``begin`` for this block, or None; either way the block is on the list of the
        next pass.  ``texel_rows``: the block multiplies the texel rows of the feature map (``a_ptr``); T is its product if it
        was launched at ``begin`` from that very matrix."""
        key = self._key(w0, w1, row, K, D)
        self._asked[key] = (w0, w1, row, K, D, bool(want_bwd))
        if texel_rows:
            self._tex_asked[key] = True
        hit = self._images.get(key)
        if hit is None or (want_bwd and hit[1] is None) or hit[2] != w0._version or hit[3] != w1._version:
            return None
        T = None
        if texel_rows:
            t = self._tex_out.pop(key, None)
            if t is not None and t[0] == a_ptr:
                T = t[1]
        return hit[0], (hit[1] if want_bwd else None), T


_PACK_TLS = threading.local()       # .plan: the PackPlan of the pass running on this thread (one thread per GPU is supported)


def defer_until_stall(fn) -> None:
    """Registers mesh-independent device work of this thread's pass (a callable issuing launches on the current stream): it
    runs at the next point where the launching thread has to wait for the device anyway (Cubify's counter read-back)."""
    lst = getattr(_PACK_TLS, "deferred", None)
    if lst is None:
        lst = _PACK_TLS.deferred = []
    lst.append(fn)


def run_deferred() -> None:
    plan = getattr(_PACK_TLS, "plan", None)
    if plan is not None:
        plan.launch_early()
    lst = getattr(_PACK_TLS, "deferred", None)
    if lst:
        _PACK_TLS.deferred = []
        for fn in lst:
            fn()


class pack_plan:
    """``with pack_plan(plan):`` -- the dense GraphConv blocks evaluated inside (on this thread) use and feed ``plan``."""

    def __init__(self, plan: Optional[PackPlan], fmap: Optional[Tensor] = None):
        self.plan, self.fmap = plan, fmap

    def __enter__(self):
        self.prev = getattr(_PACK_TLS, "plan", None)
        _PACK_TLS.plan = self.plan
        if self.plan is not None:
            self.plan.begin(self.fmap)
        return self.plan

    def __exit__(self, *exc):
        _PACK_TLS.plan = self.prev
        _PACK_TLS.deferred = []             # work registered for a stall that never came (an exception on the way) is dropped
        return False


def _project_block(a_ptr: int, lda: int, M: int, K: int, w0: Tensor, w1: Tensor, row: int, D: int, c_ptr: int, accumulate: bool,
                   want_bwd_image: bool, texel_rows: bool = False, out: Optional[list] = None):
    """C[M x 2D] (+)= A[M x K] @ [W0[row:row+K] | W1[row:row+K]].  Returns the operand image of the input gradient
    ([gz | A^T gz] @ [W0 | W1]^T block) when it was packed in the same launch, else None."""
    dev = w0.device
    p0, p1 = w0.data_ptr() + 4 * row * D, w1.data_ptr() + 4 * row * D
    if _use_tc(K, 2 * D):
        lib = _lib.load()
        want_bwd = bool(want_bwd_image and _use_tc(2 * D, K))
        plan = getattr(_PACK_TLS, "plan", None)
        if plan is not None:
            hit = plan.take(w0, w1, row, K, D, want_bwd, a_ptr, texel_rows and lda == K and not accumulate)
            if hit is not None:                         # packed with all the other blocks of this pass
                if hit[2] is not None and out is not None:
                    out.append(hit[2])                  # ... and already projected (texel rows): the caller takes this T
                else:
                    _lib.call("mrb_gemm_tc_acc", a_ptr, lda, M, K, _lib.ptr(hit[0]), 2 * D, c_ptr, 2 * D, int(accumulate))
                return hit[1]
        img = torch.empty(lib.mrb_gemm_tc_image_bytes(K, 2 * D), dtype=torch.uint8, device=dev)
        img_bwd = None
        if want_bwd_image and _use_tc(2 * D, K):
            img_bwd = torch.empty(lib.mrb_gemm_tc_image_bytes(2 * D, K), dtype=torch.uint8, device=dev)
            _lib.call("mrb_gemm_tc_pack_graphconv", p0, p1, K, D, _lib.ptr(img), _lib.ptr(img_bwd))
        else:
            _lib.call("mrb_gemm_tc_pack", p0, p1, D, 1, 1, D, K, 2 * D, _lib.ptr(img))
        _lib.call("mrb_gemm_tc_acc", a_ptr, lda, M, K, _lib.ptr(img), 2 * D, c_ptr, 2 * D, int(accumulate))
        return img_bwd
    beta = 1.0 if accumulate else 0.0
    _gemm(False, False, M, D, K, a_ptr, lda, p0, D, beta, c_ptr, 2 * D)
    _gemm(False, False, M, D, K, a_ptr, lda, p1, D, beta, c_ptr + 4 * D, 2 * D)
    return None


def _backproject_block(g_ptr: int, M: int, K: int, w0: Tensor, w1: Tensor, row: int, D: int, img_bwd, out_ptr: int, ldo: int):
    """out[M x K] = G[M x 2D] @ [W0[row:row+K] | W1[row:row+K]]^T."""
    p0, p1 = w0.data_ptr() + 4 * row * D, w1.data_ptr() + 4 * row * D
    if _use_tc(2 * D, K):
        if img_bwd is None:
            img_bwd = torch.empty(_lib.load().mrb_gemm_tc_image_bytes(2 * D, K), dtype=torch.uint8, device=w0.device)
            _lib.call("mrb_gemm_tc_pack", p0, p1, 1, D, 2, D, 2 * D, K, _lib.ptr(img_bwd))
        tc_gemm(g_ptr, 2 * D, M, 2 * D, img_bwd, K, out_ptr, ldo)
    else:
        _gemm(False, True, M, K, D, g_ptr, 2 * D, p0, D, 0.0, out_ptr, ldo)
        _gemm(False, True, M, K, D, g_ptr + 4 * D, 2 * D, p1, D, 1.0, out_ptr, ldo)


class _GraphConvSplit(torch.autograd.Function):
    """relu([parts] W0 + A ([parts] W1)) (+ residual) for a column concatenation ``parts`` of dense blocks, the vertex
    positions and a VertexAlign term -- evaluated part by part (csrc/graphconv2.cu), nothing is concatenated.

    ``spec = (main_rows, pos_row, tex_row, tex)``: first row in w0 / w1 of every dense block, of the 3 position rows (or None)
    and of the aligned-feature rows (or None) with their ``TexelTerm``."""

    @staticmethod
    def forward(ctx, topo, spec, w0, w1, pos, fmap, residual, *mains):
        main_rows, pos_row, tex_row, tex = spec
        _require_cuda(w0, "GraphConv")
        w0, w1 = _f32c(w0), _f32c(w1)
        Ktot, D = w0.shape
        dev = w0.device
        n = topo.num_vertices
        mains = [_rows(m) for m in mains]
        for m in mains:
            _require_cuda(m, "GraphConv")
        pos_c = None if pos is None else _f32c(pos.detach())
        need_gx = [ctx.needs_input_grad[7 + i] for i in range(len(mains))]
        y = None
        imgs_bwd = []
        if mains:
            y = torch.empty(n, 2 * D, dtype=torch.float32, device=dev)
            for i, (m, r) in enumerate(zip(mains, main_rows)):
                imgs_bwd.append(_project_block(m.data_ptr(), m.stride(0), n, m.shape[1], w0, w1, r, D, _lib.ptr(y), i > 0,
                                               need_gx[i]))
        T = None
        tex_img_bwd = None
        if tex is not None:
            R = tex.rows.shape[0]
            T = torch.empty(R, 2 * D, dtype=torch.float32, device=dev)
            early = []
            tex_img_bwd = _project_block(_lib.ptr(tex.rows), tex.C, R, tex.C, w0, w1, tex_row, D, _lib.ptr(T), False,
                                         ctx.needs_input_grad[5], texel_rows=True, out=early)
            if early:                                   # projected at the start of the pass (functional.PackPlan.begin)
                T = early[0]
        out = torch.empty(n, D, dtype=torch.float32, device=dev)
        mask = torch.empty(n, (D + 31) // 32, dtype=torch.int32, device=dev)
        res = None if residual is None else _rows(residual)
        wp0 = wp1 = None
        if pos_c is not None:
            wp0, wp1 = w0.data_ptr() + 4 * pos_row * D, w1.data_ptr() + 4 * pos_row * D
        _lib.call("mrb_gc_gather_fwd", _lib.ptr(topo.rowptr), _lib.ptr(topo.col), n, D, _lib.ptr(y), 2 * D, _lib.ptr(pos_c), wp0, wp1,
                  None if tex is None else _lib.ptr(tex.texrow), _lib.ptr(T), 1, _lib.ptr(mask),
                  None if res is None else res.data_ptr(), 0 if res is None else res.stride(0), _lib.ptr(out), D)
        saved = [w0, w1, mask] + ([] if pos_c is None else [pos_c]) + mains
        ctx.save_for_backward(*saved)
        ctx.topo, ctx.spec, ctx.imgs_bwd, ctx.tex_img_bwd = topo, spec, imgs_bwd, tex_img_bwd
        ctx.has_pos = pos_c is not None
        return out

    @staticmethod
    def backward(ctx, gout):
        main_rows, pos_row, tex_row, tex = ctx.spec
        w0, w1, mask = ctx.saved_tensors[:3]
        rest = list(ctx.saved_tensors[3:])
        pos_c = rest.pop(0) if ctx.has_pos else None
        mains = rest
        topo = ctx.topo
        n = topo.num_vertices
        Ktot, D = w0.shape
        dev = w0.device
        if gout.dtype != torch.float32 or gout.stride(1) != 1 or gout.stride(0) < D:
            gout = _f32c(gout)
        need_w = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        need_pos = ctx.has_pos and ctx.needs_input_grad[4]
        need_tex = tex is not None and (need_w or ctx.needs_input_grad[5])
        gy = torch.empty(n, 2 * D, dtype=torch.float32, device=dev)
        gpos = torch.empty(n, 3, dtype=torch.float32, device=dev) if need_pos else None
        gT = None
        if need_tex:
            R = tex.rows.shape[0]
            gT = torch.empty(R, 2 * D, dtype=torch.float32, device=dev)
        wp0 = wp1 = None
        if ctx.has_pos:
            wp0, wp1 = w0.data_ptr() + 4 * pos_row * D, w1.data_ptr() + 4 * pos_row * D
        _lib.call("mrb_gc_gather_bwd", _lib.ptr(topo.rowptr_t), _lib.ptr(topo.col_t), n, D, gout.data_ptr(), gout.stride(0),
                  _lib.ptr(mask), _lib.ptr(gy), wp0 if need_pos else None, wp1 if need_pos else None, _lib.ptr(gpos),
                  _lib.ptr(tex.texrow) if need_tex else None, _lib.ptr(gT), gT.shape[0] if need_tex else 0)
        gp = _lib.ptr(gy)
        gmains = []
        for i, (m, r) in enumerate(zip(mains, main_rows)):
            if ctx.needs_input_grad[7 + i]:
                K = m.shape[1]
                gx = torch.empty(n, K, dtype=torch.float32, device=dev)
                _backproject_block(gp, n, K, w0, w1, r, D, ctx.imgs_bwd[i], _lib.ptr(gx), K)
                gmains.append(gx)
            else:
                gmains.append(None)
        gw0 = gw1 = None
        if need_w:
            gw = torch.zeros(2, Ktot, D, dtype=torch.float32, device=dev)
            g0, g1 = gw.data_ptr(), gw.data_ptr() + 4 * Ktot * D
            tail_done = not ctx.has_pos
            tc_ok = _use_tc_wgrad(n, 2 * D) and D % 32 == 0
            for m, r in zip(mains, main_rows):
                K = m.shape[1]
                if tc_ok:
                    with_tail = not tail_done
                    _lib.call("mrb_gemm_tc_wgrad_split", m.data_ptr(), m.stride(0), gp, 2 * D, n, K, 2 * D, g0 + 4 * r * D,
                              g1 + 4 * r * D, D, D, _lib.ptr(pos_c) if with_tail else None, 3, 3 if with_tail else 0,
                              g0 + 4 * pos_row * D if with_tail else None, g1 + 4 * pos_row * D if with_tail else None)
                    tail_done = True
                else:
                    _gemm(True, False, K, D, n, m.data_ptr(), m.stride(0), gp, 2 * D, 0.0, g0 + 4 * r * D, D)
                    _gemm(True, False, K, D, n, m.data_ptr(), m.stride(0), gp + 4 * D, 2 * D, 0.0, g1 + 4 * r * D, D)
            if not tail_done:           # no dense block carried the 3 position rows along: pos^T gy on the CUDA cores
                _gemm(True, False, 3, D, n, _lib.ptr(pos_c), 3, gp, 2 * D, 0.0, g0 + 4 * pos_row * D, D)
                _gemm(True, False, 3, D, n, _lib.ptr(pos_c), 3, gp + 4 * D, 2 * D, 0.0, g1 + 4 * pos_row * D, D)
            if tex is not None:         # rows^T gT -> the aligned-feature rows of dW0 | dW1
                R, C = tex.rows.shape
                if _use_tc_wgrad(R, 2 * D) and D % 32 == 0:
                    _lib.call("mrb_gemm_tc_wgrad", _lib.ptr(tex.rows), C, _lib.ptr(gT), 2 * D, R, C, 2 * D, g0 + 4 * tex_row * D,
                              g1 + 4 * tex_row * D, D, D)
                else:
                    _gemm(True, False, C, D, R, _lib.ptr(tex.rows), C, _lib.ptr(gT), 2 * D, 0.0, g0 + 4 * tex_row * D, D)
                    _gemm(True, False, C, D, R, _lib.ptr(tex.rows), C, _lib.ptr(gT) + 4 * D, 2 * D, 0.0, g1 + 4 * tex_row * D, D)
            gw0, gw1 = gw[0], gw[1]
        gfmap = None
        if tex is not None and ctx.needs_input_grad[5]:
            R, C = tex.rows.shape
            g_rows = torch.empty(R, C, dtype=torch.float32, device=dev)
            _backproject_block(_lib.ptr(gT), R, C, w0, w1, tex_row, D, ctx.tex_img_bwd, _lib.ptr(g_rows), C)
            gfmap = torch.empty(tex.fmap.shape, dtype=torch.float32, device=dev)
            _lib.call("mrb_rows_to_feature_map", _lib.ptr(g_rows), C, tex.n_img, C, tex.size * tex.size, _lib.ptr(gfmap))
            if tex.fmap.dtype != torch.float32:
                gfmap = gfmap.to(tex.fmap.dtype)
        gres = gout if ctx.needs_input_grad[6] else None
        return (None, None, gw0, gw1, gpos, gfmap, gres) + tuple(gmains)


def graph_conv_parts(parts, adj: Tensor, w0: Tensor, w1: Tensor, residual: Optional[Tensor] = None) -> Tensor:
    """GraphConv (reference meshRCNN/layers.py:47-68) of ``torch.cat([...], dim=1)`` given as its parts, in the reference's
    column order: ``("x", dense SV x K matrix)``, ``("pos", SV x 3 vertex positions)``, ``("tex", TexelTerm)``.
    ``residual`` (optional, SV x D) is added after the ReLU (ResGraphConv skip, layers.py:96-100)."""
    D = w0.shape[1]
    mains, main_rows, pos, pos_row, tex, tex_row = [], [], None, None, None, None
    row = 0
    n = None
    for kind, t in parts:
        if kind == "x":
            mains.append(t)
            main_rows.append(row)
            row += t.shape[1]
            n = t.shape[0]
        elif kind == "pos":
            if pos is not None or t.shape[1] != 3:
                raise RuntimeError("graph_conv_parts: one SV x 3 position block")
            pos, pos_row = t, row
            row += 3
            n = t.shape[0]
        elif kind == "tex":
            if tex is not None:
                raise RuntimeError("graph_conv_parts: one VertexAlign term")
            tex, tex_row = t, row
            row += t.C
            n = t.texrow.shape[0]
        else:
            raise RuntimeError("graph_conv_parts: unknown part %r" % (kind,))
    if row != w0.shape[0]:
        raise RuntimeError("graph_conv_parts: parts are %d columns wide, the weights expect %d" % (row, w0.shape[0]))
    if D % 4:        # odd output widths (the 3-wide ShapeNet head): the generic path on the materialised concatenation
        if tex is not None:
            raise RuntimeError("graph_conv_parts: out_features %% 4 != 0 is not supported with a VertexAlign term")
        dense = [t for _, t in parts]
        out = graph_conv(dense[0] if len(dense) == 1 else concat_cols(dense), adj, w0, w1)
        return out if residual is None else out + residual
    topo = from_coo(adj, n)
    spec = (tuple(main_rows), pos_row, tex_row, tex)
    return _GraphConvSplit.apply(topo, spec, w0, w1, pos, None if tex is None else tex.fmap, residual, *mains)


class _PositionHead(torch.autograd.Function):
    """new_pos = pos + tanh([pos | x] W^T)  (reference layers.py:255-259 without, :335-339 with the position columns) in one
    kernel; returns new_pos."""

    @staticmethod
    def forward(ctx, x, pos, weight, x_col, p_col):
        _require_cuda(x, "position head")
        x, pos_c, w = _rows(x), _f32c(pos), _f32c(weight)
        n, Kx = x.shape
        if w.shape[0] != 3:
            raise RuntimeError("position head: the weight must be 3 x in_features")
        new_pos = torch.empty(n, 3, dtype=torch.float32, device=x.device)
        delta = torch.empty(n, 3, dtype=torch.float32, device=x.device)
        _lib.call("mrb_head_fwd", x.data_ptr(), x.stride(0), Kx, _lib.ptr(pos_c), _lib.ptr(w), w.shape[1], x_col, p_col, n,
                  _lib.ptr(new_pos), _lib.ptr(delta))
        ctx.save_for_backward(x, pos_c, w, delta)
        ctx.cols = (x_col, p_col)
        return new_pos

    @staticmethod
    def backward(ctx, g):
        x, pos_c, w, delta = ctx.saved_tensors
        x_col, p_col = ctx.cols
        n, Kx = x.shape
        dev = x.device
        g = _f32c(g)
        gpre = torch.empty(n, 3, dtype=torch.float32, device=dev)
        gx = torch.empty(n, Kx, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        gpos = torch.empty(n, 3, dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        _lib.call("mrb_head_bwd", _lib.ptr(g), _lib.ptr(delta), _lib.ptr(w), w.shape[1], x_col, p_col, n, Kx, _lib.ptr(gpre),
                  _lib.ptr(gx), Kx, _lib.ptr(gpos))
        gw = None
        if ctx.needs_input_grad[2]:
            gw = torch.empty_like(w)            # dW[:, cols] = gpre^T @ [x | pos]: the two blocks cover every column
            ldw = w.shape[1]
            _gemm(True, False, 3, Kx, n, _lib.ptr(gpre), 3, x.data_ptr(), x.stride(0), 0.0, gw.data_ptr() + 4 * x_col, ldw)
            if p_col >= 0:
                _gemm(True, False, 3, 3, n, _lib.ptr(gpre), 3, _lib.ptr(pos_c), 3, 0.0, gw.data_ptr() + 4 * p_col, ldw)
        return gx, gpos, gw, None, None


def position_head(x: Tensor, pos: Tensor, weight: Tensor, pos_first: Optional[bool]) -> Tensor:
    """``pos + tanh(linear(cat([pos, x])))`` (``pos_first=True``, Pix3D), ``pos + tanh(linear(x))`` (``pos_first=None``)."""
    Kx = x.shape[1]
    if pos_first is None:
        x_col, p_col = 0, -1
    elif pos_first:
        x_col, p_col = 3, 0
    else:
        x_col, p_col = 0, Kx
    if weight.shape[1] != Kx + (0 if p_col < 0 else 3):
        raise RuntimeError("position head: weight is 3 x %d, inputs are %d columns wide" % (weight.shape[1], Kx + (0 if p_col < 0 else 3)))
    return _PositionHead.apply(x, pos, weight, x_col, p_col)


# ----------------------------------------------------------------------------------------------------------
# VertexAlign
# ----------------------------------------------------------------------------------------------------------
def _map_tensor(f: Tensor) -> Tensor:
    """Feature maps are consumed as fp32 or bf16 NCHW (north star: "bf16 features rtol 2e-2"); anything else -> fp32."""
    if f.dtype == torch.bfloat16:
        return f if f.is_contiguous() else f.contiguous()
    return _f32c(f)


class _VertAlign(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, vert_mesh, mesh_info, *fmaps):
        _require_cuda(pos, "VertexAlign")
        pos_c = _f32c(pos.detach())
        maps = []
        for f in fmaps:
            _require_cuda(f, "VertexAlign")
            if f.dim() != 4:
                raise RuntimeError("VertexAlign: feature maps must be N x C x H x W")
            maps.append(_map_tensor(f))
        SV = pos_c.shape[0]
        ctot = sum(m.shape[1] for m in maps)
        out = torch.empty(SV, ctot, dtype=torch.float32, device=pos.device)
        off = 0
        for m in maps:
            n_img, C, Hm, Wm = m.shape
            ws = torch.empty_like(m)          # channels-last copy for the row gather
            name = "mrb_vert_align_fwd_bf16" if m.dtype == torch.bfloat16 else "mrb_vert_align_fwd"
            _lib.call(name, _lib.ptr(m), n_img, C, Hm, Wm, _lib.ptr(pos_c), _lib.ptr(vert_mesh), _lib.ptr(mesh_info), SV,
                      _lib.ptr(out) + 4 * off, ctot, _lib.ptr(ws))
            off += C
        ctx.save_for_backward(pos_c, vert_mesh, mesh_info)
        ctx.shapes = [tuple(m.shape) for m in maps]
        ctx.dtypes = [f.dtype for f in fmaps]
        return out

    @staticmethod
    def backward(ctx, gout):
        pos_c, vert_mesh, mesh_info = ctx.saved_tensors
        gout = _rows(gout)                       # usually a column slice of a stage-input gradient: read in place
        SV, ctot = gout.shape
        ldg = gout.stride(0)
        grads = []
        off = 0
        for i, shape in enumerate(ctx.shapes):
            n_img, C, Hm, Wm = shape
            if ctx.needs_input_grad[3 + i]:
                g = torch.zeros(shape, dtype=torch.float32, device=gout.device)
                _lib.call("mrb_vert_align_bwd", gout.data_ptr() + 4 * off, ldg, n_img, C, Hm, Wm, _lib.ptr(pos_c),
                          _lib.ptr(vert_mesh), _lib.ptr(mesh_info), SV, _lib.ptr(g))
                grads.append(g.to(ctx.dtypes[i]))
            else:
                grads.append(None)
            off += C
        return (None, None, None) + tuple(grads)   # no gradient to positions (reference layers.py:592)


def vert_align(img_features: Sequence[Tensor], vertex_positions: Tensor, vertices_per_mesh: Sequence[int],
               image_sizes, mesh_index: Sequence[int], topo: Optional[MeshTopology] = None) -> Tensor:
    dev = vertex_positions.device
    _require_cuda(vertex_positions, "VertexAlign")
    if sum(int(m) for m in mesh_index) != len(vertices_per_mesh):
        raise RuntimeError("VertexAlign: sum(mesh_index) must equal the number of meshes")
    if sum(vertices_per_mesh) != vertex_positions.shape[0]:
        raise RuntimeError("VertexAlign: vertices_per_mesh does not sum to the number of vertex positions")
    vert_mesh = vertex_mesh_ids(vertices_per_mesh, vertex_positions.shape[0], dev, topo)
    info = mesh_info_table(mesh_index, image_sizes, dev)
    return _VertAlign.apply(vertex_positions, vert_mesh, info, *img_features)


# ----------------------------------------------------------------------------------------------------------
# bilinear VertexAlign (opt-in; csrc/vert_align_bilinear.cu): differentiable in the vertex positions
# ----------------------------------------------------------------------------------------------------------
def _square_maps(fmaps: Sequence[Tensor], what: str) -> List[Tensor]:
    maps = []
    for f in fmaps:
        _require_cuda(f, what)
        if f.dim() != 4 or f.shape[2] != f.shape[3]:
            raise RuntimeError("VertexAlign: feature maps must be N x C x H x W with H == W (the reference indexes H with the "
                               "x coordinate)")
        maps.append(_map_tensor(f))
    return maps


def _bilinear_tables(img_features: Sequence[Tensor], vertex_positions: Tensor, vertices_per_mesh: Sequence[int],
                     mesh_index: Sequence[int], image_sizes):
    """(vert_mesh, mesh_info) of the bilinear kernels after the host-side checks that keep every index they read in range:
    each vertex's mesh has a mesh_info row, and each image that holds a mesh exists in every map.  vert_mesh is built from
    ``vertices_per_mesh`` itself (not taken from a registered topology), so it cannot name a mesh the table lacks."""
    _require_cuda(vertex_positions, "VertexAlign")
    if vertex_positions.dim() != 2 or vertex_positions.shape[1] != 3:
        raise RuntimeError("VertexAlign: vertex positions must be SV x 3")
    if len(mesh_index) != len(image_sizes):
        raise RuntimeError("VertexAlign: mesh_index and image_sizes differ in length")
    if any(int(m) < 0 for m in mesh_index) or any(int(c) < 0 for c in vertices_per_mesh):
        raise RuntimeError("VertexAlign: negative mesh or vertex count")
    if sum(int(m) for m in mesh_index) != len(vertices_per_mesh):
        raise RuntimeError("VertexAlign: sum(mesh_index) must equal the number of meshes")
    if sum(int(c) for c in vertices_per_mesh) != vertex_positions.shape[0]:
        raise RuntimeError("VertexAlign: vertices_per_mesh does not sum to the number of vertex positions")
    used = [i for i, m in enumerate(mesh_index) if int(m) > 0]
    for f in img_features:
        if used and f.dim() == 4 and used[-1] >= f.shape[0]:
            raise RuntimeError("VertexAlign: image %d holds a mesh but the feature map has %d images" % (used[-1], f.shape[0]))
    dev = vertex_positions.device
    SV = vertex_positions.shape[0]
    vert_mesh = vertex_mesh_ids(vertices_per_mesh, SV, dev) if SV else torch.empty(0, dtype=torch.int32, device=dev)
    return vert_mesh, mesh_info_table(mesh_index, image_sizes, dev)


class _VertAlignBilinear(torch.autograd.Function):
    """Bilinear VertexAlign of every map into its column block of an SV x sum(C_m) output; gradients to the maps and to the
    vertex positions (csrc/vert_align_bilinear.cu)."""

    @staticmethod
    def forward(ctx, pos, vert_mesh, mesh_info, *fmaps):
        pos_c = _f32c(pos.detach())
        maps = _square_maps(fmaps, "VertexAlign")
        SV = pos_c.shape[0]
        ctot = sum(m.shape[1] for m in maps)
        out = torch.empty(SV, ctot, dtype=torch.float32, device=pos.device)
        rows, off = [], 0
        for m in maps:
            n_img, C, S, _ = m.shape
            r = feature_rows(m)
            _lib.call("mrb_vert_align_bilinear_fwd", _lib.ptr(r), C, C, S, n_img, _lib.ptr(pos_c), _lib.ptr(vert_mesh),
                      _lib.ptr(mesh_info), SV, 0, _lib.ptr(out) + 4 * off, ctot)
            rows.append(r)
            off += C
        ctx.save_for_backward(pos_c, vert_mesh, mesh_info, *rows)
        ctx.shapes = [tuple(m.shape) for m in maps]
        ctx.dtypes = [f.dtype for f in fmaps]
        ctx.pos_dtype = pos.dtype
        return out

    @staticmethod
    def backward(ctx, gout):
        pos_c, vert_mesh, mesh_info = ctx.saved_tensors[:3]
        rows = ctx.saved_tensors[3:]
        gout = _rows(gout)
        SV, ldg = gout.shape[0], gout.stride(0)
        dev = gout.device
        gpos = torch.zeros(SV, 3, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        grads, off = [], 0
        for i, (shape, r) in enumerate(zip(ctx.shapes, rows)):
            n_img, C, S, _ = shape
            grows = torch.zeros(r.shape, dtype=torch.float32, device=dev) if ctx.needs_input_grad[3 + i] else None
            if grows is not None or gpos is not None:
                _lib.call("mrb_vert_align_bilinear_bwd", gout.data_ptr() + 4 * off, ldg, _lib.ptr(r), C, C, S, n_img,
                          _lib.ptr(pos_c), _lib.ptr(vert_mesh), _lib.ptr(mesh_info), SV, _lib.ptr(grows), C, _lib.ptr(gpos), 1)
            if grows is not None:
                g = torch.empty(shape, dtype=torch.float32, device=dev)
                _lib.call("mrb_rows_to_feature_map", _lib.ptr(grows), C, n_img, C, S * S, _lib.ptr(g))
                grads.append(g if ctx.dtypes[i] == torch.float32 else g.to(ctx.dtypes[i]))
            else:
                grads.append(None)
            off += C
        if gpos is not None and ctx.pos_dtype != torch.float32:
            gpos = gpos.to(ctx.pos_dtype)
        return (gpos, None, None) + tuple(grads)


def vert_align_bilinear(img_features: Sequence[Tensor], vertex_positions: Tensor, vertices_per_mesh: Sequence[int],
                        image_sizes, mesh_index: Sequence[int]) -> Tensor:
    """Bilinear VertexAlign (the opt-in mode of ``layers.VertexAlign``): SV x sum(C_m), differentiable in every map and in
    ``vertex_positions``.  Same projection and axis convention as ``vert_align``; each square map is then sampled like
    ``grid_sample(align_corners=True, padding_mode="border")`` -- see csrc/vert_align_bilinear.cu for the exact
    definition.  fp32 or bf16 maps; the output and the position gradient are fp32, map gradients come in the map's dtype."""
    vert_mesh, info = _bilinear_tables(img_features, vertex_positions, vertices_per_mesh, mesh_index, image_sizes)
    return _VertAlignBilinear.apply(vertex_positions, vert_mesh, info, *img_features)


def _project_texels(maps: Sequence[Tensor], w: Tensor, n_img: int):
    """T = per-texel projections of every map, packed map after map: T[r0_m + r] = rows_m[r] @ W[:, c0_m:c0_m+C_m]^T, with
    rows_m the channels-last fp32 rows of map m in (image, x1, y1) order.  Returns (T, [rows_m], [R_m])."""
    lib = _lib.load()
    dev = w.device
    D, ctot = w.shape
    rows_per_map = [n_img * m.shape[2] * m.shape[3] for m in maps]
    T = torch.empty(sum(rows_per_map), D, dtype=torch.float32, device=dev)
    rows_cl, r0, c0 = [], 0, 0
    for m, R in zip(maps, rows_per_map):
        C = m.shape[1]
        cl = torch.empty(R, C, dtype=torch.float32, device=dev)
        _lib.call("mrb_feature_map_to_rows", _lib.ptr(m), int(m.dtype == torch.bfloat16), n_img, C, R // n_img, _lib.ptr(cl))
        # T[r0:r0+R] = cl @ W[:, c0:c0+C]^T : logical operand B(k, n) = W[n, c0 + k]
        if _use_tc(C, D):
            img = torch.empty(lib.mrb_gemm_tc_image_bytes(C, D), dtype=torch.uint8, device=dev)
            _lib.call("mrb_gemm_tc_pack", w.data_ptr() + 4 * c0, None, 1, ctot, 0, 0, C, D, _lib.ptr(img))
            tc_gemm(_lib.ptr(cl), C, R, C, img, D, T.data_ptr() + 4 * r0 * D, D)
        else:
            _gemm(False, True, R, D, C, _lib.ptr(cl), C, w.data_ptr() + 4 * c0, ctot, 0.0, T.data_ptr() + 4 * r0 * D, D)
        rows_cl.append(cl)
        r0 += R
        c0 += C
    return T, rows_cl, rows_per_map


def _backproject_texels(gT: Tensor, w: Tensor, rows_cl, shapes, rows_per_map, dtypes, n_img: int, want_w: bool, want_maps):
    """Weight and map gradients from the gradient gT of the packed projections T (``_project_texels``): dW_m^T = rows_m^T @
    gT_m and d map_m = NCHW(gT_m @ W[:, c0_m:c0_m+C_m]).  Returns (gW or None, [gmap_m or None])."""
    lib = _lib.load()
    dev = gT.device
    D, ctot = w.shape
    gwt = torch.zeros(ctot, D, dtype=torch.float32, device=dev) if want_w else None
    gmaps = []
    r0 = c0 = 0
    for i, (shape, R, cl) in enumerate(zip(shapes, rows_per_map, rows_cl)):
        C = shape[1]
        gt_ptr = gT.data_ptr() + 4 * r0 * D
        if gwt is not None:             # dW_m^T (C x D) = rows_m^T @ gT_m
            if _use_tc_wgrad(R, D):
                _lib.call("mrb_gemm_tc_wgrad", _lib.ptr(cl), C, gt_ptr, D, R, C, D, gwt.data_ptr() + 4 * c0 * D, None, D, D)
            else:
                _gemm(True, False, C, D, R, _lib.ptr(cl), C, gt_ptr, D, 0.0, gwt.data_ptr() + 4 * c0 * D, D)
        if want_maps[i]:                # d rows_m (R x C) = gT_m @ W[:, c0:c0+C] : B(k, n) = W[k, c0 + n]
            g_rows = torch.empty(R, C, dtype=torch.float32, device=dev)
            if _use_tc(D, C):
                img = torch.empty(lib.mrb_gemm_tc_image_bytes(D, C), dtype=torch.uint8, device=dev)
                _lib.call("mrb_gemm_tc_pack", w.data_ptr() + 4 * c0, None, ctot, 1, 0, 0, D, C, _lib.ptr(img))
                tc_gemm(gt_ptr, D, R, D, img, C, _lib.ptr(g_rows), C)
            else:
                _gemm(False, False, R, C, D, gt_ptr, D, w.data_ptr() + 4 * c0, ctot, 0.0, _lib.ptr(g_rows), C)
            g = torch.empty(shape, dtype=torch.float32, device=dev)
            _lib.call("mrb_rows_to_feature_map", _lib.ptr(g_rows), C, n_img, C, R // n_img, _lib.ptr(g))
            gmaps.append(g if dtypes[i] == torch.float32 else g.to(dtypes[i]))
        else:
            gmaps.append(None)
        r0 += R
        c0 += C
    gw = gwt.t().contiguous() if gwt is not None else None      # nn.Linear stores out x in
    return gw, gmaps


def _linear_maps(weight: Tensor, fmaps: Sequence[Tensor]):
    """(fp32 weight, maps, n_img) of linear(VertexAlign(maps)) after the shape checks."""
    w = _f32c(weight)
    D, ctot = w.shape
    maps = _square_maps(fmaps, "VertexAlign+linear")
    n_img = maps[0].shape[0]
    if any(m.shape[0] != n_img for m in maps) or sum(m.shape[1] for m in maps) != ctot:
        raise RuntimeError("VertexAlign+linear: maps %s do not match the %d x %d weight" %
                           ([tuple(m.shape) for m in maps], D, ctot))
    if D % 4 or not 1 <= len(maps) <= 8:
        raise RuntimeError("VertexAlign+linear: out_features %% 4 == 0 and 1..8 maps required")
    return w, maps, n_img


class _VertAlignLinear(torch.autograd.Function):
    """linear(VertexAlign(maps))  =  sum over maps of  mask * (texel rows @ W_m^T)[texel(v)]   (csrc/align_proj.cu).

    The texels of every map are projected once on the tensor cores (n_img * HW_m rows instead of SV), every vertex then
    gathers and sums one D-wide row per map; the SV x sum(C_m) VertexAlign output is never formed.  Replaces
    ``self.linear(self.vertAlign(...))`` of the ShapeNet stages (reference meshRCNN/layers.py:151-155,226-230)."""

    @staticmethod
    def forward(ctx, pos, vert_mesh, mesh_info, weight, *fmaps):
        _require_cuda(pos, "VertexAlign+linear")
        dev = pos.device
        pos_c = _f32c(pos.detach())
        w, maps, n_img = _linear_maps(weight, fmaps)
        D = w.shape[0]
        sizes = (ctypes.c_int * len(maps))(*[int(m.shape[2]) for m in maps])
        T, rows_cl, rows_per_map = _project_texels(maps, w, n_img)
        SV = pos_c.shape[0]
        out = torch.empty(SV, D, dtype=torch.float32, device=dev)
        _lib.call("mrb_vert_align_proj_fwd", _lib.ptr(T), D, len(maps), sizes, n_img, _lib.ptr(pos_c), _lib.ptr(vert_mesh),
                  _lib.ptr(mesh_info), SV, _lib.ptr(out), D)
        ctx.save_for_backward(pos_c, vert_mesh, mesh_info, w, *rows_cl)
        ctx.meta = (sizes, n_img, [tuple(m.shape) for m in maps], [f.dtype for f in fmaps], rows_per_map)
        return out

    @staticmethod
    def backward(ctx, gout):
        pos_c, vert_mesh, mesh_info, w = ctx.saved_tensors[:4]
        rows_cl = ctx.saved_tensors[4:]
        sizes, n_img, shapes, dtypes, rows_per_map = ctx.meta
        dev = gout.device
        D = w.shape[0]
        gout = _rows(gout)
        SV = gout.shape[0]
        gT = torch.empty(sum(rows_per_map), D, dtype=torch.float32, device=dev)
        _lib.call("mrb_vert_align_proj_bwd", gout.data_ptr(), gout.stride(0), D, len(shapes), sizes, n_img, _lib.ptr(pos_c),
                  _lib.ptr(vert_mesh), _lib.ptr(mesh_info), SV, _lib.ptr(gT))
        gw, gmaps = _backproject_texels(gT, w, rows_cl, shapes, rows_per_map, dtypes, n_img, ctx.needs_input_grad[3],
                                        ctx.needs_input_grad[4:])
        return (None, None, None, gw) + tuple(gmaps)


class _VertAlignLinearBilinear(torch.autograd.Function):
    """linear(bilinear VertexAlign(maps)) = sum over maps of bilinear(T_m)(v): the same per-texel projections T as
    ``_VertAlignLinear``, then one bilinear sample of T_m per map, accumulated (csrc/vert_align_bilinear.cu).  The backward
    kernel gives gT and the position gradient; the weight and map gradients come from gT as in ``_VertAlignLinear``."""

    @staticmethod
    def forward(ctx, pos, vert_mesh, mesh_info, weight, *fmaps):
        _require_cuda(pos, "VertexAlign+linear")
        dev = pos.device
        pos_c = _f32c(pos.detach())
        w, maps, n_img = _linear_maps(weight, fmaps)
        D = w.shape[0]
        T, rows_cl, rows_per_map = _project_texels(maps, w, n_img)
        SV = pos_c.shape[0]
        out = torch.empty(SV, D, dtype=torch.float32, device=dev)
        r0 = 0
        for i, (m, R) in enumerate(zip(maps, rows_per_map)):
            _lib.call("mrb_vert_align_bilinear_fwd", T.data_ptr() + 4 * r0 * D, D, D, int(m.shape[2]), n_img, _lib.ptr(pos_c),
                      _lib.ptr(vert_mesh), _lib.ptr(mesh_info), SV, int(i > 0), _lib.ptr(out), D)
            r0 += R
        ctx.save_for_backward(pos_c, vert_mesh, mesh_info, w, T, *rows_cl)
        ctx.meta = (n_img, [tuple(m.shape) for m in maps], [f.dtype for f in fmaps], rows_per_map, pos.dtype)
        return out

    @staticmethod
    def backward(ctx, gout):
        pos_c, vert_mesh, mesh_info, w, T = ctx.saved_tensors[:5]
        rows_cl = ctx.saved_tensors[5:]
        n_img, shapes, dtypes, rows_per_map, pos_dtype = ctx.meta
        dev = gout.device
        D = w.shape[0]
        gout = _rows(gout)
        SV = gout.shape[0]
        want_T = ctx.needs_input_grad[3] or any(ctx.needs_input_grad[4:])
        gT = torch.zeros(sum(rows_per_map), D, dtype=torch.float32, device=dev) if want_T else None
        gpos = torch.zeros(SV, 3, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        if gT is not None or gpos is not None:
            r0 = 0
            for shape, R in zip(shapes, rows_per_map):
                _lib.call("mrb_vert_align_bilinear_bwd", gout.data_ptr(), gout.stride(0), T.data_ptr() + 4 * r0 * D, D, D,
                          shape[2], n_img, _lib.ptr(pos_c), _lib.ptr(vert_mesh), _lib.ptr(mesh_info), SV,
                          None if gT is None else gT.data_ptr() + 4 * r0 * D, D, _lib.ptr(gpos), 1)
                r0 += R
        gw, gmaps = None, [None] * len(shapes)
        if gT is not None:
            gw, gmaps = _backproject_texels(gT, w, rows_cl, shapes, rows_per_map, dtypes, n_img, ctx.needs_input_grad[3],
                                            ctx.needs_input_grad[4:])
        if gpos is not None and pos_dtype != torch.float32:
            gpos = gpos.to(pos_dtype)
        return (gpos, None, None, gw) + tuple(gmaps)


def vert_align_linear(img_features: Sequence[Tensor], vertex_positions: Tensor, vertices_per_mesh: Sequence[int],
                      image_sizes, mesh_index: Sequence[int], weight: Tensor, topo: Optional[MeshTopology] = None,
                      bilinear: bool = False) -> Tensor:
    """``F.linear(VertexAlign()(img_features, ...), weight)`` (weight: out x sum(C_m), no bias) without forming the
    SV x sum(C_m) matrix -- see ``_VertAlignLinear``.  ``bilinear=True``: the same with bilinear VertexAlign
    (``vert_align_bilinear``), differentiable in ``vertex_positions`` too (``_VertAlignLinearBilinear``)."""
    if bilinear:
        vert_mesh, info = _bilinear_tables(img_features, vertex_positions, vertices_per_mesh, mesh_index, image_sizes)
        return _VertAlignLinearBilinear.apply(vertex_positions, vert_mesh, info, weight, *img_features)
    dev = vertex_positions.device
    _require_cuda(vertex_positions, "VertexAlign")
    if sum(int(m) for m in mesh_index) != len(vertices_per_mesh):
        raise RuntimeError("VertexAlign: sum(mesh_index) must equal the number of meshes")
    if sum(vertices_per_mesh) != vertex_positions.shape[0]:
        raise RuntimeError("VertexAlign: vertices_per_mesh does not sum to the number of vertex positions")
    vert_mesh = vertex_mesh_ids(vertices_per_mesh, vertex_positions.shape[0], dev, topo)
    info = mesh_info_table(mesh_index, image_sizes, dev)
    return _VertAlignLinear.apply(vertex_positions, vert_mesh, info, weight, *img_features)


# ----------------------------------------------------------------------------------------------------------
# losses
# ----------------------------------------------------------------------------------------------------------
class _EdgeLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, adj):
        _require_cuda(pos, "edge loss")
        pos_c = _f32c(pos)
        adj_c = adj.contiguous()
        if adj_c.dtype != torch.int64:
            adj_c = adj_c.long()
        E = adj_c.shape[1]
        acc = torch.empty(1, dtype=torch.float64, device=pos.device)
        out = torch.empty(1, dtype=torch.float32, device=pos.device)
        _lib.call("mrb_edge_loss_fwd", _lib.ptr(pos_c), _lib.ptr(adj_c), E, _lib.ptr(acc), _lib.ptr(out))
        ctx.save_for_backward(pos_c, adj_c)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        pos_c, adj_c = ctx.saved_tensors
        gpos = torch.zeros_like(pos_c)
        g = _f32c(g).reshape(1)
        _lib.call("mrb_edge_loss_bwd", _lib.ptr(pos_c), _lib.ptr(adj_c), adj_c.shape[1], _lib.ptr(g), _lib.ptr(gpos))
        return gpos, None


def edge_length(pos: Tensor, adj: Tensor) -> Tensor:
    """mean over the directed edge list of |v_r - v_c|^2 (reference loss_functions.py:47-48,175-189), O(E)."""
    return _EdgeLoss.apply(pos, adj)


def face_areas(verts: Tensor, faces: Tensor, v_index: Sequence[int], f_index: Sequence[int]) -> Tensor:
    _require_cuda(verts, "surface_areas")
    dev = verts.device
    v = _f32c(verts.detach())
    f = faces.contiguous().long()
    areas = torch.empty(f.shape[0], dtype=torch.float32, device=dev)
    if f.shape[0]:
        _lib.call("mrb_face_areas", _lib.ptr(v), _lib.ptr(f), _lib.ptr(offsets_table(v_index, dev)),
                  _lib.ptr(offsets_table(f_index, dev)), len(f_index), max(f_index), _lib.ptr(areas))
    return areas


class _Sample(torch.autograd.Function):
    """Packed-batch surface sampling + unit-ball normalisation (mesh_sampling.py:6-35, process.py:7-20)."""

    @staticmethod
    def forward(ctx, verts, faces, v_off, f_off, B, max_faces, n, u, face_idx, xi2, xi1, seed, cdf):
        _require_cuda(verts, "sample")
        dev = verts.device
        v = _f32c(verts)
        f = faces.contiguous().long()
        if face_idx is None and cdf is None:
            cdf = _face_cdf(v, f, v_off, f_off, B, max_faces)
        raw = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
        cloud = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
        fidx = torch.empty(B, n, dtype=torch.int32, device=dev)
        w = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
        stats = torch.empty(B, 8, dtype=torch.float64, device=dev)
        cv = lambda t, dt: None if t is None else t.to(device=dev, dtype=dt).contiguous()
        u, xi2, xi1 = cv(u, torch.float32), cv(xi2, torch.float32), cv(xi1, torch.float32)
        face_idx = cv(face_idx, torch.int64)
        _lib.call("mrb_sample_points_fwd", _lib.ptr(v), _lib.ptr(f), _lib.ptr(v_off), _lib.ptr(f_off), _lib.ptr(cdf), B, n,
                  _lib.ptr(u), _lib.ptr(face_idx), _lib.ptr(xi2), _lib.ptr(xi1), int(seed), _lib.ptr(raw), _lib.ptr(fidx),
                  _lib.ptr(w), _lib.ptr(cloud), _lib.ptr(stats))
        ctx.save_for_backward(cloud, stats, fidx, w, f, v_off)
        ctx.dims = (B, n, tuple(v.shape))
        ctx.set_materialize_grads(False)        # autograd would otherwise zero-fill an int "gradient" for fidx every backward
        ctx.mark_non_differentiable(fidx)
        return cloud, fidx

    @staticmethod
    def backward(ctx, gcloud, _gfidx):
        if gcloud is None:
            return (None,) * 13
        cloud, stats, fidx, w, f, v_off = ctx.saved_tensors
        B, n, vshape = ctx.dims
        # rows padded to 4 floats: one 16-byte vector reduction per face corner; the V x 3 view is the gradient
        gverts = torch.zeros(vshape[0], 4, dtype=torch.float32, device=cloud.device)
        scratch = torch.empty(4 * B, dtype=torch.float64, device=cloud.device)
        _lib.call("mrb_sample_points_bwd_ld", _lib.ptr(_f32c(gcloud)), _lib.ptr(cloud), _lib.ptr(stats), _lib.ptr(fidx),
                  _lib.ptr(w), _lib.ptr(f), _lib.ptr(v_off), B, n, _lib.ptr(gverts), 4, _lib.ptr(scratch))
        return (gverts[:, :3],) + (None,) * 12


def _face_cdf(v: Tensor, f: Tensor, v_off: Tensor, f_off: Tensor, B: int, max_faces: int) -> Tensor:
    """Inclusive per-mesh CDF (fp64) of the face areas of a packed batch (``mrb_face_area_cdf``)."""
    areas = torch.empty(f.shape[0], dtype=torch.float32, device=v.device)
    cdf = torch.empty(f.shape[0], dtype=torch.float64, device=v.device)
    _lib.call("mrb_face_area_cdf", _lib.ptr(v), _lib.ptr(f), _lib.ptr(v_off), _lib.ptr(f_off), B, max_faces,
              _lib.ptr(areas), _lib.ptr(cdf))
    return cdf


def cached_face_cdf(owner, verts: Tensor, faces: Tensor, v_index: Sequence[int], f_index: Sequence[int]) -> Tensor:
    """Device-resident ground-truth sampling cache (SURVEY.md 8 f-2): the reference re-samples the static GT meshes inside
    every stage call (loss_functions.py:57-59), recomputing their face areas each time.  The area CDF of ``batch.meshes``
    is computed once per batch object and kept on it (``owner._mrb_face_cdf``), keyed by the identity and version of the
    packed tensors, so in-place edits or a new ``.to()`` copy invalidate it."""
    key = (verts.data_ptr(), verts._version, faces.data_ptr(), faces._version, tuple(verts.shape), tuple(faces.shape),
           tuple(f_index))
    hit = getattr(owner, "_mrb_face_cdf", None)
    if hit is not None and hit[0] == key:
        return hit[1]
    dev = verts.device
    cdf = _face_cdf(_f32c(verts.detach()), faces.contiguous().long(), offsets_table(v_index, dev), offsets_table(f_index, dev),
                    len(f_index), max(f_index))
    try:
        owner._mrb_face_cdf = (key, cdf)
    except AttributeError:          # objects with __slots__ / tuples: no cache
        pass
    return cdf


def _next_seeds(n: int) -> List[int]:
    """``n`` sampling seeds from torch's CPU generator (so that torch.manual_seed() makes sampling reproducible, no device
    sync) in ONE draw -- the same values as ``n`` single draws (tests/test_host_logic.py), at a sixth of the host time.  The
    rank is mixed in, so ranks that were seeded identically still draw different surface samples for their shards."""
    seeds = torch.randint(0, 2 ** 62, (n,), dtype=torch.int64).tolist()
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        mix = (torch.distributed.get_rank() * 0x9E3779B97F4A7C15) & (2 ** 62 - 1)
        seeds = [s ^ mix for s in seeds]
    return seeds


def _next_seed() -> int:
    return _next_seeds(1)[0]


def sample_points(verts: Tensor, faces: Tensor, v_index: Sequence[int], f_index: Sequence[int], n: int,
                  u: Optional[Tensor] = None, face_idx: Optional[Tensor] = None, xi2: Optional[Tensor] = None,
                  xi1: Optional[Tensor] = None, seed: Optional[int] = None, cdf_owner=None) -> Tuple[Tensor, Tensor]:
    """B x n x 3 normalised clouds (and the global face id of every point).  Randomness: Philox in-kernel from
    ``seed`` (default: drawn from torch's generator), or injected ``u``/``face_idx`` + ``xi2`` + ``xi1`` (B x n).
    ``cdf_owner``: object on which the area CDF of a *static* mesh set (ground truth, no gradient) is cached."""
    dev = verts.device
    _require_cuda(verts, "sample")
    B = len(f_index)
    if len(v_index) != B:
        raise RuntimeError("sample: v_index and f_index must have the same length")
    if B and min(f_index) <= 0:
        raise RuntimeError("sample: every mesh needs at least one face")
    if sum(v_index) != verts.shape[0] or sum(f_index) != faces.shape[0]:
        raise RuntimeError("sample: index lists do not match the packed tensors")
    if seed is None:
        seed = _next_seed() if xi2 is None else 0
    cdf = None
    if cdf_owner is not None and face_idx is None and B and not verts.requires_grad:
        cdf = cached_face_cdf(cdf_owner, verts, faces, v_index, f_index)
    return _Sample.apply(verts, faces, offsets_table(v_index, dev), offsets_table(f_index, dev), B,
                         max(f_index) if B else 0, int(n), u, face_idx, xi2, xi1, seed, cdf)


@torch.no_grad()
def sample_surface(verts: Tensor, faces: Tensor, v_index: Sequence[int], f_index: Sequence[int], n: int,
                   u: Optional[Tensor] = None, face_idx: Optional[Tensor] = None, xi2: Optional[Tensor] = None,
                   xi1: Optional[Tensor] = None, seed: Optional[int] = None, cdf_owner=None,
                   scale: Optional[Tensor] = None, v_starts: Optional[Sequence[int]] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """Eval-side surface sample (no autograd): ``(points B x n x 3, unit face normals B x n x 3, global face ids B x n)``.
    The points are those of ``sample_points`` for the same randomness arguments before its unit-ball normalisation,
    multiplied by ``scale[b]`` (optional per-mesh fp32 CUDA tensor, e.g. from ``mesh_gt_scale``).  ``v_starts``: first
    vertex row of every mesh when the listed meshes are not the whole packed buffer (meshes without faces filtered out of
    the lists); by default the running sum of ``v_index``."""
    dev = verts.device
    _require_cuda(verts, "sample_surface")
    B = len(f_index)
    if len(v_index) != B:
        raise RuntimeError("sample_surface: v_index and f_index must have the same length")
    if B and min(f_index) <= 0:
        raise RuntimeError("sample_surface: every mesh needs at least one face")
    if v_starts is None and (sum(v_index) != verts.shape[0] or sum(f_index) != faces.shape[0]):
        raise RuntimeError("sample_surface: index lists do not match the packed tensors")
    if seed is None:
        seed = _next_seed() if xi2 is None else 0
    n = int(n)
    v = _f32c(verts.detach())
    f = faces.contiguous().long()
    f_off = offsets_table(f_index, dev)
    v_off = offsets_table(v_index, dev) if v_starts is None else _device_table("off", list(v_starts) + [v.shape[0]], dev)
    cdf = None
    if face_idx is None and B:
        cdf = (cached_face_cdf(cdf_owner, verts, faces, v_index, f_index) if cdf_owner is not None and v_starts is None
               else _face_cdf(v, f, v_off, f_off, B, max(f_index)))
    points = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
    normals = torch.empty(B, n, 3, dtype=torch.float32, device=dev)
    fidx = torch.empty(B, n, dtype=torch.int32, device=dev)
    cv = lambda t, dt: None if t is None else t.to(device=dev, dtype=dt).contiguous()
    u, xi2, xi1, sc = cv(u, torch.float32), cv(xi2, torch.float32), cv(xi1, torch.float32), cv(scale, torch.float32)
    face_idx = cv(face_idx, torch.int64)
    _lib.call("mrb_sample_surface_fwd", _lib.ptr(v), _lib.ptr(f), _lib.ptr(v_off), _lib.ptr(f_off), _lib.ptr(cdf), B, n,
              _lib.ptr(u), _lib.ptr(face_idx), _lib.ptr(xi2), _lib.ptr(xi1), int(seed), _lib.ptr(sc), _lib.ptr(points),
              _lib.ptr(normals), _lib.ptr(fidx))
    return points, normals, fidx


@torch.no_grad()
def mesh_gt_scale(verts: Tensor, v_index: Sequence[int], target: float = 10.0) -> Tensor:
    """fp32 [B]: ``target / longest side of the bounding box`` of every mesh of a packed vertex buffer (the paper's GT-10
    normalisation with ``target = 10``).  A mesh of zero extent gets inf."""
    _require_cuda(verts, "mesh_gt_scale")
    dev = verts.device
    v = _f32c(verts.detach())
    if sum(v_index) != v.shape[0]:
        raise RuntimeError("mesh_gt_scale: v_index does not match the packed vertices")
    scale = torch.empty(len(v_index), dtype=torch.float32, device=dev)
    _lib.call("mrb_mesh_gt_scale", _lib.ptr(v), _lib.ptr(offsets_table(v_index, dev)), len(v_index), float(target),
              _lib.ptr(scale))
    return scale


MAX_THRESHOLDS = 8


@torch.no_grad()
def mesh_metrics(d_p: Tensor, i_p: Tensor, d_q: Tensor, i_q: Tensor, n_p: Tensor, n_q: Tensor,
                 thresholds: Sequence[float]) -> Tensor:
    """fp32 [B, 3 + 3T] per-mesh metrics from the k = 0 outputs of ``knn_search`` and the sample normals: Chamfer-L2,
    NormalConsistency, AbsNormalConsistency, then (Precision, Recall, F1) in percent for every threshold (T <= 8)."""
    _require_cuda(d_p, "mesh_metrics")
    thr = [float(t) for t in thresholds]
    if len(thr) > MAX_THRESHOLDS:
        raise ValueError("mesh_metrics: at most %d thresholds, got %d" % (MAX_THRESHOLDS, len(thr)))
    B, P = d_p.shape
    Q = d_q.shape[1]
    out = torch.empty(B, 3 + 3 * len(thr), dtype=torch.float32, device=d_p.device)
    taus = (ctypes.c_float * max(1, len(thr)))(*thr)
    _lib.call("mrb_mesh_metrics", _lib.ptr(d_p), _lib.ptr(i_p), _lib.ptr(d_q), _lib.ptr(i_q), _lib.ptr(_f32c(n_p)),
              _lib.ptr(_f32c(n_q)), B, P, Q, ctypes.addressof(taus), len(thr), _lib.ptr(out))
    return out


KNN_ALGOS = {"auto": 0, "tiled": 1, "grid": 2}


def knn_search(p: Tensor, q: Tensor, k: int = 0, algo: str = "auto"):
    """Exact nearest / k-nearest neighbours in both directions between B x P x 3 and B x Q x 3 clouds (no gradient):
    (d_p, i_p, knn_p, d_q, i_q, knn_q) -- squared distance and int32 index of the nearest point of the other cloud and
    the k nearest indices sorted by (distance, index) (None when k = 0).  ``algo``: "auto" | "tiled" | "grid"
    (mrb_knn_fwd_algo; both strategies return identical results)."""
    _require_cuda(p, "knn_search")
    _require_cuda(q, "knn_search")
    pc, qc = _f32c(p.detach()), _f32c(q.detach())
    B, P, _ = pc.shape
    Q = qc.shape[1]
    dev = p.device
    dp = torch.empty(B, P, dtype=torch.float32, device=dev)
    dq = torch.empty(B, Q, dtype=torch.float32, device=dev)
    ip = torch.empty(B, P, dtype=torch.int32, device=dev)
    iq = torch.empty(B, Q, dtype=torch.int32, device=dev)
    kp = torch.empty(B, P, k, dtype=torch.int32, device=dev) if k else None
    kq = torch.empty(B, Q, k, dtype=torch.int32, device=dev) if k else None
    ws = torch.empty(_lib.load().mrb_knn_workspace_bytes(B, P, Q), dtype=torch.uint8, device=dev)
    args = (_lib.ptr(pc), _lib.ptr(qc), B, P, Q, k, _lib.ptr(dp), _lib.ptr(ip), _lib.ptr(kp), _lib.ptr(dq), _lib.ptr(iq),
            _lib.ptr(kq), _lib.ptr(ws))
    if algo == "auto":
        _lib.call("mrb_knn_fwd", *args)
    else:
        _lib.call("mrb_knn_fwd_algo", *args, KNN_ALGOS[algo])
    return dp, ip, kp, dq, iq, kq


class _Chamfer(torch.autograd.Function):
    """Both directions of the nearest-neighbour search (+ optional k-NN index sets) and the two chamfer sums."""

    @staticmethod
    def forward(ctx, p, q, k):
        _require_cuda(p, "chamfer")
        _require_cuda(q, "chamfer")
        pc, qc = _f32c(p), _f32c(q)
        B, P, _ = pc.shape
        Q = qc.shape[1]
        dev = p.device
        dp, ip, kp, dq, iq, kq = knn_search(pc, qc, k)
        acc = torch.empty(2, dtype=torch.float64, device=dev)
        sums = torch.empty(2, dtype=torch.float32, device=dev)
        _lib.call("mrb_sum_scaled", _lib.ptr(dp), B * P, 1.0, _lib.ptr(acc), _lib.ptr(sums))
        _lib.call("mrb_sum_scaled", _lib.ptr(dq), B * Q, 1.0, _lib.ptr(acc) + 8, _lib.ptr(sums) + 4)
        ctx.save_for_backward(pc, qc, ip, iq)
        outs = [sums[0], sums[1], ip, iq]
        ctx.set_materialize_grads(False)        # no zero-filled int "gradients" for the index outputs
        ctx.mark_non_differentiable(ip, iq)
        if k:
            ctx.mark_non_differentiable(kp, kq)
            outs += [kp, kq]
        else:
            outs += [None, None]
        return tuple(outs)

    @staticmethod
    def backward(ctx, g1, g2, *_):
        if g1 is None and g2 is None:
            return None, None, None
        pc, qc, ip, iq = ctx.saved_tensors
        B, P, _ = pc.shape
        Q = qc.shape[1]
        gp = torch.zeros_like(pc) if ctx.needs_input_grad[0] else None
        gq = torch.zeros_like(qc) if ctx.needs_input_grad[1] else None
        z = lambda g: torch.zeros(1, dtype=torch.float32, device=pc.device) if g is None else _f32c(g).reshape(1)
        _lib.call("mrb_chamfer_bwd", _lib.ptr(pc), _lib.ptr(qc), B, P, Q, _lib.ptr(ip), _lib.ptr(iq), _lib.ptr(z(g1)),
                  _lib.ptr(z(g2)), 1.0, _lib.ptr(gp), _lib.ptr(gq))
        return gp, gq, None


def chamfer_knn(p: Tensor, q: Tensor, k: int = 0):
    """(loss_1, loss_2, idx_p, idx_q, knn_p, knn_q): loss_1 = sum_i min_j |p_i-q_j|^2, loss_2 the reverse direction
    (reference loss_functions.py:93-102); idx_* int32 nearest indices; knn_* the k nearest indices (:141)."""
    return _Chamfer.apply(p, q, int(k))


class _ChamferTotal(torch.autograd.Function):
    """scale * (sum_i min_j |p_i - q_j|^2 + sum_j min_i |p_i - q_j|^2) as ONE scalar (what mesh_loss needs,
    loss_functions.py:62-66) + the index outputs: the two nearest-neighbour distance arrays live in one buffer, so the sum,
    the add and the division by point_cloud_size are a single reduction launch, and the backward is one kernel."""

    @staticmethod
    def forward(ctx, p, q, k, scale):
        _require_cuda(p, "chamfer")
        _require_cuda(q, "chamfer")
        pc, qc = _f32c(p), _f32c(q)
        B, P, _ = pc.shape
        Q = qc.shape[1]
        dev = p.device
        d = torch.empty(B * (P + Q), dtype=torch.float32, device=dev)
        ip = torch.empty(B, P, dtype=torch.int32, device=dev)
        iq = torch.empty(B, Q, dtype=torch.int32, device=dev)
        kp = torch.empty(B, P, k, dtype=torch.int32, device=dev) if k else None
        kq = torch.empty(B, Q, k, dtype=torch.int32, device=dev) if k else None
        ws = torch.empty(_lib.load().mrb_knn_workspace_bytes(B, P, Q), dtype=torch.uint8, device=dev)
        _lib.call("mrb_knn_fwd", _lib.ptr(pc.detach()), _lib.ptr(qc.detach()), B, P, Q, k, d.data_ptr(), _lib.ptr(ip), _lib.ptr(kp),
                  d.data_ptr() + 4 * B * P, _lib.ptr(iq), _lib.ptr(kq), _lib.ptr(ws))
        acc = torch.empty(1, dtype=torch.float64, device=dev)
        out = torch.empty(1, dtype=torch.float32, device=dev)
        _lib.call("mrb_sum_scaled", _lib.ptr(d), B * (P + Q), float(scale), _lib.ptr(acc), _lib.ptr(out))
        ctx.save_for_backward(pc, qc, ip, iq)
        ctx.scale = float(scale)
        ctx.set_materialize_grads(False)        # no zero-filled int "gradients" for the four index outputs (4 fill launches)
        ctx.mark_non_differentiable(ip, iq)
        if k:
            ctx.mark_non_differentiable(kp, kq)
        return out[0], ip, iq, kp, kq

    @staticmethod
    def backward(ctx, g, *_):
        if g is None:
            return None, None, None, None
        pc, qc, ip, iq = ctx.saved_tensors
        B, P, _ = pc.shape
        Q = qc.shape[1]
        gp = torch.zeros_like(pc) if ctx.needs_input_grad[0] else None
        gq = torch.zeros_like(qc) if ctx.needs_input_grad[1] else None
        gs = _lib.ptr(_f32c(g).reshape(1))
        _lib.call("mrb_chamfer_bwd", _lib.ptr(pc), _lib.ptr(qc), B, P, Q, _lib.ptr(ip), _lib.ptr(iq), gs, gs, ctx.scale,
                  _lib.ptr(gp), _lib.ptr(gq))
        return gp, gq, None, None


def chamfer_total(p: Tensor, q: Tensor, k: int, scale: float):
    """(scale * (loss_1 + loss_2), idx_p, idx_q, knn_p, knn_q) -- see ``_ChamferTotal``."""
    return _ChamferTotal.apply(p, q, int(k), float(scale))


class _ScalarCombine(torch.autograd.Function):
    """sum_i w_i * x_i over 0-dim CUDA tensors in one launch (backward: one launch for all the g * w_i)."""

    @staticmethod
    def forward(ctx, weights, *xs):
        n = len(xs)
        xc = [_f32c(x.detach()).reshape(1) for x in xs]
        _require_cuda(xc[0], "weighted scalar sum")
        out = torch.empty(1, dtype=torch.float32, device=xc[0].device)
        ptrs = (ctypes.c_void_p * n)(*[x.data_ptr() for x in xc])
        w = (ctypes.c_float * n)(*[float(v) for v in weights])
        _lib.call("mrb_scalar_combine", ctypes.addressof(ptrs), ctypes.addressof(w), n, _lib.ptr(out))
        ctx.weights = tuple(float(v) for v in weights)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        n = len(ctx.weights)
        if all(v == 1.0 for v in ctx.weights):
            return (None,) + (g,) * n                       # a plain sum: every term receives g itself, no kernel
        out = torch.empty(n, dtype=torch.float32, device=g.device)
        w = (ctypes.c_float * n)(*ctx.weights)
        _lib.call("mrb_scalar_scatter", _lib.ptr(_f32c(g).reshape(1)), ctypes.addressof(w), n, _lib.ptr(out))
        return (None,) + tuple(out[i] for i in range(n))


def weighted_scalar_sum(xs: Sequence[Tensor], weights: Optional[Sequence[float]] = None) -> Tensor:
    """``sum(w * x for w, x in zip(weights, xs))`` for 0-dim CUDA tensors (loss terms) as one kernel; weights default to 1."""
    xs = list(xs)
    if len(xs) == 1 and (weights is None or float(weights[0]) == 1.0):
        return xs[0]
    if len(xs) > 16 or not all(isinstance(x, Tensor) and x.is_cuda for x in xs):
        total = None
        for i, x in enumerate(xs):
            t = x if weights is None else x * float(weights[i])
            total = t if total is None else total + t
        return total
    return _ScalarCombine.apply(tuple([1.0] * len(xs) if weights is None else weights), *xs)


def _normals_fwd(pts: Tensor, knn: Tensor, k: int, keep_eig: bool):
    """(normals B x P x 3, eig | None).  ``keep_eig``: also keep the fp64 eigen-decomposition (12 planes of B * P doubles) for
    the backward pass, which then skips the Jacobi sweeps."""
    B, P, _ = pts.shape
    n = torch.empty(B, P, 3, dtype=torch.float32, device=pts.device)
    eig = torch.empty(12, B * P, dtype=torch.float64, device=pts.device) if keep_eig else None
    _lib.call("mrb_normals_fwd_eig", _lib.ptr(pts), _lib.ptr(knn), B, P, k, _lib.ptr(n), _lib.ptr(eig))
    return n, eig


def _normals_bwd(pts: Tensor, knn: Tensor, k: int, gn: Tensor, eig: Optional[Tensor]) -> Tensor:
    """Gradient of the estimated normals w.r.t. the points.  The kernel scatters into rows padded to 4 floats (one 16-byte
    vector reduction per neighbour instead of three scalar atomics); the B x P x 3 view of that buffer is returned."""
    B, P, _ = pts.shape
    g4 = torch.zeros(B, P, 4, dtype=torch.float32, device=pts.device)
    _lib.call("mrb_normals_bwd_ld", _lib.ptr(pts), _lib.ptr(knn), B, P, k, _lib.ptr(gn), _lib.ptr(g4), 4, _lib.ptr(eig))
    return g4[..., :3]


class _NormalLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, q, knn_p, knn_q, idx_p, idx_q):
        _require_cuda(p, "normal loss")
        pc, qc = _f32c(p), _f32c(q)
        B, P, _ = pc.shape
        Q = qc.shape[1]
        if P != Q:
            # the reference gathers rows of a cloud with the *other* cloud's k-NN indices (loss_functions.py:141,146)
            raise RuntimeError("normal loss requires equally sized clouds (reference semantics)")
        k = knn_p.shape[2]
        dev = p.device
        i32 = lambda t: t.to(torch.int32).contiguous()
        knn_p, knn_q, idx_p, idx_q = i32(knn_p), i32(knn_q), i32(idx_p), i32(idx_q)
        n_p, eig_p = _normals_fwd(pc, knn_p, k, ctx.needs_input_grad[0])
        n_q, eig_q = _normals_fwd(qc, knn_q, k, ctx.needs_input_grad[1])
        ctx.eig = (eig_p, eig_q)         # plain attributes: not inputs / outputs of the node
        acc = torch.empty(2, dtype=torch.float64, device=dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        _lib.call("mrb_normal_loss_fwd", _lib.ptr(n_p), _lib.ptr(n_q), B, P, Q, _lib.ptr(idx_p), _lib.ptr(idx_q),
                  _lib.ptr(acc), _lib.ptr(out))
        ctx.save_for_backward(pc, qc, knn_p, knn_q, idx_p, idx_q, n_p, n_q)
        return out[0], out[1]

    @staticmethod
    def backward(ctx, g0, g1):
        pc, qc, knn_p, knn_q, idx_p, idx_q, n_p, n_q = ctx.saved_tensors
        B, P, _ = pc.shape
        Q = qc.shape[1]
        k = knn_p.shape[2]
        dev = pc.device
        z = lambda g: torch.zeros(1, dtype=torch.float32, device=dev) if g is None else _f32c(g).reshape(1)
        need_p, need_q = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gnp = torch.zeros_like(n_p) if need_p else None
        gnq = torch.zeros_like(n_q) if need_q else None
        _lib.call("mrb_normal_loss_bwd", _lib.ptr(n_p), _lib.ptr(n_q), B, P, Q, _lib.ptr(idx_p), _lib.ptr(idx_q),
                  _lib.ptr(z(g0)), _lib.ptr(z(g1)), _lib.ptr(gnp), _lib.ptr(gnq))
        gp = gq = None
        if need_p:
            gp = _normals_bwd(pc, knn_p, k, gnp, ctx.eig[0])
        if need_q:
            gq = _normals_bwd(qc, knn_q, k, gnq, ctx.eig[1])
        return gp, gq, None, None, None, None


class _NormalLossTotal(torch.autograd.Function):
    """scale * (sum_i |n_p[i] . n_q[idx_p[i]]| + sum_j |n_q[j] . n_p[idx_q[j]]|) as one scalar (loss_functions.py:69-72 with
    the negation and the division folded into ``scale``)."""

    @staticmethod
    def forward(ctx, p, q, knn_p, knn_q, idx_p, idx_q, scale):
        _require_cuda(p, "normal loss")
        pc, qc = _f32c(p), _f32c(q)
        B, P, _ = pc.shape
        Q = qc.shape[1]
        if P != Q:
            raise RuntimeError("normal loss requires equally sized clouds (reference semantics)")
        k = knn_p.shape[2]
        dev = p.device
        i32 = lambda t: t if (t.dtype == torch.int32 and t.is_contiguous()) else t.to(torch.int32).contiguous()
        knn_p, knn_q, idx_p, idx_q = i32(knn_p), i32(knn_q), i32(idx_p), i32(idx_q)
        n_p, eig_p = _normals_fwd(pc, knn_p, k, ctx.needs_input_grad[0])
        n_q, eig_q = _normals_fwd(qc, knn_q, k, ctx.needs_input_grad[1])
        ctx.eig = (eig_p, eig_q)         # plain attributes: not inputs / outputs of the node
        acc = torch.empty(2, dtype=torch.float64, device=dev)
        out = torch.empty(1, dtype=torch.float32, device=dev)
        _lib.call("mrb_normal_loss_total_fwd", _lib.ptr(n_p), _lib.ptr(n_q), B, P, Q, _lib.ptr(idx_p), _lib.ptr(idx_q), float(scale),
                  _lib.ptr(acc), _lib.ptr(out))
        ctx.save_for_backward(pc, qc, knn_p, knn_q, idx_p, idx_q, n_p, n_q)
        ctx.scale = float(scale)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        pc, qc, knn_p, knn_q, idx_p, idx_q, n_p, n_q = ctx.saved_tensors
        B, P, _ = pc.shape
        Q = qc.shape[1]
        k = knn_p.shape[2]
        need_p, need_q = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gnp = torch.zeros_like(n_p) if need_p else None
        gnq = torch.zeros_like(n_q) if need_q else None
        _lib.call("mrb_normal_loss_total_bwd", _lib.ptr(n_p), _lib.ptr(n_q), B, P, Q, _lib.ptr(idx_p), _lib.ptr(idx_q),
                  _lib.ptr(_f32c(g).reshape(1)), ctx.scale, _lib.ptr(gnp), _lib.ptr(gnq))
        gp = gq = None
        if need_p:
            gp = _normals_bwd(pc, knn_p, k, gnp, ctx.eig[0])
        if need_q:
            gq = _normals_bwd(qc, knn_q, k, gnq, ctx.eig[1])
        return gp, gq, None, None, None, None, None


def normal_total(p: Tensor, q: Tensor, knn_p: Tensor, knn_q: Tensor, idx_p: Tensor, idx_q: Tensor, scale: float) -> Tensor:
    return _NormalLossTotal.apply(p, q, knn_p, knn_q, idx_p, idx_q, float(scale))


def normal_distance(p: Tensor, q: Tensor, knn_p: Tensor, knn_q: Tensor, idx_p: Tensor, idx_q: Tensor):
    return _NormalLoss.apply(p, q, knn_p, knn_q, idx_p, idx_q)


@torch.no_grad()
def compute_normals(pt: Tensor, knn: Tensor) -> Tensor:
    _require_cuda(pt, "compute_normals")
    pc = _f32c(pt)
    B, P, _ = pc.shape
    knn = knn.to(torch.int32).contiguous()
    out = torch.empty(B, P, 3, dtype=torch.float32, device=pt.device)
    _lib.call("mrb_normals_fwd", _lib.ptr(pc), _lib.ptr(knn), B, P, knn.shape[2], _lib.ptr(out))
    return out


# ----------------------------------------------------------------------------------------------------------
# tensor-core projections (tcgen05): weight image packing + GEMM
# ----------------------------------------------------------------------------------------------------------
def tc_pack(src0: Tensor, src1: Optional[Tensor], stride_k: int, stride_n: int, split_axis: int, split_at: int,
            K: int, N: int) -> Tensor:
    """Packs the logical K x N weight operand B(k, n) = src[k*stride_k + n*stride_n] (two sources when split) into the
    tf32 hi/lo, K-major, 128B-swizzled image the tcgen05 kernel streams with TMA bulk copies."""
    nbytes = _lib.load().mrb_gemm_tc_image_bytes(K, N)
    image = torch.empty(nbytes, dtype=torch.uint8, device=src0.device)
    _lib.call("mrb_gemm_tc_pack", _lib.ptr(src0), _lib.ptr(src1), stride_k, stride_n, split_axis, split_at, K, N,
              _lib.ptr(image))
    return image


def tc_gemm(a_ptr: int, lda: int, M: int, K: int, image: Tensor, N: int, c_ptr: int, ldc: int) -> None:
    _lib.call("mrb_gemm_tc", a_ptr, lda, M, K, _lib.ptr(image), N, c_ptr, ldc)
