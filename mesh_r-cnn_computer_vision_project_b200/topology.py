"""Packed-mesh topology side-car.

The reference API passes adjacency around as a bare ``2 x E`` int64 COO tensor (``adj_index`` returned by
``Cubify.forward``, reference meshRCNN/layers.py:478,484, consumed by ``GraphConv.forward`` :47 and
``total_edge_length`` loss_functions.py:175).  The kernels want CSR with int32 columns.  ``Cubify`` already
produces that form on the device, so it registers it here keyed by the identity of the COO tensor it
returns; any other COO tensor is converted on the device the first time it is seen (no host sync).
"""
import weakref
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import _lib


class MeshTopology:
    """CSR adjacency (row-sorted, int32) of a packed batch of meshes, plus the CSR of its transpose (the
    backward of the neighbour sum gathers along columns; for symmetric adjacency both are the same arrays).
    Cubify also records the per-vertex mesh ids ``vert_mesh`` and the per-mesh vertex counts ``v_index`` they belong to."""

    __slots__ = ("num_vertices", "num_edges", "rowptr", "col", "rowptr_t", "col_t", "symmetric", "vert_mesh",
                 "v_index", "v_offsets", "row32", "bad_index_flags", "__weakref__")

    def __init__(self, num_vertices, num_edges, rowptr, col, rowptr_t=None, col_t=None, symmetric=False,
                 vert_mesh=None, v_offsets=None, row32=None, v_index=None):
        self.num_vertices = int(num_vertices)
        self.num_edges = int(num_edges)
        self.rowptr = rowptr
        self.col = col
        self.symmetric = bool(symmetric)
        self.rowptr_t = rowptr if symmetric else rowptr_t
        self.col_t = col if symmetric else col_t
        self.vert_mesh = vert_mesh
        self.v_index = None if v_index is None else list(v_index)
        self.v_offsets = v_offsets
        self.row32 = row32
        self.bad_index_flags = None      # device flags of mrb_coo_to_csr (foreign COO tensors only)


# Edge lists that do not come from Cubify (rebuilt eval adjacency, user tensors) are checked for out-of-range vertex ids
# when their CSR is built: mrb_coo_to_csr flags them on the device and this costs one host read per NEW tensor (the CSR is
# cached afterwards).  The reference raises IndexError for such input; set False to skip the read (flags stay available as
# ``MeshTopology.bad_index_flags``).
VALIDATE_FOREIGN_COO = True

_REGISTRY: Dict[Tuple[int, int, int], Tuple[weakref.ref, int, MeshTopology]] = {}


def _key(adj: Tensor, n: int) -> Tuple[int, int, int]:
    return (adj.data_ptr(), adj.shape[1], n)


def register(adj: Tensor, topo: MeshTopology) -> None:
    if adj.shape[1] == 0:                    # every empty tensor has data_ptr 0: never cached
        return
    if len(_REGISTRY) > 64:
        for k in [k for k, (r, _, _) in _REGISTRY.items() if r() is None]:
            del _REGISTRY[k]
    _REGISTRY[_key(adj, topo.num_vertices)] = (weakref.ref(adj), adj._version, topo)


def lookup(adj: Tensor, num_vertices: int) -> Optional[MeshTopology]:
    """The CSR registered for this COO tensor, if the tensor is still the one that was registered: same storage (the
    registered object is alive, so its address cannot have been recycled) and the version counter it had at registration
    time -- an in-place edit of the edge list (pruning / re-indexing in the eval path) invalidates the entry."""
    hit = _REGISTRY.get(_key(adj, num_vertices))
    if hit is None:
        return None
    ref, version, topo = hit
    t = ref()
    if t is None or t.data_ptr() != adj.data_ptr() or adj._version != version or t._version != version:
        return None
    return topo


def from_coo(adj: Tensor, num_vertices: int) -> MeshTopology:
    """CSR (+ transpose CSR) of an arbitrary ``2 x E`` int64 COO edge list, built on the device."""
    topo = lookup(adj, num_vertices)
    if topo is not None:
        return topo
    if not adj.is_cuda:
        raise RuntimeError("meshrcnn_b200: adjacency must be a CUDA tensor (no CPU fallback)")
    if adj.dim() != 2 or adj.shape[0] != 2:
        raise RuntimeError("meshrcnn_b200: adjacency must be 2 x E (COO)")
    adj_c = adj.contiguous().to(torch.int64)
    E = adj_c.shape[1]
    n = int(num_vertices)
    dev = adj.device
    out, flags = [], []
    for transpose in (0, 1):
        rowptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
        col = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        ws = torch.empty(2 * (n + 1) + 2, dtype=torch.int32, device=dev)
        _lib.call("mrb_coo_to_csr", _lib.ptr(adj_c), E, n, transpose, _lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(ws))
        out += [rowptr, col]
        flags.append(ws[n + 1:n + 3])        # [not row-sorted, index out of range] (device side, no sync here)
    topo = MeshTopology(n, E, out[0], out[1], out[2], out[3], symmetric=False)
    topo.bad_index_flags = torch.stack(flags)[:, 1]
    if VALIDATE_FOREIGN_COO and bool(topo.bad_index_flags.any()):      # one host sync, only for foreign edge lists
        raise IndexError("meshrcnn_b200: adjacency holds vertex ids outside [0, %d) (the reference raises IndexError "
                         "here as well)" % n)
    register(adj, topo)
    return topo
