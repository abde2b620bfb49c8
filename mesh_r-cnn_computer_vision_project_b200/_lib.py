"""ctypes binding of ``libmeshrcnn_b200.so`` (the C ABI declared in ``include/meshrcnn_b200.h``).

There is deliberately NO CPU fallback: if the CUDA library is missing or a tensor is not a CUDA tensor the call
raises.  PyTorch is used only for device memory, streams and autograd bookkeeping.
"""
import ctypes
import os
import re
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MRB_LIB_PATH") or os.path.join(_HERE, "libmeshrcnn_b200.so")   # override: diagnostic builds

_C = {"p": ctypes.c_void_p, "i": ctypes.c_int, "l": ctypes.c_longlong, "L": ctypes.c_ulonglong, "f": ctypes.c_float,
      "d": ctypes.c_double}

HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "meshrcnn_b200.h")


def parse_header(path: str = HEADER_PATH):
    """name -> (return code, argument codes) for every prototype of include/meshrcnn_b200.h -- the header is the
    single source of truth for the ctypes signatures (codes: p pointer, i int, l long long, L unsigned long long,
    f float, d double, s const char*)."""
    src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
    protos = {}
    for m in re.finditer(r"\n\s*((?:const\s+)?(?:unsigned\s+)?(?:long\s+long|int|char|void|float|double)\s*\*?)\s*"
                         r"(mrb_\w+)\s*\(([^)]*)\)\s*;", src):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        codes = ""
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    codes += "p"
                elif a.startswith("unsigned long long"):
                    codes += "L"
                elif a.startswith("long long"):
                    codes += "l"
                elif a.startswith("int"):
                    codes += "i"
                elif a.startswith("float"):
                    codes += "f"
                elif a.startswith("double"):
                    codes += "d"
                else:
                    raise RuntimeError("meshrcnn_b200: cannot parse argument %r of %s" % (a, name))
        protos[name] = ("s" if "char" in ret else ("l" if "long long" in ret else "i"), codes)
    return protos


SIGNATURES = parse_header()

_lib = None
_lock = threading.Lock()


class LibraryMissing(RuntimeError):
    pass


def load():
    """Loads (once) and returns the ctypes library.  Raises LibraryMissing if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing(
                "meshrcnn_b200: %s not found -- build it with `python -m meshrcnn_b200.build` "
                "(there is no CPU / PyTorch fallback for the hot path)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (ret, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = ctypes.c_char_p if ret == "s" else _C[ret]
            fn.argtypes = [_C[a] for a in args]
        if lib.mrb_version() != 100:
            raise RuntimeError("meshrcnn_b200: library/header version mismatch")
        _bind_fast(lib)
        _lib = lib
    return _lib


# Optional call shim (csrc/host/fastcall.c, built by meshrcnn_b200.build): entry points whose arguments are all pointers /
# int / long long are called through a plain cast instead of libffi (ctypes spends 3-5 us per call on ~15 arguments, a step
# makes ~150 calls).  Same library, same symbols; without the shim everything goes through ctypes.
_FAST = {}            # name -> address of the entry point
_fast_call = None


def _bind_fast(lib):
    global _fast_call
    if os.environ.get("MRB_NO_FASTCALL", "0") == "1":
        return
    try:
        from . import _fastcall
    except ImportError:
        return
    for name, (ret, args) in SIGNATURES.items():
        if ret == "i" and all(a in "pilL" for a in args):
            _FAST[name] = ctypes.cast(getattr(lib, name), ctypes.c_void_p).value
    _fast_call = _fastcall.call_ints


def stream_ptr() -> int:
    """Raw cudaStream_t of torch's current stream on the current device.  (torch.cuda.current_stream() costs ~14 us of
    Python per call -- 130 calls per step -- so the C accessors are used directly.)"""
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def ptr(t):
    """Raw device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("meshrcnn_b200: expected a CUDA tensor (no CPU fallback), got device %s" % t.device)
    if not t.is_contiguous():
        raise RuntimeError("meshrcnn_b200: internal error, non-contiguous tensor passed to the C ABI")
    return t.data_ptr()


def check(code: int, what: str = ""):
    if code != 0:
        msg = load().mrb_last_error()
        raise RuntimeError("meshrcnn_b200 %s failed (code %d): %s" % (what, code, msg.decode() if msg else "?"))


# kernels launched by each entry point (for the `gpu_launches` claim of bench.py; memsets not counted)
LAUNCHES = {
    "mrb_cubify_count": 4, "mrb_cubify_emit": 3, "mrb_coo_to_csr": 5, "mrb_csr_gather_fwd": 1, "mrb_relu_mask": 1, "mrb_graphconv_bwd_gather": 1,
    "mrb_segment_ids": 1, "mrb_sgemm": 1, "mrb_gemm_tc": 1, "mrb_gemm_tc_pack": 1, "mrb_gemm_tc_pack_graphconv": 1, "mrb_gemm_tc_pack_graphconv_batch": 1, "mrb_gemm_tc_wgrad": 1, "mrb_vert_align_fwd": 2, "mrb_vert_align_bwd": 1,
    "mrb_vert_align_fwd_bf16": 2, "mrb_feature_map_to_rows": 1, "mrb_rows_to_feature_map": 1, "mrb_vert_align_proj_fwd": 1,
    "mrb_vert_align_proj_bwd": 1, "mrb_vert_align_bilinear_fwd": 1, "mrb_vert_align_bilinear_bwd": 1, "mrb_gemm_tc_acc": 1, "mrb_gemm_tc_wgrad_split": 1, "mrb_vert_align_texrows": 1,
    "mrb_gc_gather_fwd": 1, "mrb_gc_gather_bwd": 1, "mrb_head_fwd": 1, "mrb_head_bwd": 1, "mrb_voxel_bce_fwd": 2, "mrb_voxel_bce_bwd": 1, "mrb_normal_loss_total_fwd": 2,
    "mrb_normal_loss_total_bwd": 1, "mrb_scalar_combine": 1, "mrb_scalar_scatter": 1, "mrb_face_areas": 1,
    "mrb_face_area_cdf": 2, "mrb_sample_points_fwd": 2, "mrb_normalize_cloud_fwd": 1, "mrb_sample_points_bwd": 2, "mrb_sample_points_bwd_ld": 2,
    "mrb_sample_surface_fwd": 1, "mrb_mesh_gt_scale": 1, "mrb_mesh_metrics": 1,
    "mrb_knn_fwd": 3, "mrb_knn_fwd_algo": 4, "mrb_sum_scaled": 2, "mrb_chamfer_bwd": 1, "mrb_normals_fwd": 1, "mrb_normals_fwd_eig": 1, "mrb_normals_bwd": 1, "mrb_normals_bwd_ld": 1,
    "mrb_normal_loss_fwd": 2, "mrb_normal_loss_bwd": 1, "mrb_edge_loss_fwd": 2, "mrb_edge_loss_bwd": 1,
}

launch_count = 0          # running total of kernel launches issued through `call`
_timing = None            # None, or {name: [(start_event, end_event), ...]} while `timed_calls()` is active


class timed_calls:
    """Context manager: brackets every C-ABI call with CUDA events on the launching stream and reports the summed
    device time per entry point (used by bench.py for the per-kernel roofline; adds ~2 event records per call, so
    it is never active inside a headline timed region)."""

    def __enter__(self):
        global _timing
        _timing = {}
        return self

    def __exit__(self, *exc):
        global _timing
        torch.cuda.synchronize()
        self.ms = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in _timing.items()}
        self.calls = {k: len(v) for k, v in _timing.items()}
        _timing = None
        return False


def call(name: str, *args):
    """Calls an int-returning entry point with the current stream appended, raising on error."""
    global launch_count
    lib = load()
    launch_count += LAUNCHES.get(name, 1)
    if _timing is None:
        addr = _FAST.get(name)
        if addr is not None:
            try:
                rc = _fast_call(addr, args + (stream_ptr(),))
            except TypeError:                  # an argument that is not an int / None (e.g. a ctypes array): let ctypes convert it
                rc = getattr(lib, name)(*args, stream_ptr())
        else:
            rc = getattr(lib, name)(*args, stream_ptr())
        if rc != 0:
            check(rc, name)
        return
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    check(getattr(lib, name)(*args, stream_ptr()), name)
    b.record()
    _timing.setdefault(name, []).append((a, b))
