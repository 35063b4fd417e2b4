"""ctypes binding of libmnf_b200.so (the C ABI declared in include/mnf_b200.h).

The product has no CPU fallback: if the shared library is missing this module raises at
first use with the build command, and every wrapper raises ``RuntimeError`` carrying
``mnf_last_error()`` when an entry point returns non-zero.
"""

from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get(
    "MNF_B200_LIB", os.path.join(os.path.dirname(_HERE), "lib", "libmnf_b200.so")
)

ABI_VERSION = 1
MAX_OPS, MAX_LIN, MAX_DIM, MAX_HIDDEN, MAX_BINS = 32, 6, 64, 128, 32

OP_AFFINE_CONST, OP_GLOW, OP_AFFINE_HALF, OP_NSF_CL, OP_NSF_AR, OP_MADE = 1, 2, 3, 4, 5, 6
FLAG_PARITY, FLAG_SCALE, FLAG_SHIFT, FLAG_MADE_SEQ = 1, 2, 4, 8
RUN_INVERSE, RUN_GENERIC, RUN_LOGPROB, RUN_STAGED = 1, 2, 4, 8

launch_count = 0  # kernels launched through this binding (bench.py reports it)


class FlowOp(C.Structure):
    """struct mnf_flow_op (include/mnf_b200.h)."""

    _fields_ = [
        ("type", C.c_int32),
        ("flags", C.c_uint32),
        ("K", C.c_int32),
        ("bound", C.c_float),
        ("n_lin", C.c_int32),
        ("sizes", C.c_int32 * (MAX_LIN + 1)),
        ("net_off", C.c_int32 * 2),
        ("aux_off", C.c_int32),
        ("edge_deriv", C.c_float),
    ]


class GatherOut(C.Structure):
    """struct mnf_gather_out."""

    _fields_ = [("n_peers", C.c_int32), ("reserved", C.c_int32), ("row_offset", C.c_int64),
                ("peer_ptrs", C.c_void_p * 8), ("multicast_ptr", C.c_void_p)]


_lib = None

_f32p = C.c_void_p  # device pointers travel as integers
_SIGS = {
    "mnf_abi_version": (C.c_int, []),
    "mnf_last_error": (C.c_char_p, []),
    "mnf_launch_count": (C.c_uint64, []),
    "mnf_device_info": (C.c_int, [C.POINTER(C.c_int)] * 4),
    "mnf_launch_stats": (C.c_int64, [C.c_char_p, C.c_int64]),
    "mnf_launch_stats_reset": (None, []),
    "mnf_flow_stack_run": (
        C.c_int,
        [C.POINTER(FlowOp), C.c_int, _f32p, C.c_int64, _f32p, _f32p, _f32p, _f32p, _f32p,
         C.c_int64, C.c_int, C.c_int, _f32p, C.POINTER(GatherOut), C.c_void_p],
    ),
    "mnf_flow_stack_backward": (
        C.c_int,
        [C.POINTER(FlowOp), C.c_int, _f32p, C.c_int64, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p,
         C.c_int64, C.c_int, C.c_int, C.c_void_p],
    ),
    "mnf_flow_stack_sample": (
        C.c_int,
        [C.POINTER(FlowOp), C.c_int, _f32p, C.c_int64, C.c_uint64, C.c_uint32, C.c_uint64, _f32p, _f32p, _f32p,
         C.c_int64, C.c_int, C.c_int, _f32p, C.c_void_p],
    ),
    "mnf_flow_stack_stage_size": (C.c_int64, [C.POINTER(FlowOp), C.c_int, C.c_int, C.c_int64]),
    "mnf_flow_stack_stage_max_rows": (C.c_int64, [C.POINTER(FlowOp), C.c_int, C.c_int, C.c_int64]),
    "mnf_flow_stack_stage": (C.c_int, [C.POINTER(FlowOp), C.c_int, _f32p, C.c_int64, C.c_int, _f32p, C.c_void_p]),
    "mnf_flow_stack_workspace": (C.c_int64, [C.c_int, C.c_int64, C.c_int]),
    "mnf_flow_stack_plan": (C.c_int, [C.POINTER(FlowOp), C.c_int, C.c_int, C.c_int64]),
    "mnf_flow_handle_create": (C.c_int, [C.POINTER(FlowOp), C.c_int, _f32p, C.c_int64, C.c_int, _f32p, _f32p, C.c_int64,
                                         C.POINTER(C.c_void_p)]),
    "mnf_flow_handle_destroy": (None, [C.c_void_p]),
    "mnf_flow_handle_log_prob": (C.c_int, [C.c_void_p, _f32p, _f32p, C.c_int64, C.c_void_p]),
    "mnf_glow_assemble": (C.c_int, [_f32p, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_void_p]),
    "mnf_actnorm_init": (
        C.c_int,
        [_f32p, C.c_int64, C.c_int, _f32p, _f32p, C.c_int, C.c_int, C.c_void_p, C.c_void_p],
    ),
}


def declared_symbols() -> list[str]:
    return sorted(_SIGS)


def register(sigs: dict) -> None:
    """Other host modules (MNF layers, MADE) add their entry points here."""
    _SIGS.update(sigs)
    if _lib is not None:
        _bind(_lib, sigs)


def _bind(lib, sigs):
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found. torch_mnf (B200) has no CPU/PyTorch fallback: build the "
                "CUDA library first with `python torch-mnf_b200/build.py`."
            )
        handle = C.CDLL(LIB_PATH)
        _bind(handle, _SIGS)
        if handle.mnf_abi_version() != ABI_VERSION:
            raise ImportError(
                f"{LIB_PATH}: ABI version {handle.mnf_abi_version()} != expected {ABI_VERSION}; rebuild"
            )
        _lib = handle
    return _lib


def launch_stats(reset: bool = False) -> dict:
    """{launch site (kernel name): launches since the last reset} from the library's own tally."""
    h = lib()
    buf = C.create_string_buffer(8192)
    h.mnf_launch_stats(buf, 8192)
    out = {}
    for item in buf.value.decode().split(";"):
        if "=" in item:
            k, v = item.rsplit("=", 1)
            out[k] = int(v)
    if reset:
        h.mnf_launch_stats_reset()
    return out


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().mnf_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


class on_device:
    """``with on_device(dev):`` -- torch.cuda.device(dev) only when dev is not already current (the context manager
    costs two cudaSetDevice calls, a tenth of a small-batch call)."""

    __slots__ = ("ctx",)

    def __init__(self, device):
        self.ctx = None if torch.cuda.current_device() == device.index else torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            return self.ctx.__exit__(*exc)
        return False


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)  # no Stream object per call (a tenth of a small-batch call)


def stream_ptr(device) -> int:
    if _raw_stream is not None:
        idx = device.index
        return _raw_stream(idx if idx is not None else torch.cuda.current_device())
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    """No CPU path: inputs must be CUDA fp32; made contiguous if needed."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is on {t.device}; torch_mnf (B200) runs only on CUDA tensors (no CPU fallback)"
        )
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")  # the reference is fp32-only too
    return t.contiguous()


def ptr(t) -> int | None:
    return None if t is None else t.data_ptr()
