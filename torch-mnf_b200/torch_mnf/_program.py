"""Host-side flow-program builder: turns a list of flow modules into the descriptor array +
packed parameter blob that ``mnf_flow_stack_run`` consumes (include/mnf_b200.h), caches it
until a parameter changes, and launches it.

Layout of the blob (fp32, device): every group starts on a 4-float boundary; a conditioner
net is stored per Linear layer as weight ``[out][in]`` (torch order) followed by bias.
"""

from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib


class ParamPacker:
    def __init__(self, device, differentiable: bool = False):
        self.device = device
        self.differentiable = differentiable  # keep the autograd graph from the nn.Parameters to the blob
        self.parts: list[torch.Tensor] = []
        self.n = 0
        self.post = []  # callables(blob) run after the blob exists (e.g. Glow assembly)

    def _pad(self):
        pad = (-self.n) % 4
        if pad:
            self.parts.append(torch.zeros(pad, device=self.device))
            self.n += pad

    def add(self, *tensors) -> int:
        """Append tensors back to back (one group); returns the group's float offset."""
        self._pad()
        off = self.n
        for t in tensors:
            if not self.differentiable:
                t = t.detach()
            if t.device != self.device:
                raise RuntimeError(f"parameter on {t.device}, input on {self.device}")
            self.parts.append(t.reshape(-1).to(torch.float32))
            self.n += t.numel()
        return off

    def reserve(self, n: int, fill=None, torch_fill=None) -> int:
        """n floats written after the blob exists by ``fill(blob, off)`` (a kernel); in differentiable mode
        ``torch_fill()`` must return the same n values as a differentiable tensor instead."""
        self._pad()
        off = self.n
        self.n += n
        if self.differentiable:
            if torch_fill is None:
                raise NotImplementedError("this flow has no differentiable parameter assembly")
            t = torch_fill().reshape(-1).to(torch.float32)
            if t.numel() != n:
                raise RuntimeError(f"torch_fill returned {t.numel()} values, expected {n}")
            self.parts.append(t)
            return off
        self.parts.append(torch.zeros(n, device=self.device))
        if fill is not None:
            self.post.append(lambda blob, off=off: fill(blob, off))
        return off

    def finish(self) -> torch.Tensor:
        self._pad()
        blob = torch.cat(self.parts) if self.parts else torch.zeros(4, device=self.device)
        for fn in self.post:
            fn(blob)
        return blob


def net_tensors(linears, masks=None):
    """[w0, b0, w1, b1, ...] for a chain of nn.Linear; MADE masks ([in,out]) folded into the weights."""
    out = []
    for i, lin in enumerate(linears):
        w = lin.weight
        if masks is not None:
            w = w * masks[i].to(w.dtype).T  # made.py:23: x @ (W.T * mask)
        out += [w, lin.bias]
    return out


def check_leaky(*nets):
    """The kernels evaluate conditioner MLPs with the reference's LeakyReLU slope (models/mlp.py:4: leaky_a=0.2)."""
    for net in nets:
        a = getattr(net, "leaky_a", 0.2) if net is not None else 0.2
        if a != 0.2:
            raise NotImplementedError(
                f"conditioner MLP with leaky_a={a}: the CUDA kernels implement LeakyReLU(0.2) only (models/mlp.py:4)")


def new_op(type_, flags=0, K=0, bound=0.0, sizes=(), net_off=(0, 0), aux_off=0, edge_deriv=0.0):
    if len(sizes) - 1 > _lib.MAX_LIN:
        raise ValueError(f"conditioner has {len(sizes) - 1} Linear layers; at most {_lib.MAX_LIN} supported")
    op = _lib.FlowOp()
    op.type, op.flags, op.K, op.bound = type_, flags, K, float(bound)
    op.n_lin = max(len(sizes) - 1, 0)
    for i, s in enumerate(sizes):
        op.sizes[i] = int(s)
    op.net_off[0], op.net_off[1] = int(net_off[0]), int(net_off[1])
    op.aux_off, op.edge_deriv = int(aux_off), float(edge_deriv)
    return op


def spline_edge_derivative(min_deriv: float = 1e-3) -> float:
    """min_d + softplus(log(exp(1 - min_d) - 1)) evaluated in fp32 (spline_flow.py:46-49,104)."""
    c = torch.tensor(math.log(math.exp(1 - min_deriv) - 1), dtype=torch.float32)
    return float(min_deriv + torch.nn.functional.softplus(c))


_version_of = __import__("operator").attrgetter("_version")


def _tensors_of(flows):
    out = []
    for f in flows:
        out += list(f.parameters()) + list(f.buffers())
    return out


#: bumped by anything that rewrites parameters behind autograd's back without touching ``_version`` (CUDA-graph replays
#: of a captured optimizer step, torch_mnf.graphs): every cached blob / plan / descriptor includes it in its key
_param_epoch = 0


def bump_param_epoch() -> None:
    global _param_epoch
    _param_epoch += 1


def param_epoch() -> int:
    return _param_epoch


_data_ptr_of = __import__("operator").methodcaller("data_ptr")

#: per-module caches that hold ctypes descriptors / device blobs: never copied or pickled with the module
CACHE_KEYS = ("_prog", "_single_prog", "_tc_plan", "_fused_plan", "_rnvp_struct_cache", "_std_base", "_last_kl_terms",
              "_kl_plan")


def state_without_caches(module):
    """``__getstate__`` of the drop-in modules: the module's ``__dict__`` minus the launch caches (ctypes structs with
    raw device pointers cannot be pickled or deep-copied; the reference's modules can, so ours must too)."""
    return {k: v for k, v in module.__dict__.items() if k not in CACHE_KEYS}


def _state_key(flows, device, tensors):
    """Per-call fingerprint of everything the packed blob depends on: in-place updates bump ``_version``;
    re-assigned storage (``.to()``, ``p.data = ...``, ``load_state_dict(assign=True)``) shows in the data pointers of
    EVERY tensor; kernels that write parameters behind autograd's back bump ``_program_salt`` (ActNorm init) or the
    global parameter epoch (CUDA-graph replays of an optimizer step)."""
    return (
        str(device), tuple(map(_version_of, tensors)), tuple(map(_data_ptr_of, tensors)),
        tuple(f.__dict__.get("_program_salt", 0) for f in flows), _param_epoch,
    )


class _FlowStackFn(torch.autograd.Function):
    """Differentiable launch of a flow program: forward = mnf_flow_stack_run keeping every flow's output,
    backward = mnf_flow_stack_backward.  The parameter blob is an autograd function of the nn.Parameters
    (torch.cat of views, MADE masks and the Glow assembly applied by torch), so d loss / d blob is chained
    to them by torch."""

    @staticmethod
    def forward(ctx, prog, inverse, x, blob):
        B, D = x.shape
        lib = _lib.lib()
        n = prog._n_ops
        ld = torch.empty(B, device=x.device, dtype=torch.float32)
        inter = torch.empty((n, B, D), device=x.device, dtype=torch.float32)
        ws = FlowProgram._workspace(lib, n, B, D, x.device, have_y=True)
        with torch.cuda.device(x.device):
            rc = lib.mnf_flow_stack_run(prog._ops, n, blob.data_ptr(), blob.numel(), x.data_ptr(), None,
                                        ld.data_ptr(), None, inter.data_ptr(), B, D,
                                        _lib.RUN_INVERSE if inverse else 0, _lib.ptr(ws), None, _lib.stream_ptr(x.device))
        _lib.check(rc, "mnf_flow_stack_run")
        _lib.launch_count += 1
        ctx.prog, ctx.inverse = prog, inverse
        ctx.save_for_backward(x, inter, blob)
        return ld, inter

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_ld, g_inter):
        x, inter, blob = ctx.saved_tensors
        prog = ctx.prog
        B, D = x.shape
        lib = _lib.lib()
        g_blob = torch.zeros_like(blob)
        g_x = torch.empty_like(x) if ctx.needs_input_grad[2] else None
        g_ld = g_ld.contiguous() if g_ld is not None else None
        g_inter = g_inter.contiguous() if g_inter is not None else None
        with torch.cuda.device(x.device):
            rc = lib.mnf_flow_stack_backward(prog._ops, prog._n_ops, blob.data_ptr(), blob.numel(), g_blob.data_ptr(),
                                             x.data_ptr(), inter.data_ptr(), None, _lib.ptr(g_ld), _lib.ptr(g_inter),
                                             _lib.ptr(g_x), B, D, _lib.RUN_INVERSE if ctx.inverse else 0,
                                             _lib.stream_ptr(x.device))
        _lib.check(rc, "mnf_flow_stack_backward")
        _lib.launch_count += 1
        return None, None, g_x, g_blob


class BoundLogProb:
    """``f(x) -> log p(x)`` through ``mnf_flow_handle_log_prob``: the program, its packed parameters and its staged net
    image are bound once, a call is one C function of five arguments -- no cache-key check over the parameters, no
    marshalling of descriptors.  Contract (as for a captured CUDA graph): the parameters must not change while the
    object is in use; build a new one after an update.  Additive API, not part of the reference."""

    def __init__(self, prog, device, dim, max_rows):
        lib = _lib.lib()
        prog._build(device)
        if not 0 < prog._n_ops <= _lib.MAX_OPS:
            raise NotImplementedError(f"a bound program holds between 1 and {_lib.MAX_OPS} flows")
        self.device, self.dim, self.max_rows = prog._blob.device, dim, int(max_rows)
        self._blob = prog._blob
        self._staged = prog._staged_image(lib, 1, dim, None)
        # dim 2: the kernels a bound call can reach need at most the weight image of the tensor-core kernel, whatever the
        # batch; other dims (MADE density in log-prob mode) park max_rows points in the workspace
        need = lib.mnf_flow_stack_workspace(prog._n_ops, 0 if dim == 2 else self.max_rows, dim)
        self._ws = torch.empty(need, device=self.device, dtype=torch.float32) if need > 0 else None
        ws_rows = (1 << 62) if dim == 2 else self.max_rows
        self._handle = C.c_void_p()
        rc = lib.mnf_flow_handle_create(prog._ops, prog._n_ops, self._blob.data_ptr(), self._blob.numel(), dim,
                                        _lib.ptr(self._staged), _lib.ptr(self._ws), ws_rows if self._ws is not None else 0,
                                        C.byref(self._handle))
        _lib.check(rc, "mnf_flow_handle_create")
        self._call = lib.mnf_flow_handle_log_prob
        self._stream = _lib.stream_ptr

    def __call__(self, x, out=None):
        if out is None:
            out = torch.empty(x.shape[0], device=x.device, dtype=torch.float32)
        rc = self._call(self._handle, x.data_ptr(), out.data_ptr(), x.shape[0], self._stream(x.device))
        if rc:
            _lib.check(rc, "mnf_flow_handle_log_prob")
        return out

    def __del__(self):
        h, self._handle = getattr(self, "_handle", None), None
        if h:
            try:
                _lib.lib().mnf_flow_handle_destroy(h)
            except Exception:  # noqa: BLE001  (interpreter shutdown)
                pass


class FlowProgram:
    """Cached (descriptors, blob) for a sequence of flow modules."""

    def __init__(self, flows):
        self.flows = list(flows)
        self._refresh_tensors()
        self._key = None
        self._ops = None
        self._blob = None

    def _build(self, device):
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        key = _state_key(self.flows, device, self._tensors)
        if key == self._key:
            return
        # something changed: re-enumerate (Module.to() re-creates buffers, load_state_dict(assign=True) replaces the
        # Parameter objects -- both bump the flows' _program_salt through the hooks in flows/_base.py, so the stale
        # list can never produce a matching key)
        self._refresh_tensors()
        key = _state_key(self.flows, device, self._tensors)
        pk = ParamPacker(device)
        ops = [f._emit(pk) for f in self.flows]
        with torch.no_grad():
            blob = pk.finish()
        self._ops = (_lib.FlowOp * max(len(ops), 1))(*ops)
        self._n_ops = len(ops)
        self._blob = blob
        self._staged = {}  # dim -> pre-staged shared-memory image of the nets (or False), rebuilt with the blob
        self._key = key

    def _staged_image(self, lib, n_rows, dim, kernel):
        """Per-parameter-version image of a dim-2 program (mnf_flow_stack_stage), cached until a parameter changes: the
        conditioner tables of the piecewise-linear kernel (any batch size) or, for the shapes without them, the
        shared-memory layout of the nets (batches below 65536 rows)."""
        if dim != 2 or kernel is not None or not 0 < self._n_ops <= _lib.MAX_OPS:
            return None
        img = self._staged.get(dim)
        if img is None:
            size = lib.mnf_flow_stack_stage_size(self._ops, self._n_ops, dim, self._blob.numel())
            self._staged["max_rows"] = lib.mnf_flow_stack_stage_max_rows(self._ops, self._n_ops, dim, self._blob.numel())
            img = False
            if size > 0:
                img = torch.empty(size, device=self._blob.device, dtype=torch.float32)
                with torch.cuda.device(self._blob.device):
                    rc = lib.mnf_flow_stack_stage(self._ops, self._n_ops, self._blob.data_ptr(), self._blob.numel(), dim,
                                                  img.data_ptr(), _lib.stream_ptr(self._blob.device))
                _lib.check(rc, "mnf_flow_stack_stage")
            self._staged[dim] = img
        return img if img is not False and n_rows <= self._staged["max_rows"] else None

    @staticmethod
    def _workspace(lib, n_ops, n_rows, dim, dev, have_y=False, kernel=None):
        if have_y and dim != 2:
            return None  # only log-prob-only runs (no y buffer) of the MADE kernel park points in the workspace
        need = lib.mnf_flow_stack_workspace(n_ops, n_rows, dim)
        return torch.empty(need, device=dev, dtype=torch.float32) if need > 0 else None

    def plan(self, device, dim) -> int:
        """1 if the dim-2 register-resident kernel will run this program, else 0 (generic)."""
        self._build(device)
        n = min(self._n_ops, _lib.MAX_OPS)
        return _lib.lib().mnf_flow_stack_plan(self._ops, n, dim, self._blob.numel())

    def _refresh_tensors(self):
        self._tensors = _tensors_of(self.flows)
        self._salts = tuple(f.__dict__.get("_program_salt", 0) for f in self.flows)

    def needs_grad(self, x) -> bool:
        if not torch.is_grad_enabled():
            return False
        if x.requires_grad:
            return True
        if self._salts != tuple(f.__dict__.get("_program_salt", 0) for f in self.flows):
            self._refresh_tensors()  # parameters were replaced (load_state_dict(assign=True), .to()): re-read flags
        return any(p.requires_grad for p in self._tensors)

    def run_autograd(self, x, inverse: bool):
        """(log_det [B], outputs of every flow [n_ops, B, D]) with the autograd graph attached
        (mnf_flow_stack_backward).  One chunk only: at most MNF_MAX_OPS flows."""
        x = _lib.require_cuda_f32(x, "input")
        if x.dim() != 2:
            raise ValueError(f"flows take [batch, dim] inputs, got shape {tuple(x.shape)}")
        self._build(x.device)
        if not 0 < self._n_ops <= _lib.MAX_OPS:
            raise NotImplementedError(f"autograd through {self._n_ops} flows: between 1 and {_lib.MAX_OPS} supported")
        pk = ParamPacker(self._blob.device, differentiable=True)
        for f in self.flows:
            f._emit(pk)
        blob = pk.finish()
        if blob.numel() != self._blob.numel():
            raise RuntimeError("differentiable parameter blob does not match the cached layout")
        return _FlowStackFn.apply(self, inverse, x, blob)

    @torch.no_grad()
    def sample(self, n_rows: int, dim: int, device, seed: int, row_offset: int = 0, want_x: bool = True,
               want_log_prob: bool = True, want_z: bool = False, kernel=None):
        """(x, log_prob, z) of ``n_rows`` standard-normal base draws pushed through the flows (mnf_flow_stack_sample):
        z of global row row_offset + r from Philox(seed, stream 0), x its forward pass, log_prob = log N(z) - log_det.
        Outputs not asked for are None.  kernel as for ``run``.  Single-chunk programs only."""
        self._build(device)
        if not 0 < self._n_ops <= _lib.MAX_OPS:
            raise NotImplementedError(f"sampling through {self._n_ops} flows: between 1 and {_lib.MAX_OPS} supported")
        lib = _lib.lib()
        dev = self._blob.device
        x = torch.empty(n_rows, dim, device=dev, dtype=torch.float32) if want_x else None
        lp = torch.empty(n_rows, device=dev, dtype=torch.float32) if want_log_prob else None
        z = torch.empty(n_rows, dim, device=dev, dtype=torch.float32) if want_z else None
        flags = 0
        if kernel == "generic":
            flags |= _lib.RUN_GENERIC
        elif kernel is not None:
            flags |= ((int(kernel) + 1) << 4) & 0x70
        ws = self._staged_image(lib, n_rows, dim, kernel)
        if ws is not None:
            flags |= _lib.RUN_STAGED
        else:
            ws = self._workspace(lib, self._n_ops, n_rows, dim, dev, have_y=want_x, kernel=kernel)
        with _lib.on_device(dev):
            rc = lib.mnf_flow_stack_sample(self._ops, self._n_ops, self._blob.data_ptr(), self._blob.numel(),
                                           int(seed) & (2**64 - 1), 0, int(row_offset), _lib.ptr(x), _lib.ptr(lp),
                                           _lib.ptr(z), n_rows, dim, flags, _lib.ptr(ws), _lib.stream_ptr(dev))
        _lib.check(rc, "mnf_flow_stack_sample")
        _lib.launch_count += 1
        return x, lp, z

    @torch.no_grad()
    def run(self, x, inverse: bool, want_inter: bool = False, want_base_lp: bool = False, out=None,
            log_det=None, kernel=None, log_prob_only=False, log_prob_out=None, gather=None):
        """kernel: None = library default, "generic" = interpreter, 0/1/2 = dim-2 kernel variant.
        log_prob_only: return (None, None, None, log_det + standard-normal log-density) without
        storing the transformed points (single-chunk programs only).
        gather: optional _lib.GatherOut -- also store the log-probs into peer ranks' buffers (fused gather)."""
        x = _lib.require_cuda_f32(x, "input")
        if x.dim() != 2:
            raise ValueError(f"flows take [batch, dim] inputs, got shape {tuple(x.shape)}")
        B, D = x.shape
        dev = x.device
        self._build(dev)
        lib = _lib.lib()
        n = self._n_ops
        if log_prob_only and 0 < n <= _lib.MAX_OPS:
            lp = log_prob_out if log_prob_out is not None else torch.empty(B, device=dev, dtype=torch.float32)
            flags = (_lib.RUN_INVERSE if inverse else 0) | _lib.RUN_LOGPROB
            if kernel == "generic":
                flags |= _lib.RUN_GENERIC
            elif kernel is not None:
                flags |= ((int(kernel) + 1) << 4) & 0x70
            ws = self._staged_image(lib, B, D, kernel)
            if ws is not None:
                flags |= _lib.RUN_STAGED
            else:
                ws = self._workspace(lib, n, B, D, dev, kernel=kernel)
            with _lib.on_device(dev):
                rc = lib.mnf_flow_stack_run(self._ops, n, self._blob.data_ptr(), self._blob.numel(), x.data_ptr(),
                                            None, None, lp.data_ptr(), None, B, D, flags, _lib.ptr(ws),
                                            C.byref(gather) if gather is not None else None, _lib.stream_ptr(dev))
            _lib.check(rc, "mnf_flow_stack_run")
            _lib.launch_count += 1
            return None, None, None, lp
        y = out if out is not None else torch.empty_like(x)
        ld = log_det if log_det is not None else torch.empty(B, device=dev, dtype=torch.float32)
        lp = torch.empty(B, device=dev, dtype=torch.float32) if want_base_lp else None
        inter = torch.empty((n, B, D), device=dev, dtype=torch.float32) if want_inter else None
        if n == 0:
            y.copy_(x)
            ld.zero_()
        stream = _lib.stream_ptr(dev)
        ws = self._workspace(lib, min(n, _lib.MAX_OPS), B, D, dev, have_y=True, kernel=kernel)
        flags = _lib.RUN_INVERSE if inverse else 0
        if kernel == "generic":
            flags |= _lib.RUN_GENERIC
        elif kernel is not None:
            flags |= ((int(kernel) + 1) << 4) & 0x70
        staged = self._staged_image(lib, B, D, kernel)
        if staged is not None:
            ws, flags = staged, flags | _lib.RUN_STAGED
        with torch.cuda.device(dev):
            # stacks longer than MNF_MAX_OPS run in chunks, log-dets summed across chunks
            done, src, first = 0, x, True
            order = list(range(0, n, _lib.MAX_OPS))
            if inverse:
                order = order[::-1]
            for start in order:
                cnt = min(_lib.MAX_OPS, n - start)
                ops_ptr = C.cast(C.byref(self._ops, start * C.sizeof(_lib.FlowOp)), C.POINTER(_lib.FlowOp))
                last = done + cnt == n
                ld_chunk = ld if first else torch.empty_like(ld)
                rc = lib.mnf_flow_stack_run(
                    ops_ptr, cnt, self._blob.data_ptr(), self._blob.numel(), src.data_ptr(), y.data_ptr(),
                    ld_chunk.data_ptr(), _lib.ptr(lp) if last else None,
                    inter[done:].data_ptr() if inter is not None else None, B, D, flags, _lib.ptr(ws), None, stream,
                )
                _lib.check(rc, "mnf_flow_stack_run")
                _lib.launch_count += 1
                if not first:
                    ld += ld_chunk
                first, src, done = False, y, done + cnt
        return y, ld, inter, lp
