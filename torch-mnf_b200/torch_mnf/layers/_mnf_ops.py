"""Host-side wrappers of the MNF entry points of libmnf_b200.so (include/mnf_b200.h):
noise bookkeeping (injected tape or in-kernel Philox), RNVP stacks, and the struct marshalling."""

from __future__ import annotations

import ctypes as C

import torch

from .. import _lib

RNVP_MAX_NET = 4
_vp, _u64, _u32, _i64, _int = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int64, C.c_int


class RnvpFlow(C.Structure):
    """struct mnf_rnvp_flow."""

    _fields_ = [
        ("n_net", C.c_int32),
        ("net_sizes", C.c_int32 * RNVP_MAX_NET),
        ("net_w", C.c_void_p * RNVP_MAX_NET),
        ("net_b", C.c_void_p * RNVP_MAX_NET),
        ("t_w", C.c_void_p), ("t_b", C.c_void_p), ("s_w", C.c_void_p), ("s_b", C.c_void_p),
    ]


class KlArgs(C.Structure):
    """struct mnf_kl_args."""

    _fields_ = [
        ("conv", C.c_int32), ("n_out", C.c_int32), ("n_in", C.c_int32), ("ksize", C.c_int32),
        ("W_mean", _vp), ("W_log_var", _vp), ("b_mean", _vp), ("b_log_var", _vp),
        ("q0_log_var", _vp), ("r0_c", _vp), ("r0_b1", _vp), ("r0_b2", _vp),
        ("z", _vp), ("zT", _vp), ("ld_q", _vp), ("ld_r", _vp), ("eps_w", _vp), ("eps_b", _vp),
        ("seed", C.c_uint64), ("noise_stream", C.c_uint32),
        ("workspace", _vp), ("out", _vp),
    ]


KL_MAX_FLOWS = 4


class KlFusedArgs(C.Structure):
    """struct mnf_kl_fused_args."""

    _fields_ = [
        ("kl", KlArgs), ("q0_mean", _vp), ("eps_z", _vp), ("z_stream", C.c_uint32),
        ("n_flows_q", C.c_int32), ("n_flows_r", C.c_int32), ("reserved", C.c_int32),
        ("flows", RnvpFlow * (2 * KL_MAX_FLOWS)), ("masks", _vp * (2 * KL_MAX_FLOWS)),
        ("mask_streams", C.c_uint32 * (2 * KL_MAX_FLOWS)),
    ]


_lib.register({
    "mnf_kl_div_fused": (_int, [C.POINTER(KlFusedArgs), _vp]),
    "mnf_kl_div_fused_multi": (_int, [C.POINTER(C.POINTER(KlFusedArgs)), _int, _vp]),
    "mnf_sample_z0": (_int, [_vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int, _vp]),
    "mnf_rnvp_forward": (_int, [C.POINTER(RnvpFlow), _int, _vp, _vp, C.POINTER(C.c_void_p), _u64, _u32, _u64,
                                _i64, _int, _vp, _vp, _vp]),
    "mnf_linear_forward": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int,
                                  _int, _int, _vp]),
    "mnf_linear_forward_affine": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int,
                                         _int, _int, _vp, _vp, _vp]),
    "mnf_linear_sample_weights": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u32, _u64, _vp, _vp, _i64, _int,
                                         _int, _vp]),
    "mnf_linear_function_forward": (_int, [_vp, _int, _vp, _vp, _vp, _i64, _i64, _int, _int, _int, _vp, _vp, _vp]),
    "mnf_conv2d_forward": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int,
                                  _int, _int, _int, _int, _vp]),
    "mnf_conv2d_forward_ps": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int,
                                     _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_conv2d_forward_geom": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int,
                                       _int, _int, _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_kl_div": (_int, [C.POINTER(KlArgs), _vp]),
    "mnf_linear_tc_workspace": (_i64, [_i64, _i64, _int, _int]),
    "mnf_linear_forward_tc": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int,
                                     _int, _int, _vp, _vp]),
    "mnf_linear_forward_tc_affine": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int,
                                            _int, _int, _vp, _vp, _vp, _vp]),
    "mnf_mc_moments": (_int, [_vp, _i64, _i64, _int, _int, _vp, _vp]),
    "mnf_mc_class_moments": (_int, [_vp, _i64, _i64, _int, _vp, _vp, _vp]),
    "mnf_rnvp_tc_workspace": (_i64, [_int, _i64, _int]),
    "mnf_rnvp_forward_tc": (_int, [C.POINTER(RnvpFlow), _int, _vp, _vp, C.POINTER(C.c_void_p), _u64, _u32, _u64, _i64,
                                   _int, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _u32, _int, _vp]),
    "mnf_conv2d_moments": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _vp]),
    "mnf_conv2d_moments_ps": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _int,
                                     _vp]),
    "mnf_conv2d_moments_geom": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _int, _int,
                                       _int, _int, _int, _vp]),
    "mnf_conv_noise_relu_pool": (_int, [_vp, _vp, _i64, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int, _int, _vp]),
    "mnf_conv_noise_relu_pool_z": (_int, [_vp, _vp, _i64, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int, _int, _vp, _i64,
                                          _vp]),
    "mnf_conv2d_forward_tc_z": (_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int,
                                       _int, _int, _int, _vp, _vp]),
    "mnf_conv_tc_workspace": (_i64, [_i64, _int, _int, _int, _int, _int]),
    "mnf_conv2d_forward_tc": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _u64, _u32, _u64, _vp, _i64, _int, _int, _int, _int,
                                     _int, _vp, _vp]),
    "mnf_conv_tc_stage": (_int, [_vp] * 10 + [_i64, _int, _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_tc_linear": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _int, _int, _int, _vp]),
    "mnf_tc_eligible": (_int, [_vp, _vp, _i64, _int, _int]),
})


class Noise:
    """Noise source of ONE layer call.  With a tape (any object with ``normal(shape)`` /
    ``bernoulli(shape)``, e.g. oracle.noise.NoiseTape) every draw is taken from it in the
    reference's order; without one the kernels draw from Philox and ``draw`` only hands out the
    per-draw stream ids."""

    def __init__(self, tape, device, row_offset: int = 0, seed: int | None = None):
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if tape is None and seed is None and device.type == "cuda" and torch.cuda.is_current_stream_capturing():
            # CUDA-graph capture: a Philox seed passed by value would be frozen into the graph and every replay would
            # repeat the same z / masks / eps.  Materialise the draws with torch's graph-safe generator instead (its
            # offset advances per replay), in the reference's draw order.
            from ._train import DeviceTape

            tape = DeviceTape(device)
        self.tape, self.device, self.row_offset = tape, device, int(row_offset)
        self.streams = 0
        if tape is None and seed is None:
            seed = int(torch.randint(0, 2**62, (1,)).item())  # follows torch.manual_seed
        self.seed = seed or 0
        self.keep = []  # injected tensors must outlive the asynchronous launches

    def _next_stream(self):
        s = self.streams
        self.streams += 1
        return s

    def normal(self, shape):
        """-> (device tensor or None, noise stream id)."""
        sid = self._next_stream()
        if self.tape is None:
            return None, sid
        t = self.tape.normal(tuple(shape)).to(self.device, torch.float32).contiguous()
        self.keep.append(t)
        return t, sid

    def bernoulli(self, shape):
        sid = self._next_stream()
        if self.tape is None:
            return None, sid
        t = self.tape.bernoulli(tuple(shape)).to(self.device, torch.float32).contiguous()
        self.keep.append(t)
        return t, sid


def _p(t):
    return None if t is None else t.data_ptr()


def _param(t, device, name):
    if t.device != device:
        raise RuntimeError(f"{name} is on {t.device} but the input is on {device}")
    t = t.detach()
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


def sample_z0(q0_mean, q0_log_var, n_rows, noise: Noise):
    dev = noise.device
    dim = q0_mean.numel()
    eps, sid = noise.normal((n_rows, dim) if n_rows != -1 else (dim,))
    rows = max(n_rows, 1)
    z = torch.empty((rows, dim), device=dev, dtype=torch.float32)
    qm, qv = _param(q0_mean, dev, "q0_mean"), _param(q0_log_var, dev, "q0_log_var")
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_sample_z0(qm.data_ptr(), qv.data_ptr(), _p(eps), noise.seed, sid, noise.row_offset,
                                      z.data_ptr(), rows, dim, _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_sample_z0")
    _lib.launch_count += 1
    return z


def _rnvp_struct(flow, dev, keep):
    from .._program import check_leaky

    check_leaky(flow.net)
    lin = flow.net.linears()
    if len(lin) > RNVP_MAX_NET:
        raise ValueError(f"RNVP conditioner with {len(lin)} layers; at most {RNVP_MAX_NET} supported")
    # fast path: the descriptor only holds raw pointers, so it stays valid while the parameters keep their storage
    # (optimizer steps update in place); rebuilding it was a third of the host time of a kl_div() call
    tensors = [t for m in lin for t in (m.weight, m.bias)] + [flow.t.weight, flow.t.bias, flow.s.weight, flow.s.bias]
    key = (str(dev), tuple(t.data_ptr() for t in tensors))
    cached = flow.__dict__.get("_rnvp_struct_cache")
    if cached is not None and cached[0] == key:
        return cached[1], cached[2]
    plain = all(t.device == dev and t.dtype == torch.float32 and t.is_contiguous() for t in tensors)
    st = RnvpFlow()
    st.n_net = len(lin)
    for i, m in enumerate(lin):
        w, b = _param(m.weight, dev, "net.weight"), _param(m.bias, dev, "net.bias")
        keep += [w, b]
        st.net_sizes[i], st.net_w[i], st.net_b[i] = m.out_features, w.data_ptr(), b.data_ptr()
    for name, mod in (("t", flow.t), ("s", flow.s)):
        w, b = _param(mod.weight, dev, name + ".weight"), _param(mod.bias, dev, name + ".bias")
        keep += [w, b]
        setattr(st, name + "_w", w.data_ptr())
        setattr(st, name + "_b", b.data_ptr())
    maxh = max(m.out_features for m in lin)
    if plain:
        flow.__dict__["_rnvp_struct_cache"] = (key, st, maxh)
    return st, maxh


@torch.no_grad()
def rnvp_stack_inplace(flows, z, noise: Noise, want_inter=False):
    """Runs the RNVP flows in place on z [R, dim]; returns (log_det [R], intermediates or None)."""
    dev = z.device
    R, dim = z.shape
    n = len(flows)
    keep = []
    structs, maxh = [], 1
    for f in flows:
        st, h = _rnvp_struct(f, dev, keep)
        structs.append(st)
        maxh = max(maxh, h)
    arr = (RnvpFlow * max(n, 1))(*structs)
    masks, first_sid = [], None
    for _ in range(n):
        m, sid = noise.bernoulli((R, dim))
        masks.append(m)
        first_sid = sid if first_sid is None else first_sid
    mask_arr = None
    if n and masks[0] is not None:
        mask_arr = (C.c_void_p * n)(*[m.data_ptr() for m in masks])
    ld = torch.empty(R, device=dev, dtype=torch.float32)
    ws = torch.empty(2 * R * maxh, device=dev, dtype=torch.float32)
    inter = torch.empty((n, R, dim), device=dev, dtype=torch.float32) if want_inter else None
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_rnvp_forward(arr, n, z.data_ptr(), ld.data_ptr(), mask_arr, noise.seed, first_sid or 0,
                                         noise.row_offset, R, dim, ws.data_ptr(), _p(inter), _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_rnvp_forward")
    _lib.launch_count += 2 * n
    return ld, inter


def rnvp_tc_ok(flows, dim) -> bool:
    return (len(flows) >= 1 and dim % 16 == 0 and dim >= 32
            and all(len(f.net.linears()) == 1 and f.net.linears()[0].out_features <= 64 for f in flows))


@torch.no_grad()
def rnvp_stack_tc(flows, z, noise: Noise, x=None, x_rows=None, xz_out=None, q0=None, n_rows=None, z_is_scratch=False):
    """Tensor-core variant of rnvp_stack_inplace; optionally leaves tf32(x*z_final) in xz_out.  With q0 =
    (q0_mean, q0_log_var) the base sample z0 is drawn inside the call (z may be None) -- draw order as in
    MNFLinear.sample_z: normal[R, dim] first, then one Bernoulli mask per flow."""
    dev = noise.device
    n = len(flows)
    eps_z, eps_sid, q0m, q0v = None, 0, None, None
    if q0 is not None:
        q0m, q0v = _param(q0[0], dev, "q0_mean"), _param(q0[1], dev, "q0_log_var")
        R, dim = n_rows, q0m.numel()
        eps_z, eps_sid = noise.normal((R, dim))
        z = torch.empty((R, dim), device=dev, dtype=torch.float32)
    R, dim = z.shape
    keep = []
    arr = (RnvpFlow * n)(*[_rnvp_struct(f, dev, keep)[0] for f in flows])
    masks, first_sid = [], None
    for _ in range(n):
        m, sid = noise.bernoulli((R, dim))
        masks.append(m)
        first_sid = sid if first_sid is None else first_sid
    mask_arr = (C.c_void_p * n)(*[m.data_ptr() for m in masks]) if masks[0] is not None else None
    ld = torch.empty(R, device=dev, dtype=torch.float32)
    lib = _lib.lib()
    ws = torch.empty(lib.mnf_rnvp_tc_workspace(n, R, dim), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        rc = lib.mnf_rnvp_forward_tc(arr, n, z.data_ptr(), ld.data_ptr(), mask_arr, noise.seed, first_sid or 0,
                                     noise.row_offset, R, dim, _p(x), x_rows or (x.size(0) if x is not None else 1),
                                     _p(xz_out), ws.data_ptr(), _p(q0m), _p(q0v), _p(eps_z), eps_sid, int(z_is_scratch),
                                     _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_rnvp_forward_tc")
    return ld, z


def rnvp_stack(flows, z, tape, want_inter):
    """NormalizingFlow([RNVP...]).forward: returns (list incl. the input, log_det[B]).  With grad enabled and
    trainable parameters (or a z that requires grad) the differentiable primitives of layers/_train.py run, as the
    reference's version is differentiable (rnvp.py:25-39 under torch autograd)."""
    z = _lib.require_cuda_f32(z, "input")
    flows = list(flows)
    if torch.is_grad_enabled() and (z.requires_grad or any(p.requires_grad for f in flows for p in f.parameters())):
        from . import _train

        t = _train._tape(tape, z.device)
        xs, ld = [z], torch.zeros(z.size(0), device=z.device)
        for f in flows:
            mask = _train._draw(t, "bernoulli", z.shape, z.device)
            nxt, l = _train.rnvp_flow(f, xs[-1], mask)
            xs.append(nxt)
            ld = ld + l
        return (xs if want_inter else [z, xs[-1]]), ld
    noise = tape if isinstance(tape, Noise) else Noise(tape, z.device)
    out = z.clone()
    ld, inter = rnvp_stack_inplace(list(flows), out, noise, want_inter)
    xs = [z] + (list(inter.unbind(0)) if inter is not None else [out])
    return xs, ld


TC_MIN_WORK = 1 << 24  # n_rows * n_in * n_out below which the fp32 SIMT kernel is used


def use_tensor_cores(layer, n_rows, precision):
    """precision: "fp32" (exact SIMT path), "tf32" (tcgen05), or "auto" (tf32 for large aligned shapes)."""
    n_out, n_in = layer.W_mean.shape
    if precision == "fp32":
        return False
    ok = n_in % 4 == 0 and n_in >= 32 and n_out >= 8
    if precision == "tf32":
        if not ok:
            raise ValueError(f"tf32 tensor-core path needs n_in % 4 == 0, n_in >= 32, n_out >= 8 (got {n_in}, {n_out})")
        return True
    return ok and n_rows * n_in * n_out >= TC_MIN_WORK and n_in >= 128 and n_out >= 32


@torch.no_grad()
def linear_forward(layer, x, z, noise: Noise, x_rows=None, relu=False, precision="auto", staged_ws=None, n_rows=None,
                   affine=None):
    """staged_ws: tensor-core workspace whose first n_rows*n_in floats already hold tf32(x*z) (z is then None).
    affine: optional (col_scale, col_shift) [n_out] applied after the noise and ReLU (a folded eval-mode BatchNorm1d)."""
    dev = x.device
    scale, shift = affine if affine is not None else (None, None)
    R = z.size(0) if z is not None else n_rows
    n_in, n_out = layer.W_mean.shape[1], layer.W_mean.shape[0]
    eps, sid = noise.normal((R, n_out))
    out = torch.empty((R, n_out), device=dev, dtype=torch.float32)
    args = [_param(t, dev, n) for t, n in ((layer.W_mean, "W_mean"), (layer.W_log_var, "W_log_var"),
                                           (layer.b_mean, "b_mean"), (layer.b_log_var, "b_log_var"))]
    if staged_ws is not None or use_tensor_cores(layer, R, precision):
        xr = x_rows or x.size(0)
        ws = staged_ws if staged_ws is not None else torch.empty(
            _lib.lib().mnf_linear_tc_workspace(xr, R, n_in, n_out), device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            rc = _lib.lib().mnf_linear_forward_tc_affine(x.data_ptr(), xr, _p(z), *(a.data_ptr() for a in args),
                                                         _p(eps), noise.seed, sid, noise.row_offset, out.data_ptr(), R,
                                                         n_in, n_out, int(relu), _p(scale), _p(shift), ws.data_ptr(),
                                                         _lib.stream_ptr(dev))
        _lib.check(rc, "mnf_linear_forward_tc")
        _lib.launch_count += 5
        return out
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_linear_forward_affine(x.data_ptr(), x_rows or x.size(0), z.data_ptr(),
                                                  *(a.data_ptr() for a in args), _p(eps), noise.seed, sid, noise.row_offset,
                                                  out.data_ptr(), R, n_in, n_out, int(relu), _p(scale), _p(shift),
                                                  _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_linear_forward")
    _lib.launch_count += 1
    return out


#: bytes of one chunk's weight image [S_c, n_out, n_in] when function samples run without a tape: small enough to stay
#: in the B200's 126 MB L2 between the weight draw that writes it and the function GEMM that reads it
FUNCTION_IMAGE_BYTES = 64 << 20


def function_chunk(weights_per_sample: int) -> int:
    """Samples per chunk of a function-sample call: FUNCTION_IMAGE_BYTES of weights, at least one sample, at most the
    65535 of one function GEMM launch."""
    return max(1, min(65535, FUNCTION_IMAGE_BYTES // (4 * weights_per_sample)))


def check_function_args(n_samples, sample_offset, chunk=None):
    """ValueError for n_samples < 1, chunk < 1 or a negative sample_offset -- before any device work."""
    if int(n_samples) < 1:
        raise ValueError(f"n_samples must be positive, got {n_samples}")
    if chunk is not None and int(chunk) < 1:
        raise ValueError(f"chunk must be positive, got {chunk}")
    if int(sample_offset) < 0:
        raise ValueError(f"sample_offset must be non-negative, got {sample_offset}")


def function_input(x, n_in, n_samples):
    """x [B, n_in] (shared by the samples) or [n_samples, B, n_in] (one block per sample), CUDA fp32, contiguous."""
    if not isinstance(x, torch.Tensor):
        raise TypeError("input must be a torch.Tensor")
    if x.dim() == 2:
        ok = x.size(1) == n_in
    elif x.dim() == 3:
        ok = x.size(0) == n_samples and x.size(2) == n_in
    else:
        ok = False
    if not ok:
        raise ValueError(f"input of shape {tuple(x.shape)}: expected [B, {n_in}] or [{n_samples}, B, {n_in}]")
    return _lib.require_cuda_f32(x, "input")


#: rows of the z draw of a function-sample call at the least: mnf_rnvp_forward runs one row on its cluster kernel and at
#: most 4 rows of a wide layer on the GEMV form, both summing in another order than the tiled GEMM, so fewer rows would
#: make a sample's z depend on how many samples the call draws
Z_MIN_ROWS = 5


@torch.no_grad()
def linear_function_z(layer, n_samples, noise: Noise, sample_offset=0):
    """z [S, n_in] of S posterior function samples: rows sample_offset .. sample_offset + S - 1 of MNFLinear.sample_z
    (normal[S, n_in], one Bernoulli[S, n_in] per q-flow).  Without a tape at least Z_MIN_ROWS rows are drawn (the extra
    rows are the next samples' z and are dropped), so a sample's z does not depend on S."""
    rows = n_samples if noise.tape is not None else max(n_samples, Z_MIN_ROWS)
    return conv_sample_z_rows(layer, rows, noise, sample_offset)[:n_samples]


@torch.no_grad()
def linear_sample_weights(layer, z, noise: Noise, sample_offset=0):
    """Posterior weight draws of an MNFLinear for the S rows of z (linear_function_z): (W [S, n_out, n_in], b [S, n_out])
    from the next two draws of noise, normal[S, n_out, n_in] (E) and normal[S, n_out] (e); Philox elements are keyed by
    the global sample index sample_offset + s."""
    dev = noise.device
    n_out, n_in = layer.W_mean.shape
    n_samples = z.size(0)
    eps_w, sid_w = noise.normal((n_samples, n_out, n_in))
    eps_b, sid_b = noise.normal((n_samples, n_out))
    W = torch.empty((n_samples, n_out, n_in), device=dev, dtype=torch.float32)
    b = torch.empty((n_samples, n_out), device=dev, dtype=torch.float32)
    args = [_param(getattr(layer, n), dev, n) for n in ("W_mean", "W_log_var", "b_mean", "b_log_var")]
    with _lib.on_device(dev):
        rc = _lib.lib().mnf_linear_sample_weights(*(a.data_ptr() for a in args), z.data_ptr(), _p(eps_w), _p(eps_b),
                                                  noise.seed, sid_w, sid_b, int(sample_offset), W.data_ptr(),
                                                  b.data_ptr(), n_samples, n_in, n_out, _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_linear_sample_weights")
    _lib.launch_count += 1
    return W, b


@torch.no_grad()
def linear_function_forward(x, W, b, relu=False, affine=None, out=None):
    """out [S, B, n_out] = x_s @ W[s]^T + b[s] (then ReLU, then the folded batch norm ``affine`` = (col_scale,
    col_shift)); x [B, n_in] shared by the samples or [S, B, n_in]."""
    dev = x.device
    S, n_out, n_in = W.shape
    B = x.size(-2)
    scale, shift = affine if affine is not None else (None, None)
    if out is None:
        out = torch.empty((S, B, n_out), device=dev, dtype=torch.float32)
    with _lib.on_device(dev):
        rc = _lib.lib().mnf_linear_function_forward(x.data_ptr(), int(x.dim() == 3), W.data_ptr(), b.data_ptr(),
                                                    out.data_ptr(), S, B, n_in, n_out, int(relu), _p(scale), _p(shift),
                                                    _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_linear_function_forward")
    _lib.launch_count += 1
    return out


def mc_moments(y, n_unique, n_samples, sums, softmax=False, entropy_sums=None):
    """sums [2, n_unique, n_cols] fp64 += (sum_s f(y), sum_s f(y)^2) over the samples of the sample-major y
    [n_samples * n_unique, n_cols]; f = identity or a per-row softmax (mnf_mc_moments).  entropy_sums [n_unique] fp64
    (needs softmax): also += sum_s H(softmax(y[s * n_unique + b])), the per-sample entropies (mnf_mc_class_moments)."""
    dev = y.device
    n_cols = y.size(1)
    if y.shape != (n_samples * n_unique, n_cols) or sums.shape != (2, n_unique, n_cols):
        raise ValueError(f"mc_moments: y {tuple(y.shape)} / sums {tuple(sums.shape)} do not match "
                         f"{n_samples} samples of {n_unique} rows")
    if sums.dtype != torch.float64 or not sums.is_contiguous() or sums.device != dev:
        raise ValueError("mc_moments: sums must be a contiguous float64 tensor on the device of y")
    if entropy_sums is not None:
        if not softmax:
            raise ValueError("mc_moments: entropy_sums needs softmax=True (entropies of class probabilities)")
        if (entropy_sums.shape != (n_unique,) or entropy_sums.dtype != torch.float64
                or not entropy_sums.is_contiguous() or entropy_sums.device != dev):
            raise ValueError(f"mc_moments: entropy_sums must be a contiguous float64 [{n_unique}] tensor on the device "
                             f"of y (got {tuple(entropy_sums.shape)} {entropy_sums.dtype} on {entropy_sums.device})")
    y = _lib.require_cuda_f32(y, "y")
    with _lib.on_device(dev):
        if entropy_sums is None:
            rc = _lib.lib().mnf_mc_moments(y.data_ptr(), n_unique, n_samples, n_cols, int(softmax), sums.data_ptr(),
                                           _lib.stream_ptr(dev))
        else:
            rc = _lib.lib().mnf_mc_class_moments(y.data_ptr(), n_unique, n_samples, n_cols, sums.data_ptr(),
                                                 entropy_sums.data_ptr(), _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_mc_moments" if entropy_sums is None else "mnf_mc_class_moments")
    _lib.launch_count += 1
    return sums


@torch.no_grad()
def conv_forward(layer, x, z, noise: Noise, n_imgs=None, relu_pool=False, drawn=None, out=None):
    """drawn = (eps or None, stream id, row offset): use this noise instead of drawing (a slice of a larger draw)."""
    dev = x.device
    x_imgs, c_in, H, W = x.shape
    R = n_imgs or x_imgs
    c_out, ks = layer.W_mean.shape[0], layer.W_mean.shape[2]
    OH, OW = layer.output_size(H, W)
    eps, sid, row_offset = drawn if drawn is not None else (*noise.normal((R, c_out, OH, OW)), noise.row_offset)
    shape = (R, c_out, OH // 2, OW // 2) if relu_pool else (R, c_out, OH, OW)
    if out is None:
        out = torch.empty(shape, device=dev, dtype=torch.float32)
    args = [_param(t, dev, n) for t, n in ((layer.W_mean, "W_mean"), (layer.W_log_var, "W_log_var"),
                                           (layer.b_log_var, "b_log_var"))]
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_conv2d_forward_geom(x.data_ptr(), x_imgs, z.data_ptr(), *(a.data_ptr() for a in args),
                                                _p(eps), noise.seed, sid, row_offset, out.data_ptr(), R, c_in, H, W,
                                                c_out, ks, int(relu_pool), layer.padding, layer.stride, layer.dilation,
                                                layer.groups, _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_conv2d_forward_geom")
    _lib.launch_count += 1
    return out


def _conv_args(layer, dev):
    return [_param(t, dev, n) for t, n in ((layer.W_mean, "W_mean"), (layer.W_log_var, "W_log_var"),
                                           (layer.b_log_var, "b_log_var"))]


@torch.no_grad()
def conv_sample_z_rows(layer, n_z, noise: Noise, z_offset=0):
    """n_z independent draws of MNFConv2d.sample_z (mnf_conv.py:80-88), one per Monte-Carlo sample: [n_z, n_out].
    Draw order: normal[n_z, n_out], then one Bernoulli[n_z, n_out] per q-flow.  Philox draws are keyed by the global
    sample index z_offset + i, so a sharded prediction sees the z rows a single-device call would."""
    keep, noise.row_offset = noise.row_offset, int(z_offset)
    try:
        z = sample_z0(layer.q0_mean, layer.q0_log_var, n_z, noise)
        rnvp_stack_inplace(list(layer.flow_q.flows), z, noise)
    finally:
        noise.row_offset = keep
    return z


@torch.no_grad()
def conv_moments(layer, x, z):
    """(mean, sd) [B, c_out, OH, OW] of MNFConv2d.forward without its noise (mnf_conv.py:69-75): the part of the layer
    that does not depend on the Monte-Carlo sample when z is shared by the call.  z = None: unit scale."""
    dev = x.device
    B, c_in, H, W = x.shape
    c_out, ks = layer.W_mean.shape[0], layer.W_mean.shape[2]
    OH, OW = layer.output_size(H, W)
    mean = torch.empty((B, c_out, OH, OW), device=dev, dtype=torch.float32)
    sd = torch.empty_like(mean)
    args = _conv_args(layer, dev)
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_conv2d_moments_geom(x.data_ptr(), _p(z), *(a.data_ptr() for a in args), mean.data_ptr(),
                                                sd.data_ptr(), B, c_in, H, W, c_out, ks, layer.padding, layer.stride,
                                                layer.dilation, layer.groups, _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_conv2d_moments_geom")
    _lib.launch_count += 1
    return mean, sd


def conv_noise_relu_pool(mean, sd, noise: Noise, n_rows, z_rows=None, rows_per_z=1):
    """maxpool2(relu(mean[r % B] + sd[r % B] * eps[r])) for n_rows rows: the per-sample tail of an MNFConv2d."""
    dev = mean.device
    B, c_out, OH, OW = mean.shape
    eps, sid = noise.normal((n_rows, c_out, OH, OW))
    out = torch.empty((n_rows, c_out, OH // 2, OW // 2), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_conv_noise_relu_pool_z(mean.data_ptr(), sd.data_ptr(), B, _p(eps), noise.seed, sid,
                                                   noise.row_offset, out.data_ptr(), n_rows, c_out, OH, OW, _p(z_rows),
                                                   rows_per_z, _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_conv_noise_relu_pool")
    _lib.launch_count += 1
    return out


def conv_mc_relu_pool(layer, x, z, noise: Noise, n_rows, z_rows=None, rows_per_z=1):
    """maxpool2(relu(MNFConv2d(x.repeat(...)))) for n_rows = len(x) * S rows: mean and variance are evaluated once
    per distinct image (z is shared by the call), only the noise / ReLU / pool tail runs per sample.
    z_rows [n_z, c_out] (with z = None): per-sample z, row r scaled by z_rows[r // rows_per_z] (SURVEY 8f-4)."""
    mean, sd = conv_moments(layer, x, z)
    return conv_noise_relu_pool(mean, sd, noise, n_rows, z_rows, rows_per_z)


@torch.no_grad()
def conv_forward_tc(layer, x, z, noise: Noise, z_rows=None, rows_per_z=1):
    """maxpool2(relu(MNFConv2d(x))) on the TF32 tensor cores (implicit GEMM, or im2col + GEMMs for other geometries).
    z_rows [n_z, c_out] (with z = None): per-sample z, image r scaled by z_rows[r // rows_per_z].
    Padding, stride, dilation and groups are not supported here: the tensor-core conv serves MNFLeNet's plain layers."""
    if layer.padding != 0 or layer.stride != 1:
        raise ValueError(f"the tensor-core conv supports padding=0, stride=1 only (got padding={layer.padding}, "
                         f"stride={layer.stride})")
    if layer.dilation != 1 or layer.groups != 1:
        raise ValueError(f"the tensor-core conv supports dilation=1, groups=1 only (got dilation={layer.dilation}, "
                         f"groups={layer.groups})")
    dev = x.device
    R, c_in, H, W = x.shape
    c_out, ks = layer.W_mean.shape[0], layer.W_mean.shape[2]
    OH, OW = H - ks + 1, W - ks + 1
    eps, sid = noise.normal((R, c_out, OH, OW))
    out = torch.empty((R, c_out, OH // 2, OW // 2), device=dev, dtype=torch.float32)
    lib = _lib.lib()
    ws = torch.empty(lib.mnf_conv_tc_workspace(R, c_in, H, W, c_out, ks), device=dev, dtype=torch.float32)
    args = _conv_args(layer, dev)
    with torch.cuda.device(dev):
        rc = lib.mnf_conv2d_forward_tc_z(x.data_ptr(), _p(z), _p(z_rows), rows_per_z, *(a.data_ptr() for a in args),
                                         _p(eps), noise.seed, sid, noise.row_offset, out.data_ptr(), R, c_in, H, W, c_out,
                                         ks, ws.data_ptr(), _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_conv2d_forward_tc")
    _lib.launch_count += 3
    return out


def _kl_fused_plan(layer, conv, dev):
    """Prefilled mnf_kl_fused_args of a layer (every parameter pointer, shapes, flow descriptors), cached while the
    parameters keep their storage; None when the layer is outside the fused entry point's shape class."""
    fq, fr = list(layer.flow_q.flows), list(layer.flow_r.flows)
    names = ("W_mean", "W_log_var", "b_log_var", "q0_mean", "q0_log_var", "r0_c", "r0_b1", "r0_b2") + (() if conv else ("b_mean",))
    tensors = [getattr(layer, n) for n in names]
    for f in fq + fr:
        tensors += [t for m in f.net.linears() for t in (m.weight, m.bias)] + [f.t.weight, f.t.bias, f.s.weight, f.s.bias]
    key = (str(dev), conv, tuple(t.data_ptr() for t in tensors))
    cached = layer.__dict__.get("_kl_plan")
    if cached is not None and cached[0] == key:
        return cached[1]
    plan = None
    n_out, n_in = layer.W_mean.shape[0], layer.W_mean.shape[1]
    ks = layer.W_mean.shape[2] if conv else 1
    dim = n_out if conv else n_in
    ok = (len(fq) <= KL_MAX_FLOWS and len(fr) <= KL_MAX_FLOWS and dim <= 11000
          and all(len(f.net.linears()) == 1 and f.net.linears()[0].out_features <= 64 for f in fq + fr)
          and all(t.device == dev and t.dtype == torch.float32 and t.is_contiguous() for t in tensors))
    if ok:
        a = KlFusedArgs()
        k = a.kl
        k.conv, k.n_out, k.n_in, k.ksize = int(conv), n_out, n_in, ks
        for n in ("W_mean", "W_log_var", "b_log_var", "q0_log_var", "r0_c", "r0_b1", "r0_b2"):
            setattr(k, n, getattr(layer, n).data_ptr())
        k.b_mean = None if conv else layer.b_mean.data_ptr()
        a.q0_mean = layer.q0_mean.data_ptr()
        a.n_flows_q, a.n_flows_r = len(fq), len(fr)
        keep = []
        for i, f in enumerate(fq):
            a.flows[i] = _rnvp_struct(f, dev, keep)[0]
        for i, f in enumerate(fr):
            a.flows[KL_MAX_FLOWS + i] = _rnvp_struct(f, dev, keep)[0]
        fan = n_in * ks * ks
        # Philox stream numbering of a call without a tape (the draw order of kl_div below)
        a.z_stream = 0
        for i in range(len(fq)):
            a.mask_streams[i] = 1 + i
        a.kl.noise_stream = 1 + len(fq)  # eps_w; eps_b (conv) is noise_stream + 1 inside the library
        for i in range(len(fr)):
            a.mask_streams[KL_MAX_FLOWS + i] = 3 + len(fq) + i
        plan = (a, dim, fan, max(n_out, fan), len(fq), len(fr))
    layer.__dict__["_kl_plan"] = (key, plan, {})
    return plan


def _kl_philox_args(layer, plan, stream, out_ptr, dev):
    """The layer's cached argument block pointed at this stream's scratch buffers, a fresh seed and `out_ptr` [5]."""
    a, dim, fan, rows, nq, nr = plan
    scratch = layer.__dict__["_kl_plan"][2]
    buf = scratch.get(stream)
    if buf is None:
        buf = scratch[stream] = torch.empty(2 * dim + 8 + 2 * rows + 64, device=dev, dtype=torch.float32)
    base = buf.data_ptr()
    k = a.kl
    k.z, k.zT, k.ld_q, k.ld_r = base, base + 4 * dim, base + 8 * dim, base + 8 * dim + 4
    k.workspace, k.out = base + 4 * (2 * dim + 8), out_ptr
    k.seed = int(torch.randint(0, 2**62, (1,)).item())  # follows torch.manual_seed
    return a


@torch.no_grad()
def kl_div_multi(layers):
    """Sum of kl_div() over several MNF layers in THREE launches (mnf_kl_div_fused_multi): same draws, same values as
    calling the layers one after the other without a tape.  Returns None when a layer is outside the fused entry point's
    shape class (the caller then loops)."""
    from .mnf_conv import MNFConv2d

    dev = layers[0].W_mean.device
    if dev.type != "cuda" or torch.cuda.is_current_stream_capturing():
        return None
    plans = [_kl_fused_plan(layer, isinstance(layer, MNFConv2d), dev) for layer in layers]
    if any(p is None for p in plans) or any(layer.W_mean.device != dev for layer in layers):
        return None
    stream = _lib.stream_ptr(dev)
    out = torch.empty((len(layers), 5), device=dev, dtype=torch.float32)
    ptrs = (C.POINTER(KlFusedArgs) * len(layers))()
    for i, (layer, plan) in enumerate(zip(layers, plans)):
        ptrs[i] = C.pointer(_kl_philox_args(layer, plan, stream, out.data_ptr() + 20 * i, dev))
    with _lib.on_device(dev):
        rc = _lib.lib().mnf_kl_div_fused_multi(ptrs, len(layers), stream)
    _lib.check(rc, "mnf_kl_div_fused_multi")
    _lib.launch_count += 3 * ((len(layers) + 3) // 4)
    for i, layer in enumerate(layers):
        layer.__dict__["_last_kl_terms"] = out[i]  # kl, kl_W, kl_b, log_q, log_r
    return out[:, 0].sum()


@torch.no_grad()
def kl_div(layer, conv: bool, tape=None):
    """Shared driver of MNFLinear.kl_div / MNFConv2d.kl_div (draw order: SURVEY.md 8c)."""
    dev = layer.W_mean.device
    if dev.type != "cuda":
        raise RuntimeError("torch_mnf (B200) runs only on CUDA parameters (no CPU fallback)")
    plan = _kl_fused_plan(layer, conv, dev)
    if plan is not None and tape is None and not torch.cuda.is_current_stream_capturing():
        # Philox mode, the common call: nothing but the seed and the result buffer changes between calls -- the noise
        # stream numbering (z0 = 0, flow_q masks 1.., eps_w, eps_b, flow_r masks) is fixed by the layer's shape and was
        # written into the cached argument block, the scratch buffers live with it (one set per CUDA stream)
        stream = _lib.stream_ptr(dev)
        out = torch.empty(5, device=dev, dtype=torch.float32)
        a = _kl_philox_args(layer, plan, stream, out.data_ptr(), dev)
        with _lib.on_device(dev):
            rc = _lib.lib().mnf_kl_div_fused(C.byref(a), stream)
        _lib.check(rc, "mnf_kl_div_fused")
        _lib.launch_count += 3
        layer.__dict__["_last_kl_terms"] = out  # kl, kl_W, kl_b, log_q, log_r
        return out[0]
    noise = Noise(tape, dev)
    n_out = layer.W_mean.shape[0]
    n_in = layer.W_mean.shape[1]
    ks = layer.W_mean.shape[2] if conv else 1
    dim = n_out if conv else n_in
    if plan is not None:
        # three launches for the whole call (mnf_kl_div_fused): z0 + flow_q + flow_r in one cluster kernel, the weight
        # pass, the final reduction.  Draw order as below: z0, flow_q masks, eps_w, eps_b, flow_r masks.
        a, dim, fan, rows, nq, nr = plan
        a = KlFusedArgs.from_buffer_copy(a)  # the cached block keeps its Philox defaults
        eps_z, a.z_stream = noise.normal((dim,) if conv else (1, dim))
        a.eps_z = _p(eps_z)
        for i in range(nq):
            m, a.mask_streams[i] = noise.bernoulli((1, dim))
            a.masks[i] = _p(m)
        eps_w, sid = noise.normal((fan,) if conv else (n_out, n_in))
        eps_b = None
        if conv:
            eps_b, _ = noise.normal(())
        else:
            noise._next_stream()
        for i in range(nr):
            m, a.mask_streams[KL_MAX_FLOWS + i] = noise.bernoulli((1, dim))
            a.masks[KL_MAX_FLOWS + i] = _p(m)
        buf = torch.empty(2 * dim + 8 + 2 * rows + 64 + 8, device=dev, dtype=torch.float32)
        base = buf.data_ptr()
        k = a.kl
        k.z, k.zT, k.ld_q, k.ld_r = base, base + 4 * dim, base + 8 * dim, base + 8 * dim + 4
        k.workspace = base + 4 * (2 * dim + 8)
        out = buf[2 * dim + 8 + 2 * rows + 64:2 * dim + 8 + 2 * rows + 64 + 5]
        k.out = out.data_ptr()
        k.eps_w, k.eps_b = _p(eps_w), _p(eps_b)
        k.seed, k.noise_stream = noise.seed, sid
        with _lib.on_device(dev):
            rc = _lib.lib().mnf_kl_div_fused(C.byref(a), _lib.stream_ptr(dev))
        _lib.check(rc, "mnf_kl_div_fused")
        _lib.launch_count += 3
        layer.__dict__["_last_kl_terms"] = out  # kl, kl_W, kl_b, log_q, log_r
        return out[0]
    z = sample_z0(layer.q0_mean, layer.q0_log_var, -1 if conv else 1, noise)  # conv draws randn_like[n_out]
    ld_q, _ = rnvp_stack_inplace(list(layer.flow_q.flows), z, noise)
    fan = n_in * ks * ks
    eps_w, sid = noise.normal((fan,) if conv else (n_out, n_in))
    eps_b = None
    if conv:
        eps_b, _ = noise.normal(())
    else:
        noise._next_stream()  # keep stream numbering identical between the two layer kinds
    zT = z.clone()
    ld_r, _ = rnvp_stack_inplace(list(layer.flow_r.flows), zT, noise)
    rows = max(n_out, fan)
    ws = torch.empty(2 * rows, device=dev, dtype=torch.float32)
    out = torch.empty(5, device=dev, dtype=torch.float32)
    keep = [_param(getattr(layer, n), dev, n) for n in
            ("W_mean", "W_log_var", "b_log_var", "q0_log_var", "r0_c", "r0_b1", "r0_b2")]
    a = KlArgs()
    a.conv, a.n_out, a.n_in, a.ksize = int(conv), n_out, n_in, ks
    a.W_mean, a.W_log_var, a.b_log_var, a.q0_log_var, a.r0_c, a.r0_b1, a.r0_b2 = (t.data_ptr() for t in keep)
    bm = None if conv else _param(layer.b_mean, dev, "b_mean")
    a.b_mean = _p(bm)
    a.z, a.zT, a.ld_q, a.ld_r = z.data_ptr(), zT.data_ptr(), ld_q.data_ptr(), ld_r.data_ptr()
    a.eps_w, a.eps_b = _p(eps_w), _p(eps_b)
    a.seed, a.noise_stream = noise.seed, sid
    a.workspace, a.out = ws.data_ptr(), out.data_ptr()
    with torch.cuda.device(dev):
        rc = _lib.lib().mnf_kl_div(C.byref(a), _lib.stream_ptr(dev))
    _lib.check(rc, "mnf_kl_div")
    _lib.launch_count += 2
    layer.__dict__["_last_kl_terms"] = out  # kl, kl_W, kl_b, log_q, log_r
    return out[0]
