"""Training path of the MNF layers: autograd Functions over the exact-fp32 primitives of csrc/mnf_train.cu
(include/mnf_b200.h, "Training path").  The reference differentiates MNFLinear.forward / kl_div with torch autograd
(tests/test_mnf_mnist.py:28-43); here every matrix product, the RNVP update, the local-reparameterisation output and
the weight-sized KL terms have hand-written forward and backward kernels, torch autograd only links them and handles
the O(n) vector glue (bias KL, r(z|W) moments).

Noise is materialised in this mode (a tape, or torch's CUDA generator) so that backward sees the draws forward used;
the draw order is the reference's (SURVEY.md 8c)."""

from __future__ import annotations

import ctypes as C

import torch

from .. import _lib

_vp, _i64, _int, _f = C.c_void_p, C.c_int64, C.c_int, C.c_float
_lib.register({
    "mnf_gemm_f32": (_int, [_int, _int, _i64, _int, _int, _vp, _i64, _vp, _i64, _vp, _f, _vp, _i64, _vp]),
    "mnf_gemm_f32_batched": (_int, [_int, _int, _int, _i64, _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _f, _vp,
                                    _i64, _i64, _vp]),
    "mnf_ew": (_int, [_int, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "mnf_colsum": (_int, [_vp, _vp, _i64, _int, _vp, _vp]),
    "mnf_rnvp_gate_forward": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "mnf_rnvp_gate_backward": (_int, [_vp] * 9 + [_i64, _int, _vp]),
    "mnf_kl_rows_forward": (_int, [_vp] * 7 + [_int, _int, _vp]),
    "mnf_kl_rows_backward": (_int, [_vp] * 11 + [_int, _int, _vp]),
    "mnf_im2col_t": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _vp]),
    "mnf_col2im_t": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _vp]),
    "mnf_im2col_t_ps": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_col2im_t_ps": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_im2col_t_geom": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_col2im_t_geom": (_int, [_vp, _vp, _i64, _int, _int, _int, _int, _int, _int, _int, _vp]),
    "mnf_swap01": (_int, [_vp, _vp, _i64, _i64, _i64, _vp]),
    "mnf_rowsum": (_int, [_vp, _i64, _i64, _vp, _vp]),
})

EW_MUL, EW_MUL_ROWVEC, EW_FMA, EW_SQUARE, EW_EXP, EW_LEAKY, EW_LEAKY_BWD, EW_NOISE_OUT, EW_GVAR, EW_LIN_IN_BWD, EW_Z0 = range(1, 12)
EW_MUL_COLVEC, EW_ADD_2MUL, EW_ADD_COLVEC, EW_RELU, EW_RELU_BWD = 12, 13, 14, 15, 16


def _p(t):
    return None if t is None else t.data_ptr()


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


def needs_grad(module, *tensors) -> bool:
    return torch.is_grad_enabled() and (
        any(t is not None and t.requires_grad for t in tensors) or any(p.requires_grad for p in module.parameters()))


class DeviceTape:
    """Noise source of the training path when no tape is injected: torch's generator on the layer's device."""

    def __init__(self, device):
        self.device = device

    def normal(self, shape):
        return torch.randn(tuple(shape), device=self.device, dtype=torch.float32)

    def bernoulli(self, shape):
        return torch.bernoulli(torch.full(tuple(shape), 0.5, device=self.device, dtype=torch.float32))


def _tape(noise, device):
    from . import _mnf_ops as ops

    if isinstance(noise, ops.Noise):
        noise = noise.tape
    return noise if noise is not None else DeviceTape(device)


def _draw(tape, kind, shape, device):
    return getattr(tape, kind)(tuple(shape)).to(device, torch.float32).contiguous()


# ------------------------------------------------------------------------------------------------------------------
# raw primitive launches
# ------------------------------------------------------------------------------------------------------------------
def gemm(A, B, trans_a=False, trans_b=False, bias=None, out=None, beta=0.0):
    """op(A) @ op(B) + bias + beta*out with A, B as stored (row-major 2-D, unit inner stride)."""
    M, K = (A.shape[1], A.shape[0]) if trans_a else A.shape
    N = B.shape[0] if trans_b else B.shape[1]
    if out is None:
        out = torch.empty((M, N), device=A.device, dtype=torch.float32)
    with torch.cuda.device(A.device):
        rc = _lib.lib().mnf_gemm_f32(int(trans_a), int(trans_b), M, N, K, A.data_ptr(), A.stride(0), B.data_ptr(),
                                     B.stride(0), _p(bias), float(beta), out.data_ptr(), out.stride(0),
                                     _lib.stream_ptr(A.device))
    _lib.check(rc, "mnf_gemm_f32")
    _lib.launch_count += 1
    return out


def gemm_grouped(A, B, groups, trans_a=False, trans_b=False):
    """The block-diagonal product of a grouped convolution: A and B are split along their rows into `groups` equal
    blocks and out[block g] = op(A_g) @ op(B_g), all blocks in one launch (mnf_gemm_f32_batched).  groups = 1 is
    gemm(A, B, trans_a, trans_b)."""
    if groups == 1:
        return gemm(A, B, trans_a=trans_a, trans_b=trans_b)
    ra, rb = A.shape[0] // groups, B.shape[0] // groups  # rows of one block of A and of B as stored
    M, K = (A.shape[1], ra) if trans_a else (ra, A.shape[1])
    N = rb if trans_b else B.shape[1]
    out = torch.empty((groups * M, N), device=A.device, dtype=torch.float32)
    with torch.cuda.device(A.device):
        rc = _lib.lib().mnf_gemm_f32_batched(int(trans_a), int(trans_b), groups, M, N, K, A.data_ptr(), A.stride(0),
                                             ra * A.stride(0), B.data_ptr(), B.stride(0), rb * B.stride(0), None, 0.0,
                                             out.data_ptr(), out.stride(0), M * out.stride(0), _lib.stream_ptr(A.device))
    _lib.check(rc, "mnf_gemm_f32_batched")
    _lib.launch_count += 1
    return out


def ew(op, a, b=None, c=None, d=None, ncols=1, two=False):
    out = torch.empty_like(a)
    out2 = torch.empty_like(a) if two else None
    with torch.cuda.device(a.device):
        rc = _lib.lib().mnf_ew(op, a.data_ptr(), _p(b), _p(c), _p(d), out.data_ptr(), _p(out2), a.numel(), ncols,
                               _lib.stream_ptr(a.device))
    _lib.check(rc, "mnf_ew")
    _lib.launch_count += 1
    return (out, out2) if two else out


def colsum(a, b=None):
    R, N = a.shape
    out = torch.empty(N, device=a.device, dtype=torch.float32)
    with torch.cuda.device(a.device):
        rc = _lib.lib().mnf_colsum(a.data_ptr(), _p(b), R, N, out.data_ptr(), _lib.stream_ptr(a.device))
    _lib.check(rc, "mnf_colsum")
    _lib.launch_count += 1
    return out


def _call(name, *args, device):
    with torch.cuda.device(device):
        rc = getattr(_lib.lib(), name)(*args, _lib.stream_ptr(device))
    _lib.check(rc, name)
    _lib.launch_count += 1


def _conv_out(n, ks, pad, stride, dilation=1):
    return (n + 2 * pad - dilation * (ks - 1) - 1) // stride + 1


def im2col_t(x, ks, pad=0, stride=1, dilation=1):
    R, c_in, H, W = x.shape
    P = R * _conv_out(H, ks, pad, stride, dilation) * _conv_out(W, ks, pad, stride, dilation)
    out = torch.empty((c_in * ks * ks, P), device=x.device, dtype=torch.float32)
    if dilation == 1:
        _call("mnf_im2col_t_ps", x.data_ptr(), out.data_ptr(), R, c_in, H, W, ks, pad, stride, device=x.device)
    else:
        _call("mnf_im2col_t_geom", x.data_ptr(), out.data_ptr(), R, c_in, H, W, ks, pad, stride, dilation,
              device=x.device)
    return out


def col2im_t(g_cols_t, shape, ks, pad=0, stride=1, dilation=1):
    R, c_in, H, W = shape
    out = torch.empty(shape, device=g_cols_t.device, dtype=torch.float32)
    if dilation == 1:
        _call("mnf_col2im_t_ps", g_cols_t.data_ptr(), out.data_ptr(), R, c_in, H, W, ks, pad, stride,
              device=g_cols_t.device)
    else:
        _call("mnf_col2im_t_geom", g_cols_t.data_ptr(), out.data_ptr(), R, c_in, H, W, ks, pad, stride, dilation,
              device=g_cols_t.device)
    return out


def swap01(t, d0, d1, inner):
    """[d0, d1, inner] -> [d1, d0, inner] (contiguous copy)."""
    out = torch.empty(d1 * d0 * inner, device=t.device, dtype=torch.float32)
    _call("mnf_swap01", t.data_ptr(), out.data_ptr(), d0, d1, inner, device=t.device)
    return out


def rowsum(a):
    out = torch.empty(a.size(0), device=a.device, dtype=torch.float32)
    _call("mnf_rowsum", a.data_ptr(), a.size(0), a.size(1), out.data_ptr(), device=a.device)
    return out


# ------------------------------------------------------------------------------------------------------------------
# autograd Functions
# ------------------------------------------------------------------------------------------------------------------
class LinearFn(torch.autograd.Function):
    """a @ W.T + b (nn.Linear) on mnf_gemm_f32; backward = dgrad + wgrad GEMMs and a column sum."""

    @staticmethod
    def forward(ctx, a, W, b):
        a, W = _c(a), _c(W)
        ctx.save_for_backward(a, W)
        return gemm(a, W, trans_b=True, bias=b)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        a, W = ctx.saved_tensors
        g = _c(g)
        ga = gemm(g, W) if ctx.needs_input_grad[0] else None
        gW = gemm(g, a, trans_a=True) if ctx.needs_input_grad[1] else None
        gb = colsum(g) if ctx.needs_input_grad[2] else None
        return ga, gW, gb


class MulFn(torch.autograd.Function):
    """a * m for a fixed 0/1 mask m (RNVP's z2 = mask * z, rnvp.py:30)."""

    @staticmethod
    def forward(ctx, a, m):
        ctx.save_for_backward(m)
        return ew(EW_MUL, _c(a), m)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        (m,) = ctx.saved_tensors
        return ew(EW_MUL, _c(g), m), None


class LeakyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a):
        a = _c(a)
        ctx.save_for_backward(a)
        return ew(EW_LEAKY, a)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        (a,) = ctx.saved_tensors
        return ew(EW_LEAKY_BWD, _c(g), a)


class ReluFn(torch.autograd.Function):
    """nn.ReLU between the MaskedLinear layers of a standalone MADE (made.py:43)."""

    @staticmethod
    def forward(ctx, a):
        a = _c(a)
        ctx.save_for_backward(a)
        return ew(EW_RELU, a)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        (a,) = ctx.saved_tensors
        return ew(EW_RELU_BWD, _c(g), a)


class SampleZ0Fn(torch.autograd.Function):
    """q0_mean + exp(q0_log_var / 2) * eps (mnf_linear.py:61-64)."""

    @staticmethod
    def forward(ctx, q0_mean, q0_log_var, eps):
        ctx.save_for_backward(q0_log_var, eps)
        return _z0(q0_mean, q0_log_var, eps)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        q0_log_var, eps = ctx.saved_tensors
        g = _c(g)
        g_mean = colsum(g)
        g_lv = colsum(g, eps) * (0.5 * torch.exp(0.5 * q0_log_var))
        return g_mean, g_lv, None


def _z0(q0_mean, q0_log_var, eps):
    out = torch.empty_like(eps)
    with torch.cuda.device(eps.device):
        rc = _lib.lib().mnf_ew(EW_Z0, _c(q0_mean).data_ptr(), _c(q0_log_var).data_ptr(), eps.data_ptr(), None,
                               out.data_ptr(), None, eps.numel(), eps.size(-1), _lib.stream_ptr(eps.device))
    _lib.check(rc, "mnf_ew")
    _lib.launch_count += 1
    return out


class RnvpGateFn(torch.autograd.Function):
    """(z, mask, shift, scale) -> (z_out, log_det) of rnvp.py:33-40."""

    @staticmethod
    def forward(ctx, z, mask, shift, scale):
        z, shift, scale = _c(z), _c(shift), _c(scale)
        R, n = z.shape
        z_out = torch.empty_like(z)
        ld = torch.empty(R, device=z.device, dtype=torch.float32)
        with torch.cuda.device(z.device):
            rc = _lib.lib().mnf_rnvp_gate_forward(z.data_ptr(), mask.data_ptr(), shift.data_ptr(), scale.data_ptr(),
                                                  z_out.data_ptr(), ld.data_ptr(), R, n, _lib.stream_ptr(z.device))
        _lib.check(rc, "mnf_rnvp_gate_forward")
        _lib.launch_count += 1
        ctx.save_for_backward(z, mask, shift, scale)
        return z_out, ld

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_out, g_ld):
        z, mask, shift, scale = ctx.saved_tensors
        R, n = z.shape
        g_out = _c(g_out) if g_out is not None else None
        g_ld = _c(g_ld) if g_ld is not None else None
        g_shift, g_scale, g_z = torch.empty_like(z), torch.empty_like(z), torch.empty_like(z)
        with torch.cuda.device(z.device):
            rc = _lib.lib().mnf_rnvp_gate_backward(z.data_ptr(), mask.data_ptr(), shift.data_ptr(), scale.data_ptr(),
                                                   _p(g_out), _p(g_ld), g_shift.data_ptr(), g_scale.data_ptr(),
                                                   g_z.data_ptr(), R, n, _lib.stream_ptr(z.device))
        _lib.check(rc, "mnf_rnvp_gate_backward")
        _lib.launch_count += 1
        return g_z, None, g_shift, g_scale


class MnfLinearOutFn(torch.autograd.Function):
    """mean = (x*z) W_mean^T + b_mean, var = x^2 exp(W_log_var)^T + exp(b_log_var), out = mean + sqrt(var) eps
    (mnf_linear.py:47-57) with a hand-written adjoint."""

    @staticmethod
    def forward(ctx, x, z, W_mean, W_log_var, b_mean, b_log_var, eps):
        x, z, W_mean, W_log_var = _c(x), _c(z), _c(W_mean), _c(W_log_var)
        xz = ew(EW_MUL, x, z)
        x2 = ew(EW_SQUARE, x)
        Wv = ew(EW_EXP, W_log_var)
        bv = ew(EW_EXP, _c(b_log_var))
        mean = gemm(xz, W_mean, trans_b=True, bias=b_mean)
        var = gemm(x2, Wv, trans_b=True, bias=bv)
        ctx.save_for_backward(x, z, W_mean, xz, x2, Wv, bv, var, eps)
        return ew(EW_NOISE_OUT, mean, var, eps)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, z, W_mean, xz, x2, Wv, bv, var, eps = ctx.saved_tensors
        g = _c(g)
        g_var = ew(EW_GVAR, g, var, eps)
        gW_mean = gemm(g, xz, trans_a=True)
        gW_lv = ew(EW_MUL, gemm(g_var, x2, trans_a=True), Wv)
        gb_mean = colsum(g)
        gb_lv = ew(EW_MUL, colsum(g_var), bv)
        gxz = gemm(g, W_mean)
        gx2 = gemm(g_var, Wv)
        gx, gz = ew(EW_LIN_IN_BWD, gxz, gx2, z, x, two=True)
        return (gx if ctx.needs_input_grad[0] else None), gz, gW_mean, gW_lv, gb_mean, gb_lv, None


class KlRowsFn(torch.autograd.Function):
    """(z [n_in], W_mean, W_log_var, r0_c, eps_w) -> (pre [n_out], kl_rows [n_out]): the weight-sized part of
    MNFLinear.kl_div (mnf_linear.py:67-79)."""

    @staticmethod
    def forward(ctx, z, W_mean, W_log_var, r0_c, eps_w):
        z, W_mean, W_log_var, r0_c = _c(z), _c(W_mean), _c(W_log_var), _c(r0_c)
        n_out, n_in = W_mean.shape
        pre = torch.empty(n_out, device=z.device, dtype=torch.float32)
        kl_rows = torch.empty_like(pre)
        with torch.cuda.device(z.device):
            rc = _lib.lib().mnf_kl_rows_forward(z.data_ptr(), W_mean.data_ptr(), W_log_var.data_ptr(), r0_c.data_ptr(),
                                                eps_w.data_ptr(), pre.data_ptr(), kl_rows.data_ptr(), n_out, n_in,
                                                _lib.stream_ptr(z.device))
        _lib.check(rc, "mnf_kl_rows_forward")
        _lib.launch_count += 1
        ctx.save_for_backward(z, W_mean, W_log_var, r0_c, eps_w)
        return pre, kl_rows

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_pre, g_kl):
        z, W_mean, W_log_var, r0_c, eps_w = ctx.saved_tensors
        n_out, n_in = W_mean.shape
        zeros = torch.zeros(n_out, device=z.device, dtype=torch.float32)
        g_pre = _c(g_pre) if g_pre is not None else zeros
        g_kl = _c(g_kl) if g_kl is not None else zeros
        gWm, gWlv = torch.empty_like(W_mean), torch.empty_like(W_mean)
        gz, gc = torch.empty_like(z), torch.empty_like(z)
        with torch.cuda.device(z.device):
            rc = _lib.lib().mnf_kl_rows_backward(z.data_ptr(), W_mean.data_ptr(), W_log_var.data_ptr(), r0_c.data_ptr(),
                                                 eps_w.data_ptr(), g_pre.data_ptr(), g_kl.data_ptr(), gWm.data_ptr(),
                                                 gWlv.data_ptr(), gz.data_ptr(), gc.data_ptr(), n_out, n_in,
                                                 _lib.stream_ptr(z.device))
        _lib.check(rc, "mnf_kl_rows_backward")
        _lib.launch_count += 1
        return gz, gWm, gWlv, gc, None


# ------------------------------------------------------------------------------------------------------------------
# layer-level training paths
# ------------------------------------------------------------------------------------------------------------------
def rnvp_flow(flow, z, mask):
    """RNVP.forward (rnvp.py:26-40) -> (z_out, log_det[R])."""
    from .._program import check_leaky

    check_leaky(flow.net)
    y = MulFn.apply(z, mask)
    lins = flow.net.linears()
    for i, lin in enumerate(lins):
        y = LinearFn.apply(y, lin.weight, lin.bias)
        if i + 1 < len(lins):
            y = LeakyFn.apply(y)
    shift = LinearFn.apply(y, flow.t.weight, flow.t.bias)
    scale = LinearFn.apply(y, flow.s.weight, flow.s.bias)
    return RnvpGateFn.apply(z, mask, shift, scale)


def rnvp_stack(flows, z, tape):
    ld = None
    for f in flows:
        mask = _draw(tape, "bernoulli", z.shape, z.device)
        z, l = rnvp_flow(f, z, mask)
        ld = l if ld is None else ld + l
    if ld is None:
        ld = torch.zeros(z.size(0), device=z.device)
    return z, ld


def sample_z(layer, n_rows, tape, dim):
    """(z_T [n_rows, dim], log_det_q [n_rows]) of MNFLinear.sample_z / MNFConv2d.sample_z."""
    dev = layer.W_mean.device
    eps = _draw(tape, "normal", (n_rows, dim) if n_rows != -1 else (dim,), dev).reshape(max(n_rows, 1), dim)
    z0 = SampleZ0Fn.apply(layer.q0_mean, layer.q0_log_var, eps)
    return rnvp_stack(list(layer.flow_q.flows), z0, tape)


def linear_forward(layer, x, noise=None, relu=False):
    """MNFLinear.forward (mnf_linear.py:47-57), differentiable."""
    x = _lib.require_cuda_f32(x, "input")
    tape = _tape(noise, x.device)
    z, _ = sample_z(layer, x.size(0), tape, layer.n_in)
    eps = _draw(tape, "normal", (x.size(0), layer.n_out), x.device)
    out = MnfLinearOutFn.apply(x, z, layer.W_mean, layer.W_log_var, layer.b_mean, layer.b_log_var, eps)
    return torch.relu(out) if relu else out


def linear_kl_div(layer, noise=None):
    """MNFLinear.kl_div (mnf_linear.py:66-90), differentiable.  The [n_out, n_in]-sized work runs in the kl_rows
    kernels; the vector-sized glue (bias KL, r(z|W) moments) is left to torch."""
    dev = layer.W_mean.device
    if dev.type != "cuda":
        raise RuntimeError("torch_mnf (B200) runs only on CUDA parameters (no CPU fallback)")
    tape = _tape(noise, dev)
    z, ld_q = sample_z(layer, 1, tape, layer.n_in)
    eps_w = _draw(tape, "normal", (layer.n_out, layer.n_in), dev)
    pre, kl_rows = KlRowsFn.apply(z[0], layer.W_mean, layer.W_log_var, layer.r0_c, eps_w)
    kl_W = kl_rows.sum()
    kl_b = 0.5 * torch.sum(-layer.b_log_var + layer.b_log_var.exp() + layer.b_mean**2 - 1)
    log_q = -ld_q.squeeze() - 0.5 * layer.q0_log_var.sum()
    a = torch.tanh(pre).mean()
    mean_r, log_var_r = layer.r0_b1 * a, layer.r0_b2 * a
    z_r, ld_r = rnvp_stack(list(layer.flow_r.flows), z, tape)
    log_r = ld_r.squeeze() + 0.5 * torch.sum(-log_var_r.exp() * (z_r[0] - mean_r) ** 2 + log_var_r)
    return kl_W + kl_b + log_q - log_r


# ------------------------------------------------------------------------------------------------------------------
# MNFConv2d
# ------------------------------------------------------------------------------------------------------------------
class MnfConvOutFn(torch.autograd.Function):
    """mean = conv(x, W_mean * z[c]), var = conv(x^2, exp(W_log_var)) + exp(b_log_var), out = mean + sqrt(var) eps
    (mnf_conv.py:68-79) as im2col GEMMs in the [c_out, R*OH*OW] layout, with a hand-written adjoint.  pad / stride /
    dilation / groups: geometry of the convolution (plain ints, no gradient).  With groups, the rows of the im2col
    matrix and of the weights split into per-group blocks and every product is a batched, block-diagonal GEMM."""

    @staticmethod
    def forward(ctx, x, z, W_mean, W_log_var, b_log_var, eps, pad=0, stride=1, dilation=1, groups=1):
        x, z = _c(x), _c(z)
        R, c_in, H, W = x.shape
        c_out, ks = W_mean.shape[0], W_mean.shape[2]
        S = _conv_out(H, ks, pad, stride, dilation) * _conv_out(W, ks, pad, stride, dilation)
        fan = (c_in // groups) * ks * ks
        cols = im2col_t(x, ks, pad, stride, dilation)
        cols2 = ew(EW_SQUARE, cols)
        Wm = _c(W_mean).view(c_out, fan)
        Wz = ew(EW_MUL_COLVEC, Wm, z, ncols=fan)
        Wv = ew(EW_EXP, _c(W_log_var).view(c_out, fan))
        bv = ew(EW_EXP, _c(b_log_var))
        mean = swap01(gemm_grouped(Wz, cols, groups), c_out, R, S).view(eps.shape)
        var_t = ew(EW_ADD_COLVEC, gemm_grouped(Wv, cols2, groups), bv, ncols=R * S)
        var = swap01(var_t, c_out, R, S).view(eps.shape)
        ctx.save_for_backward(z, Wm, cols, cols2, Wz, Wv, bv, var, eps)
        ctx.geom = (tuple(x.shape), ks, W_mean.shape, pad, stride, dilation, groups)
        return ew(EW_NOISE_OUT, mean, var, eps)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        z, Wm, cols, cols2, Wz, Wv, bv, var, eps = ctx.saved_tensors
        xshape, ks, wshape, pad, stride, dilation, groups = ctx.geom
        R, c_out = xshape[0], wshape[0]
        P = cols.shape[1]
        S = P // R
        g = _c(g)
        g_var = ew(EW_GVAR, g, var, eps)
        g_t = swap01(g, R, c_out, S).view(c_out, P)
        gv_t = swap01(g_var, R, c_out, S).view(c_out, P)
        gWz = gemm_grouped(g_t, cols, groups, trans_b=True)
        gW_mean = ew(EW_MUL_COLVEC, gWz, z, ncols=Wm.shape[1]).view(wshape)
        gz = rowsum(ew(EW_MUL, gWz, Wm))
        gW_lv = ew(EW_MUL, gemm_grouped(gv_t, cols2, groups, trans_b=True), Wv).view(wshape)
        gb_lv = ew(EW_MUL, rowsum(gv_t), bv)
        gx = None
        if ctx.needs_input_grad[0]:
            g_cols = ew(EW_ADD_2MUL, gemm_grouped(Wz, g_t, groups, trans_a=True),
                        gemm_grouped(Wv, gv_t, groups, trans_a=True), cols)
            gx = col2im_t(g_cols, xshape, ks, pad, stride, dilation)
        return gx, gz, gW_mean, gW_lv, gb_lv, None, None, None, None, None


def conv_forward(layer, x, noise=None, relu_pool=False):
    """MNFConv2d.forward (mnf_conv.py:67-79), differentiable."""
    x = _lib.require_cuda_f32(x, "input")
    tape = _tape(noise, x.device)
    z, _ = sample_z(layer, -1, tape, layer.n_out)
    OH, OW = layer.output_size(x.size(2), x.size(3))
    eps = _draw(tape, "normal", (x.size(0), layer.n_out, OH, OW), x.device)
    out = MnfConvOutFn.apply(x, z[0], layer.W_mean, layer.W_log_var, layer.b_log_var, eps, layer.padding, layer.stride,
                             layer.dilation, layer.groups)
    return torch.nn.functional.max_pool2d(torch.relu(out), 2) if relu_pool else out


def conv_kl_div(layer, noise=None):
    """MNFConv2d.kl_div (mnf_conv.py:90-133), differentiable.  The flows and the two r0_c contractions run on the
    CUDA primitives; the remaining terms are elementwise over the (small) conv weights and left to torch."""
    dev = layer.W_mean.device
    if dev.type != "cuda":
        raise RuntimeError("torch_mnf (B200) runs only on CUDA parameters (no CPU fallback)")
    tape = _tape(noise, dev)
    n_out = layer.n_out
    z, ld_q = sample_z(layer, -1, tape, n_out)
    W_var, b_var = layer.W_log_var.exp(), layer.b_log_var.exp()
    Wz = layer.W_mean * z.view(-1, 1, 1, 1)
    kl_W = 0.5 * torch.sum(-layer.W_log_var + W_var + Wz**2 - 1)
    kl_b = 0.5 * torch.sum(-layer.b_log_var + b_var - 1)  # the reference's b_mean is a fixed zero
    log_q = -ld_q.squeeze() - 0.5 * layer.q0_log_var.sum()
    c_row = layer.r0_c.view(1, -1)
    act_mean = LinearFn.apply(Wz.reshape(-1, n_out), c_row, None)[:, 0]            # eq. (11)
    act_std = LinearFn.apply(W_var.sqrt().reshape(-1, n_out), c_row, None)[:, 0]   # eq. (12)
    eps_w = _draw(tape, "normal", act_std.shape, dev)
    act = act_mean + act_std * eps_w
    eps_b = _draw(tape, "normal", (), dev)
    act = act + torch.sum(b_var * layer.r0_c**2).sqrt() * eps_b
    a = act.mean()
    mean_r, log_var_r = layer.r0_b1 * a, layer.r0_b2 * a
    z_r, ld_r = rnvp_stack(list(layer.flow_r.flows), z, tape)
    log_r = ld_r.squeeze() + 0.5 * torch.sum(-log_var_r.exp() * (z_r[0] - mean_r) ** 2 + log_var_r)
    return kl_W + kl_b + log_q - log_r
