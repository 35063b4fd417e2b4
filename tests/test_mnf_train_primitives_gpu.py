"""The training primitives of csrc/mnf_train.cu, each against a plain fp64 restatement of its operation, at the sizes
where the kernels change how they split the work: the 64 x 64 GEMM tile and its 16-deep k-slice, the 148 * 16 block
cap of the elementwise grid-stride loop (606 208 elements), the 128-block row split of mnf_colsum (8 192 rows), the
64-block row split of mnf_kl_rows_backward (2 048 rows) and the one-warp-per-row kernels at widths around 32.

Two kinds of data:
* exact data -- small integers, so that every fp32 partial sum is representable and the result cannot depend on the
  summation order: the kernel must match fp64 bit for bit.  Only this catches a single dropped or doubled row, tile or
  chunk at a large size;
* random normal data -- |err| <= c * u * m elementwise, u = 2^-24, where m is the fp64 sum of the absolute values of
  the terms that make up the result (|A| |B| for a product) and c = 8 + 4 sqrt(K) for sums of K terms.  A bound relative
  to max |ref| would be flaky or loose once K is large.  Where fp32 rounds a factor such as 1 - sigmoid(20) to 0, the
  bound is the absolute one that the fp64 magnitudes imply."""

import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
U = 2.0**-24
EW_CAP = 148 * 16 * 256  # elements beyond which every elementwise kernel runs its grid-stride loop


def _lib():
    import torch_mnf.layers  # noqa: F401  (registers the training entry points)
    from torch_mnf import _lib

    return _lib


def _call(name, *args):
    lib = _lib()
    rc = getattr(lib.lib(), name)(*args, lib.stream_ptr(torch.device(DEV, torch.cuda.current_device())))
    assert rc == 0, f"{name} returned {rc}: {lib.lib().mnf_last_error()}"


def _p(t):
    return None if t is None else t.data_ptr()


def _c(K):
    return 8 + 4 * math.sqrt(max(K, 1))


def _within(got, ref, mag, c, what):
    """|got - ref| <= c * u * mag elementwise (fp64 ref and mag).  NaN in got fails: the outputs start as NaN, so an
    element the kernel never wrote shows."""
    err = (got.double() - ref).abs()
    bound = c * U * mag
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = int(torch.argmax(bad.flatten().int()))
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the bound; worst at {i}: "
                             f"got {got.flatten()[i].item()!r}, ref {ref.flatten()[i].item()!r}, "
                             f"err {err.flatten()[i].item():.3e} > {bound.flatten()[i].item():.3e}")


def _bitwise(got, ref, what):
    ref32 = ref.float()
    assert torch.equal(ref32.double(), ref), f"{what}: the reference is not exact in fp32"
    if not torch.equal(got, ref32):
        bad = got != ref32
        i = int(torch.argmax(bad.flatten().int()))
        raise AssertionError(f"{what}: {int(bad.sum())} elements differ; first at {i}: got {got.flatten()[i].item()!r}, "
                             f"want {ref32.flatten()[i].item()!r}")


def _ints(shape, lo, hi, g):
    return torch.randint(lo, hi + 1, tuple(shape), device=DEV, generator=g).float()


def _padded(rows, cols, pad, fill=float("nan")):
    """A [rows, cols] view with leading dimension cols + pad of a buffer whose padding holds `fill`."""
    buf = torch.full((max(rows, 1), cols + pad), fill, device=DEV)
    return buf[:rows, :cols]


def _addr(t):
    """Device address of a view's first element -- also for an empty view, where torch's data_ptr() is NULL."""
    return t.untyped_storage().data_ptr() + t.storage_offset() * t.element_size()


# ---- mnf_gemm_f32 -----------------------------------------------------------------------------------------------------
GEMM_M = (1, 63, 64, 65, 1000)
GEMM_N = (1, 63, 64, 65, 257)


def _gemm_case(M, N, K, ta, tb, kind, g, pad):
    """Operands as stored (A [K, M] when ta, B [N, K] when tb) in padded views, filled with exact or random data."""
    a_shape = (K, M) if ta else (M, K)
    b_shape = (N, K) if tb else (K, N)
    A, B = _padded(*a_shape, pad), _padded(*b_shape, pad)
    if kind == "exact":
        A.copy_(_ints(a_shape, -4, 4, g)), B.copy_(_ints(b_shape, -4, 4, g))
        bias, C0 = _ints((N,), -64, 64, g), _ints((M, N), -64, 64, g)
    else:
        A.copy_(torch.randn(a_shape, device=DEV, generator=g)), B.copy_(torch.randn(b_shape, device=DEV, generator=g))
        bias, C0 = torch.randn(N, device=DEV, generator=g), torch.randn(M, N, device=DEV, generator=g)
    opA = (A.t() if ta else A).double()
    opB = (B.t() if tb else B).double()
    return A, B, bias, C0, opA @ opB, opA.abs() @ opB.abs()


@pytest.mark.parametrize("K", [0, 1, 15, 16, 17, 4097])
@pytest.mark.parametrize("kind", ["exact", "random"])
def test_gemm_f32_matches_fp64(K, kind):
    """Every transposition, M and N around the 64-wide tile, K around the 16-deep slice; leading dimensions wider than
    the logical width (NaN in the gap: a read there would poison the result, a write there would show); bias present
    and absent; beta 0, 0.5 and 1.  With beta = 0 a NaN-filled C must not leak into the result (the BLAS contract).
    With K = 0 the result is bias + beta C.  Operands go through the raw ABI as (address, leading dimension)."""
    g = torch.Generator(device=DEV).manual_seed(1000 + K)
    for M in GEMM_M:
        for N in GEMM_N:
            for ta in (False, True):
                for tb in (False, True):
                    pad = max((M + N + K) % 3 * 5, int(K == 0))  # dense and padded leading dimensions
                    A, B, bias, C0, prod, mag = _gemm_case(M, N, K, ta, tb, kind, g, pad)
                    for use_bias in (False, True):
                        for beta in (0.0, 0.5, 1.0):
                            cbuf = torch.full((M, N + 3), -7.0, device=DEV)
                            out = cbuf[:, :N]
                            out.copy_(C0 if beta != 0.0 else torch.full_like(C0, float("nan")))
                            _call("mnf_gemm_f32", int(ta), int(tb), M, N, K, _addr(A), A.stride(0), _addr(B),
                                  B.stride(0), bias.data_ptr() if use_bias else None, beta, _addr(out), out.stride(0))
                            ref = prod + (bias.double() if use_bias else 0.0) + beta * C0.double()
                            what = f"gemm M={M} N={N} K={K} ta={ta} tb={tb} bias={use_bias} beta={beta}"
                            if kind == "exact":
                                _bitwise(out, ref, what)
                            else:
                                m = mag + (bias.double().abs() if use_bias else 0.0) + beta * C0.double().abs()
                                _within(out, ref, m, _c(K), what)
                            assert bool((cbuf[:, N:] == -7.0).all()), f"{what}: wrote past the logical width of C"


# ---- mnf_ew -----------------------------------------------------------------------------------------------------------
EW_SIZES = (1, 255, 257, EW_CAP + 1000)


def _ew_operands(n, ncols, g):
    a = torch.randn(n, device=DEV, generator=g)
    b = torch.randn(n, device=DEV, generator=g)
    c = torch.randn(n, device=DEV, generator=g)
    d = torch.randn(n, device=DEV, generator=g)
    bpos = torch.exp(torch.randn(n, device=DEV, generator=g))  # variances
    bz = torch.where(torch.rand(n, device=DEV, generator=g) < 0.2, torch.zeros_like(b), b)  # exact zeros
    vec_row = torch.randn(ncols, device=DEV, generator=g)  # [col] operands: ncols entries
    vec_row2 = torch.randn(ncols, device=DEV, generator=g)
    vec_col = torch.randn((n + ncols - 1) // ncols, device=DEV, generator=g)  # [row] operand: one entry per row
    return a, b, c, d, bpos, bz, vec_row, vec_row2, vec_col


def _ew_ref(op, n, ncols, a, b, c, d, bpos, bz, vec_row, vec_row2, vec_col):
    """(operands (a, b, c, d), fp64 results, fp64 magnitudes, c) of op; magnitude = the sum of |terms|."""
    A, B, Cc, D = a.double(), b.double(), c.double(), d.double()
    idx = torch.arange(n, device=DEV)
    col, row = idx % ncols, idx // ncols
    if op == 1:
        return (a, b, None, None), [A * B], [(A * B).abs()], 2
    if op == 2:
        r = A * vec_row.double()[col]
        return (a, vec_row, None, None), [r], [r.abs()], 2
    if op == 3:
        return (a, b, c, None), [A + B * Cc], [A.abs() + (B * Cc).abs()], 2
    if op == 4:
        return (a, None, None, None), [A * A], [A * A], 2
    if op == 5:
        return (a, None, None, None), [A.exp()], [A.exp()], 8
    if op == 6:
        r = torch.where(A > 0, A, 0.2 * A)
        return (a, None, None, None), [r], [r.abs()], 2
    if op == 7:
        r = A * torch.where(bz.double() > 0, 1.0, 0.2)
        return (a, bz, None, None), [r], [r.abs()], 2
    if op == 8:
        s = bpos.double().sqrt() * Cc
        return (a, bpos, c, None), [A + s], [A.abs() + s.abs()], 4
    if op == 9:
        r = A * Cc / (2 * bpos.double().sqrt())
        return (a, bpos, c, None), [r], [r.abs()], 4
    if op == 10:
        return (a, b, c, d), [A * Cc + 2 * D * B, A * D], [(A * Cc).abs() + (2 * D * B).abs(), (A * D).abs()], 2
    if op == 11:
        s = (0.5 * vec_row2.double()[col]).exp() * Cc
        r = vec_row.double()[col] + s
        return (vec_row, vec_row2, c, None), [r], [vec_row.double()[col].abs() + s.abs()], 8
    if op == 12:
        r = A * vec_col.double()[row]
        return (a, vec_col, None, None), [r], [r.abs()], 2
    if op == 13:
        return (a, b, c, None), [A + 2 * B * Cc], [A.abs() + (2 * B * Cc).abs()], 2
    if op == 14:
        r = A + vec_col.double()[row]
        return (a, vec_col, None, None), [r], [A.abs() + vec_col.double()[row].abs()], 2
    if op == 15:
        return (a, None, None, None), [A.clamp_min(0)], [A.abs()], 1
    if op == 16:
        r = torch.where(bz.double() > 0, A, 0.0)
        return (a, bz, None, None), [r], [r.abs()], 1
    raise ValueError(op)


BROADCAST_OPS = (2, 11, 12, 14)  # MUL_ROWVEC, Z0, MUL_COLVEC, ADD_COLVEC


@pytest.mark.parametrize("n", EW_SIZES)
@pytest.mark.parametrize("op", range(1, 17))
def test_ew_op_matches_fp64(op, n):
    g = torch.Generator(device=DEV).manual_seed(17 * op + n)
    for ncols in ((1, 3, 32, 257) if op in BROADCAST_OPS else (1,)):
        (a, b, c, d), refs, mags, k = _ew_ref(op, n, ncols, *_ew_operands(n, ncols, g))
        out = torch.full((n,), float("nan"), device=DEV)
        out2 = torch.full((n,), float("nan"), device=DEV) if op == 10 else None
        _call("mnf_ew", op, _p(a), _p(b), _p(c), _p(d), out.data_ptr(), _p(out2), n, ncols)
        for got, ref, mag, what in zip((out, out2), refs, mags, ("out", "out2")):
            _within(got, ref, mag, k, f"ew op {op} n={n} ncols={ncols} {what}")


@pytest.mark.parametrize("slope_op,act", [(7, lambda t: F.leaky_relu(t, 0.2)), (16, torch.relu)])
def test_activation_backward_matches_autograd_at_zero(slope_op, act):
    """LEAKY_BWD / RELU_BWD against torch autograd of leaky_relu(., 0.2) / relu, with pre-activations exactly 0, -0 and
    on either side."""
    pre = torch.tensor([0.0, -0.0, 1e-30, -1e-30, 2.5, -2.5, 0.0, 7.0], device=DEV).repeat(33)
    grad = torch.randn(pre.numel(), device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    x = pre.double().requires_grad_()
    act(x).backward(grad.double())
    out = torch.full_like(grad, float("nan"))
    _call("mnf_ew", slope_op, grad.data_ptr(), pre.data_ptr(), None, None, out.data_ptr(), None, pre.numel(), 1)
    _within(out, x.grad, x.grad.abs(), 2, f"ew op {slope_op} vs autograd")  # 0.2f is not 0.2: 2 u, not 1
    assert torch.equal(out == 0, x.grad == 0)


# ---- mnf_colsum / mnf_rowsum / mnf_swap01 -----------------------------------------------------------------------------
@pytest.mark.parametrize("R", [0, 1, 63, 64, 65, 8191, 8192, 8193, 100003])
def test_colsum_matches_fp64(R):
    """Exact data must give the fp64 sums bit for bit at every row split; random data the summation bound.  R = 0 passes
    the address of an empty view and must give zeros."""
    g = torch.Generator(device=DEV).manual_seed(R)
    for N in (1, 127, 128, 129, 1000):
        for with_b in (False, True):
            for kind in ("exact", "random"):
                shape = (max(R, 1), N)
                if kind == "exact":
                    a, b = _ints(shape, -8, 8, g)[:R], _ints(shape, -4, 4, g)[:R]
                else:
                    a, b = torch.randn(shape, device=DEV, generator=g)[:R], torch.randn(shape, device=DEV, generator=g)[:R]
                b = b if with_b else None
                got = torch.full((N,), float("nan"), device=DEV)
                _call("mnf_colsum", _addr(a), _addr(b) if with_b else None, R, N, got.data_ptr())
                terms = a.double() * (b.double() if with_b else 1.0)
                ref = terms.sum(0)
                what = f"colsum R={R} N={N} b={with_b} {kind}"
                if R == 0:
                    assert torch.equal(got, torch.zeros(N, device=DEV)), what
                elif kind == "exact":
                    _bitwise(got, ref, what)
                else:
                    _within(got, ref, terms.abs().sum(0), _c(R), what)


@pytest.mark.parametrize("cols", [1, 31, 32, 33, 5000])
def test_rowsum_matches_fp64(cols):
    from torch_mnf.layers import _train

    g = torch.Generator(device=DEV).manual_seed(cols)
    for rows in (1, 7, 1000):
        a = _ints((rows, cols), -8, 8, g)
        _bitwise(_train.rowsum(a), a.double().sum(1), f"rowsum exact {rows}x{cols}")
        a = torch.randn(rows, cols, device=DEV, generator=g)
        _within(_train.rowsum(a), a.double().sum(1), a.double().abs().sum(1), _c(cols), f"rowsum {rows}x{cols}")


@pytest.mark.parametrize("d0,d1,inner", [(1, 1, 1), (1, 5, 1), (5, 1, 1), (3, 4, 1), (3, 4, 7), (1, 9, 13), (9, 1, 13),
                                         (64, 33, 1), (7, 130, 33), (300, 41, 57)])
def test_swap01_is_permute(d0, d1, inner):
    from torch_mnf.layers import _train

    t = torch.randn(d0, d1, inner, device=DEV)
    got = _train.swap01(t, d0, d1, inner).view(d1, d0, inner)
    assert torch.equal(got, t.permute(1, 0, 2))


# ---- mnf_rnvp_gate_forward / _backward --------------------------------------------------------------------------------
def _rnvp_ref(z, m, shift, scale, go, gl):
    """fp64 autograd of gate = sigmoid(scale), z' = (1-m) z gate + (1-gate) shift + m z, ld = sum (1-m) log gate."""
    z, shift, scale = (t.double().requires_grad_() for t in (z, shift, scale))
    m = m.double()
    gate = torch.sigmoid(scale)
    zo = (1 - m) * z * gate + (1 - gate) * shift + m * z
    ld = ((1 - m) * torch.log(gate)).sum(1)
    loss = (zo * go.double()).sum() if go is not None else 0.0
    loss = loss + ((ld * gl.double()).sum() if gl is not None else 0.0)
    grads = torch.autograd.grad(loss, (z, shift, scale), allow_unused=True)
    gz, gs, gc = (torch.zeros_like(t) if gr is None else gr for gr, t in zip(grads, (z, shift, scale)))
    return zo.detach(), ld.detach(), gz, gs, gc, gate.detach()


@pytest.mark.parametrize("rows", [1, 7, 4097])
@pytest.mark.parametrize("dim", [1, 31, 32, 33, 256, 1000])
def test_rnvp_gate_matches_fp64_autograd(dim, rows):
    """Random, all-0 and all-1 masks; N(0, 2) scales and scales up to |20| (where fp32 rounds 1 - gate to 0); both
    gradients, and grad_out = NULL or grad_log_det = NULL."""
    g = torch.Generator(device=DEV).manual_seed(dim * 10007 + rows)
    z, shift = torch.randn(rows, dim, device=DEV, generator=g), torch.randn(rows, dim, device=DEV, generator=g)
    go, gl = torch.randn(rows, dim, device=DEV, generator=g), torch.randn(rows, device=DEV, generator=g)
    masks = {"random": torch.bernoulli(torch.full((rows, dim), 0.5, device=DEV), generator=g),
             "zeros": torch.zeros(rows, dim, device=DEV), "ones": torch.ones(rows, dim, device=DEV)}
    scales = {"normal": 2 * torch.randn(rows, dim, device=DEV, generator=g),
              "wide": 40 * torch.rand(rows, dim, device=DEV, generator=g) - 20}
    scales["wide"][0, 0] = 20.0
    for mk, m in masks.items():
        for sk, scale in scales.items():
            what = f"rnvp dim={dim} rows={rows} mask={mk} scale={sk}"
            zo, ld = torch.full_like(z, float("nan")), torch.full((rows,), float("nan"), device=DEV)
            _call("mnf_rnvp_gate_forward", z.data_ptr(), m.data_ptr(), shift.data_ptr(), scale.data_ptr(),
                  zo.data_ptr(), ld.data_ptr(), rows, dim)
            r_zo, r_ld, _, _, _, gate = _rnvp_ref(z, m, shift, scale, go, gl)
            Z, S, M = z.double().abs(), shift.double().abs(), m.double()
            _within(zo, r_zo, Z + S, 8, what + " z_out")
            _within(ld, r_ld, ((1 - M) * (1 + gate.log().abs())).sum(1), _c(dim), what + " log_det")
            for g_out, g_ld in ((go, gl), (go, None), (None, gl)):
                gs, gsc, gz = (torch.full_like(z, float("nan")) for _ in range(3))
                _call("mnf_rnvp_gate_backward", z.data_ptr(), m.data_ptr(), shift.data_ptr(), scale.data_ptr(),
                      _p(g_out), _p(g_ld), gs.data_ptr(), gsc.data_ptr(), gz.data_ptr(), rows, dim)
                _, _, r_gz, r_gs, r_gsc, _ = _rnvp_ref(z, m, shift, scale, g_out, g_ld)
                GO = g_out.double().abs() if g_out is not None else torch.zeros_like(Z)
                GL = (g_ld.double().abs()[:, None] * (1 - M)) if g_ld is not None else torch.zeros_like(Z)
                sub = f"{what} grad_out={'NULL' if g_out is None else 'set'} grad_ld={'NULL' if g_ld is None else 'set'}"
                _within(gs, r_gs, GO, 8, sub + " grad_shift")
                _within(gz, r_gz, GO, 8, sub + " grad_z")
                _within(gsc, r_gsc, GO * (Z + S) + GL, 16, sub + " grad_scale")


# ---- mnf_kl_rows_forward / _backward ----------------------------------------------------------------------------------
def _kl_inputs(n_out, n_in, g):
    z = 1 + 0.3 * torch.randn(n_in, device=DEV, generator=g)
    Wm = 0.5 * torch.randn(n_out, n_in, device=DEV, generator=g)
    Wlv = torch.randn(n_out, n_in, device=DEV, generator=g) - 1
    c = torch.randn(n_in, device=DEV, generator=g)
    eps = torch.randn(n_out, n_in, device=DEV, generator=g)
    return z, Wm, Wlv, c, eps


def _kl_run(z, Wm, Wlv, c, eps, gp, gk):
    n_out, n_in = Wm.shape
    pre, kl = torch.full((n_out,), float("nan"), device=DEV), torch.full((n_out,), float("nan"), device=DEV)
    _call("mnf_kl_rows_forward", z.data_ptr(), Wm.data_ptr(), Wlv.data_ptr(), c.data_ptr(), eps.data_ptr(),
          pre.data_ptr(), kl.data_ptr(), n_out, n_in)
    gWm, gWlv = torch.full_like(Wm, float("nan")), torch.full_like(Wm, float("nan"))
    gz, gc = torch.full_like(z, float("nan")), torch.full_like(z, float("nan"))
    _call("mnf_kl_rows_backward", z.data_ptr(), Wm.data_ptr(), Wlv.data_ptr(), c.data_ptr(), eps.data_ptr(),
          gp.data_ptr(), gk.data_ptr(), gWm.data_ptr(), gWlv.data_ptr(), gz.data_ptr(), gc.data_ptr(), n_out, n_in)
    return pre, kl, gWm, gWlv, gz, gc


@pytest.mark.parametrize("n_in", [1, 127, 128, 129, 1000])
@pytest.mark.parametrize("n_out", [1, 31, 33, 2049, 5000])
def test_kl_rows_match_fp64_autograd(n_out, n_in):
    """pre[j] = sum_i (W_mean z + exp(W_log_var / 2) eps) c_i and klrow[j] = 0.5 sum_i (-W_log_var + exp(W_log_var) +
    (W_mean z)^2 - 1), and their adjoint, against fp64 autograd; also with g_pre = 0, which is what the module passes
    when only kl_rows reaches the loss."""
    g = torch.Generator(device=DEV).manual_seed(n_out * 7919 + n_in)
    z, Wm, Wlv, c, eps = _kl_inputs(n_out, n_in, g)
    gp_rand, gk = torch.randn(n_out, device=DEV, generator=g), torch.randn(n_out, device=DEV, generator=g)
    for gp in (gp_rand, torch.zeros_like(gp_rand)):
        what = f"kl_rows n_out={n_out} n_in={n_in} g_pre={'0' if not gp.any() else 'random'}"
        pre, kl, gWm, gWlv, gz, gc = _kl_run(z, Wm, Wlv, c, eps, gp, gk)
        Z, W, LV, Cc, E = (t.double().requires_grad_() for t in (z, Wm, Wlv, c, eps))
        wm = W * Z
        sd = torch.exp(0.5 * LV)
        r_pre = ((wm + sd * E) * Cc).sum(1)
        r_kl = 0.5 * (-LV + LV.exp() + wm**2 - 1).sum(1)
        GP, GK = gp.double(), gk.double()
        r_gWm, r_gWlv, r_gz, r_gc = torch.autograd.grad((r_pre * GP).sum() + (r_kl * GK).sum(), (W, LV, Z, Cc))
        with torch.no_grad():
            aZ, aW, aC, aE, sdd = Z.abs(), W.abs(), Cc.abs(), E.abs(), sd.detach()
            _within(pre, r_pre.detach(), ((aW * aZ + sdd * aE) * aC).sum(1), _c(n_in), what + " pre")
            _within(kl, r_kl.detach(), 0.5 * (LV.abs() + LV.exp() + wm**2 + 1).sum(1), _c(n_in), what + " kl_rows")
            g_wm = GK.abs()[:, None] * aW * aZ + GP.abs()[:, None] * aC  # |d / d(W_mean z)|
            _within(gWm, r_gWm, g_wm * aZ, 8, what + " grad_W_mean")
            _within(gWlv, r_gWlv, 0.5 * GK.abs()[:, None] * (LV.exp() + 1) + 0.5 * GP.abs()[:, None] * aC * sdd * aE,
                    8, what + " grad_W_log_var")
            _within(gz, r_gz, (g_wm * aW).sum(0), _c(n_out), what + " grad_z")
            _within(gc, r_gc, (GP.abs()[:, None] * (aW * aZ + sdd * aE)).sum(0), _c(n_out), what + " grad_r0_c")


def test_kl_rows_empty_problems():
    """n_out = 0: nothing to write forward, and the adjoint's grad_z / grad_r0_c are zero.  n_in = 0: pre and kl_rows
    are empty sums, 0."""
    lib = _lib()
    buf = torch.zeros(64, device=DEV)
    z, gz, gc = torch.randn(5, device=DEV), torch.full((5,), float("nan"), device=DEV), torch.full((5,), 7.0, device=DEV)
    p = buf.data_ptr()
    _call("mnf_kl_rows_forward", z.data_ptr(), p, p, z.data_ptr(), p, p, p, 0, 5)
    _call("mnf_kl_rows_backward", z.data_ptr(), p, p, z.data_ptr(), p, p, p, p, p, gz.data_ptr(), gc.data_ptr(), 0, 5)
    assert torch.equal(gz, torch.zeros(5, device=DEV)) and torch.equal(gc, torch.zeros(5, device=DEV))
    pre, kl = torch.full((3,), float("nan"), device=DEV), torch.full((3,), float("nan"), device=DEV)
    _call("mnf_kl_rows_forward", p, p, p, p, p, pre.data_ptr(), kl.data_ptr(), 3, 0)
    assert torch.equal(pre, torch.zeros(3, device=DEV)) and torch.equal(kl, torch.zeros(3, device=DEV))
    _call("mnf_kl_rows_backward", p, p, p, p, p, p, p, p, p, p, p, 3, 0)
    _call("mnf_kl_rows_forward", p, p, p, p, p, p, p, 0, 0)
    torch.cuda.synchronize()
    assert lib.lib().mnf_kl_rows_forward(p, p, p, p, p, p, p, -1, 0, None) == -1
