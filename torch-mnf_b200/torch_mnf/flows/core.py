"""Flow containers (reference: flows/core.py:10-55), fused into one CUDA launch per call."""

from __future__ import annotations

import math
from collections.abc import Sequence

import torch
from torch import Tensor, nn
from torch.distributions import Distribution, Independent, MultivariateNormal, Normal

from .. import _lib
from .._program import FlowProgram, state_without_caches
from ._base import Flow


class NormalizingFlow(nn.Module):
    """A sequence of flows.  ``forward`` / ``inverse`` return ``(list, log_det[B])`` where the
    list holds the input followed by the output of every flow (core.py:17-35).

    All flows run in ONE kernel launch: the point stays in registers from the first flow to
    the last and the log-det is accumulated on chip.  ``return_intermediates=False`` (an
    additive option) skips writing the per-flow outputs to HBM; the list is then
    ``[input, final]`` so ``xs[-1]`` / ``zs[-1]`` keep working.

    Stacks made only of ``RNVP`` flows (the MNF q/r flows) go through the MNF RNVP kernel and
    accept a ``noise`` tape for their Bernoulli masks.
    """

    def __init__(self, flows: Sequence[nn.Module], return_intermediates: bool = True) -> None:
        super().__init__()
        self.flows = nn.ModuleList(flows)
        self.return_intermediates = return_intermediates
        self.__dict__["_prog"] = None

    __getstate__ = state_without_caches  # copy.deepcopy / pickle drop the launch caches (ctypes descriptors)

    def _flow_list(self) -> list:
        """The flows as a plain list (read from the module dicts directly: nn.Module.__getattr__ is on every
        small-batch call's critical path)."""
        return list(self._modules["flows"]._modules.values())

    def _program(self) -> FlowProgram:
        prog = self.__dict__.get("_prog")
        flows = self._flow_list()
        if prog is None or prog.flows != flows:  # (list comparison: identity first, no __eq__ on nn.Module)
            for f in flows:
                if not isinstance(f, Flow):
                    raise TypeError(f"{type(f).__name__} is not a torch_mnf flow")
            prog = FlowProgram(flows)
            self.__dict__["_prog"] = prog
        return prog

    def _is_rnvp_stack(self) -> bool:
        from .rnvp import RNVP

        return len(self.flows) > 0 and all(isinstance(f, RNVP) for f in self.flows)

    def _maf_density_stack(self, v: Tensor, inverse: bool, log_prob_only: bool = False, out=None):
        """Stacks made only of MAF (inverse) / IAF (forward) flows in their one-pass direction take a tensor-core
        path when eligible (flows/maf.py::_tc_mode): the fused persistent tcgen05 kernel for dim-64 stacks, the
        per-layer TF32 GEMM chain otherwise.  -> (outputs list, log_det, log_prob or None) or None."""
        from .maf import IAF, MAF, density_stack

        flows = self._flow_list()
        if not flows or not all(isinstance(f, MAF) for f in flows):
            return None
        if any(isinstance(f, IAF) != (not inverse) for f in flows):
            return None
        order = flows[::-1] if inverse else flows
        got = density_stack(order, v, self.__dict__, want_inter=self.return_intermediates and not log_prob_only,
                            want_z=not log_prob_only, want_log_prob=log_prob_only,
                            log_prob_out=out if (out is not None and out.is_contiguous()) else None)
        if got is None:
            return None
        z, ld, inter, lp = got
        if log_prob_only:
            if out is not None and lp is not out:
                out.copy_(lp)
                lp = out
            return None, ld, lp
        outs = [v] + (list(inter.unbind(0)) if inter is not None else [z])
        return outs, ld, None

    def _data_dependent_init(self, v: Tensor, inverse: bool) -> None:
        """ActNorm initialises itself from the first batch IT sees, i.e. the output of the flows that run before
        it in this direction (affine_constant_flow.py:42-50 inside core.py:30-33's loop).  Flows with a pending
        init get that input from a one-off run of the preceding sub-stack."""
        order = self._flow_list()
        if inverse:
            order.reverse()
        for i, f in enumerate(order):
            pending = getattr(f, "_init_pending", None)
            if pending is None or not pending(inverse):
                continue
            inp = v.detach()
            if i > 0:
                head = order[:i][::-1] if inverse else order[:i]
                with torch.no_grad():
                    inp = FlowProgram(head).run(inp, inverse)[0]
            f._before_run(inp, inverse)

    def _run(self, v: Tensor, inverse: bool, want_lp: bool = False):
        if not want_lp:
            got = self._maf_density_stack(v, inverse)
            if got is not None:
                return got[0], got[1], None
        self._data_dependent_init(v, inverse)
        prog = self._program()
        if len(self.flows) and prog.needs_grad(v):  # training: mnf_flow_stack_run + mnf_flow_stack_backward
            ld, inter = prog.run_autograd(v, inverse)
            outs = [v] + (list(inter.unbind(0)) if self.return_intermediates else [inter[-1]])
            lp = None
            if want_lp:  # standard-normal base density of the result, differentiable through torch
                z = inter[-1]
                lp = -0.5 * z.square().sum(1) - 0.5 * z.size(1) * math.log(2 * math.pi)
            return outs, ld, lp
        y, ld, inter, lp = prog.run(
            v, inverse, want_inter=self.return_intermediates, want_base_lp=want_lp
        )
        outs = [v] + (list(inter.unbind(0)) if inter is not None else [y])
        if inter is not None and len(self.flows) == 0:
            outs = [v]
        return outs, ld, lp

    def forward(self, z: Tensor, noise=None) -> tuple[list[Tensor], Tensor]:  # z -> x
        if self._is_rnvp_stack():
            from .rnvp import rnvp_stack_forward

            return rnvp_stack_forward(list(self.flows), z, noise, self.return_intermediates)
        outs, ld, _ = self._run(z, inverse=False)
        return outs, ld

    def inverse(self, x: Tensor) -> tuple[list[Tensor], Tensor]:  # x -> z
        if self._is_rnvp_stack():
            raise NotImplementedError("RNVP has no inverse (reference: flows/rnvp.py)")
        outs, ld, _ = self._run(x, inverse=True)
        return outs, ld


def _is_std_normal(base, dim: int) -> bool:
    try:
        if isinstance(base, MultivariateNormal):
            return (
                base.loc.numel() == dim
                and bool((base.loc == 0).all())
                and bool((base.covariance_matrix == torch.eye(dim, device=base.loc.device)).all())
            )
        if isinstance(base, Independent) and isinstance(base.base_dist, Normal):
            n = base.base_dist
            return n.loc.numel() == dim and bool((n.loc == 0).all()) and bool((n.scale == 1).all())
    except Exception:
        return False
    return False


class NormalizingFlowModel(NormalizingFlow):
    """(base distribution, flows) pair (core.py:38-55)."""

    def __init__(self, base: Distribution, flows: Sequence[nn.Module], return_intermediates: bool = True) -> None:
        super().__init__(flows, return_intermediates)
        self.base = base
        self.__dict__["_std_base"] = {}

    def _base_is_std(self, dim):
        cache = self.__dict__.setdefault("_std_base", {})
        if dim not in cache:
            cache[dim] = _is_std_normal(self.base, dim)
        return cache[dim]

    def base_log_prob(self, x: Tensor) -> Tensor:
        """base.log_prob(inverse(x)[-1]) (core.py:46-49).  For a standard-normal base the
        density is evaluated inside the flow kernel (no second pass over z)."""
        if self._base_is_std(x.size(-1)):
            keep, self.return_intermediates = self.return_intermediates, False
            try:
                _, _, lp = self._run(x, inverse=True, want_lp=True)
            finally:
                self.return_intermediates = keep
            return lp
        zs, _ = self.inverse(x)
        z = zs[-1]
        loc = getattr(self.base, "loc", None)
        return self.base.log_prob(z if loc is None or loc.device == z.device else z.to(loc.device)).to(z.device)

    def log_prob(self, x: Tensor, out: Tensor | None = None, gather=None) -> Tensor:
        """log p(x) = log_det(inverse) + base_log_prob in ONE pass (the reference's callers
        run the inverse twice, tests/test_flows.py:22-24).  For a standard-normal base nothing but
        the [B] result is written to HBM; ``out`` lets the caller place it (e.g. in its slice of an
        all-gather buffer); ``gather`` (a ``_lib.GatherOut``) makes the kernel store the result into the other
        ranks' buffers as well (peer memory / NVLS multicast), see ``torch_mnf.distributed.PeerGather``."""
        if self._base_is_std(x.size(-1)) and 0 < len(self.flows) <= _lib.MAX_OPS and not (
            torch.is_grad_enabled() and self._program().needs_grad(x)
        ):
            if gather is None:
                got = self._maf_density_stack(x, True, log_prob_only=True, out=out)
                if got is not None:
                    return got[2]
            self._data_dependent_init(x, True)
            return self._program().run(x, inverse=True, log_prob_only=True, log_prob_out=out, gather=gather)[3]
        if self._base_is_std(x.size(-1)) and len(self.flows):  # training: one differentiable pass
            _, ld, lp = self._run(x, inverse=True, want_lp=True)
            return ld + lp
        zs, ld = self.inverse(x)
        return ld + self.base_log_prob(x)

    def log_prob_fn(self, max_rows: int = 65535):
        """``f(x [B, dim] CUDA fp32 contiguous, out=None) -> log p(x)`` with the model bound once (standard-normal base,
        at most ``max_rows`` rows per call): for call sites that evaluate a FIXED model over and over, where the module
        call's host work -- checking ~150 parameter tensors for changes, marshalling the descriptors -- is most of a
        small-batch call (BASELINE config 1).  The parameters must not change while ``f`` is in use.  Additive API."""
        from .._program import BoundLogProb

        p = next(self.parameters())
        dim = int(self.base.event_shape[0])
        if not self._base_is_std(dim):
            raise NotImplementedError("log_prob_fn needs a standard-normal base distribution")
        if any(getattr(f, "data_dep_init_done", True) is False for f in self.flows):
            raise RuntimeError("run the data-dependent initialisation (one forward / inverse call) before binding the model")
        return BoundLogProb(self._program(), p.device, dim, max_rows)

    def sample_and_log_prob(self, *num_samples: int, seed: int | None = None, row_offset: int = 0) -> tuple[Tensor, Tensor]:
        """``(x [*n, dim], log_prob [*n])``: draws from the model together with their log-density log q(x) =
        log N(z) - log_det(forward), without the inverse pass ``log_prob(x)`` would take.  Additive API.

        With a standard-normal base, z of global row ``row_offset + r`` comes from Philox4x32-10 keyed by ``seed``
        (``seed=None``: a seed drawn from torch's generator, so ``torch.manual_seed`` fixes it), the same numbers as
        every Philox draw of the library for those indices; dim-2 stacks of the table kernel draw, transform and score
        in one launch.  A batch sharded over ranks reproduces the single call bit for bit when every rank passes the
        same seed and its slice as offset::

            lo, hi = torch_mnf.distributed.shard_range(n, world, rank)
            x, lp = model.sample_and_log_prob(hi - lo, seed=seed, row_offset=lo)

        With grad enabled and trainable parameters, x and log_prob carry reparameterisation gradients (the same z, no
        gradient of its own; backward through mnf_flow_stack_backward), e.g. for reverse-KL fitting.  Under CUDA-graph
        capture with ``seed=None`` z is drawn by torch's graph-safe generator, so that every replay draws anew.  Any
        other base is sampled by torch.distributions (``seed`` is then a ValueError)."""
        return self._sample(num_samples, seed, row_offset, want_log_prob=True)

    def _sample(self, num_samples, seed, row_offset, want_log_prob):
        n = tuple(num_samples[0]) if len(num_samples) == 1 and not isinstance(num_samples[0], int) else tuple(num_samples)
        rows = math.prod(n)
        dim = int(self.base.event_shape[0]) if len(self.base.event_shape) == 1 else None
        p = next(self.parameters(), None)
        std = p is not None and p.is_cuda and dim is not None and self._base_is_std(dim)
        if any(getattr(f, "data_dep_init_done", True) is False for f in self.flows):
            raise RuntimeError("run the data-dependent initialisation (one forward / inverse call) before binding the model")
        if not std:
            if seed is not None:
                raise ValueError("seed= draws a standard-normal base with Philox; this model's base is sampled by "
                                 "torch.distributions")
            z = self.base.sample(n)
            if p is not None and z.device != p.device:
                z = z.to(p.device)
            z = z.float().reshape(-1, z.size(-1))
            xs, ld = self.forward(z)
            loc = getattr(self.base, "loc", None)
            lp = self.base.log_prob(z if loc is None or loc.device == z.device else z.to(loc.device)).to(z.device) - ld
            return xs[-1].reshape(*n, -1), lp.reshape(n)
        if not 0 < len(self.flows) <= _lib.MAX_OPS:
            raise NotImplementedError(f"sampling through {len(self.flows)} flows: between 1 and {_lib.MAX_OPS} supported")
        prog = self._program()
        capturing = seed is None and torch.cuda.is_current_stream_capturing()
        if seed is None and not capturing:
            seed = int(torch.randint(0, 2**62, (1,)).item())  # follows torch.manual_seed, as _mnf_ops.Noise
        grad = prog.needs_grad(p.detach())
        if capturing or grad:
            if capturing:  # a seed passed by value would be frozen into the graph: torch's generator advances per replay
                z = torch.randn(rows, dim, device=p.device, dtype=torch.float32)
            else:
                _, _, z = prog.sample(rows, dim, p.device, seed, row_offset, want_x=False, want_log_prob=False, want_z=True)
            if grad:  # reparameterisation gradients through mnf_flow_stack_backward
                ld, inter = prog.run_autograd(z, inverse=False)
                x = inter[-1]
            else:
                x, ld, _, _ = prog.run(z, inverse=False)
            lp = -0.5 * z.square().sum(1) - 0.5 * dim * math.log(2 * math.pi) - ld
        else:
            x, lp, _ = prog.sample(rows, dim, p.device, seed, row_offset, want_log_prob=want_log_prob)
        return x.reshape(*n, dim), (lp.reshape(n) if lp is not None else None)

    def sample(self, *num_samples: int, seed: int | None = None) -> Tensor:
        """core.py:51-55.  A standard-normal base is drawn directly on the flows' device (no host round trip);
        any other base is sampled by torch.distributions and moved over.  ``seed`` (additive): the Philox draw of
        ``sample_and_log_prob(..., seed=seed)``, whose x this returns (without computing log-densities)."""
        if seed is not None:
            return self._sample(num_samples, seed, 0, want_log_prob=False)[0]
        p = next(self.parameters(), None)
        n = tuple(num_samples[0]) if len(num_samples) == 1 and not isinstance(num_samples[0], int) else num_samples
        dim = int(self.base.event_shape[0]) if len(self.base.event_shape) == 1 else None
        if p is not None and p.is_cuda and dim is not None and self._base_is_std(dim):
            z = torch.randn(*n, dim, device=p.device, dtype=torch.float32)
        else:
            z = self.base.sample(*num_samples)
            if p is not None and z.device != p.device:
                z = z.to(p.device)
        xs, _ = self.forward(z.float().reshape(-1, z.size(-1)))
        return xs[-1].reshape(z.shape)
