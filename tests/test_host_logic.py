"""Host-side logic that needs no GPU: drop-in API surface, state_dict compatibility with the
reference (golden fixtures hold reference state_dicts), flow-program packing, kernel planning."""

import pytest
import torch

from oracle import flows_cpu
from tests.helpers import build_flow, golden_sd, golden_spec, load_flow_model, load_golden

CASES = ["rnvp9_moons", "nsfcl3_stack", "nsfcl_d4", "nsfar2_d3", "maf9_d64", "maf3_d8", "maf_iaf_d2",
         "affine_misc_d4"]


@pytest.mark.parametrize("name", CASES)
def test_reference_state_dict_loads_strict(name):
    g = load_golden(name)
    model = load_flow_model(golden_spec(g), golden_sd(g), device="cpu")
    keys = {k for k in golden_sd(g) if not k.endswith(".P")}
    assert set(model.state_dict().keys()) == keys


def test_public_names_match_reference():
    import torch_mnf.flows as nf
    import torch_mnf.layers as L
    import torch_mnf.models as M

    for n in ["ActNormFlow", "AffineConstantFlow", "AffineHalfFlow", "NormalizingFlow", "NormalizingFlowModel",
              "Glow", "IAF", "MAF", "RNVP", "NSF_AR", "NSF_CL"]:  # flows/__init__.py:17-23
        assert hasattr(nf, n)
    for n in ["MADE", "MaskedLinear", "MNFConv2d", "MNFLinear"]:  # layers/__init__.py:1-3
        assert hasattr(L, n)
    for n in ["MLP", "MNFFeedForward", "MNFLeNet"]:
        assert hasattr(M, n)


def test_made_masks_equal_oracle_and_reference():
    from torch_mnf.layers import MADE

    made = MADE(64, [24, 24, 24], 128, natural_ordering=True)
    ref = golden_sd(load_golden("maf9_d64"))
    for i, m in enumerate(flows_cpu.made_masks(64, [24, 24, 24], 128, natural=True)):
        assert torch.equal(made[2 * i].mask, torch.from_numpy(m))
        assert torch.equal(made[2 * i].mask, ref[f"flows.0.net.{2 * i}.mask"])
    made = MADE(6, [7, 5], 12, num_masks=3)  # random ordering + mask cycling keeps the autoregressive property
    for _ in range(4):
        made.update_masks()
        m = [layer.mask.float() for layer in made if hasattr(layer, "mask")]
        conn = (m[0] @ m[1] @ m[2])[:, :6]  # input i -> output j path count
        order = torch.from_numpy(made.m[-1])
        for i in range(6):
            for j in range(6):
                if order[i] >= order[j]:
                    assert conn[i, j] == 0


def test_flow_program_packing_and_plan():
    from torch_mnf import _lib
    from torch_mnf._program import FlowProgram

    specs = [{"type": "AffineHalfFlow", "dim": 2, "parity": bool(i % 2), "scale": True, "shift": True,
              "h_sizes": [24, 24, 24]} for i in range(9)]
    flows = [build_flow(s) for s in specs]
    prog = FlowProgram(flows)
    prog._build(torch.device("cpu"))
    assert prog._n_ops == 9 and prog._blob.numel() % 4 == 0
    per_net = 24 + 24 + 2 * (24 * 24 + 24) + 24 + 1
    assert prog._blob.numel() >= 18 * per_net
    for k in range(9):
        op = prog._ops[k]
        assert op.type == _lib.OP_AFFINE_HALF and op.n_lin == 4 and list(op.sizes[:5]) == [1, 24, 24, 24, 1]
        assert op.net_off[0] % 4 == 0 and op.net_off[1] % 4 == 0
        assert bool(op.flags & _lib.FLAG_PARITY) == bool(k % 2)
        w0 = flows[k].s_net[0].weight.detach().reshape(-1)
        assert torch.equal(prog._blob[op.net_off[0]: op.net_off[0] + 24], w0)
    assert prog.plan(torch.device("cpu"), 2) == 1  # BASELINE config 1 -> table kernel
    key = prog._key
    prog._build(torch.device("cpu"))
    assert prog._key is key  # cached
    with torch.no_grad():
        flows[3].t_net[2].bias.add_(1.0)
    prog._build(torch.device("cpu"))
    assert prog._key != key  # parameter change invalidates the packed blob
    wide = FlowProgram([build_flow({"type": "NSF_CL", "dim": 4, "K": 5, "B": 3, "n_h": 8})])
    assert wide.plan(torch.device("cpu"), 4) == 0  # dim 4 -> generic interpreter


def test_maf_masks_are_folded_into_packed_weights():
    from torch_mnf._program import FlowProgram

    f = build_flow({"type": "MAF", "dim": 8, "parity": True, "h_sizes": [16, 16]})
    prog = FlowProgram([f])
    prog._build(torch.device("cpu"))
    lin0 = f.net[0]
    packed = prog._blob[prog._ops[0].net_off[0]: prog._ops[0].net_off[0] + 16 * 8].view(16, 8)
    assert torch.equal(packed, (lin0.weight * lin0.mask.float().T).detach())


def test_shard_range_covers_rows_exactly():
    from torch_mnf.distributed import shard_range

    for n in (0, 1, 7, 500, 1 << 24):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1


def test_differentiable_blob_matches_cached_layout_and_reaches_parameters():
    """Training path: the blob handed to mnf_flow_stack_backward is an autograd function of the nn.Parameters with the
    SAME layout as the cached inference blob (MADE masks applied by torch), so d loss / d blob lands on them."""
    from torch_mnf._program import FlowProgram, ParamPacker

    flows = [build_flow({"type": "MAF", "dim": 8, "parity": True, "h_sizes": [16, 16]}),
             build_flow({"type": "NSF_CL", "dim": 8, "K": 5, "B": 3, "n_h": 8}),
             build_flow({"type": "AffineConstantFlow", "dim": 8, "scale": True, "shift": False})]
    prog = FlowProgram(flows)
    prog._build(torch.device("cpu"))
    with torch.enable_grad():  # the suite's default is inference mode (tests/conftest.py)
        pk = ParamPacker(torch.device("cpu"), differentiable=True)
        ops = [f._emit(pk) for f in flows]
        blob = pk.finish()
        assert blob.requires_grad and torch.equal(blob.detach(), prog._blob)
        assert [o.net_off[0] for o in ops] == [prog._ops[k].net_off[0] for k in range(3)]
        w = torch.arange(blob.numel(), dtype=torch.float32)
        (blob * w).sum().backward()
        assert prog.needs_grad(torch.zeros(2, 8))
    lin0 = flows[0].net[0]
    off = ops[0].net_off[0]
    expect = w[off: off + 16 * 8].view(16, 8) * lin0.mask.float().T  # masked entries receive no gradient
    assert torch.equal(lin0.weight.grad, expect)
    assert flows[2].s.grad is not None and flows[1].f1[0].weight.grad is not None
    with torch.no_grad():
        assert not prog.needs_grad(torch.zeros(2, 8))


def test_glow_torch_assembly_matches_oracle():
    """Glow's differentiable assembly (training path) == the oracle's W, and its inverse / log-det are consistent."""
    g = load_golden("nsfcl3_stack")
    sd = golden_sd(g)
    glow = build_flow({"type": "Glow", "dim": 2})
    glow.load_state_dict({k[len("flows.1."):]: v for k, v in sd.items() if k.startswith("flows.1.") and not k.endswith(".P")})
    glow.P.copy_(sd["flows.1.P"])
    with torch.enable_grad():
        out = glow._assemble_torch()
    W = flows_cpu.glow_W(flows_cpu.sub(sd, "flows.1."))
    torch.testing.assert_close(out[:4].detach().view(2, 2), W, rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(out[4:8].detach().view(2, 2) @ W, torch.eye(2), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(out[8].detach(), torch.log(torch.abs(sd["flows.1.S"])).sum(), rtol=1e-6, atol=1e-7)
    with torch.enable_grad():
        out.sum().backward()
    assert all(p.grad is not None for p in (glow.L, glow.S, glow.U))


def test_sync_actnorm_init_single_process():
    import torch_mnf.flows as nf
    from torch_mnf.distributed import sync_actnorm_init

    model = nf.NormalizingFlow([nf.ActNormFlow(3), nf.Glow(3)])
    called = []
    assert sync_actnorm_init(model, init_fn=lambda m: called.append(1)) == 1
    assert called == [1] and model.flows[0].data_dep_init_done
    assert sync_actnorm_init(model, init_fn=lambda m: called.append(2)) == 1 and called == [1]  # already initialised
    assert sync_actnorm_init(nf.NormalizingFlow([nf.Glow(3)])) == 0


# ---------------------------------------------------------------------------------------
# cache hygiene (ADVICE r1): launch caches must neither break copy/pickle nor survive parameter changes
# ---------------------------------------------------------------------------------------
def test_modules_deepcopy_and_pickle_with_populated_caches():
    """After a call the modules hold ctypes descriptors with raw pointers (RnvpFlow structs, MADE plans, flow
    programs).  ctypes objects with pointers cannot be pickled, so the caches must be dropped by __getstate__ --
    the reference's modules copy and pickle fine (EMA copies, torch.save(model))."""
    import copy
    import ctypes
    import io
    import pickle

    import torch_mnf.flows as nf
    from torch_mnf._program import FlowProgram
    from torch_mnf.layers import MNFLinear
    from torch_mnf.layers._mnf_ops import RnvpFlow
    from torch_mnf.layers.made import MadeLayer

    with pytest.raises(ValueError):  # the failure mode being guarded against
        pickle.dumps(RnvpFlow())
    layer = MNFLinear(8, 4)
    for f in list(layer.flow_q.flows) + list(layer.flow_r.flows):
        f.__dict__["_rnvp_struct_cache"] = (("cuda:0", (1, 2)), RnvpFlow(), 50)
    layer.__dict__["_last_kl_terms"] = torch.zeros(5)
    stack = nf.NormalizingFlowModel(torch.distributions.MultivariateNormal(torch.zeros(4), torch.eye(4)),
                                    [nf.MAF(4, parity=bool(i % 2), h_sizes=(8, 8)) for i in range(2)])
    stack.__dict__["_prog"] = FlowProgram(list(stack.flows))
    stack.__dict__["_tc_plan"] = (True, (MadeLayer * 1)(MadeLayer()))
    stack.flows[0].__dict__["_tc_plan"] = (MadeLayer * 1)(MadeLayer())
    stack.flows[0].__dict__["_single_prog"] = FlowProgram([stack.flows[0]])
    for m in (layer, stack):
        c = copy.deepcopy(m)
        assert set(c.state_dict()) == set(m.state_dict())
        for k, v in m.state_dict().items():
            assert torch.equal(c.state_dict()[k], v)
        buf = io.BytesIO()
        torch.save(m, buf)
        buf.seek(0)
        r = torch.load(buf, weights_only=False)
        assert set(r.state_dict()) == set(m.state_dict())
        for mod in c.modules():
            assert not any(isinstance(v, (ctypes.Structure, ctypes.Array)) for v in mod.__dict__.values())
    assert stack.__dict__["_prog"] is not None  # the original keeps its caches
    assert copy.deepcopy(stack)._program() is not stack._program()


def test_flow_program_key_sees_every_kind_of_parameter_change():
    """(versions, all data pointers, per-flow salt, parameter epoch): in-place updates, `p.data = ...` on ANY tensor,
    load_state_dict(assign=True), Module.to() and CUDA-graph replays all invalidate the packed blob."""
    import torch_mnf.flows as nf
    from torch_mnf import _program
    from torch_mnf._program import FlowProgram, _state_key

    flows = [nf.AffineHalfFlow(2, parity=bool(i % 2), h_sizes=(4, 4)) for i in range(3)]
    prog = FlowProgram(flows)
    dev = torch.device("cpu")

    def key():
        k = _state_key(prog.flows, dev, prog._tensors)
        if k != getattr(key, "last", None):  # what FlowProgram._build does on a mismatch
            prog._refresh_tensors()
            k = _state_key(prog.flows, dev, prog._tensors)
        key.last = k
        return k

    k0 = key()
    assert key() == k0
    with torch.no_grad():
        flows[1].s_net[2].weight.add_(1.0)  # in-place: version counter
    k1 = key()
    assert k1 != k0
    mid = flows[1].t_net[2].weight  # neither the first nor the last tensor of the program
    v = mid._version
    mid.data = mid.data.clone()
    assert mid._version == v
    k2 = key()
    assert k2 != k1
    sd = {k: v.clone() + 1 for k, v in flows[2].state_dict().items()}
    old = flows[2].s_net[0].weight
    flows[2].load_state_dict(sd, assign=True)
    assert flows[2].s_net[0].weight is not old
    k3 = key()
    assert k3 != k2
    assert any(t is flows[2].s_net[0].weight for t in prog._tensors)  # the list was re-read from the modules
    flows[0].requires_grad_(False), flows[1].requires_grad_(False), flows[2].requires_grad_(False)
    with torch.enable_grad():
        assert not prog.needs_grad(torch.zeros(1, 2))
    flows[0].double().float()  # Module._apply
    k4 = key()
    assert k4 != k3
    _program.bump_param_epoch()
    assert key() != k4


def test_made_plan_key_sees_pointer_changes_and_epoch():
    import torch_mnf.flows as nf
    from torch_mnf import _program
    from torch_mnf.layers.made import MadeStackPlan

    f = nf.MAF(8, parity=False, h_sizes=(8, 8))
    plan = MadeStackPlan([f])

    def key():
        ts = plan._tensors()
        return (tuple(t._version for t in ts), tuple(t.data_ptr() for t in ts), _program.param_epoch())

    k0 = key()
    w = f.net[2].weight
    w.data = w.data.clone()
    assert key() != k0
    k1 = key()
    _program.bump_param_epoch()
    assert key() != k1


def test_non_default_leaky_slope_is_rejected_not_ignored():
    import torch_mnf.flows as nf
    from torch_mnf._program import ParamPacker
    from torch_mnf.models import MLP

    f = nf.NSF_CL(2, K=4, B=3, n_h=4, net_class=lambda *s: MLP(*s, leaky_a=0.1))
    with pytest.raises(NotImplementedError, match="leaky_a"):
        f._emit(ParamPacker(torch.device("cpu")))
    nf.NSF_CL(2, K=4, B=3, n_h=4)._emit(ParamPacker(torch.device("cpu")))


def test_kl_fused_plan_numbering_matches_the_draw_order_and_follows_parameter_storage():
    """The cached argument block of mnf_kl_div_fused carries the Philox stream ids of a tape-less call; they must be the
    ids a Noise object hands out in kl_div's draw order (z0, flow_q masks, eps_w, eps_b, flow_r masks), and the block must
    be rebuilt when any parameter gets new storage."""
    from torch_mnf.layers import MNFConv2d, MNFLinear
    from torch_mnf.layers import _mnf_ops as ops

    dev = torch.device("cpu")
    for layer, conv in ((MNFLinear(12, 7, n_flows_q=2, n_flows_r=3), False), (MNFConv2d(3, 5, 3), True)):
        plan = ops._kl_fused_plan(layer, conv, dev)
        assert plan is not None
        a, dim, fan, rows, nq, nr = plan
        assert (dim, fan) == ((5, 27) if conv else (12, 12)) and rows == max(layer.W_mean.shape[0], fan)
        noise = ops.Noise(None, dev, seed=1)
        _, z_sid = noise.normal((dim,))
        q_sids = [noise.bernoulli((1, dim))[1] for _ in range(nq)]
        _, w_sid = noise.normal((fan,))
        noise._next_stream()  # eps_b (conv) or the skipped id (linear)
        r_sids = [noise.bernoulli((1, dim))[1] for _ in range(nr)]
        assert a.z_stream == z_sid and a.kl.noise_stream == w_sid
        assert [a.mask_streams[i] for i in range(nq)] == q_sids
        assert [a.mask_streams[ops.KL_MAX_FLOWS + i] for i in range(nr)] == r_sids
        assert a.n_flows_q == nq and a.n_flows_r == nr and a.kl.conv == int(conv)
        assert ops._kl_fused_plan(layer, conv, dev) is plan  # cached
        layer.flow_r.flows[0].t.weight.data = layer.flow_r.flows[0].t.weight.data.clone()
        again = ops._kl_fused_plan(layer, conv, dev)
        assert again is not plan and again[0].flows[ops.KL_MAX_FLOWS].t_w == layer.flow_r.flows[0].t.weight.data_ptr()
    # outside the fused entry point's shape class: two-layer conditioners -> the multi-launch path
    wide = MNFLinear(12, 7, h_sizes=(8, 8))
    assert ops._kl_fused_plan(wide, False, dev) is None


def test_table_kernel_planning_and_buffer_sizes():
    """Host side of csrc/flow_pl.cu (no launch): which programs have a piecewise-linear form, and that the staged image
    of any of them fits the workspace mnf_flow_stack_workspace() asks callers to provide."""
    from tests.helpers import build_flow
    from torch_mnf import _lib
    from torch_mnf._program import FlowProgram

    lib = _lib.lib()
    cpu = torch.device("cpu")

    def prog_of(specs):
        prog = FlowProgram([build_flow(s) for s in specs])
        prog._build(cpu)
        return prog

    def stage_size(prog, dim=2):
        return lib.mnf_flow_stack_stage_size(prog._ops, prog._n_ops, dim, prog._blob.numel())

    nsf = lambda K, h: {"type": "NSF_CL", "dim": 2, "K": K, "B": 3, "n_h": h}  # noqa: E731
    aff = lambda hs, p=False, scale=True, shift=True: {"type": "AffineHalfFlow", "dim": 2, "parity": p, "scale": scale,  # noqa: E731
                                                       "shift": shift, "h_sizes": hs}
    act = {"type": "ActNormFlow", "dim": 2, "scale": True, "shift": True}
    glow = {"type": "AffineConstantFlow", "dim": 2, "scale": True, "shift": False}  # (Glow's blob is assembled by a kernel: no CPU build)
    hdr, bp, rows = 256, 512, 512  # flow_pl.cu: header floats, padded breakpoints and rows per table
    # config 2: six spline tables of stride 52 floats; config 1: nine (s, t) tables of stride 12
    assert stage_size(prog_of([act, glow, nsf(8, 16)] * 3)) == hdr + 6 * (bp + rows * 52)
    assert stage_size(prog_of([aff([24, 24, 24], bool(i % 2)) for i in range(9)])) == hdr + 9 * (bp + rows * 12)
    # any depth 1..5 and width <= 64, every instantiated bin count; conditioner-free flows add no table
    for specs in ([aff([40])], [aff([32, 16]), glow], [aff([64] * 5)], [nsf(4, 12)], [nsf(5, 8)], [nsf(16, 64)], [nsf(10, 20), act],
                  [aff([16, 16, 16], scale=False), nsf(8, 16)]):
        prog = prog_of(specs)
        size = stage_size(prog)
        assert size > hdr, specs
        assert size <= lib.mnf_flow_stack_workspace(prog._n_ops, 1 << 20, 2), specs
        assert prog.plan(cpu, 2) == 1, specs
    # outside the table kernel: bins it is not instantiated for, widths above 64 (both still have other kernels or the
    # interpreter), other dims
    assert stage_size(prog_of([nsf(7, 16)])) == 0
    assert stage_size(prog_of([aff([96, 96])])) == 0
    wide = prog_of([{"type": "NSF_CL", "dim": 4, "K": 8, "B": 3, "n_h": 16}])
    assert stage_size(wide, dim=4) == 0 and lib.mnf_flow_stack_workspace(1, 1 << 20, 4) == 0
