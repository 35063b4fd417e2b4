"""mnf_flow_stack_sample without a GPU: argument checks, the binding, and the compiler's report for the table kernel's
draw instantiations."""

import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _affine_program():
    from torch_mnf import _lib

    ops = (_lib.FlowOp * 1)()
    ops[0].type = _lib.OP_AFFINE_CONST
    ops[0].aux_off = 0
    return ops


def _sample(flags, x=None, lp=None, z=None, n_rows=8):
    from torch_mnf import _lib

    lib = _lib.lib()
    return lib.mnf_flow_stack_sample(_affine_program(), 1, 1 << 12, 16, 1, 0, 0, x, lp, z, n_rows, 2, flags, None, None)


def test_sample_symbol_is_declared_and_bound():
    from torch_mnf import _lib

    assert "mnf_flow_stack_sample" in _lib.declared_symbols()
    fn = _lib.lib().mnf_flow_stack_sample
    assert len(fn.argtypes) == 15 and fn.restype is ctypes.c_int


@pytest.mark.parametrize("flags", ["inverse", "logprob", 0x100, 0x80])
def test_sample_rejects_flags_outside_the_forward_direction(flags):
    from torch_mnf import _lib

    f = {"inverse": _lib.RUN_INVERSE, "logprob": _lib.RUN_LOGPROB}.get(flags, flags)
    assert _sample(f, x=1 << 12) == -1
    assert b"flags" in _lib.lib().mnf_last_error()


def test_sample_needs_an_output():
    from torch_mnf import _lib

    assert _sample(0) == -1
    assert b"no output" in _lib.lib().mnf_last_error()
    assert _sample(0, n_rows=0) == 0  # an empty batch is a no-op, as for mnf_flow_stack_run


def _ptxas_report():
    log = os.path.join(ROOT, "torch-mnf_b200", "build", "flow_pl.ptxas.log")
    if not os.path.exists(log):
        pytest.skip("no compiler report: build the library first (python torch-mnf_b200/build.py)")
    out, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(_ZN3mnf3fpl14flow_pl_kernel\w+)'", line)
        if m:
            cur = m.group(1)
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            out.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out.setdefault(cur, {})["regs"] = int(m.group(1))
            cur = None
    return out


def test_draw_instantiations_need_no_more_registers_or_spills():
    """flow_pl_kernel<K, false, true> draws its points instead of loading them: it must not cost the point loop
    registers or local-memory traffic over the forward instantiation <K, false>."""
    rep = _ptxas_report()
    draws = {k: v for k, v in rep.items() if "Lb0ELb1EEEv" in k}
    assert len(draws) == 7, sorted(rep)
    for k, v in draws.items():
        fwd = rep[k.replace("Lb0ELb1EEEv", "Lb0ELb0EEEv")]
        assert v["regs"] <= fwd["regs"], (k, v, fwd)
        assert v["spill"][0] <= fwd["spill"][0] and v["spill"][1] <= fwd["spill"][1], (k, v, fwd)
    assert draws["_ZN3mnf3fpl14flow_pl_kernelILi8ELb0ELb1EEEvNS0_6ParamsE"] == {"spill": (0, 0), "regs": 64}
