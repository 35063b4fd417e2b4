"""The dim-2 dispatch of mnf_flow_stack_run without a GPU: which programs mnf_flow_stack_plan sends to the dim-2 kernels,
and the refusal of a conditioner-net program that comes without a workspace (checked before any device query)."""

import pytest

N_PARAMS = 1 << 16  # the descriptors' offsets only need to lie inside the blob; nothing is read from it here


def _affine_half(parity):
    from torch_mnf import _lib
    from torch_mnf._program import new_op

    flags = _lib.FLAG_SCALE | _lib.FLAG_SHIFT | (_lib.FLAG_PARITY if parity else 0)
    return new_op(_lib.OP_AFFINE_HALF, flags, sizes=(1, 24, 24, 24, 1), net_off=(0, 1024))


def _program(name):
    """Descriptors of BASELINE config 1 (AffineHalfFlow x 9, h = 24), config 2 ([ActNorm, Glow, NSF_CL(K = 8, n_h = 16)]
    x 3) and of [ActNorm, Glow] x 3, a stack without conditioner nets."""
    from torch_mnf import _lib
    from torch_mnf._program import new_op

    actnorm = new_op(_lib.OP_AFFINE_CONST, aux_off=0)
    glow = new_op(_lib.OP_GLOW, aux_off=4)
    nsf = new_op(_lib.OP_NSF_CL, K=8, bound=3.0, sizes=(1, 16, 16, 16, 23), net_off=(0, 2048), edge_deriv=1.0)
    ops = {"cfg1": [_affine_half(i % 2) for i in range(9)],
           "cfg2": [actnorm, glow, nsf] * 3,
           "conditioner_free": [actnorm, glow] * 3}[name]
    return (_lib.FlowOp * len(ops))(*ops), len(ops)


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "conditioner_free"])
def test_plan_sends_dim2_stacks_to_the_dim2_kernels(name):
    from torch_mnf import _lib

    ops, n = _program(name)
    assert _lib.lib().mnf_flow_stack_plan(ops, n, 2, N_PARAMS) == 1


def test_run_without_workspace_is_refused_for_conditioner_nets():
    from torch_mnf import _lib

    lib = _lib.lib()
    ops, n = _program("cfg1")
    fake = 1 << 12  # device pointers are never dereferenced: the call must fail on its arguments alone
    rc = lib.mnf_flow_stack_run(ops, n, fake, N_PARAMS, fake, fake, fake, None, None, 8, 2, 0, None, None, None)
    assert rc == -1  # MNF_E_ARG
    assert b"mnf_flow_stack_workspace" in lib.mnf_last_error()
