"""b200zkp_dev_quotient_values on circuits that hold plonky2's interpolation gates (the gate set of a recursive verifier): the
middle of prove() on the device — wires commitment -> Z / partial products -> their commitment -> quotient values -> quotient
commitment — bit for bit against tests/interpolation_ref.py (oracle/vanishing_ref.py with the two gates), the verifier's identity on the committed quotient, and the argument
checks of the two gate kinds."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
P = 0xFFFFFFFF00000001
HIGH, LOW = 14, 15


def _common(zp, c):
    return zp.CommonCircuitData(c.n_log, [(g, c.selector_indices[i], c.groups[c.selector_indices[i]], c.gate_params[i])
                                          for i, g in enumerate(c.gates)],
                                c.num_selectors, quotient_degree_factor=8, k_is=np.array(c.k_is, np.uint64))


def _prove_middle(ctx, c, wires, betas, gammas, alphas, r, h):
    import torch
    from intmax_zkp_core_b200 import device as D, prover as zp
    dev = lambda cols: torch.from_numpy(np.array(cols, np.uint64).view(np.int64)).cuda()
    wire_vals = dev(wires)
    com_cs = D.commit_device(ctx, dev(c.constants + c.sigmas), r, h)
    com_w = D.commit_device(ctx, wire_vals, r, h)
    zpp_vals = zp.zs_partial_products_device(ctx, wire_vals[:80], dev(c.sigmas), np.array(c.k_is, np.uint64), betas, gammas, 8)
    com_z = D.commit_device(ctx, zpp_vals, r, h)
    q = zp.compute_quotient_values_device(ctx, _common(zp, c), com_cs.lde, com_w.lde, com_z.lde, betas, gammas, alphas, c.pi_hash)
    com_q = zp.commit_quotient_device(ctx, q, c.n_log, r, h)
    ctx.synchronize()
    return com_cs, com_w, com_z, q, com_q


@pytest.mark.parametrize("n_log,interpolation", [(5, (LOW, 4)), (6, (LOW, 4)), (5, (HIGH, 3)), (6, (HIGH, 2))])
def test_quotient_values_match_oracle(n_log, interpolation):
    from intmax_zkp_core_b200 import device as D
    import interpolation_ref as I
    from helpers import bitrev_perm
    c = I.recursion_circuit(n_log, seed=n_log, interpolation=interpolation)
    assert interpolation[0] in c.gates
    r, h = 3, 4
    rnd = random.Random(n_log + 17)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    ctx = D.torch_context(0)
    com_cs, com_w, com_z, q, com_q = _prove_middle(ctx, c, c.wires, betas, gammas, alphas, r, h)
    got = q.cpu().numpy().view(np.uint64)
    inv = np.argsort(bitrev_perm(n_log + r))
    nat = lambda com: [row[inv] for row in com.lde.cpu().numpy().view(np.uint64)]      # leaf order -> natural order
    want = I.quotient_values(c, nat(com_cs), nat(com_w), nat(com_z), betas, gammas, alphas, 8, r, 3)
    assert (got == np.array(want, np.uint64)).all()
    co = lambda com: com.coeffs.cpu().numpy().view(np.uint64)
    qc = com_q.coeffs.cpu().numpy().view(np.uint64).reshape(2, 8 << n_log)
    assert I.check_quotient_identity(c, co(com_cs), co(com_w), co(com_z), qc, betas, gammas, alphas, 8, rnd.randrange(2, P))
    ctx.close()


@pytest.mark.parametrize("n_log", [8, 12])
def test_recursion_circuit_closes_the_identity(n_log):
    """the 14-gate recursion set; one changed LowDegree coefficient or power wire breaks the identity"""
    from intmax_zkp_core_b200 import device as D
    import interpolation_ref as I
    c = I.recursion_circuit(n_log, seed=40 + n_log, n_poseidon=64)
    assert len(c.gates) == 14
    r, h = 3, 4
    rnd = random.Random(n_log)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zeta = rnd.randrange(2, P)
    ctx = D.torch_context(0)
    co = lambda com: com.coeffs.cpu().numpy().view(np.uint64)
    com_cs, com_w, com_z, q, com_q = _prove_middle(ctx, c, c.wires, betas, gammas, alphas, r, h)
    qc = com_q.coeffs.cpu().numpy().view(np.uint64).reshape(2, 8 << n_log)
    assert I.check_quotient_identity(c, co(com_cs), co(com_w), co(com_z), qc, betas, gammas, alphas, 8, zeta)
    row = c.row_gate.index(c.gates.index(LOW))
    L = I.interpolation_layout(LOW, 4)
    for j in (L["coeff"](5), L["eval_pow"](3) + 1):
        bad = np.array(c.wires, np.uint64)
        bad[j][row] = (int(bad[j][row]) + 1) % P
        com_cs, com_b, com_z, qb, com_qb = _prove_middle(ctx, c, bad, betas, gammas, alphas, r, h)
        qbc = com_qb.coeffs.cpu().numpy().view(np.uint64).reshape(2, 8 << n_log)
        assert not I.check_quotient_identity(c, co(com_cs), co(com_b), co(com_z), qbc, betas, gammas, alphas, 8, zeta), j
    ctx.close()


def test_interpolation_argument_errors():
    import torch
    from intmax_zkp_core_b200 import device as D, prover as zp
    from intmax_zkp_core_b200._lib import B200ZkpError
    ctx = D.torch_context(0)
    t = lambda k: torch.zeros((k, 64), dtype=torch.int64, device="cuda")
    run = lambda common: zp.compute_quotient_values_device(ctx, common, t(83), t(135), t(20), [1, 2], [3, 4], [5, 6], [0, 0, 0, 0])
    for kind, bits in ((LOW, 0), (HIGH, 0), (LOW, 5), (HIGH, 6)):
        common = zp.CommonCircuitData(3, [(zp.GATE_NOOP, 0, (0, 2)), (kind, 0, (0, 2), (bits,))], 1)
        with pytest.raises(B200ZkpError) as e:
            run(common)
        assert e.value.code == -1, (kind, bits)
    common = zp.CommonCircuitData(3, [(zp.GATE_NOOP, 0, (0, 2)), (13, 0, (0, 2))], 1)      # 13 is not assigned
    with pytest.raises(B200ZkpError) as e:
        run(common)
    assert e.value.code == -4
    # the largest instances are accepted
    for kind, bits in ((LOW, 4), (HIGH, 5)):
        run(zp.CommonCircuitData(3, [(zp.GATE_NOOP, 0, (0, 2)), (kind, 0, (0, 2), (bits,))], 1))
    ctx.synchronize()
    ctx.close()
