"""b200zkp_dev_quotient_values and prover.prove on circuits that hold plonky2_u32's gates (the gate set of a verifier circuit built
with the ecdsa feature, tests/u32_ref.py): the quotient bit for bit against the reference, the verifier's identity on the
committed quotient, whole proofs word for word against tests/plonk_ref.py (plain and zero-knowledge), and the argument checks."""
import copy
import ctypes as C
import gc
import random

import numpy as np
import pytest

from test_gpu_interpolation import _prove_middle
from test_gpu_prove import PIS, _device_prove, _ref_form
from test_gpu_zk import KEY, _assert_same_proof, _zk_prove

pytestmark = pytest.mark.gpu
P = 0xFFFFFFFF00000001


def _coeffs(com):
    return com.coeffs.cpu().numpy().view(np.uint64)


@pytest.mark.parametrize("n_log", [5, 6])
def test_quotient_values_match_reference(n_log):
    from intmax_zkp_core_b200 import device as D
    import u32_ref as U
    from helpers import bitrev_perm
    c = U.ecdsa_circuit(n_log, seed=n_log)
    assert len(c.gates) == 20
    r, h = 3, 4
    rnd = random.Random(n_log + 31)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    ctx = D.torch_context(0)
    com_cs, com_w, com_z, q, com_q = _prove_middle(ctx, c, c.wires, betas, gammas, alphas, r, h)
    got = q.cpu().numpy().view(np.uint64)
    inv = np.argsort(bitrev_perm(n_log + r))
    nat = lambda com: [row[inv] for row in com.lde.cpu().numpy().view(np.uint64)]      # leaf order -> natural order
    want = U.quotient_values(c, nat(com_cs), nat(com_w), nat(com_z), betas, gammas, alphas, 8, r, 3)
    assert (got == np.array(want, np.uint64)).all()
    qc = _coeffs(com_q).reshape(2, 8 << n_log)
    assert U.check_quotient_identity(c, _coeffs(com_cs), _coeffs(com_w), _coeffs(com_z), qc, betas, gammas, alphas, 8,
                                     rnd.randrange(2, P))
    ctx.close()


@pytest.mark.parametrize("n_log", [8, 12])
def test_ecdsa_circuit_closes_the_identity(n_log):
    """the 20-gate ecdsa set; one changed U32Arithmetic limb or Comparison bit breaks the identity"""
    from intmax_zkp_core_b200 import device as D
    import u32_ref as U
    c = U.ecdsa_circuit(n_log, seed=40 + n_log, n_poseidon=64)
    r, h = 3, 4
    rnd = random.Random(n_log)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zeta = rnd.randrange(2, P)
    ctx = D.torch_context(0)
    com_cs, com_w, com_z, q, com_q = _prove_middle(ctx, c, c.wires, betas, gammas, alphas, r, h)
    qc = _coeffs(com_q).reshape(2, 8 << n_log)
    assert U.check_quotient_identity(c, _coeffs(com_cs), _coeffs(com_w), _coeffs(com_z), qc, betas, gammas, alphas, 8, zeta)
    for j, row in ((U.arithmetic_layout(3)["limb"](2, 30), c.u32_rows[0]), (U.comparison_layout(32, 16)["bit"](1), c.u32_rows[5])):
        bad = np.array(c.wires, np.uint64)
        bad[j][row] = (int(bad[j][row]) + 1) % P
        com_cs, com_b, com_z, qb, com_qb = _prove_middle(ctx, c, bad, betas, gammas, alphas, r, h)
        qbc = _coeffs(com_qb).reshape(2, 8 << n_log)
        assert not U.check_quotient_identity(c, _coeffs(com_cs), _coeffs(com_b), _coeffs(com_z), qbc, betas, gammas, alphas, 8, zeta), j
    ctx.close()


def _ecdsa(n_log, seed, n_poseidon=None):
    import plonk_ref as R
    import u32_ref as U
    return R.with_public_inputs(U.ecdsa_circuit(n_log, seed=seed, n_poseidon=n_poseidon), PIS)


def test_device_proof_equals_reference_prover(oracle):
    import plonk_ref as R
    import u32_ref as U
    from intmax_zkp_core_b200 import device as D
    c = _ecdsa(5, 25)
    tctx = D.torch_context(0)
    data, pw = _device_prove(tctx, c, PIS)
    want = R.prove(c, PIS, R.fri_args(5), True, ref=U)
    assert [int(v) for v in data.circuit_digest.elements] == want["circuit_digest"]
    assert (data.constants_sigmas_commitment._cap.elements == want["constants_sigmas_cap"]).all()
    _assert_same_proof(_ref_form(pw), want)
    assert R.verify(_ref_form(pw), PIS, c, data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements,
                    R.fri_args(5), True, ref=U)
    del data, pw
    tctx.close()


def test_device_zk_proof_equals_reference_prover(oracle):
    import plonk_ref as R
    import u32_ref as U
    import zk_ref as Z
    from intmax_zkp_core_b200 import device as D
    c = Z.blind(_ecdsa(5, 26, n_poseidon=4), 2, 2, seed=26)
    tctx = D.torch_context(0)
    data, pw = _zk_prove(tctx, c, KEY)
    assert data.zero_knowledge
    got = _ref_form(pw)
    want = Z.prove(c, PIS, R.fri_args(5), True, KEY, ref=U)
    assert [int(v) for v in data.circuit_digest.elements] == want["circuit_digest"]
    _assert_same_proof(got, want)
    assert Z.verify(got, PIS, c, data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements, R.fri_args(5),
                    True, ref=U)
    del data, pw
    tctx.close()


def test_ecdsa_circuit_proof_passes_the_reference_verifier(oracle):
    import plonk_ref as R
    import u32_ref as U
    from intmax_zkp_core_b200 import device as D
    n_log = 12
    c = _ecdsa(n_log, 52, n_poseidon=64)
    tctx = D.torch_context(0)
    data, pw = _device_prove(tctx, c, PIS)
    fri = R.fri_args(n_log)
    digest, cs_cap = data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements
    check = lambda form: R.verify(form, PIS, c, digest, cs_cap, fri, True, ref=U)
    form = _ref_form(pw)
    assert check(form)
    bad = copy.deepcopy(form)
    j = U.comparison_layout(32, 16)["result"]
    bad["openings"]["wires"][j] = ((bad["openings"]["wires"][j][0] + 1) % P, bad["openings"]["wires"][j][1])
    assert not check(bad)
    del data, pw
    tctx.close()


def test_u32_argument_errors():
    import torch
    from intmax_zkp_core_b200 import device as D, prover as zp
    from intmax_zkp_core_b200._lib import B200ZkpError
    ctx = D.torch_context(0)
    t = lambda k: torch.zeros((k, 64), dtype=torch.int64, device="cuda")
    run = lambda gates, ns=1: zp.compute_quotient_values_device(ctx, zp.CommonCircuitData(3, gates, ns), t(ns + 82), t(135), t(20),
                                                                [1, 2], [3, 4], [5, 6], [0, 0, 0, 0])
    one = lambda kind, params: [(zp.GATE_NOOP, 0, (0, 2)), (kind, 0, (0, 2), params)]
    bad = [(zp.GATE_U32_ARITHMETIC, (0,)), (zp.GATE_U32_ARITHMETIC, (4,)), (zp.GATE_U32_ARITHMETIC, (2**31,)),
           (zp.GATE_U32_ADD_MANY, (0, 1)), (zp.GATE_U32_ADD_MANY, (17, 1)), (zp.GATE_U32_ADD_MANY, (16, 0)),
           (zp.GATE_U32_ADD_MANY, (16, 4)), (zp.GATE_U32_ADD_MANY, (1, 2**30)),
           (zp.GATE_U32_SUBTRACTION, (0,)), (zp.GATE_U32_SUBTRACTION, (7,)), (zp.GATE_U32_SUBTRACTION, (2**31,)),
           (zp.GATE_U32_RANGE_CHECK, (0,)), (zp.GATE_U32_RANGE_CHECK, (8,)), (zp.GATE_U32_RANGE_CHECK, (2**32 - 1,)),
           (zp.GATE_COMPARISON, (0, 1)), (zp.GATE_COMPARISON, (64, 22)), (zp.GATE_COMPARISON, (32, 0)),
           (zp.GATE_COMPARISON, (4, 5)), (zp.GATE_COMPARISON, (32, 8)), (zp.GATE_COMPARISON, (63, 20)),
           (zp.GATE_COMPARISON, (63, 26))]
    for kind, params in bad:
        with pytest.raises(B200ZkpError) as e:
            run(one(kind, params))
        assert e.value.code == -1, (kind, params)
    with pytest.raises(B200ZkpError) as e:
        run(one(13, ()))                                          # 13 is not assigned
    assert e.value.code == -4
    for kind, params in ((zp.GATE_U32_ARITHMETIC, (3,)), (zp.GATE_U32_ADD_MANY, (16, 3)), (zp.GATE_U32_SUBTRACTION, (6,)),
                         (zp.GATE_U32_RANGE_CHECK, (7,)), (zp.GATE_COMPARISON, (63, 21)), (zp.GATE_COMPARISON, (1, 1))):
        run(one(kind, params))                                    # the largest (and smallest) instances are accepted
    # the 20 gates of the ecdsa set are accepted; a description of 33 gates is refused by the library itself
    import u32_ref as U
    c = U.ecdsa_circuit(5, seed=1)
    run([(g, c.selector_indices[i], c.groups[c.selector_indices[i]], c.gate_params[i]) for i, g in enumerate(c.gates)],
        c.num_selectors)
    with pytest.raises(ValueError):
        zp.CommonCircuitData(3, [(zp.GATE_NOOP, 0, (0, 33))] * 33, 1)
    d = zp._VanishingDesc()
    d.degree_bits, d.quotient_degree_bits, d.quotient_degree_factor = 3, 3, 8
    d.num_routed_wires, d.num_challenges, d.num_selectors, d.n_gates = 80, 2, 1, 33
    k, ch = zp.get_unique_coset_shifts(80), np.array([1, 2], np.uint64)
    d.k_is, d.betas, d.gammas, d.alphas = k.ctypes.data, ch.ctypes.data, ch.ctypes.data, ch.ctypes.data
    cs, w, z, out = t(83), t(135), t(20), t(2)
    ptr = lambda x: C.c_void_p(x.data_ptr())
    assert ctx._lib.b200zkp_dev_quotient_values(ctx._h, C.byref(d), ptr(cs), 64, ptr(w), 64, ptr(z), 64, ptr(out), 64) == -1
    d.n_gates = 32
    for i in range(32):
        d.gate_group_end[i] = 32
    assert ctx._lib.b200zkp_dev_quotient_values(ctx._h, C.byref(d), ptr(cs), 64, ptr(w), 64, ptr(z), 64, ptr(out), 64) == 0
    ctx.synchronize()
    ctx.close()


def test_u32_prove_leaves_no_live_buffer(oracle):
    from intmax_zkp_core_b200 import device as D
    c = _ecdsa(6, 3)
    tctx = D.torch_context(0)
    data, pw = _device_prove(tctx, c, PIS)
    assert pw.proof.opening_proof.query_round_proofs
    del data, pw
    gc.collect()
    live, cached = C.c_uint64(), C.c_uint64()
    tctx.check(tctx._lib.b200zkp_ctx_buffer_bytes(tctx._h, C.byref(live), C.byref(cached)))
    assert live.value == 0
    tctx.close()
