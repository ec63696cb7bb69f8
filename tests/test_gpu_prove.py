"""The whole of plonky2's prove() on the device (prover.prove): commitments from HBM into batch handles
(b200zkp_batch_from_device), the opening set in one call (b200zkp_batch_openings), and the proof word for word against the
restated prover tests/plonk_ref.py, or accepted by its restated verifier at circuit-like sizes."""
import ctypes as C
import gc

import numpy as np
import pytest

from helpers import P, rand_field

pytestmark = pytest.mark.gpu
HIGH, LOW = 14, 15
PIS = [3, 1, 4, 1, 5, 2**64 - 1]


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.uint64)).view(np.int64)).cuda()


def _host(t):
    return t.cpu().numpy().view(np.uint64)


# ------------------------------------------------------------------------------------------------ b200zkp_batch_from_device
@pytest.mark.parametrize("n_log,k,r,h,is_coeffs", [(5, 7, 3, 4, False), (5, 7, 3, 4, True), (10, 135, 3, 4, False),
                                                   (3, 1, 1, 4, True), (8, 20, 2, 0, False)])
def test_from_device_equals_host_commit(ctx, n_log, k, r, h, is_coeffs):
    import intmax_zkp_core_b200 as z
    rng = np.random.default_rng(n_log * 7 + k)
    data = rand_field(rng, (k, 1 << n_log), canonical=False)
    data[0, :4] = [P, 2**64 - 1, P - 1, 0]
    host = (z.PolynomialBatch.from_coeffs if is_coeffs else z.PolynomialBatch.from_values)(data, r, False, h, ctx=ctx)
    dev = z.PolynomialBatch.from_device(_dev(data), r, False, h, is_coeffs=is_coeffs, ctx=ctx)
    assert dev._cap == host._cap
    assert (dev.polynomials == host.polynomials).all()
    assert (dev.merkle_tree.leaves == host.merkle_tree.leaves).all()
    assert (dev.merkle_tree.digests == host.merkle_tree.digests).all()
    assert (_host(dev.coeffs) == host.polynomials).all()
    assert dev.lde.shape == (k, 1 << (n_log + r))
    rows, sib = dev.rows([0, 5])
    want_rows, want_sib = host.rows([0, 5])
    assert (rows == want_rows).all() and (sib == want_sib).all()


def test_from_device_argument_errors_leave_out_null(ctx):
    import torch
    t = torch.zeros((4, 16), dtype=torch.int64, device="cuda")
    for args in ((t.data_ptr(), 0, 4, 0, 1, 0), (t.data_ptr(), 0, 4, 4, 1, 6), (t.data_ptr(), 0, 30, 4, 3, 0),
                 (t.data_ptr(), 0, 4, 4, 9, 0), (None, 0, 4, 4, 1, 0)):
        h = C.c_void_p(12345)
        ptr, is_coeffs, n_log, k, r, cap = args
        rc = ctx._lib.b200zkp_batch_from_device(ctx._h, C.c_void_p(ptr) if ptr else None, is_coeffs, n_log, k, r, cap, None, C.byref(h))
        assert rc == -1 and h.value is None, args


# ------------------------------------------------------------------------------------------------ b200zkp_batch_openings
def test_batch_openings_equals_per_batch_evaluation(ctx, oracle):
    import intmax_zkp_core_b200 as z
    import intmax_zkp_core_b200.fri as zf
    from oracle import fri_ref as F
    rng = np.random.default_rng(8)
    n_log = 11
    data = [rand_field(rng, (k, 1 << n_log), canonical=False) for k in (3, 4, 2)]
    batches = [z.PolynomialBatch.from_coeffs(d, 2, False, 3, ctx=ctx) for d in data]
    zeta = (int(rng.integers(1, P, dtype=np.uint64)), int(rng.integers(1, P, dtype=np.uint64)))
    points = [zeta, (5, 0), F.escale(zeta, F.root(n_log))]
    polys = [[(0, 0), (0, 2), (1, 2), (1, 3), (2, 1)], [], [(1, 2), (2, 0)]]        # (1, 2) at both points, one empty batch
    inst = zf.FriInstanceInfo([zf.FriBatchInfo(pt, [zf.FriPolynomialInfo(o, i) for o, i in ps]) for pt, ps in zip(points, polys)])
    before = ctx.launch_count
    got = zf.batch_openings(inst, batches)
    assert ctx.launch_count - before == 2
    for pt, ps, vals in zip(points, polys, got):
        assert len(vals) == len(ps)
        per_batch = [b.eval_ext2(np.array(pt, np.uint64)) for b in batches]
        for (o, i), v in zip(ps, vals):
            assert v == tuple(int(x) for x in per_batch[o][i])
            canon = np.where(data[o][i] >= np.uint64(P), data[o][i] - np.uint64(P), data[o][i])
            assert v == tuple(int(x) for x in oracle.eval_ext2(canon, np.array(pt, np.uint64)))


def test_batch_openings_argument_errors(ctx):
    import intmax_zkp_core_b200 as z
    import intmax_zkp_core_b200.fri as zf
    a = z.PolynomialBatch.from_coeffs(np.ones((2, 8), np.uint64), 1, False, 0, ctx=ctx)
    b = z.PolynomialBatch.from_coeffs(np.ones((1, 16), np.uint64), 1, False, 0, ctx=ctx)
    other = z.Context(0)
    c = z.PolynomialBatch.from_coeffs(np.ones((1, 8), np.uint64), 1, False, 0, ctx=other)
    out = np.zeros(16, np.uint64)

    def run(inst, oracles, n_oracles=None, null_oracles=False):
        args = list(zf._instance_args(inst, oracles))
        if n_oracles is not None:
            args[1] = n_oracles
        if null_oracles:
            args[0] = None
        return ctx._lib.b200zkp_batch_openings(ctx._h, *args, out.ctypes.data_as(C.c_void_p))

    one = lambda o, i: zf.FriInstanceInfo([zf.FriBatchInfo((1, 2), [zf.FriPolynomialInfo(o, i)])])
    assert run(one(0, 1), [a]) == 0
    assert run(one(0, 1), [a], null_oracles=True) == -1
    assert run(one(0, 1), [a], n_oracles=0) == -1
    assert run(zf.FriInstanceInfo([zf.FriBatchInfo((1, 2), [])]), [a]) == -1        # nothing to open
    assert run(one(1, 0), [a, c]) == -1                                              # oracle of another ctx
    assert run(one(1, 0), [a, b]) == -1                                              # degrees differ
    assert run(one(1, 0), [a]) == -1                                                 # oracle index out of range
    assert run(one(0, 2), [a]) == -1                                                 # polynomial index out of range
    del c
    other.close()


# ------------------------------------------------------------------------------------------------ prove()
def _device_prove(ctx, c, pis, wires=None, mul_by_x=True):
    from intmax_zkp_core_b200 import fri as zf, prover as zp
    common = zp.CommonCircuitData(c.n_log, [(g, c.selector_indices[i], c.groups[c.selector_indices[i]], c.gate_params[i])
                                            for i, g in enumerate(c.gates)],
                                  c.num_selectors, quotient_degree_factor=8, k_is=np.array(c.k_is, np.uint64))
    data = zp.circuit_data(ctx, common, _dev(c.constants + c.sigmas), zf.standard_recursion_fri_config())
    proof = zp.prove(ctx, data, _dev(c.wires if wires is None else wires), pis, mul_by_x)
    return data, proof


def _pairs(a):
    return [(int(x), int(y)) for x, y in np.asarray(a).reshape(-1, 2)]


def _ref_form(pw):
    """the device proof in tests/plonk_ref.py's form"""
    p = pw.proof
    op = p.opening_proof
    fields = ("constants", "plonk_sigmas", "wires", "plonk_zs", "plonk_zs_next", "partial_products", "quotient_polys")
    return dict(wires_cap=p.wires_cap.elements, plonk_zs_partial_products_cap=p.plonk_zs_partial_products_cap.elements,
                quotient_polys_cap=p.quotient_polys_cap.elements,
                openings={f: list(getattr(p.openings, f)) for f in fields},
                opening_proof=dict(caps=[cp.elements for cp in op.commit_phase_merkle_caps], final_poly=_pairs(op.final_poly),
                                   pow_witness=op.pow_witness,
                                   rounds=[dict(initial=[(row, pr.siblings) for row, pr in r.initial_trees_proof.evals_proofs],
                                                steps=[(s.evals, s.merkle_proof.siblings) for s in r.steps])
                                           for r in op.query_round_proofs]))


def _circuit(kind, n_log, seed, n_poseidon=None):
    import interpolation_ref as I
    import plonk_ref as R
    from oracle import vanishing_ref as V
    if kind == "extended":
        c, ref = V.Circuit(n_log, seed=seed, extended=True, n_poseidon=n_poseidon), V
    else:
        c, ref = I.recursion_circuit(n_log, seed=seed, n_poseidon=n_poseidon, interpolation=kind), I
    return R.with_public_inputs(c, PIS), ref


@pytest.mark.parametrize("n_log", [5, 6])
@pytest.mark.parametrize("kind", ["extended", (LOW, 4), (HIGH, 3)])
def test_device_proof_equals_reference_prover(ctx, oracle, kind, n_log):
    import plonk_ref as R
    from intmax_zkp_core_b200 import device as D
    c, ref = _circuit(kind, n_log, seed=20 + n_log)
    tctx = D.torch_context(0)
    data, pw = _device_prove(tctx, c, PIS)
    got = _ref_form(pw)
    want = R.prove(c, PIS, R.fri_args(n_log), True, ref=ref)
    assert [int(v) for v in data.circuit_digest.elements] == want["circuit_digest"]
    assert (data.constants_sigmas_commitment._cap.elements == want["constants_sigmas_cap"]).all()
    for key in ("wires_cap", "plonk_zs_partial_products_cap", "quotient_polys_cap"):
        assert (got[key] == want[key]).all(), key
    assert got["openings"] == want["openings"]
    g, w = got["opening_proof"], want["opening_proof"]
    assert len(g["caps"]) == len(w["caps"]) and all((a == b).all() for a, b in zip(g["caps"], w["caps"]))
    assert g["final_poly"] == w["final_poly"] and g["pow_witness"] == w["pow_witness"]
    assert len(g["rounds"]) == len(w["rounds"]) == 28
    for rg, rw in zip(g["rounds"], w["rounds"]):
        assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for a, b in zip(rg["initial"], rw["initial"]))
        assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for a, b in zip(rg["steps"], rw["steps"]))
    assert pw.public_inputs == [v % P for v in PIS]
    del data, pw
    tctx.close()


@pytest.mark.parametrize("n_log", [8, 12])
def test_recursion_circuit_proof_passes_the_reference_verifier(ctx, oracle, n_log):
    import copy
    import plonk_ref as R
    from intmax_zkp_core_b200 import device as D
    c, ref = _circuit((LOW, 4), n_log, seed=40 + n_log, n_poseidon=64)
    assert len(c.gates) == 14
    tctx = D.torch_context(0)
    data, pw = _device_prove(tctx, c, PIS)
    fri = R.fri_args(n_log)
    assert fri["arities"] == data.fri_params.reduction_arity_bits
    digest, cs_cap = data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements
    check = lambda form: R.verify(form, PIS, c, digest, cs_cap, fri, True, ref=ref)
    form = _ref_form(pw)
    assert check(form)
    bad = copy.deepcopy(form)
    bad["openings"]["wires"][9] = ((bad["openings"]["wires"][9][0] + 1) % P, bad["openings"]["wires"][9][1])
    assert not check(bad)
    wires = np.array(c.wires, np.uint64)
    wires[100][5] = (int(wires[100][5]) + 1) % P
    _, pw_bad = _device_prove(tctx, c, PIS, wires=wires)
    assert not check(_ref_form(pw_bad))
    del data, pw, pw_bad
    tctx.close()


def test_prove_leaves_no_live_buffer(oracle):
    from intmax_zkp_core_b200 import device as D
    c, _ = _circuit((LOW, 4), 6, seed=3)
    tctx = D.torch_context(0)
    data, pw = _device_prove(tctx, c, PIS)
    assert pw.proof.opening_proof.query_round_proofs
    del data, pw
    gc.collect()
    live, cached = C.c_uint64(), C.c_uint64()
    tctx.check(tctx._lib.b200zkp_ctx_buffer_bytes(tctx._h, C.byref(live), C.byref(cached)))
    assert live.value == 0
    tctx.close()
