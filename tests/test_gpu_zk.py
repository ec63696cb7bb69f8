"""Zero-knowledge prove() on the device: b200zkp_dev_random_field against tests/chacha_ref.py word for word, salted proofs against
the zk reference prover of tests/zk_ref.py word for word, and a blinded recursion circuit whose proof the zk verifier accepts."""
import copy
import ctypes as C
import gc

import numpy as np
import pytest

import chacha_ref as CR
from helpers import P
from test_gpu_prove import HIGH, LOW, PIS, _circuit, _dev, _host, _ref_form

pytestmark = pytest.mark.gpu
KEY = bytes(range(32))
OTHER_KEY = bytes(range(100, 132))


# ------------------------------------------------------------------------------------------------ b200zkp_dev_random_field
@pytest.mark.parametrize("first,count", [(0, 1), (3, 1), (1, 2), (2, 7), (0, 4096), (5, 4093), (1000003, 65537),
                                         (0, 1 << 22), (4 * 777 + 1, (1 << 22) - 3), (2**34 - 6, 6)])
def test_random_field_equals_chacha_ref(ctx, first, count):
    import torch
    from intmax_zkp_core_b200 import prover as zp
    nonce = CR.nonce_for_oracle(2)
    buf = torch.full((count + 8,), 0x5A5A, dtype=torch.int64, device="cuda")      # 8 guard words after the range
    torch.cuda.synchronize()
    zp.random_field_device(ctx, KEY, nonce, count, first=first, out=buf[:count])
    ctx.synchronize()
    got = _host(buf)
    assert (got[:count] == CR.elements(KEY, nonce, first, count)).all()
    assert (got[:count] < P).all()
    assert (got[count:] == 0x5A5A).all()
    fresh = zp.random_field_device(ctx, KEY, nonce, count, first=first)
    ctx.synchronize()
    assert fresh.shape == (count,) and fresh.dtype == torch.int64 and (_host(fresh) == got[:count]).all()


def test_random_field_argument_errors(ctx):
    import torch
    from intmax_zkp_core_b200 import prover as zp
    out = torch.zeros(64, dtype=torch.int64, device="cuda")
    lib, h, o = ctx._lib, ctx._h, C.c_void_p(out.data_ptr())
    before = ctx.launch_count
    assert lib.b200zkp_dev_random_field(h, None, bytes(12), 0, 4, o) == -1
    assert lib.b200zkp_dev_random_field(h, KEY, None, 0, 4, o) == -1
    assert lib.b200zkp_dev_random_field(h, KEY, bytes(12), 0, 4, None) == -1
    assert lib.b200zkp_dev_random_field(h, KEY, bytes(12), 2**34 - 3, 4, o) == -1          # block 2^32 would be needed
    assert lib.b200zkp_dev_random_field(h, KEY, bytes(12), 2**34, 1, o) == -1
    assert lib.b200zkp_dev_random_field(h, KEY, bytes(12), 1, 2**64 - 1, o) == -1         # first + count wraps
    assert lib.b200zkp_dev_random_field(h, None, None, 0, 0, None) == 0                    # count 0: nothing to do
    assert ctx.launch_count == before                                                      # nothing was launched
    ctx.synchronize()
    assert not bool(out.any())
    assert lib.b200zkp_dev_random_field(h, KEY, bytes(12), 2**34 - 4, 4, o) == 0           # the last block is fine
    assert ctx.launch_count == before + 1
    with pytest.raises(ValueError):
        zp.random_field_device(ctx, KEY[:31], bytes(12), 4)
    with pytest.raises(ValueError):
        zp.random_field_device(ctx, KEY, bytes(11), 4)
    with pytest.raises(ValueError):
        zp.random_field_device(ctx, KEY, bytes(12), 4, out=out)
    ctx.synchronize()


# ------------------------------------------------------------------------------------------------ zk prove()
def _zk_prove(ctx, c, key, wires=None, zero_knowledge=True):
    from intmax_zkp_core_b200 import fri as zf, prover as zp
    common = zp.CommonCircuitData(c.n_log, [(g, c.selector_indices[i], c.groups[c.selector_indices[i]], c.gate_params[i])
                                            for i, g in enumerate(c.gates)],
                                  c.num_selectors, quotient_degree_factor=8, k_is=np.array(c.k_is, np.uint64))
    data = zp.circuit_data(ctx, common, _dev(c.constants + c.sigmas), zf.standard_recursion_fri_config(),
                           zero_knowledge=zero_knowledge)
    proof = zp.prove(ctx, data, _dev(c.wires if wires is None else wires), PIS, True, salt_key=key)
    return data, proof


def _blinded(kind, n_log, seed, regular, pairs, n_poseidon=8):
    import zk_ref as Z
    c, ref = _circuit(kind, n_log, seed, n_poseidon=n_poseidon)
    return Z.blind(c, regular, pairs, seed=seed), ref


def _assert_same_proof(g, w):
    for key in ("wires_cap", "plonk_zs_partial_products_cap", "quotient_polys_cap"):
        assert (np.asarray(g[key]) == np.asarray(w[key])).all(), key
    assert g["openings"] == w["openings"]
    go, wo = g["opening_proof"], w["opening_proof"]
    assert len(go["caps"]) == len(wo["caps"]) and all((a == b).all() for a, b in zip(go["caps"], wo["caps"]))
    assert go["final_poly"] == wo["final_poly"] and go["pow_witness"] == wo["pow_witness"]
    assert len(go["rounds"]) == len(wo["rounds"]) == 28
    for rg, rw in zip(go["rounds"], wo["rounds"]):
        assert [len(a[0]) for a in rg["initial"]] == [len(b[0]) for b in rw["initial"]]
        assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for a, b in zip(rg["initial"], rw["initial"]))
        assert all((a[0] == b[0]).all() and (a[1] == b[1]).all() for a, b in zip(rg["steps"], rw["steps"]))


@pytest.mark.parametrize("n_log", [5, 6])
@pytest.mark.parametrize("kind", ["extended", (LOW, 4), (HIGH, 3)])
def test_device_zk_proof_equals_reference_prover(oracle, kind, n_log):
    import plonk_ref as R
    import zk_ref as Z
    from intmax_zkp_core_b200 import device as D
    c, ref = _blinded(kind, n_log, 30 + n_log, 2, 2)
    tctx = D.torch_context(0)
    data, pw = _zk_prove(tctx, c, KEY)
    assert data.zero_knowledge and data.fri_params.hiding
    got = _ref_form(pw)
    want = Z.prove(c, PIS, R.fri_args(n_log), True, KEY, ref=ref)
    assert [int(v) for v in data.circuit_digest.elements] == want["circuit_digest"]
    assert (data.constants_sigmas_commitment._cap.elements == want["constants_sigmas_cap"]).all()
    _assert_same_proof(got, want)
    widths = [len(row) for row, _ in got["opening_proof"]["rounds"][0]["initial"]]
    assert widths[1:] == [135 + 4, 20 + 4, 16 + 4]
    assert Z.verify(got, PIS, c, data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements, R.fri_args(n_log),
                    True, ref=ref)
    del data, pw
    tctx.close()


def test_blinded_recursion_circuit_proof_passes_the_zk_verifier(oracle):
    import plonk_ref as R
    import zk_ref as Z
    from intmax_zkp_core_b200 import device as D
    n_log = 14
    fri = R.fri_args(n_log)
    regular, z_pairs = Z.blinding_counts(n_log, fri)
    c, ref = _blinded((LOW, 4), n_log, 54, regular, z_pairs, n_poseidon=64)
    assert len(c.gates) == 14 and len(c.blinding_rows[0]) == regular and len(c.blinding_rows[1]) == z_pairs
    tctx = D.torch_context(0)
    data, pw = _zk_prove(tctx, c, None)
    assert fri["arities"] == data.fri_params.reduction_arity_bits
    digest, cs_cap = data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements
    check = lambda form: Z.verify(form, PIS, c, digest, cs_cap, fri, True, ref=ref)
    form = _ref_form(pw)
    assert check(form)
    bad = copy.deepcopy(form)
    row, sib = bad["opening_proof"]["rounds"][5]["initial"][1]
    row = np.array(row)
    row[-2] = (int(row[-2]) + 1) % P                    # one salt word of an opened wires leaf
    bad["opening_proof"]["rounds"][5]["initial"][1] = (row, sib)
    assert not check(bad)
    bad = copy.deepcopy(form)
    bad["openings"]["partial_products"][4] = ((bad["openings"]["partial_products"][4][0] + 1) % P,
                                              bad["openings"]["partial_products"][4][1])
    assert not check(bad)
    assert not check(Z.strip_salts(form))
    del data, pw
    tctx.close()


def test_zk_proofs_of_one_witness(oracle):
    import plonk_ref as R
    import zk_ref as Z
    from intmax_zkp_core_b200 import device as D
    c, ref = _blinded((LOW, 4), 6, 7, 3, 2)
    fri = R.fri_args(6)
    tctx = D.torch_context(0)
    caps = ("wires_cap", "plonk_zs_partial_products_cap", "quotient_polys_cap")
    data, a = _zk_prove(tctx, c, KEY)
    _, b = _zk_prove(tctx, c, OTHER_KEY)
    _, a2 = _zk_prove(tctx, c, KEY)
    _, d1 = _zk_prove(tctx, c, None)            # a fresh key from the OS for every proof
    _, d2 = _zk_prove(tctx, c, None)
    fa, fb, fa2, fd1, fd2 = (_ref_form(p) for p in (a, b, a2, d1, d2))
    check = lambda form: Z.verify(form, PIS, c, data.circuit_digest.elements, data.constants_sigmas_commitment._cap.elements, fri,
                                  True, ref=ref)
    for f in (fa, fb, fd1, fd2):
        assert check(f)
    for x, y in ((fa, fb), (fd1, fd2), (fa, fd1)):
        for k in caps:
            assert not (x[k] == y[k]).all(), k
    _assert_same_proof(fa, fa2)                 # the same key gives the same proof
    del data, a, b, a2, d1, d2
    tctx.close()


def test_salt_key_arguments(oracle):
    from intmax_zkp_core_b200 import device as D, prover as zp
    c, _ = _circuit((LOW, 4), 5, seed=3)
    tctx = D.torch_context(0)
    with pytest.raises(ValueError):
        _zk_prove(tctx, c, KEY, zero_knowledge=False)
    data, pw = _zk_prove(tctx, c, None, zero_knowledge=False)          # the non-zk proof is unchanged
    assert not data.zero_knowledge and not data.fri_params.hiding
    assert [len(row) for row, _ in pw.proof.opening_proof.query_round_proofs[0].initial_trees_proof.evals_proofs][1] == 135
    b, _ = _blinded((LOW, 4), 5, 3, 1, 1)
    with pytest.raises(ValueError):
        _zk_prove(tctx, b, KEY[:16])
    with pytest.raises(ValueError):
        zp.prove(tctx, data, _dev(c.wires), PIS, True, salt_key=KEY)
    del data, pw
    tctx.close()


def test_zk_prove_leaves_no_live_buffer(oracle):
    from intmax_zkp_core_b200 import device as D
    c, _ = _blinded((LOW, 4), 6, 3, 2, 2)
    tctx = D.torch_context(0)
    data, pw = _zk_prove(tctx, c, None)
    assert pw.proof.opening_proof.query_round_proofs
    del data, pw
    gc.collect()
    live, cached = C.c_uint64(), C.c_uint64()
    tctx.check(tctx._lib.b200zkp_ctx_buffer_bytes(tctx._h, C.byref(live), C.byref(cached)))
    assert live.value == 0
    tctx.close()
