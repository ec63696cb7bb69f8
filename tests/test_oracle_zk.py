"""Zero-knowledge prove() on the CPU: the ChaCha20 field-element stream of tests/chacha_ref.py (RFC 8439, the `cryptography`
package's keystream, pinned elements), blinding rows that keep a circuit satisfied (tests/zk_ref.py), and reference zk proofs
that the zk verifier accepts and rejects."""
import copy
import random

import numpy as np
import pytest

import chacha_ref as CR
import plonk_ref as R
import zk_ref as Z
from helpers import P
from oracle import perm_ref as PR
from oracle import vanishing_ref as V
from test_oracle_vanishing import coset_ifft

KEY = bytes(range(32))
PIS = [3, 1, 4, 1, 5, 2**64 - 1]


# ------------------------------------------------------------------------------------------------ the stream
def test_chacha_block_rfc8439_2_3_2():
    got = CR.keystream(KEY, bytes.fromhex("000000090000004a00000000"), 1, 1)
    assert got.hex() == ("10f1e7e4d13b5915500fdd1fa32071c4c7d1f4c733c068030422aa9ac3d46c4e"
                         "d2826446079faa0914c2d705d98b02a2b5129cd1de164eb9cbd083e8a2503c4e")


def test_chacha_keystream_equals_cryptography():
    pytest.importorskip("cryptography")
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms
    rng = np.random.default_rng(1)
    for key, nonce, first in ((KEY, CR.nonce_for_oracle(1), 0), (rng.bytes(32), rng.bytes(12), 7), (rng.bytes(32), bytes(12), 2**32 - 3000)):
        # cryptography's ChaCha20 takes the 32-bit block counter (little-endian) followed by the 96-bit nonce
        enc = Cipher(algorithms.ChaCha20(key, first.to_bytes(4, "little") + nonce), mode=None).encryptor()
        assert enc.update(bytes(64 * 3000)) == CR.keystream(key, nonce, first, 3000)


def test_element_mapping_is_pinned():
    nonce = CR.nonce_for_oracle(1)
    assert CR.elements(KEY, nonce, 0, 8).tolist() == [
        8800410126362406528, 3025112885576137351, 5241065360682113419, 15666533705488274408, 2193322543829132463,
        10939588473935877749, 18151928148028613924, 9262513928936287863]
    assert CR.elements(KEY, nonce, 1000003, 1).tolist() == [7686018197023369210]
    # an element is its 16 keystream bytes as lo + 2^64 hi, reduced
    ks = CR.keystream(KEY, nonce, 0, 1)
    for j in range(4):
        v = int.from_bytes(ks[16 * j:16 * j + 16], "little") % P
        assert CR.elements(KEY, nonce, j, 1)[0] == v
    # a sub-range is a slice of the whole
    whole = CR.elements(KEY, nonce, 0, 64)
    assert (CR.elements(KEY, nonce, 5, 50) == whole[5:55]).all()


# ------------------------------------------------------------------------------------------------ blinding rows
def test_blinding_counts():
    # standard_recursion_config's FRI at 2^14: arity bits [4, 4, 4], final polynomial of 2^2 coefficients
    fri = R.fri_args(14)
    assert fri["arities"] == [4, 4, 4]
    fri_openings = 28 * (1 + 2 * 3 * 15 + 2 * 4)
    assert Z.blinding_counts(14, fri) == (2 + fri_openings, 4 + fri_openings)
    regular, z = Z.blinding_counts(14, fri)
    assert (regular, z) == (2774, 2776)
    assert 1 << 13 < regular + 2 * z <= 1 << 14          # 8326 rows: a 2^14-row circuit keeps 8058 rows for its gates


def _identity(oracle, c, seed):
    """check_quotient_identity for circuit c with random challenges, at two random points"""
    rnd = random.Random(seed)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zs_pp = PR.partial_products_and_zs([c.wires[j] for j in range(V.NUM_ROUTED)], c.sigmas, c.k_is, betas, gammas, 8)
    coeffs = {k: [oracle.ifft(np.array(col, np.uint64)) for col in cols]
              for k, cols in dict(cs=c.constants + c.sigmas, wires=c.wires, zpp=zs_pp).items()}
    ldes = {k: [oracle.coset_lde(col, 3) for col in cols] for k, cols in coeffs.items()}
    q = V.quotient_values(c, ldes["cs"], ldes["wires"], ldes["zpp"], betas, gammas, alphas, 8, 3, 3)
    qc = [coset_ifft(oracle, col) for col in q]
    return all(V.check_quotient_identity(c, coeffs["cs"], coeffs["wires"], coeffs["zpp"], qc, betas, gammas, alphas, 8,
                                         rnd.randrange(2, P)) for _ in range(2))


def test_blinded_circuit_satisfies_the_quotient_identity(oracle):
    c = V.Circuit(4, seed=3, n_poseidon=4)
    b = Z.blind(c, 2, 2, seed=1)
    regular, pairs = b.blinding_rows
    assert len(regular) == 2 and len(pairs) == 2
    for a, r in pairs:
        assert all(b.wires[j][a] == b.wires[j][r] for j in range(V.NUM_ROUTED))
        assert b.sigmas[5][a] == b.k_is[5] * pow(V.root(4), r, P) % P
    assert b.wires != c.wires and b.sigmas != c.sigmas
    assert _identity(oracle, b, 5)
    # one routed wire of a pair no longer equal to its copy: the permutation argument fails
    bad = copy.deepcopy(b)
    a, r = pairs[1]
    bad.wires[7][r] = (bad.wires[7][r] + 1) % P
    assert not _identity(oracle, bad, 5)


def test_blind_refuses_rows_that_are_not_noops():
    c = V.Circuit(4, seed=3)
    noops = sum(1 for g in c.row_gate if c.gates[g] == V.NOOP)
    with pytest.raises(ValueError):
        Z.blind(c, noops + 1, 0)


# ------------------------------------------------------------------------------------------------ reference zk proofs
@pytest.fixture(scope="module")
def zk_proof(oracle):
    c = R.with_public_inputs(Z.blind(V.Circuit(5, seed=11, n_poseidon=8), 2, 2, seed=2), PIS)
    fri = R.fri_args(5, pow_bits=8)
    proof = Z.prove(c, PIS, fri, True, KEY)
    check = lambda p: Z.verify(p, PIS, c, proof["circuit_digest"], proof["constants_sigmas_cap"], fri, True)
    return c, fri, proof, check


def test_reference_zk_proof_is_accepted(zk_proof):
    c, fri, proof, check = zk_proof
    assert check(proof)
    rnd0 = proof["opening_proof"]["rounds"][0]["initial"]
    nc = c.num_selectors + V.NUM_GATE_CONSTANTS
    assert [len(row) for row, _ in rnd0] == [nc + V.NUM_ROUTED, V.NUM_WIRES + 4, 2 * 10 + 4, 2 * 8 + 4]
    # the salt words are the stream's, at the opened leaf's natural row
    x = proof["opening_proof"]["rounds"][0]["x_index"]
    N_log = c.n_log + fri["rate_bits"]
    nat = int(format(x, f"0{N_log}b")[::-1], 2)
    salts = Z.salts(KEY, c.n_log, fri["rate_bits"])
    for o in range(1, 4):
        assert (np.asarray(rnd0[o][0])[-4:] == salts[o - 1][:, nat]).all()
    # the salts change every blinded cap against the unsalted proof of the same witness
    plain = R.prove(c, PIS, fri, True)
    for key in ("wires_cap", "plonk_zs_partial_products_cap", "quotient_polys_cap"):
        assert not (plain[key] == proof[key]).all(), key


def test_reference_zk_proof_with_a_changed_salt_word_is_rejected(zk_proof):
    _, _, proof, check = zk_proof
    for o in (1, 2, 3):
        bad = copy.deepcopy(proof)
        row = np.array(bad["opening_proof"]["rounds"][3]["initial"][o][0])
        row[-1] = (int(row[-1]) + 1) % P
        bad["opening_proof"]["rounds"][3]["initial"][o] = (row, bad["opening_proof"]["rounds"][3]["initial"][o][1])
        assert not check(bad), o


def test_reference_zk_proof_without_salts_is_rejected(zk_proof):
    _, _, proof, check = zk_proof
    stripped = Z.strip_salts(proof)
    o = stripped["openings"]
    ks = [len(o["constants"]) + len(o["plonk_sigmas"]), len(o["wires"]), len(o["plonk_zs"]) + len(o["partial_products"]),
          len(o["quotient_polys"])]
    assert not Z.leaf_shapes_ok(stripped, ks)
    assert not check(stripped)
