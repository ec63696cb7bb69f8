"""GPU parity tests proper: every call goes through the C ABI (include/b200zkp.h) on cuda:0 and is compared
bit-for-bit with the oracle on the same inputs, with the committed golden vectors, with the reference's own
Poseidon fixtures, and — at BASELINE.json's full size — through size-independent properties."""
import numpy as np
import pytest

from helpers import P, bitrev, bitrev_perm, hex_to_elements, hostile_columns, rand_field

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def z():
    import intmax_zkp_core_b200 as z
    return z


# ------------------------------------------------------------------------------------------------ field primitives
def test_field_primitives_edge_cases(z, ctx):
    """The PTX carry-chain primitives against Python integers, with operands built to take the rare borrow
    (lo < x3) and carry (t + x2*eps >= 2^64) corrections and the wrap of lazy additions."""
    import ctypes as C
    rng = np.random.default_rng(99)
    M = 2**64
    special = [0, 1, 2, 2**32 - 1, 2**32, 2**32 + 1, P - 1, P, P + 1, M - 1, M - 2**32, M - 2**32 + 1, 2**63, 2**33 - 1,
               0xFFFFFFFF00000000, 0x00000000FFFFFFFF, 0xFFFFFFFEFFFFFFFF, 0x0000000100000000]
    a = np.array([x for x in special for _ in special] + [int(v) for v in rng.integers(0, M, size=4000, dtype=np.uint64)], dtype=np.uint64)
    b = np.array([y for _ in special for y in special] + [int(v) for v in rng.integers(0, M, size=4000, dtype=np.uint64)], dtype=np.uint64)
    # half of the random pairs get a tiny low word / huge high word to force borrows in reduce128
    a[400:2000] &= np.uint64(0xFFFF)
    b[400:1200] |= np.uint64(0xFFFFFFFF00000000)

    def run(op):
        out = np.empty_like(a)
        ctx.check(ctx._lib.b200zkp_field_op(ctx._h, op, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), a.size,
                                            out.ctypes.data_as(C.c_void_p)))
        return [int(v) for v in out]

    A, B = [int(v) for v in a], [int(v) for v in b]
    assert run(0) == [x * y % P for x, y in zip(A, B)]
    assert run(1) == [(x + y) % P for x, y in zip(A, B)]
    assert run(2) == [(x - y) % P for x, y in zip(A, B)]
    assert run(3) == [(x + (y << 64)) % P for x, y in zip(A, B)]
    assert run(4) == [(x + y) % P for x, y in zip(A, B)]
    m31 = (1 << 31) - 1
    assert run(5) == [((x & m31) + (((x >> 32) & m31) << 22) + ((y & m31) << 43) + ((y >> 1) % P)) % P for x, y in zip(A, B)]
    assert run(6) == [pow(x, 7, P) for x in A]
    assert run(7) == [((x ^ y) + x * y) % P for x, y in zip(A, B)]


# ------------------------------------------------------------------------------------------------ Poseidon
def test_permute_matches_oracle(z, ctx, oracle):
    rng = np.random.default_rng(21)
    states = np.concatenate([
        np.zeros((1, 12), np.uint64), np.arange(12, dtype=np.uint64)[None], np.full((1, 12), P - 1, np.uint64),
        np.full((1, 12), 2**64 - 1, np.uint64), np.full((1, 12), P, np.uint64),
        rng.integers(0, 2**64, size=(1000, 12), dtype=np.uint64)])
    got = z.PoseidonPermutation.permute(states, ctx)
    assert (got == oracle.permute_many(states)).all()
    assert (got < np.uint64(P)).all()
    assert int(got[1][0]) == 15442313428170673822            # SURVEY.md App. B


def test_reference_fixtures_on_gpu(z, ctx, golden):
    """The reference's own Poseidon KATs, computed by the CUDA kernels."""
    k = golden["reference_poseidon_kats"]
    zero = z.HashOut([0, 0, 0, 0])
    assert [int(x) for x in z.PoseidonHash.two_to_one(zero, zero, ctx).elements] == k["two_to_one_zero_zero"]["elements"]
    s = zero
    for i, h in enumerate(k["zero_hash_chain"]["hex"]):
        assert s.to_hex() == h, f"zero-hash chain entry {i}"
        s = z.PoseidonHash.two_to_one(s, s, ctx)
    for sk, hx in zip(k["accounts"]["sk"], k["accounts"]["address_hex"]):
        assert z.PoseidonHash.two_to_one(sk, sk, ctx).to_hex() == hx

    def u(x):
        return np.array([x, 0, 0, 0], dtype=np.uint64)

    def leaf(key, v):
        return z.PoseidonHash.hash_pad(np.concatenate([key, v, np.array([1], np.uint64)]), ctx).elements

    t = k["tx_hashes"]
    e3, e4 = t["smt_entries"]
    r2a = leaf(u(e3["key"][1]), leaf(u(e3["key"][2]), u(e3["value"])))
    r2b = leaf(u(e4["key"][1]), leaf(u(e4["key"][2]), u(e4["value"])))
    diff_root = z.PoseidonHash.two_to_one(leaf(u(e4["key"][0]), r2b), leaf(u(e3["key"][0]), r2a), ctx)
    for nonce, hx in zip(t["nonces"], t["tx_hex"]):
        assert z.PoseidonHash.two_to_one(diff_root, nonce, ctx).to_hex() == hx


@pytest.mark.parametrize("L", [0, 1, 3, 4, 5, 7, 8, 9, 12, 16, 17, 20, 32, 135, 139, 256])
def test_sponge_lengths(z, ctx, oracle, L):
    rng = np.random.default_rng(L)
    rows = rng.integers(0, 2**64, size=(37, L), dtype=np.uint64)
    a = z.PoseidonHash.hash_no_pad_batch(rows, ctx)
    b = z.PoseidonHash.hash_or_noop_batch(rows, ctx)
    for i in range(rows.shape[0]):
        assert (a[i] == oracle.hash_no_pad(rows[i])).all()
        assert (b[i] == oracle.hash_or_noop(rows[i])).all()


def test_two_to_one_batch(z, ctx, oracle):
    rng = np.random.default_rng(22)
    l, r = rng.integers(0, 2**64, size=(300, 4), dtype=np.uint64), rng.integers(0, 2**64, size=(300, 4), dtype=np.uint64)
    got = z.PoseidonHash.two_to_one_batch(l, r, ctx)
    for i in range(0, 300, 7):
        assert (got[i] == oracle.two_to_one(l[i], r[i])).all()


# ------------------------------------------------------------------------------------------------ NTT / LDE
@pytest.mark.parametrize("n_log", [0, 1, 2, 3, 5, 8, 9, 10, 12, 15, 16, 17])
def test_transforms_match_oracle(z, ctx, oracle, n_log):
    rng = np.random.default_rng(30 + n_log)
    k = 5 if n_log <= 12 else 2
    v = rng.integers(0, 2**64, size=(k, 1 << n_log), dtype=np.uint64)        # non-canonical inputs allowed
    assert (z.fft_batch(v, ctx) == np.stack([oracle.fft(c) for c in v])).all()
    assert (z.ifft_batch(v, ctx) == np.stack([oracle.ifft(c) for c in v])).all()
    for r in ((0, 1, 3) if n_log <= 12 else (3,)):
        assert (z.coset_lde_batch(v, r, ctx) == np.stack([oracle.coset_lde(c, r) for c in v])).all()


@pytest.mark.parametrize("n_log", [21, 24, 25])
def test_transforms_three_and_four_passes(z, ctx, oracle, n_log):
    """3 passes of 7/8 bits (2^21, 2^24: config #5's column size) and 4 passes (2^25) against the oracle's radix-2 transform."""
    rng = np.random.default_rng(n_log)
    v = rng.integers(0, 2**64, size=(1, 1 << n_log), dtype=np.uint64)
    assert (z.fft_batch(v, ctx)[0] == oracle.fft(v[0])).all()
    assert (z.ifft_batch(v, ctx)[0] == oracle.ifft(v[0])).all()
    if n_log == 21:
        lde = z.coset_lde_batch(v, 1, ctx)[0]
        assert (lde == oracle.coset_lde(v[0], 1)).all()


@pytest.mark.parametrize("n_log,k", [(11, 5), (12, 3), (13, 4), (14, 2), (15, 2), (16, 3), (17, 2), (19, 1), (20, 2)])
def test_second_generation_passes(z, oracle, n_log, k, monkeypatch):
    """ntt_ct_kernels.cuh (block-twiddle passes, TMA-staged tiles) against the oracle and against the first-generation
    passes: inverse transform in natural order; coset LDE blocks in leaf order with the coset loop (2^r <= 8 blocks), without
    it (16 blocks), with plain-load staging instead of TMA, and for a sub-range of the blocks (a multi-GPU rank's share)."""
    import ctypes as C
    import torch
    rng = np.random.default_rng(500 + n_log)
    n = 1 << n_log
    v = rng.integers(0, 2**64, size=(k, n), dtype=np.uint64)
    v[0, :4] = [2**64 - 1, P, P - 1, 0]
    ctxs = {}
    for name, env in (("tma", {}), ("plain", {"B200ZKP_NTT_TMA": "0"}), ("gen1", {"B200ZKP_NTT_CT": "0"})):
        for key in ("B200ZKP_NTT_TMA", "B200ZKP_NTT_CT"):
            monkeypatch.delenv(key, raising=False)
        for key, val in env.items():
            monkeypatch.setenv(key, val)
        ctxs[name] = z.Context(0)
    want_c = np.stack([oracle.ifft(c) for c in v]) if n_log <= 17 else None
    got = {name: z.ifft_batch(v, c) for name, c in ctxs.items()}
    assert (got["tma"] == got["gen1"]).all() and (got["plain"] == got["gen1"]).all()
    if want_c is not None:
        assert (got["tma"] == want_c).all()
    vt = torch.from_numpy(v.view(np.int64)).cuda()
    perm = None
    for r, b0, b1 in ((3, 0, 8), (3, 2, 4), (1, 0, 2), (4, 0, 16), (0, 0, 1)):
        if n_log >= 19 and r == 4:
            continue
        outs = {}
        for name, c in ctxs.items():
            lde = torch.zeros((k, (b1 - b0) * n), dtype=torch.int64, device="cuda")
            c.check(c._lib.b200zkp_dev_lde(c._h, C.c_void_p(vt.data_ptr()), n, C.c_void_p(lde.data_ptr()), (b1 - b0) * n, n_log, k, r, b0, b1))
            c.synchronize()
            outs[name] = lde.cpu().numpy().view(np.uint64)
        assert (outs["tma"] == outs["gen1"]).all(), (r, b0, b1)
        assert (outs["plain"] == outs["gen1"]).all(), (r, b0, b1)
        if n_log <= 14:
            perm = bitrev_perm(n_log + r)
            for c in range(k):
                assert (outs["tma"][c] == oracle.coset_lde(v[c], r)[perm][b0 * n:b1 * n]).all(), (r, b0, b1)
    # a whole commitment through each generation
    caps = {name: z.PolynomialBatch.from_values(v, 3, False, min(4, n_log), ctx=c).merkle_tree.cap.elements for name, c in ctxs.items()}
    assert (caps["tma"] == caps["gen1"]).all() and (caps["plain"] == caps["gen1"]).all()
    for c in ctxs.values():
        c.close()


def test_transform_roundtrip_large(z, ctx):
    rng = np.random.default_rng(31)
    v = rand_field(rng, (3, 1 << 20))
    assert (z.fft_batch(z.ifft_batch(v, ctx), ctx) == v).all()


# ------------------------------------------------------------------------------------------------ commitments
SHAPES = [  # n_log, k, rate_bits, cap_height
    (0, 5, 3, 3), (1, 3, 1, 0), (2, 3, 1, 0), (3, 9, 3, 2), (4, 135, 3, 4), (5, 20, 3, 4), (6, 16, 3, 4),
    (7, 85, 3, 4), (8, 2, 0, 0), (9, 7, 2, 11), (10, 135, 3, 4), (12, 20, 3, 4), (13, 3, 1, 5), (1, 1, 3, 4),
]


def _compare(batch, ref, k):
    assert (batch.merkle_tree.cap.elements == ref["cap"]).all(), "cap"
    assert (batch.polynomials == ref["coeffs"]).all(), "coeffs"
    assert (batch.merkle_tree.leaves == ref["leaves"]).all(), "leaves"
    assert (batch.merkle_tree.digests == ref["digests"]).all(), "digests"


@pytest.mark.parametrize("n_log,k,r,h", SHAPES)
def test_from_values_matches_oracle(z, ctx, oracle, n_log, k, r, h):
    v = oracle.synthetic_values(k, 1 << n_log, seed=n_log)
    b = z.PolynomialBatch.from_values(v, r, False, h, ctx=ctx)
    _compare(b, oracle.commit(v, r, h), k)


@pytest.mark.parametrize("n_log,k,r,h", [(4, 16, 3, 4), (9, 16, 3, 4), (11, 5, 2, 3)])
def test_from_coeffs_matches_oracle(z, ctx, oracle, n_log, k, r, h):
    v = oracle.synthetic_values(k, 1 << n_log, seed=77)
    b = z.PolynomialBatch.from_coeffs(v, r, False, h, ctx=ctx)
    _compare(b, oracle.commit(v, r, h, is_coeffs=True), k)


@pytest.mark.parametrize("n_log,k,r,h", [(3, 20, 3, 4), (8, 3, 2, 2)])
def test_blinding_with_given_salt(z, ctx, oracle, n_log, k, r, h):
    v = oracle.synthetic_values(k, 1 << n_log, seed=5)
    salt = oracle.synthetic_values(4, 1 << (n_log + r), seed=7)
    b = z.PolynomialBatch.from_values(v, r, True, h, salt=salt, ctx=ctx)
    ref = oracle.commit(v, r, h, salt=salt)
    _compare(b, ref, k)
    assert (b.get_lde_values(3) == ref["leaves"][bitrev(3, n_log + r)][:k]).all()   # salt stripped


@pytest.mark.parametrize("n_log,k,r,h,coeffs,salted", [(10, 135, 3, 4, False, False), (13, 20, 3, 4, False, False),
                                                        (9, 16, 3, 4, True, False), (6, 5, 2, 3, False, True), (0, 3, 3, 3, False, False)])
def test_copy_back_commit(z, ctx, oracle, n_log, k, r, h, coeffs, salted):
    """b200zkp_commit_copy_back: every plonky2 field on the host in one call (D2H overlapped with hashing)."""
    v = oracle.synthetic_values(k, 1 << n_log, seed=11)
    salt = oracle.synthetic_values(4, 1 << (n_log + r), seed=13) if salted else None
    ctor = z.PolynomialBatch.from_coeffs if coeffs else z.PolynomialBatch.from_values
    b = ctor(v, r, salted, h, salt=salt, ctx=ctx, copy_back=True)
    assert b._polys is not None and b.merkle_tree._leaves is not None      # filled by the call itself
    _compare(b, oracle.commit(v, r, h, is_coeffs=coeffs, salt=salt), k)
    # the device copy stays usable
    rows, _ = b.rows([0, (1 << (n_log + r)) - 1])
    assert (rows[0] == b.merkle_tree.leaves[0]).all() and (rows[1] == b.merkle_tree.leaves[-1]).all()


def test_golden_vectors_on_gpu(z, ctx, oracle, golden):
    for case in golden["commit_vectors"]["cases"]:
        n = 1 << case["n_log"]
        v = oracle.synthetic_values(case["k"], n)
        salt = oracle.synthetic_values(4, n << case["rate_bits"], seed=case["salt_seed"]) if case["salt_seed"] else None
        ctor = z.PolynomialBatch.from_coeffs if case["is_coeffs"] else z.PolynomialBatch.from_values
        b = ctor(v, case["rate_bits"], salt is not None, case["cap_height"], salt=salt, ctx=ctx)
        assert [[int(x) for x in row] for row in b.merkle_tree.cap.elements] == case["cap"]
        assert [int(x) for x in b.polynomials[0][:3]] == case["coeffs_col0_head"]
        lv = b.merkle_tree.leaves
        assert [int(x) for x in lv[0][:3]] == case["leaf0_head"]
        assert int(lv[-1][-1]) == case["leaf_last_tail"]
        d = b.merkle_tree.digests
        assert ([int(x) for x in np.bitwise_xor.reduce(d, axis=0)] if d.size else [0, 0, 0, 0]) == case["digests_xor"]


def test_hostile_inputs(z, ctx, oracle):
    for n in (8, 512):
        v = hostile_columns(n)
        b = z.PolynomialBatch.from_values(v, 3, False, 2, ctx=ctx)
        _compare(b, oracle.commit(v, 3, 2), v.shape[0])


def test_rows_proofs_and_lde_values(z, ctx, oracle):
    n_log, k, r, h = 7, 11, 3, 4
    v = oracle.synthetic_values(k, 1 << n_log, seed=9)
    b = z.PolynomialBatch.from_values(v, r, False, h, ctx=ctx)
    ref = oracle.commit(v, r, h)
    N = 1 << (n_log + r)
    idx = [0, 1, N // 2, N - 1, 37, 38, 1000]
    rows, sib = b.rows(idx)
    for q, i in enumerate(idx):
        assert (rows[q] == ref["leaves"][i]).all()
        assert (sib[q] == oracle.merkle_prove(ref["digests"], N, h, i)).all()
        assert oracle.merkle_verify(rows[q], i, sib[q], b.merkle_tree.cap.elements)
        z.verify_merkle_proof_to_cap(rows[q], i, b.merkle_tree.cap, z.MerkleProof(sib[q]), ctx)
    with pytest.raises(ValueError):
        z.verify_merkle_proof_to_cap(rows[0], 1, b.merkle_tree.cap, z.MerkleProof(sib[0]), ctx)
    for index, step in ((0, 1), (5, 1), (3, 8), (N - 1, 1)):
        assert (b.get_lde_values(index, step) == ref["leaves"][bitrev(index * step, n_log + r)]).all()
    assert (b.merkle_tree.get(5) == ref["leaves"][5]).all()
    assert (b.merkle_tree.prove(5).siblings == oracle.merkle_prove(ref["digests"], N, h, 5)).all()


def test_dev_gather_matches_batch_rows(z, ctx, oracle):
    """b200zkp_dev_gather on a batch's own device buffers: device indices in, device rows and proofs out, the same
    words as PolynomialBatch.rows; an index past the last leaf is reduced modulo the number of leaves."""
    import ctypes as C
    import torch
    n_log, k, r, h = 7, 11, 3, 4
    N, depth = 1 << (n_log + r), n_log + r - h
    b = z.PolynomialBatch.from_values(oracle.synthetic_values(k, 1 << n_log, seed=9), r, False, h, ctx=ctx)
    idx = np.array([0, 1, N // 2, N - 1, 37, 38, 1000], np.uint64)
    rows, sib = b.rows(idx)
    _, lde, digests, _ = b.device_ptrs()
    d_idx = torch.from_numpy(np.array([*idx, N + 37], np.uint64).view(np.int64)).cuda()
    d_rows = torch.zeros((idx.size + 1, k), dtype=torch.int64, device="cuda")
    d_sib = torch.zeros((idx.size + 1, depth, 4), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    p = lambda t: C.c_void_p(t.data_ptr())
    ctx.check(ctx._lib.b200zkp_dev_gather(ctx._h, C.c_void_p(lde), N, k, C.c_void_p(digests), N, h, p(d_idx), idx.size + 1,
                                          p(d_rows), p(d_sib)))
    ctx.synchronize()
    got_rows, got_sib = d_rows.cpu().numpy().view(np.uint64), d_sib.cpu().numpy().view(np.uint64)
    assert (got_rows[:-1] == rows).all() and (got_sib[:-1] == sib).all()
    assert (got_rows[-1] == rows[4]).all() and (got_sib[-1] == sib[4]).all()


@pytest.mark.parametrize("N,L,h", [(1, 5, 0), (2, 3, 1), (16, 4, 2), (16, 5, 0), (64, 32, 4), (256, 135, 4),
                                   (1024, 9, 10), (4096, 2, 3), (8, 0, 1)])
def test_merkle_tree_new(z, ctx, oracle, N, L, h):
    rng = np.random.default_rng(N + L)
    leaves = rng.integers(0, 2**64, size=(N, L), dtype=np.uint64)
    t = z.MerkleTree.new(leaves, h, ctx=ctx)
    dig, cap = oracle.merkle_new(leaves, h)
    assert (t.cap.elements == cap).all()
    assert (t.digests == dig).all()
    for i in {0, N - 1, N // 3}:
        assert (t.prove(i).siblings == oracle.merkle_prove(dig, N, h, i)).all()


def test_error_behaviour(z, ctx):
    from intmax_zkp_core_b200._lib import u64p
    import ctypes as C
    lib = ctx._lib
    h = C.c_void_p()
    buf = np.zeros(64, np.uint64)
    p = buf.ctypes.data_as(C.c_void_p)
    assert lib.b200zkp_commit_from_values(ctx._h, p, 3, 2, 3, 9, None, C.byref(h)) == -1      # cap_height > log2 N
    assert b"cap_height" in lib.b200zkp_last_error(ctx._h)
    assert lib.b200zkp_commit_from_values(ctx._h, p, 3, 0, 3, 1, None, C.byref(h)) == -1      # k == 0
    assert lib.b200zkp_commit_from_values(ctx._h, None, 3, 2, 3, 1, None, C.byref(h)) == -1   # null input
    assert lib.b200zkp_merkle_new(ctx._h, p, 6, 2, 1, C.byref(h)) == -1                       # not a power of two
    assert lib.b200zkp_merkle_new(ctx._h, p, 8, 2, 4, C.byref(h)) == -1
    assert lib.b200zkp_commit_from_values(ctx._h, p, 30, 1, 3, 1, None, C.byref(h)) == -1     # beyond two-adicity
    with pytest.raises(z.B200ZkpError):
        z.PolynomialBatch.from_values(np.zeros((1, 8), np.uint64), 3, False, 2, ctx=ctx).rows([1 << 20])


# ------------------------------------------------------------------------------------------------ device-resident API
def test_device_api_and_single_rank_shard(z, ctx, oracle):
    import torch
    from intmax_zkp_core_b200 import device as D
    n_log, k, r, h = 9, 13, 3, 4
    v = oracle.synthetic_values(k, 1 << n_log, seed=4)
    ref = oracle.commit(v, r, h)
    tctx = D.torch_context(0)
    vt = torch.from_numpy(v.view(np.int64)).cuda()
    out = D.commit_device(tctx, vt, r, h)
    tctx.synchronize()
    assert (out.cap.cpu().numpy().view(np.uint64) == ref["cap"]).all()
    assert (out.coeffs.cpu().numpy().view(np.uint64) == ref["coeffs"]).all()
    assert (out.lde.cpu().numpy().view(np.uint64).T == ref["leaves"]).all()
    assert (out.digests.cpu().numpy().view(np.uint64) == ref["digests"]).all()
    # the partitioned path with a communicator of one rank (b200zkp_comm_init_all over one ctx)
    comm = D.Comm.init_all([tctx])
    sh = D.ShardedCommitment(comm, n_log, k, r, h)
    cap = sh.run(vt)
    tctx.synchronize()
    assert (cap.cpu().numpy().view(np.uint64) == ref["cap"]).all()
    assert (sh.lde.cpu().numpy().view(np.uint64).T == ref["leaves"]).all()
    rows, sib = sh.rows([0, 77, (1 << (n_log + r)) - 1])
    assert (rows[1] == ref["leaves"][77]).all() and oracle.merkle_verify(rows[1], 77, sib[1], ref["cap"])
    sh.close()
    comm.close()
    # leaf-range shards computed one at a time on one GPU must tile the full commitment (world = 4 layout)
    for rank in range(4):
        lay = D.shard_layout(n_log, k, r, h, rank, 4)
        lde = torch.empty((k, lay["N_local"]), dtype=torch.int64, device="cuda")
        dig = torch.empty((2 * (lay["N_local"] - (1 << lay["cap_height_local"])), 4), dtype=torch.int64, device="cuda")
        capl = torch.empty((1 << lay["cap_height_local"], 4), dtype=torch.int64, device="cuda")
        lib = tctx._lib
        tctx.check(lib.b200zkp_dev_lde(tctx._h, D._ptr(out.coeffs), 1 << n_log, D._ptr(lde), lay["N_local"], n_log, k, r,
                                       lay["block_begin"], lay["block_end"]))
        tctx.check(lib.b200zkp_dev_merkle(tctx._h, D._ptr(lde), 1, lay["N_local"], k, lay["N_local"],
                                          lay["cap_height_local"], D._ptr(dig), D._ptr(capl)))
        tctx.synchronize()
        assert (lde.cpu().numpy().view(np.uint64).T == ref["leaves"][lay["leaf_begin"]:lay["leaf_end"]]).all()
        assert (capl.cpu().numpy().view(np.uint64) == ref["cap"][lay["cap_begin"]:lay["cap_end"]]).all()
    tctx.close()


# ------------------------------------------------------------------------------------------------ full size
def test_full_size_properties(z, ctx, oracle):
    """BASELINE.json config #3 (2^20 x 135, rate_bits 3, cap_height 4): too big for the single-threaded oracle
    end to end, so check size-independent properties: (1) the multithreaded CPU restatement's cap on a
    k-subset is out of budget too, so use (a) Horner evaluation of the returned coefficients at the LDE
    points of opened rows, (b) iNTT correctness via values == forward transform of coefficients on sampled
    columns, (c) every opened row's Merkle path verifies against the cap with the ORACLE's hash."""
    import torch
    from intmax_zkp_core_b200 import device as D
    n_log, k, r, h = 20, 135, 3, 4
    n, N = 1 << n_log, 1 << (n_log + r)
    v = oracle.synthetic_values(k, n)
    b = z.PolynomialBatch.from_values(v, r, False, h, ctx=ctx)
    cap = b.merkle_tree.cap.elements
    idx = [0, 1, N - 1, 123456, 7654321, N // 2 + 17]
    rows, sib = b.rows(idx)
    coeffs = b.polynomials
    # (b) forward transform of the coefficients gives back the values (columns 0, 67, 134)
    cols = [0, 67, 134]
    assert (z.fft_batch(coeffs[cols], ctx) == v[cols]).all()
    # (a) opened rows are evaluations of those coefficients at 7 * w_N^bitrev(j)
    for q, j in enumerate(idx[:3]):
        i = bitrev(j, n_log + r)
        for c in (0, 134):
            assert int(rows[q][c]) == oracle.eval_at_lde_point(coeffs[c], r, i)
    # (c) Merkle paths (leaf hash over 135 columns = 17 permutations, then 19 levels) verify with the oracle
    for q, j in enumerate(idx):
        assert sib[q].shape[0] == n_log + r - h
        assert oracle.merkle_verify(rows[q], j, sib[q], cap)
    # determinism / device-resident path gives the same cap
    tctx = D.torch_context(0)
    out = D.commit_device(tctx, torch.from_numpy(v.view(np.int64)).cuda(), r, h)
    tctx.synchronize()
    assert (out.cap.cpu().numpy().view(np.uint64) == cap).all()
    tctx.close()


def test_benchmark_shape_against_the_cpu_port(z, ctx, oracle):
    """All 16 cap entries, every digest, every coefficient and every LDE word of a 2^18 x 135 commitment (the benchmarked column
    count, 1/4 of its rows; 3 passes of 6 bits in the second-generation transforms) against the multithreaded CPU port
    (oracle/cpu_baseline.c: plonky2's own algorithm — radix-2 fft_classic, transpose + reverse_index_bits, recursive
    fill_subtree — written independently of the kernels).  bench.py runs the same comparison on the full 2^20 x 135 input
    (`parity_check`)."""
    import os
    n_log, k, r, h = 18, 135, 3, 4
    v = oracle.synthetic_values(k, 1 << n_log)
    oracle.baseline_set_threads(len(os.sched_getaffinity(0)))
    ref, _ = oracle.baseline_commit(v, r, h)
    b = z.PolynomialBatch.from_values(v, r, False, h, ctx=ctx)
    assert (b.merkle_tree.cap.elements == ref["cap"]).all()
    assert (b.polynomials == ref["coeffs"]).all()
    assert (b.merkle_tree.digests == ref["digests"]).all()
    assert (b.merkle_tree.leaves == ref["leaves"]).all()


# ------------------------------------------------------------------------------------------------ openings (N3)
@pytest.mark.parametrize("n_log,k", [(0, 3), (3, 5), (10, 135), (13, 20), (17, 7)])
def test_eval_ext2_matches_oracle(z, ctx, oracle, n_log, k):
    rng = np.random.default_rng(n_log + k)
    v = rng.integers(0, 2**64, size=(k, 1 << n_log), dtype=np.uint64)
    b = z.PolynomialBatch.from_coeffs(v, 1, False, 0, ctx=ctx)
    for zeta in (rng.integers(0, 2**64, size=2, dtype=np.uint64), np.array([5, 0], np.uint64), np.array([0, 0], np.uint64),
                 np.array([2**64 - 1, P - 1], np.uint64)):
        got = b.eval_ext2(zeta)
        for c in range(k):
            assert (got[c] == oracle.eval_ext2(v[c], zeta)).all(), (c, zeta)


# ------------------------------------------------------------------------------------------------ property-based
def test_hypothesis_commit_shapes(z, ctx, oracle):
    """Random (n, k, rate_bits, cap_height, from_values / from_coeffs, salted) with full-range u64 inputs
    (non-canonical values included) against the oracle — SURVEY.md section 4(d)."""
    from hypothesis import given, settings, strategies as st, HealthCheck

    @settings(max_examples=40, deadline=None, suppress_health_check=list(HealthCheck))
    @given(st.integers(0, 7), st.integers(1, 12), st.integers(0, 3), st.integers(0, 10), st.booleans(), st.booleans(),
           st.integers(0, 2**32 - 1))
    def run(n_log, k, r, h, coeffs, salted, seed):
        h = min(h, n_log + r)
        rng = np.random.default_rng(seed)
        v = rng.integers(0, 2**64, size=(k, 1 << n_log), dtype=np.uint64)
        salt = rng.integers(0, 2**64, size=(4, 1 << (n_log + r)), dtype=np.uint64) if salted else None
        ctor = z.PolynomialBatch.from_coeffs if coeffs else z.PolynomialBatch.from_values
        b = ctor(v, r, salted, h, salt=salt, ctx=ctx)
        ref = oracle.commit(v, r, h, is_coeffs=coeffs, salt=salt)
        assert (b.merkle_tree.cap.elements == ref["cap"]).all()
        assert (b.merkle_tree.leaves == ref["leaves"]).all()
        assert (b.polynomials == ref["coeffs"]).all()
        assert (b.merkle_tree.digests == ref["digests"]).all()

    run()
