"""Device buffers go back to the ctx's pool: after every handle is freed and every call has returned, no bytes handed out by
the pool are still live (b200zkp_ctx_buffer_bytes).  Covers the handles (batches, Merkle trees, FRI state, sharded
commitments) and the entry points that only allocate scratch, on success and on an error after the allocation."""
import ctypes as C
import gc

import numpy as np
import pytest

from helpers import P, rand_field

pytestmark = pytest.mark.gpu

ERR_UNSUPPORTED = -4


@pytest.fixture(scope="module")
def z():
    import intmax_zkp_core_b200 as z
    return z


@pytest.fixture()
def bctx(z):
    """a fresh ctx per test: its counters see this test's buffers only"""
    c = z.Context(0)
    yield c
    c.close()


def buffer_bytes(ctx):
    gc.collect()    # a PolynomialBatch and its merkle_tree refer to each other: dropped batches are freed by the cycle collector
    live, cached = C.c_uint64(), C.c_uint64()
    ctx.check(ctx._lib.b200zkp_ctx_buffer_bytes(ctx._h, C.byref(live), C.byref(cached)))
    return live.value, cached.value


def live(ctx):
    return buffer_bytes(ctx)[0]


@pytest.mark.parametrize("coeffs,salted,copy_back", [(False, False, False), (True, False, False), (False, True, False),
                                                     (True, True, False), (False, False, True), (True, True, True)])
def test_batch_returns_every_buffer(z, bctx, coeffs, salted, copy_back):
    n_log, k, r, h = 9, 20, 3, 2
    rng = np.random.default_rng(n_log + k)
    v = rand_field(rng, (k, 1 << n_log), canonical=False)
    salt = rand_field(rng, (4, 1 << (n_log + r))) if salted else None
    ctor = z.PolynomialBatch.from_coeffs if coeffs else z.PolynomialBatch.from_values
    b = ctor(v, r, salted, h, salt=salt, ctx=bctx, copy_back=copy_back)
    assert live(bctx) > 0
    assert b.polynomials.shape == (k, 1 << n_log) and b.merkle_tree.leaves.shape[0] == 1 << (n_log + r)
    b.merkle_tree.digests
    b.rows([0, 5, (1 << (n_log + r)) - 1])
    b.get_lde_values(3, 2)
    b.eval_ext2([5, 7])
    del b
    assert live(bctx) == 0


def test_copy_back_without_handle(z, bctx):
    n_log, k, r, h = 8, 16, 2, 1
    N = 1 << (n_log + r)
    v = rand_field(np.random.default_rng(3), (k, 1 << n_log))
    polys, leaves = np.empty((k, 1 << n_log), np.uint64), np.empty((N, k), np.uint64)
    digests, cap = np.empty((2 * (N - (1 << h)), 4), np.uint64), np.empty((1 << h, 4), np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    bctx.check(bctx._lib.b200zkp_commit_copy_back(bctx._h, p(v), 0, n_log, k, r, h, None, p(polys), p(leaves), p(digests), p(cap), None))
    assert live(bctx) == 0


def test_repeated_commit_does_not_grow_the_pool(z, bctx):
    v = rand_field(np.random.default_rng(1), (24, 1 << 11))
    z.PolynomialBatch.from_values(v, 3, False, 4, ctx=bctx)       # (freed at once: no reference kept)
    first = buffer_bytes(bctx)
    assert first[0] == 0 and first[1] > 0
    for _ in range(3):
        z.PolynomialBatch.from_values(v, 3, False, 4, ctx=bctx)
        now = buffer_bytes(bctx)
        assert now[0] == 0 and now[0] + now[1] <= first[0] + first[1]


def test_merkle_tree_returns_every_buffer(z, bctx):
    leaves = np.random.default_rng(5).integers(0, 2**64, size=(1024, 9), dtype=np.uint64)
    t = z.MerkleTree.new(leaves, 3, ctx=bctx)
    t.digests
    t.prove_many([0, 17, 1023])
    assert live(bctx) > 0
    del t
    assert live(bctx) == 0


def test_fri_returns_every_buffer(z, bctx):
    import intmax_zkp_core_b200.fri as zf
    rng = np.random.default_rng(9)
    n_log, r, h = 10, 3, 2
    gpu = [z.PolynomialBatch.from_coeffs(rand_field(rng, (kk, 1 << n_log)), r, False, h, ctx=bctx) for kk in (3, 2)]
    polys = [zf.FriPolynomialInfo(o, i) for o, kk in enumerate((3, 2)) for i in range(kk)]
    instance = zf.FriInstanceInfo([zf.FriBatchInfo((5, 6), polys), zf.FriBatchInfo((7, 8), polys[3:])])
    st = zf.FriCommitPhase.from_oracles(instance, gpu, (11, 12), True, ctx=bctx)
    for ab in (2, 2):
        st.commit_layer(ab, h)
        st.fold((int(rng.integers(1, P, dtype=np.uint64)), 3))
    st.final_poly()
    st.coeffs()
    st.query(0, [0, 3, (1 << (n_log + r - 2)) - 1], 2, n_log + r - 2 - h)
    st.query(1, [1], 2, n_log + r - 4 - h)
    st.close()
    del gpu
    assert live(bctx) == 0
    st = zf.FriCommitPhase.from_coeffs(rand_field(rng, (1 << 8, 2)), 2, ctx=bctx)
    st.commit_layer(3, 1)
    st.close()
    assert live(bctx) == 0


def test_scratch_entry_points_return_every_buffer(z, bctx):
    from intmax_zkp_core_b200 import prover as Z
    from oracle import perm_ref as PR
    rng = np.random.default_rng(13)
    # hashes and permutations past the 64 KB mailbox take the device-buffer path
    rows = rand_field(rng, (4096, 8))
    z.PoseidonHash.hash_no_pad_batch(rows, bctx)
    z.PoseidonHash.hash_or_noop_batch(rows, bctx)
    z.PoseidonPermutation.permute(rand_field(rng, (1024, 12)), bctx)
    z.PoseidonHash.two_to_one_batch(rand_field(rng, (3000, 4)), rand_field(rng, (3000, 4)), bctx)
    z.PoseidonHash.two_to_one([1, 2, 3, 4], [5, 6, 7, 8], bctx)
    assert live(bctx) == 0
    for n_log in (4, 12):
        x = rand_field(rng, (3, 1 << n_log))
        z.plonky2.fft_batch(x, bctx)
        z.plonky2.ifft_batch(x, bctx)
        z.plonky2.coset_ifft_batch(x, 7, bctx)
        z.plonky2.coset_lde_batch(x, 2, bctx)
        assert live(bctx) == 0
    wires, sigmas, k_is = PR.valid_permutation_instance(12, 6, seed=3)
    Z.zs_partial_products(np.array(wires, np.uint64), np.array(sigmas, np.uint64), np.array(k_is, np.uint64), [3, 4], [5, 6], 8, bctx)
    assert live(bctx) == 0
    b = z.PolynomialBatch.from_coeffs(rand_field(rng, (5, 1 << 12)), 1, False, 0, ctx=bctx)
    held = live(bctx)
    b.eval_ext2([9, 10])
    b.rows([1, 2, 3])
    assert live(bctx) == held
    del b
    assert live(bctx) == 0


def test_pow_grind_failure_returns_its_buffer(z, bctx):
    state = np.arange(12, dtype=np.uint64)
    wit = C.c_uint64()
    rc = bctx._lib.b200zkp_pow_grind(bctx._h, state.ctypes.data_as(C.c_void_p), 5, 7, 40, 1000, C.byref(wit))
    assert rc == ERR_UNSUPPORTED
    assert live(bctx) == 0


def test_one_rank_sharded_commit_returns_every_buffer(z, oracle):
    import torch
    from intmax_zkp_core_b200 import device as D
    n_log, k, r, h = 9, 13, 3, 4
    v = oracle.synthetic_values(k, 1 << n_log, seed=4)
    ref = oracle.commit(v, r, h)
    tctx = D.torch_context(0)
    comm = D.Comm.init_all([tctx])
    assert live(tctx) == 0
    # device inputs
    sh = D.ShardedCommitment(comm, n_log, k, r, h)
    sh.run(torch.from_numpy(v.view(np.int64)).cuda())
    tctx.synchronize()
    assert (sh.cap.cpu().numpy().view(np.uint64) == ref["cap"]).all()
    sh.rows([0, 77])
    sh.close()
    assert live(tctx) == 0
    # host inputs (upload staging on the copy stream)
    cap = np.empty((1 << h, 4), np.uint64)
    hh = C.c_void_p()
    comm.check(tctx._lib.b200zkp_sharded_commit_from_values(comm._h, v.ctypes.data_as(C.c_void_p), n_log, k, r, h,
                                                            cap.ctypes.data_as(C.c_void_p), C.byref(hh)))
    assert (cap == ref["cap"]).all()
    tctx._lib.b200zkp_sharded_free(hh)
    assert live(tctx) == 0
    comm.close()
    tctx.close()
