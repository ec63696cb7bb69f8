"""Kernel-body logic on the CPU: tests/emu/emu.cpp compiles the CUDA kernel bodies (csrc/*.cuh) with g++ under
B200ZKP_HOST_EMU and steps the threads of each CTA in a loop.  This checks the index logic of the NTT passes,
the Poseidon arithmetic and the digest slot formula against the oracle without a GPU.  It is NOT a product
path (the library has no CPU mode); the GPU parity tests proper are in test_gpu_*.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import P, bitrev_perm, hostile_columns, rand_field

HERE = os.path.dirname(os.path.abspath(__file__))
u64p = C.POINTER(C.c_uint64)


def ptr(a):
    return a.ctypes.data_as(u64p)


@pytest.fixture(scope="module")
def emu():
    so = os.path.join(HERE, "emu", "libemu.so")
    src = os.path.join(HERE, "emu", "emu.cpp")
    csrc = os.path.join(os.path.dirname(HERE), "intmax_zkp_core_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc)]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src])
    lib = C.CDLL(so)
    lib.emu_node_slot.restype = C.c_uint64
    lib.emu_node_slot.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint64]
    lib.emu_sponge.argtypes = [u64p, C.c_uint64, C.c_uint32, C.c_uint32, u64p]
    lib.emu_ct_plan_tma.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_int]
    return lib


def test_permutation_body(emu, oracle):
    rng = np.random.default_rng(11)
    states = [np.zeros(12, np.uint64), np.arange(12, dtype=np.uint64), np.full(12, P - 1, np.uint64),
              np.full(12, 2**64 - 1, np.uint64), np.full(12, P, np.uint64)]
    states += [rng.integers(0, 2**64, size=12, dtype=np.uint64) for _ in range(400)]
    # words 0 / 6 / 3 / 9 feed the split-basis components with the largest gains
    for w in (0, 3, 6, 9):
        st = np.zeros(12, np.uint64); st[w] = 2**64 - 1; states.append(st)
        st = np.full(12, 2**64 - 1, np.uint64); st[w] = 0; states.append(st)
    for st in states:
        got = st.copy()
        emu.emu_permute(ptr(got))
        assert (got == oracle.permute(st)).all()


def test_sponge_body(emu, oracle):
    rng = np.random.default_rng(12)
    for L in (0, 1, 3, 4, 5, 7, 8, 9, 12, 16, 17, 20, 135, 139):
        x = rng.integers(0, 2**64, size=max(L, 1), dtype=np.uint64)
        out = np.zeros(4, np.uint64)
        emu.emu_sponge(ptr(x), 1, L, 1, ptr(out))
        assert (out == oracle.hash_or_noop(x[:L])).all(), L
        emu.emu_sponge(ptr(x), 1, L, 0, ptr(out))
        assert (out == oracle.hash_no_pad(x[:L])).all(), L
    # strided (column-major) leaf
    m = rng.integers(0, 2**64, size=(20, 6), dtype=np.uint64)
    out = np.zeros(4, np.uint64)
    flat = np.ascontiguousarray(m)
    emu.emu_sponge(C.cast(C.addressof(ptr(flat).contents) + 8 * 2, u64p), 6, 20, 1, ptr(out))
    assert (out == oracle.hash_or_noop(m[:, 2])).all()


def test_sponge_in_pieces(emu, oracle):
    """merkle::sponge_absorb (the resumable leaf hash of the partitioned commitment): any cut at multiples of the rate gives
    hash_no_pad of the whole leaf, ragged tail included"""
    rng = np.random.default_rng(14)
    u32p = C.POINTER(C.c_uint32)
    for L, cuts in ((135, [8, 16, 64, 128]), (135, [128]), (135, list(range(8, 135, 8))), (20, [16]), (16, [8]), (9, [8]), (24, [])):
        x = rng.integers(0, P, size=L, dtype=np.uint64)
        out = np.zeros(4, np.uint64)
        cu = np.array(cuts + [0], np.uint32)
        emu.emu_sponge_pieces(ptr(x), 1, L, cu.ctypes.data_as(u32p), len(cuts), ptr(out))
        assert (out == oracle.hash_no_pad(x)).all(), (L, cuts)


def test_digest_slots_match_recursive_layout(emu, oracle):
    """node_slot (index formula used by the kernels) == where plonky2's recursive fill puts each digest."""
    rng = np.random.default_rng(13)
    for (N, h) in ((16, 0), (16, 2), (32, 1), (8, 3)):
        leaves = rand_field(rng, (N, 6))
        dig, cap = oracle.merkle_new(leaves, h)
        sub_log = (N.bit_length() - 1) - h
        sub = 1 << sub_log
        for s in range(1 << h):
            layer = [oracle.hash_or_noop(leaves[s * sub + m]) for m in range(sub)]
            for i in range(sub_log):
                for m, d in enumerate(layer):
                    assert (dig[emu.emu_node_slot(sub_log, s, i, m)] == d).all()
                layer = [oracle.two_to_one(layer[2 * q], layer[2 * q + 1]) for q in range(len(layer) // 2)]
            assert (cap[s] == layer[0]).all()


@pytest.mark.parametrize("n_log", [0, 1, 2, 3, 4, 6, 8, 9, 10, 11, 12, 16, 17, 19, 20])
def test_ntt_pass_bodies(emu, oracle, n_log):
    rng = np.random.default_rng(100 + n_log)
    k = 3 if n_log < 14 else 1
    n = 1 << n_log
    v = rng.integers(0, 2**64, size=(k, n), dtype=np.uint64)       # includes non-canonical inputs
    out = np.zeros_like(v)
    emu.emu_ntt(ptr(v), ptr(out), n_log, k)
    assert (out == np.stack([oracle.fft(c) for c in v])).all()
    emu.emu_intt(ptr(v), ptr(out), n_log, k)
    assert (out == np.stack([oracle.ifft(c) for c in v])).all()
    for r in ((0, 1, 3) if n_log < 12 else (3,)):
        N = n << r
        lde = np.zeros((k, N), np.uint64)
        emu.emu_lde(ptr(v), ptr(lde), n_log, k, r)
        perm = bitrev_perm(n_log + r)
        for c in range(k):
            assert (lde[c] == oracle.coset_lde(v[c], r)[perm]).all()


@pytest.mark.parametrize("n_log", [11, 12, 13, 14, 15, 16, 17, 18])
def test_ct_pass_bodies(emu, oracle, n_log):
    """second-generation passes (ntt_ct_kernels.cuh): inverse transform in natural order, coset LDE blocks in leaf order"""
    rng = np.random.default_rng(200 + n_log)
    k = 2 if n_log < 15 else 1
    n = 1 << n_log
    v = rng.integers(0, 2**64, size=(k, n), dtype=np.uint64)       # includes non-canonical inputs
    v[0, :4] = [2**64 - 1, P, P - 1, 0]
    out = np.zeros_like(v)
    assert emu.emu_ct_intt(ptr(v), ptr(out), n_log, k) == 1
    assert (out == np.stack([oracle.ifft(c) for c in v])).all()
    cases = [(3, 0, 8)] if n_log > 13 else [(3, 0, 8), (3, 2, 4), (1, 0, 2), (0, 0, 1), (3, 5, 6), (4, 0, 16)]
    for r, b0, b1 in cases:
        N = n << r
        lde = np.zeros((k, (b1 - b0) * n), np.uint64)
        assert emu.emu_ct_lde(ptr(v), ptr(lde), n_log, k, r, b0, b1) == 1
        perm = bitrev_perm(n_log + r)
        for c in range(k):
            assert (lde[c] == oracle.coset_lde(v[c], r)[perm][b0 * n:b1 * n]).all(), (r, b0, b1)


@pytest.mark.parametrize("n_log", [11, 12, 13, 14, 15, 16, 17, 19, 20])
def test_ct_plan_other_paths(emu, n_log):
    """The plans test_gpu_parity.py::test_second_generation_passes counts on to reach the other transform paths on one
    context: make_plan refuses an odd output column stride (the last pass moves pairs of elements), so b200zkp_dev_intt and
    b200zkp_dev_lde fall back to the four-step kernels (ntt_kernels.cuh); and with 16 coset blocks the first pass reads the
    one input block for every block (block stride 0), so it stages with plain loads while the other strided passes keep TMA."""
    n, k = 1 << n_log, 2
    strided = (1 << ((n_log + 7) // 8 - 1)) - 1          # every pass but the last (which never uses TMA)
    assert emu.emu_ct_plan_tma(n_log, k, n, 1, 1) == strided
    assert emu.emu_ct_plan_tma(n_log, k, n + 1, 1, 1) == -1
    for nb in (1, 2, 8, 16):
        assert emu.emu_ct_plan_tma(n_log, k, nb * n, nb, 0) == (strided & ~1 if nb == 16 else strided), nb
        assert emu.emu_ct_plan_tma(n_log, k, nb * n + 1, nb, 0) == -1, nb


def owned_columns(k, G, g):
    """partition of the columns over G ranks (sharded.inl): groups of L = max(8, G) columns, w = L / G of each group per rank"""
    L = max(8, G)
    w = L // G
    return [c for c in range(k) if (c % L) // w == g]


@pytest.mark.parametrize("n_log,k,G", [(11, 7, 2), (12, 21, 4), (13, 11, 2), (11, 19, 8)])
def test_ct_pull_pass_bodies(emu, oracle, n_log, k, G):
    """partitioned LDE (sharded.inl): the first pass gathers the columns of a group range from per-rank coefficient windows
    (KIND_PULL_LOOP, stepped on the host with the plain-load staging), later passes walk the same columns in place; rank g keeps
    coset blocks [g * 2^r / G, (g + 1) * 2^r / G).  Also: the columns of one source only (the shard-by-shard pipeline)."""
    rng = np.random.default_rng(300 + n_log)
    n, r = 1 << n_log, 3
    L = max(8, G)
    w = L // G
    kp = -(-k // L) * w
    c = rng.integers(0, 2**64, size=(k, n), dtype=np.uint64)
    win = [np.zeros((kp, n), np.uint64) for _ in range(G)]
    for q in range(G):
        cols = owned_columns(k, G, q)
        win[q][:len(cols)] = c[cols]
    srcs = (u64p * G)(*[ptr(x) for x in win])
    bpr = (1 << r) // G
    for g in (0, G - 1):
        b0, b1 = g * bpr, (g + 1) * bpr
        want = np.zeros((k, (b1 - b0) * n), np.uint64)
        assert emu.emu_ct_lde(ptr(c), ptr(want), n_log, k, r, b0, b1) == 1
        # group by group (the host-input pipeline), gathering
        copy = np.zeros((k, n), np.uint64)
        lde = np.zeros_like(want)
        for col0 in range(0, k, L):
            cnt = min(L, k - col0)
            assert emu.emu_ct_lde_cols(srcs, G, w, k, col0, cnt, 0, 0, 1, ptr(copy), ptr(lde), n_log, r, b0, b1) == 1
        assert (copy == c).all()
        assert (lde == want).all()
        # an arbitrary column range in one go (device inputs), gathering
        copy2 = np.zeros((k, n), np.uint64)
        lde2 = np.zeros_like(want)
        cut = min(k, 5)
        assert emu.emu_ct_lde_cols(srcs, G, w, k, 0, cut, 0, 0, 1, ptr(copy2), ptr(lde2), n_log, r, b0, b1) == 1
        if k > cut:
            assert emu.emu_ct_lde_cols(srcs, G, w, k, cut, k - cut, 0, 0, 1, ptr(copy2), ptr(lde2), n_log, r, b0, b1) == 1
        assert (copy2 == c).all() and (lde2 == want).all()
        # shard by shard from the gathered matrix (no gather): the columns of one source at a time
        lde3 = np.zeros_like(want)
        for q in range(G):
            cnt = len(owned_columns(k, G, q))
            if cnt:
                assert emu.emu_ct_lde_cols(srcs, G, w, k, 0, -(-cnt // w) * w, 1, q, 0, ptr(copy), ptr(lde3), n_log, r, b0, b1) == 1
        assert (lde3 == want).all()


def test_ntt_hostile_columns(emu, oracle):
    v = hostile_columns(64)
    out = np.zeros_like(v)
    emu.emu_intt(ptr(v), ptr(out), 6, v.shape[0])
    assert (out == np.stack([oracle.ifft(c) for c in v])).all()


def test_permutation_argument_rows(emu):
    """perm::row_chunk_products + perm::inverse (row N1a) against the pure-Python restatement oracle/perm_ref.py"""
    from oracle import perm_ref as PR
    import random
    emu.emu_inverse.restype = C.c_uint64
    emu.emu_inverse.argtypes = [C.c_uint64]
    rnd = random.Random(3)
    for x in [1, 2, P - 1, 7, 2**32, 2**32 - 1] + [rnd.randrange(1, P) for _ in range(50)]:
        assert emu.emu_inverse(x) * x % P == 1
    assert emu.emu_inverse(0) == 0
    for R, degree, n_log, Cn in ((12, 8, 5, 2), (80, 8, 4, 2), (7, 3, 3, 1), (5, 8, 2, 3)):
        wires, sigmas, k_is = PR.valid_permutation_instance(R, n_log, seed=R)
        betas = [rnd.randrange(P) for _ in range(Cn)]
        gammas = [rnd.randrange(P) for _ in range(Cn)]
        n = 1 << n_log
        chunks = (R + degree - 1) // degree
        running = np.zeros(Cn * chunks * n, np.uint64)
        w = np.array(wires, np.uint64)
        s = np.array(sigmas, np.uint64)
        emu.emu_perm_rows(ptr(w), ptr(s), ptr(np.array(k_is, np.uint64)), ptr(np.array(betas, np.uint64)),
                          ptr(np.array(gammas, np.uint64)), n_log, R, degree, Cn, ptr(running))
        running = running.reshape(Cn, chunks, n)
        cols = PR.partial_products_and_zs(wires, sigmas, k_is, betas, gammas, degree)
        num_prods = chunks - 1
        for c in range(Cn):
            z = cols[c]
            for i in range(n):
                for l in range(num_prods):
                    assert int(running[c, l, i]) * z[i] % P == cols[Cn + c * num_prods + l][i]
                assert int(running[c, chunks - 1, i]) * z[i] % P == (z[i + 1] if i + 1 < n else 1)


@pytest.mark.parametrize("n_log,extended", [(3, False), (5, True)])
def test_quotient_point_body(emu, oracle, n_log, extended):
    """row N1b: the per-point body of vanishing_kernels.cuh against oracle/vanishing_ref.py on a satisfied synthetic circuit
    (extended: with rows of all thirteen gate kinds)"""
    import random
    from oracle import perm_ref as PR
    from oracle import vanishing_ref as V
    r = 3
    c = V.Circuit(n_log, seed=1, extended=extended)
    rnd = random.Random(8)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zs_pp = PR.partial_products_and_zs([c.wires[j] for j in range(80)], c.sigmas, c.k_is, betas, gammas, 8)
    lde = lambda cols: [oracle.coset_lde(oracle.ifft(np.array(col, np.uint64)), r) for col in cols]
    l_cs, l_w, l_z = lde(c.constants + c.sigmas), lde(c.wires), lde(zs_pp)
    want = np.array(V.quotient_values(c, l_cs, l_w, l_z, betas, gammas, alphas, 8, r, 3), np.uint64)
    perm = bitrev_perm(n_log + r)
    leaf = lambda cols: np.ascontiguousarray(np.stack([col[perm] for col in cols]))
    gates = np.array([[g, c.selector_indices[i], *c.groups[c.selector_indices[i]], *(list(c.gate_params[i]) + [0, 0, 0])[:3]]
                      for i, g in enumerate(c.gates)], np.uint32)
    out = np.zeros((2, 1 << (n_log + r)), np.uint64)
    u32p = C.POINTER(C.c_uint32)
    a = lambda v: np.array(v, np.uint64)
    cs_l, w_l, z_l = leaf(l_cs), leaf(l_w), leaf(l_z)
    emu.emu_quotient_values(ptr(cs_l), ptr(w_l), ptr(z_l), n_log, 3, c.num_selectors, 2, 8, gates.ctypes.data_as(u32p), len(c.gates),
                            ptr(a(c.k_is)), ptr(a(betas)), ptr(a(gammas)), ptr(a(alphas)), ptr(a(c.pi_hash)), ptr(out))
    assert (out == want).all()
