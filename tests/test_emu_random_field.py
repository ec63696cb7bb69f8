"""rnd::random_field_body (csrc/random_kernels.cuh), the body of b200zkp_dev_random_field stepped block by block on the CPU by
tests/emu/emu_random.cpp, against tests/chacha_ref.py word for word: ranges that start or end inside a ChaCha block, ranges that cross many
blocks, single elements, and the 2^34 element limit of the 32-bit block counter."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import chacha_ref as CR
from helpers import P

HERE = os.path.dirname(os.path.abspath(__file__))
KEY = bytes(range(32))
u64p = C.POINTER(C.c_uint64)


def ptr(a):
    return a.ctypes.data_as(u64p)


@pytest.fixture(scope="module")
def emu():
    """tests/emu/emu_random.cpp built with g++ (rebuilt when it or a kernel header is newer)"""
    so = os.path.join(HERE, "emu", "libemu_random.so")
    src = os.path.join(HERE, "emu", "emu_random.cpp")
    csrc = os.path.join(os.path.dirname(HERE), "intmax_zkp_core_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("random_kernels.cuh", "goldilocks.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", tmp, src])
        os.replace(tmp, so)
    lib = C.CDLL(so)
    lib.emu_random_field.restype = C.c_int
    lib.emu_random_field.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, u64p]
    return lib


def _run(emu, key, nonce, first, count):
    out = np.full(max(count, 1) + 1, 0xDEADBEEF, np.uint64)         # one guard word past the range
    rc = emu.emu_random_field(key, nonce, first, count, ptr(out))
    return rc, out


@pytest.mark.parametrize("first,count", [(0, 1), (3, 1), (0, 4), (1, 2), (1, 3), (2, 7), (5, 11), (0, 4096), (3, 4093),
                                         (1000001, 3001), (4 * 12345 + 2, 1), (2**34 - 5, 5), (2**34 - 1, 1)])
def test_random_field_body_equals_chacha_ref(emu, first, count):
    for nonce in (CR.nonce_for_oracle(1), bytes.fromhex("000000090000004a00000000")):
        rc, out = _run(emu, KEY, nonce, first, count)
        assert rc == 0
        want = CR.elements(KEY, nonce, first, count)
        assert (out[:count] == want).all(), (first, count)
        assert out[count] == 0xDEADBEEF                              # nothing written past the range
        assert (out[:count] < P).all()


def test_random_field_body_limits(emu):
    rc, out = _run(emu, KEY, bytes(12), 0, 0)
    assert rc == 0 and out[0] == 0xDEADBEEF                          # count 0 writes nothing
    assert _run(emu, KEY, bytes(12), 2**34 - 4, 5)[0] == -1         # block 2^32 would be needed
    assert _run(emu, KEY, bytes(12), 2**34, 1)[0] == -1


def test_random_field_body_other_keys(emu):
    rng = np.random.default_rng(5)
    for _ in range(4):
        key, nonce = rng.bytes(32), rng.bytes(12)
        first, count = int(rng.integers(0, 10**6)), int(rng.integers(1, 600))
        rc, out = _run(emu, key, nonce, first, count)
        assert rc == 0 and (out[:count] == CR.elements(key, nonce, first, count)).all()
