"""TEST INFRASTRUCTURE: the ChaCha20 field-element stream of b200zkp_dev_random_field, restated with numpy.

    ChaCha20 is the RFC 8439 block function: 20 rounds, a 256-bit key, a 32-bit block counter and a 96-bit nonce.
    Element j of the stream (key, nonce) is made from keystream bytes [16 j, 16 j + 16): block j / 4, words 4 (j % 4) ..
    4 (j % 4) + 3.  Those bytes are read as little-endian u64 lo, hi, and element j = (lo + 2^64 hi) mod p.

The block function is vectorised over blocks with numpy uint32 (wrapping adds, xors, rotations)."""
from __future__ import annotations

import numpy as np

P = 0xFFFFFFFF00000001
SIGMA = (0x61707865, 0x3320646E, 0x79622D32, 0x6B206574)       # "expand 32-byte k"


def _rotl(x: np.ndarray, n: int) -> np.ndarray:
    return (x << np.uint32(n)) | (x >> np.uint32(32 - n))


def _quarter(s, a, b, c, d):
    s[a] += s[b]; s[d] ^= s[a]; s[d] = _rotl(s[d], 16)
    s[c] += s[d]; s[b] ^= s[c]; s[b] = _rotl(s[b], 12)
    s[a] += s[b]; s[d] ^= s[a]; s[d] = _rotl(s[d], 8)
    s[c] += s[d]; s[b] ^= s[c]; s[b] = _rotl(s[b], 7)


def blocks(key: bytes, nonce: bytes, counters) -> np.ndarray:
    """the ChaCha20 blocks of (key, nonce) at the given 32-bit counters: (len(counters), 16) uint32 words"""
    assert len(key) == 32 and len(nonce) == 12
    ctr = np.asarray(counters, dtype=np.uint64)
    assert ctr.ndim == 1 and (ctr < 2**32).all()
    k = np.frombuffer(key, dtype="<u4").astype(np.uint32)
    nw = np.frombuffer(nonce, dtype="<u4").astype(np.uint32)
    m = ctr.size
    init = np.empty((16, m), dtype=np.uint32)
    init[0:4] = np.array(SIGMA, dtype=np.uint32)[:, None]
    init[4:12] = k[:, None]
    init[12] = ctr.astype(np.uint32)
    init[13:16] = nw[:, None]
    s = [init[i].copy() for i in range(16)]
    with np.errstate(over="ignore"):
        for _ in range(10):
            _quarter(s, 0, 4, 8, 12); _quarter(s, 1, 5, 9, 13); _quarter(s, 2, 6, 10, 14); _quarter(s, 3, 7, 11, 15)
            _quarter(s, 0, 5, 10, 15); _quarter(s, 1, 6, 11, 12); _quarter(s, 2, 7, 8, 13); _quarter(s, 3, 4, 9, 14)
        out = np.stack(s) + init
    return np.ascontiguousarray(out.T)


def keystream(key: bytes, nonce: bytes, first_block: int, n_blocks: int) -> bytes:
    """n_blocks * 64 keystream bytes from block counter first_block on"""
    return blocks(key, nonce, np.arange(first_block, first_block + n_blocks, dtype=np.uint64)).astype("<u4").tobytes()


def elements(key: bytes, nonce: bytes, first: int, count: int) -> np.ndarray:
    """elements [first, first + count) of the stream (key, nonce): canonical uint64"""
    if count == 0:
        return np.zeros(0, dtype=np.uint64)
    b0, b1 = first // 4, (first + count + 3) // 4
    w = blocks(key, nonce, np.arange(b0, b1, dtype=np.uint64)).reshape(-1, 4).astype(np.uint64)
    w = w[first - 4 * b0:first - 4 * b0 + count]
    lo = w[:, 0] | (w[:, 1] << np.uint64(32))
    hi = w[:, 2] | (w[:, 3] << np.uint64(32))
    # (lo + 2^64 hi) mod p with 2^64 = 2^32 - 1 (mod p), in Python integers for clarity
    return np.array([(int(l) + int(h) * 0xFFFFFFFF) % P for l, h in zip(lo.tolist(), hi.tolist())], dtype=np.uint64)


def nonce_for_oracle(index: int) -> bytes:
    """the nonce prove() uses for the salt of PlonkOracle `index`: le32(index) || 8 zero bytes"""
    return int(index).to_bytes(4, "little") + bytes(8)
