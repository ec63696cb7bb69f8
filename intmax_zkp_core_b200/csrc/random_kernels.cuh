// F::rand_vec on the device: Goldilocks elements from a ChaCha20 keystream (the salts of a blinded PolynomialBatch).
//
// The stream (key, nonce) is defined exactly, so the device, tests/chacha_ref.py and a Rust caller all produce the same words:
//   - ChaCha20 is the RFC 8439 block function: 20 rounds, a 256-bit key, a 32-bit block counter starting at 0, a 96-bit nonce.
//   - Element j is made from keystream bytes [16 j, 16 j + 16): block j / 4, words 4 (j % 4) .. 4 (j % 4) + 3.
//   - Those bytes are read as little-endian u64 lo, hi, and element j = (lo + 2^64 hi) mod p, canonical.
// Reducing 128 uniform bits mod p leaves a statistical distance from uniform below 2^-64 per element.  plonky2's
// F::rand (gen_range on thread_rng) is exactly uniform; the streams differ, and either is a valid salt.
// One thread per ChaCha block: the four elements of a block are stored next to each other, so a warp writes 1 KB runs.
#pragma once
#include "goldilocks.cuh"

namespace rnd {

using gl::u32;
using gl::u64;

// the ChaCha20 inputs that stay fixed over a launch: key words 4..11 and nonce words 13..15 of the initial state
struct ChaChaKey {
    u32 key[8];
    u32 nonce[3];
};

// blocks of the stream are counted in 32 bits: elements [first, first + count) need first + count <= 2^34
GL_HD bool range_ok(u64 first, u64 count) {
    const u64 limit = (u64)1 << 34;
    return first <= limit && count <= limit - first;
}

GL_FN u32 rotl(u32 x, u32 n) {
#ifdef B200ZKP_HOST_EMU
    return (x << n) | (x >> (32 - n));
#else
    return __funnelshift_l(x, x, n);
#endif
}

GL_FN void quarter(u32& a, u32& b, u32& c, u32& d) {
    a += b; d ^= a; d = rotl(d, 16);
    c += d; b ^= c; b = rotl(b, 12);
    a += b; d ^= a; d = rotl(d, 8);
    c += d; b ^= c; b = rotl(b, 7);
}

// RFC 8439 section 2.3: the 16 output words of block `counter`
GL_FN void chacha20_block(const ChaChaKey& k, u32 counter, u32 out[16]) {
    u32 x[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u,
                 k.key[0], k.key[1], k.key[2], k.key[3], k.key[4], k.key[5], k.key[6], k.key[7],
                 counter, k.nonce[0], k.nonce[1], k.nonce[2]};
#pragma unroll
    for (int i = 0; i < 10; i++) {
        quarter(x[0], x[4], x[8], x[12]);
        quarter(x[1], x[5], x[9], x[13]);
        quarter(x[2], x[6], x[10], x[14]);
        quarter(x[3], x[7], x[11], x[15]);
        quarter(x[0], x[5], x[10], x[15]);
        quarter(x[1], x[6], x[11], x[12]);
        quarter(x[2], x[7], x[8], x[13]);
        quarter(x[3], x[4], x[9], x[14]);
    }
    out[0] = x[0] + 0x61707865u; out[1] = x[1] + 0x3320646eu; out[2] = x[2] + 0x79622d32u; out[3] = x[3] + 0x6b206574u;
#pragma unroll
    for (int i = 0; i < 8; i++) out[4 + i] = x[4 + i] + k.key[i];
    out[12] = x[12] + counter;
#pragma unroll
    for (int i = 0; i < 3; i++) out[13 + i] = x[13 + i] + k.nonce[i];
}

// four keystream words (w0 lowest) -> (lo + 2^64 hi) mod p, canonical
GL_FN u64 element_of_words(u32 w0, u32 w1, u32 w2, u32 w3) {
    const u64 lo = ((u64)w1 << 32) | w0, hi = ((u64)w3 << 32) | w2;
    return gl::canon_cc(gl::reduce128(lo, hi));
}

// thread t: block first / 4 + t, its elements that fall in [first, first + count) to out[element - first]
GL_FN void random_field_body(const ChaChaKey& k, u64 first, u64 count, u64* __restrict__ out, u64 t) {
    const u64 block = (first >> 2) + t;
    u32 w[16];
    chacha20_block(k, (u32)block, w);
    const u64 end = first + count;
#pragma unroll
    for (int e = 0; e < 4; e++) {
        const u64 j = (block << 2) + e;
        if (j >= first && j < end) out[j - first] = element_of_words(w[4 * e], w[4 * e + 1], w[4 * e + 2], w[4 * e + 3]);
    }
}

// number of blocks (threads) that cover [first, first + count), count > 0
GL_HD u64 blocks_of_range(u64 first, u64 count) { return ((first + count + 3) >> 2) - (first >> 2); }

#ifndef B200ZKP_HOST_EMU
__global__ void __launch_bounds__(256) random_field_kernel(const ChaChaKey k, u64 first, u64 count, u64 n_blocks,
                                                           u64* __restrict__ out) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_blocks) random_field_body(k, first, count, out, t);
}
#endif

}  // namespace rnd
