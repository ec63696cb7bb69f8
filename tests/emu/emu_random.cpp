// TEST HARNESS (not product): the body of b200zkp_dev_random_field (csrc/random_kernels.cuh) compiled with g++ under
// B200ZKP_HOST_EMU, its "threads" stepped in a loop, so the ChaCha20 block function, the element mapping and the masking of
// unaligned ranges can be checked on a machine without a GPU.  The product library never defines B200ZKP_HOST_EMU.
#define B200ZKP_HOST_EMU 1
#define __restrict__
#include <cstring>

#include "../../intmax_zkp_core_b200/csrc/random_kernels.cuh"

using gl::u64;

extern "C" {
// rnd::random_field_body stepped over every block of [first, first + count); key / nonce as bytes.  Returns -1 where the
// entry point returns B200ZKP_ERR_BAD_ARG for the range.
int emu_random_field(const unsigned char* key, const unsigned char* nonce, u64 first, u64 count, u64* out) {
    if (!count) return 0;
    if (!rnd::range_ok(first, count)) return -1;
    rnd::ChaChaKey k;
    for (int i = 0; i < 8; i++) memcpy(&k.key[i], key + 4 * i, 4);        // (little-endian host)
    for (int i = 0; i < 3; i++) memcpy(&k.nonce[i], nonce + 4 * i, 4);
    const u64 n_blocks = rnd::blocks_of_range(first, count);
    for (u64 t = 0; t < n_blocks; t++) rnd::random_field_body(k, first, count, out, t);
    return 0;
}
}
