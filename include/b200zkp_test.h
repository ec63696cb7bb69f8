/* b200zkp_test — probes and micro-benchmarks exported by libb200zkp.so for tests/ and bench.py only.
 * NOT part of the drop-in surface a plonky2 patch binds (include/b200zkp.h is); kept in the same library so the
 * probes exercise exactly the device functions the product kernels inline. */
#ifndef B200ZKP_TEST_H
#define B200ZKP_TEST_H
#include "b200zkp.h"

#ifdef __cplusplus
extern "C" {
#endif

/* device field primitives, element-wise over `count` pairs (test probe for the carry / borrow paths):
 * op 0 mul, 1 add, 2 sub, 3 reduce128(lo = a, hi = b), 4 a + canon(b) lazily,
 * 5 limb recombination O0 + O1*2^22 + O2*2^43 + rc with O0 = a[0:31], O1 = a[32:63], O2 = b[0:31], rc = canon(b >> 1),
 * 6 a^7, 7 (a ^ b) + a * b; every result canonical */
int b200zkp_field_op(b200zkp_ctx* ctx, int op, const uint64_t* a, const uint64_t* b, uint64_t count, uint64_t* out);
/* integer-pipe micro-benchmark (SURVEY.md 8d): runs `iters` dependent-chain rounds of the chosen
 * instruction mix on every SM and returns giga thread-instructions per second in *out_gips.
 * kind: 0 IMAD.WIDE.U32, 1 IADD3, 2 IMAD (32-bit), 3 alternating IMAD.WIDE/LOP3, 4 LOP3, 5 IMAD.HI.U32,
 *       6 alternating IMAD/LOP3, 7 IADD3 + IADD3.X carry pairs, 8 IMAD.WIDE.U32 without accumulator,
 *       9 DFMA, 10 alternating DFMA/IMAD.WIDE.U32, 11 alternating DFMA/IMAD, 12 alternating DFMA/LOP3,
 *       13 alternating IMAD.WIDE.U32/IMAD, 14 alternating IMAD.WIDE.U32 (no accumulator)/LOP3, 15 IMAD.WIDE.U32 : LOP3 = 1 : 3,
 *       16 three-input IADD3 with a uniform operand, 17 alternating three-input IADD3/IMAD,
 *       18 IMAD.WIDE : IMAD : LOP3 : IADD3 = 1 : 2 : 2 : 3, 19 IMAD.WIDE : LOP3 : IMAD = 1 : 2 : 1 */
int b200zkp_int_pipe_bench(b200zkp_ctx* ctx, int kind, uint32_t iters, double* out_gips);
/* device memory of the ctx's buffer pool: *live = bytes handed out and not yet returned (scratch of a call in flight and the
 * buffers of live handles), *cached = bytes kept for reuse (b200zkp_ctx_trim returns them to the driver).  A leak check. */
int b200zkp_ctx_buffer_bytes(b200zkp_ctx* ctx, uint64_t* live, uint64_t* cached);

#ifdef __cplusplus
}
#endif
#endif /* B200ZKP_TEST_H */
