//! NOT BUILT IN THIS ENVIRONMENT (no Rust toolchain) — see INTEGRATION.md.
//! Raw bindings to include/b200zkp.h, one `extern "C"` item per declared entry point used by the plonky2 patch.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct b200zkp_ctx { _p: [u8; 0] }
#[repr(C)] pub struct b200zkp_batch { _p: [u8; 0] }
#[repr(C)] pub struct b200zkp_fri { _p: [u8; 0] }
#[repr(C)] pub struct b200zkp_tree { _p: [u8; 0] }
#[repr(C)] pub struct b200zkp_comm { _p: [u8; 0] }
#[repr(C)] pub struct b200zkp_sharded { _p: [u8; 0] }

pub const B200ZKP_COMM_ID_BYTES: usize = 128;
pub const B200ZKP_SALT_SIZE: u32 = 4; // plonky2 fri/oracle.rs SALT_SIZE
pub const B200ZKP_MAX_GATES: usize = 32; // 16 before the plonky2_u32 gates (b200zkp_vanishing_desc layout changed)
/// gate kinds of `b200zkp_vanishing_desc::gate_kind` (include/b200zkp.h B200ZKP_GATE_*); parameters in `gate_params`
pub const B200ZKP_GATE_NOOP: u32 = 0;
pub const B200ZKP_GATE_CONSTANT: u32 = 1;
pub const B200ZKP_GATE_PUBLIC_INPUT: u32 = 2;
pub const B200ZKP_GATE_ARITHMETIC: u32 = 3;
pub const B200ZKP_GATE_POSEIDON: u32 = 4;
pub const B200ZKP_GATE_ARITHMETIC_EXTENSION: u32 = 5;
pub const B200ZKP_GATE_MUL_EXTENSION: u32 = 6;
pub const B200ZKP_GATE_BASE_SUM: u32 = 7; // { B, num_limbs }
pub const B200ZKP_GATE_REDUCING: u32 = 8; // { num_coeffs }
pub const B200ZKP_GATE_REDUCING_EXTENSION: u32 = 9; // { num_coeffs }
pub const B200ZKP_GATE_RANDOM_ACCESS: u32 = 10; // { bits, num_copies, num_extra_constants }
pub const B200ZKP_GATE_EXPONENTIATION: u32 = 11; // { num_power_bits }
pub const B200ZKP_GATE_POSEIDON_MDS: u32 = 12;
// 13 is not assigned
pub const B200ZKP_GATE_INTERPOLATION_HIGH_DEGREE: u32 = 14;
pub const B200ZKP_GATE_INTERPOLATION_LOW_DEGREE: u32 = 15;
// plonky2_u32 / plonky2_ecdsa gates
pub const B200ZKP_GATE_U32_ARITHMETIC: u32 = 16; // { num_ops }
pub const B200ZKP_GATE_U32_ADD_MANY: u32 = 17; // { num_addends, num_ops }
pub const B200ZKP_GATE_U32_SUBTRACTION: u32 = 18; // { num_ops }
pub const B200ZKP_GATE_U32_RANGE_CHECK: u32 = 19; // { num_input_limbs }
pub const B200ZKP_GATE_COMPARISON: u32 = 20; // { num_bits, num_chunks }

/// include/b200zkp.h `b200zkp_vanishing_desc` (row N1b: what compute_quotient_polys reads of CommonCircuitData)
#[repr(C)]
pub struct b200zkp_vanishing_desc {
    pub degree_bits: u32,
    pub quotient_degree_bits: u32,
    pub quotient_degree_factor: u32,
    pub num_routed_wires: u32,
    pub num_challenges: u32,
    pub num_selectors: u32,
    pub n_gates: u32,
    pub gate_kind: [u32; B200ZKP_MAX_GATES],
    pub gate_selector_index: [u32; B200ZKP_MAX_GATES],
    pub gate_group_begin: [u32; B200ZKP_MAX_GATES],
    pub gate_group_end: [u32; B200ZKP_MAX_GATES],
    pub gate_params: [[u32; 3]; B200ZKP_MAX_GATES],
    pub k_is: *const u64,
    pub betas: *const u64,
    pub gammas: *const u64,
    pub alphas: *const u64,
    pub public_inputs_hash: [u64; 4],
}

extern "C" {
    pub fn b200zkp_ctx_create(device: c_int, stream: *mut c_void, out: *mut *mut b200zkp_ctx) -> c_int;
    pub fn b200zkp_ctx_destroy(ctx: *mut b200zkp_ctx);
    pub fn b200zkp_last_error(ctx: *const b200zkp_ctx) -> *const c_char;

    pub fn b200zkp_commit_from_values(ctx: *mut b200zkp_ctx, values: *const u64, n_log: u32, k: u32, rate_bits: u32,
        cap_height: u32, salt: *const u64, out: *mut *mut b200zkp_batch) -> c_int;
    pub fn b200zkp_commit_from_coeffs(ctx: *mut b200zkp_ctx, coeffs: *const u64, n_log: u32, k: u32, rate_bits: u32,
        cap_height: u32, salt: *const u64, out: *mut *mut b200zkp_batch) -> c_int;
    pub fn b200zkp_batch_free(b: *mut b200zkp_batch);
    pub fn b200zkp_batch_cap(b: *mut b200zkp_batch, out: *mut u64) -> c_int;
    pub fn b200zkp_batch_shape(b: *const b200zkp_batch, shape: *mut u32) -> c_int;
    pub fn b200zkp_batch_coeffs(b: *mut b200zkp_batch, out: *mut u64) -> c_int;
    pub fn b200zkp_batch_leaves(b: *mut b200zkp_batch, out: *mut u64) -> c_int;
    pub fn b200zkp_batch_digests(b: *mut b200zkp_batch, out: *mut u64) -> c_int;
    pub fn b200zkp_batch_rows(b: *mut b200zkp_batch, idx: *const u64, n_idx: u64, rows: *mut u64, siblings: *mut u64) -> c_int;
    pub fn b200zkp_batch_lde_values(b: *mut b200zkp_batch, index: u64, step: u64, out: *mut u64) -> c_int;

    pub fn b200zkp_merkle_new(ctx: *mut b200zkp_ctx, leaves: *const u64, n_leaves: u64, leaf_len: u32, cap_height: u32,
        out: *mut *mut b200zkp_tree) -> c_int;
    pub fn b200zkp_tree_free(t: *mut b200zkp_tree);
    pub fn b200zkp_tree_cap(t: *mut b200zkp_tree, out: *mut u64) -> c_int;
    pub fn b200zkp_tree_digests(t: *mut b200zkp_tree, out: *mut u64) -> c_int;
    pub fn b200zkp_tree_prove(t: *mut b200zkp_tree, idx: *const u64, n_idx: u64, siblings: *mut u64) -> c_int;

    pub fn b200zkp_hash_no_pad(ctx: *mut b200zkp_ctx, input: *const u64, count: u64, len: u32, out: *mut u64) -> c_int;
    pub fn b200zkp_two_to_one(ctx: *mut b200zkp_ctx, left: *const u64, right: *const u64, count: u64, out: *mut u64) -> c_int;
    // opening proof (prove_openings / fri_proof): see include/b200zkp.h and INTEGRATION.md
    pub fn b200zkp_batch_eval_ext2(b: *mut b200zkp_batch, zeta: *const u64, out: *mut u64) -> c_int;
    // the whole prove() on the device: commitments of matrices already in HBM, OpeningSet::new in one call
    pub fn b200zkp_batch_from_device(ctx: *mut b200zkp_ctx, in_dev: *const u64, is_coeffs: c_int, n_log: u32, k: u32,
        rate_bits: u32, cap_height: u32, salt_dev: *const u64, out: *mut *mut b200zkp_batch) -> c_int;
    // zero_knowledge: F::rand_vec on the device, out_dev[e] = element (first + e) of the ChaCha20 stream (key, nonce)
    pub fn b200zkp_dev_random_field(ctx: *mut b200zkp_ctx, key: *const u8, nonce: *const u8, first: u64, count: u64,
        out_dev: *mut u64) -> c_int;
    pub fn b200zkp_batch_openings(ctx: *mut b200zkp_ctx, oracles: *const *mut b200zkp_batch, n_oracles: u32, n_points: u32,
        points: *const u64, point_n_polys: *const u32, poly_oracle: *const u32, poly_index: *const u32, out: *mut u64) -> c_int;
    pub fn b200zkp_fri_begin(ctx: *mut b200zkp_ctx, oracles: *const *mut b200zkp_batch, n_oracles: u32, n_points: u32,
        points: *const u64, point_n_polys: *const u32, poly_oracle: *const u32, poly_index: *const u32, alpha: *const u64,
        flags: u32, out: *mut *mut b200zkp_fri) -> c_int;
    pub fn b200zkp_fri_free(f: *mut b200zkp_fri);
    pub fn b200zkp_fri_shape(f: *const b200zkp_fri, shape: *mut u32) -> c_int;
    pub fn b200zkp_fri_commit_layer(f: *mut b200zkp_fri, arity_bits: u32, cap_height: u32, cap_out: *mut u64) -> c_int;
    pub fn b200zkp_fri_fold(f: *mut b200zkp_fri, beta: *const u64) -> c_int;
    pub fn b200zkp_fri_final_poly(f: *mut b200zkp_fri, out: *mut u64) -> c_int;
    pub fn b200zkp_fri_query(f: *mut b200zkp_fri, layer: u32, idx: *const u64, n_idx: u64, evals: *mut u64, siblings: *mut u64) -> c_int;
    pub fn b200zkp_pow_grind(ctx: *mut b200zkp_ctx, state: *const u64, witness_pos: u32, response_pos: u32,
        min_leading_zeros: u32, max_candidates: u64, witness: *mut u64) -> c_int;
    // row N1c: PolynomialValues::coset_ifft(shift) in place, k columns of 2^n_log values
    pub fn b200zkp_coset_intt(ctx: *mut b200zkp_ctx, data: *mut u64, n_log: u32, k: u32, shift: u64) -> c_int;
    pub fn b200zkp_dev_coset_intt(ctx: *mut b200zkp_ctx, values: *const u64, in_stride: u64, coeffs: *mut u64, out_stride: u64,
        scratch: *mut u64, n_log: u32, k: u32, shift: u64) -> c_int;
    // row N1a: prover.rs wires_permutation_partial_products_and_zs for every challenge, columns in committed order
    pub fn b200zkp_partial_products_and_zs(ctx: *mut b200zkp_ctx, wires: *const u64, sigmas: *const u64, n_log: u32,
        num_routed: u32, degree: u32, k_is: *const u64, betas: *const u64, gammas: *const u64, num_challenges: u32,
        out: *mut u64) -> c_int;
    pub fn b200zkp_dev_partial_products_and_zs(ctx: *mut b200zkp_ctx, wires_dev: *const u64, wires_col_stride: u64,
        sigmas_dev: *const u64, sigmas_col_stride: u64, n_log: u32, num_routed: u32, degree: u32, k_is: *const u64,
        betas: *const u64, gammas: *const u64, num_challenges: u32, out_dev: *mut u64, out_col_stride: u64) -> c_int;
    // Fiat-Shamir transcript: any number of duplexing steps in one launch (iop/challenger.rs)
    pub fn b200zkp_duplex_chain(ctx: *mut b200zkp_ctx, state: *mut u64, inputs: *const u64, n_inputs: u64, n_squeeze: u32,
        squeezed: *mut u64) -> c_int;
    // row N1b: compute_quotient_polys up to its coset_ifft, on the device-resident LDEs
    pub fn b200zkp_dev_quotient_values(ctx: *mut b200zkp_ctx, desc: *const b200zkp_vanishing_desc, constants_sigmas: *const u64,
        cs_stride: u64, wires: *const u64, wires_stride: u64, zs_partial_products: *const u64, zpp_stride: u64,
        out_dev: *mut u64, out_stride: u64) -> c_int;
    pub fn b200zkp_ctx_trim(ctx: *mut b200zkp_ctx) -> c_int;
    pub fn b200zkp_ctx_set_pool_limit(ctx: *mut b200zkp_ctx, bytes: u64) -> c_int;

    // one commitment partitioned over every GPU of the box, driven by this (single, rayon) process: NCCL inside the library
    pub fn b200zkp_comm_init_all(ctxs: *const *mut b200zkp_ctx, n: c_int, out: *mut *mut b200zkp_comm) -> c_int;
    pub fn b200zkp_comm_unique_id(id: *mut u8) -> c_int;
    pub fn b200zkp_comm_init_rank(ctx: *mut b200zkp_ctx, id: *const u8, rank: c_int, world: c_int, out: *mut *mut b200zkp_comm) -> c_int;
    pub fn b200zkp_comm_destroy(comm: *mut b200zkp_comm);
    pub fn b200zkp_comm_last_error(comm: *const b200zkp_comm) -> *const c_char;
    pub fn b200zkp_comm_shape(comm: *const b200zkp_comm, shape: *mut i32) -> c_int;
    pub fn b200zkp_comm_set_exchange_group(comm: *mut b200zkp_comm, peers_per_group: u32) -> c_int;
    pub fn b200zkp_comm_set_peer_exchange(comm: *mut b200zkp_comm, enabled: c_int) -> c_int;
    pub fn b200zkp_comm_peer_exchange(comm: *const b200zkp_comm) -> c_int;
    pub fn b200zkp_sharded_create(comm: *mut b200zkp_comm, n_log: u32, k: u32, rate_bits: u32, cap_height: u32,
        out: *mut *mut b200zkp_sharded) -> c_int;
    pub fn b200zkp_sharded_free(sh: *mut b200zkp_sharded);
    pub fn b200zkp_sharded_layout(sh: *const b200zkp_sharded, local: c_int, lay: *mut u64) -> c_int;
    pub fn b200zkp_sharded_columns(sh: *const b200zkp_sharded, local: c_int, cols: *mut u32, capacity: u32, n_cols: *mut u32) -> c_int;
    pub fn b200zkp_sharded_commit(sh: *mut b200zkp_sharded, inputs: *const *const u64, inputs_on_device: c_int, is_coeffs: c_int,
        cap_out: *mut u64) -> c_int;
    pub fn b200zkp_sharded_commit_from_values(comm: *mut b200zkp_comm, values: *const u64, n_log: u32, k: u32, rate_bits: u32,
        cap_height: u32, cap_out: *mut u64, out: *mut *mut b200zkp_sharded) -> c_int;
    pub fn b200zkp_sharded_synchronize(sh: *mut b200zkp_sharded) -> c_int;
    pub fn b200zkp_sharded_device_ptrs(sh: *mut b200zkp_sharded, local: c_int, coeffs: *mut *const u64, lde: *mut *const u64,
        digests: *mut *const u64, cap: *mut *const u64) -> c_int;
    pub fn b200zkp_sharded_rows(sh: *mut b200zkp_sharded, idx: *const u64, n_idx: u64, rows: *mut u64, siblings: *mut u64) -> c_int;
}
