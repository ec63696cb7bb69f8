// Replacement bodies for two steps of plonky2 @ f99ed9c `plonky2/src/plonk/prover.rs` (rows N1a and N1c of SURVEY.md 8f).
// NOT COMPILED HERE (no Rust toolchain in this image): a sketch for the maintainer who applies the [patch] recipe of
// INTEGRATION.md; the same C ABI calls are exercised from Python (intmax_zkp_core_b200/prover.py) and C++
// (host/prover_api.hpp), which is what the parity tests run.
use b200zkp_sys as sys;
use plonky2_field::extension::Extendable;
use plonky2_field::polynomial::{PolynomialCoeffs, PolynomialValues};
use plonky2_field::types::Field;
use plonky2_util::log2_strict;
use rand::rngs::OsRng;
use rand::RngCore;

use crate::fri::oracle::CTX;            // the thread-local b200zkp_ctx of oracle_gpu.rs (made pub(crate) there)
use crate::hash::hash_types::RichField;
use crate::iop::witness::MatrixWitness;
use crate::plonk::circuit_data::{CommonCircuitData, ProverOnlyCircuitData};
use crate::plonk::config::GenericConfig;

/// all_wires_permutation_partial_products + the `pop()` / `concat()` that moves every Z to the front: returns the
/// `zs_partial_products` batch of prove() (Z of every challenge, then the partial products challenge by challenge).
fn zs_partial_products<F: RichField + Extendable<D>, C: GenericConfig<D, F = F>, const D: usize>(
    witness: &MatrixWitness<F>,
    betas: &[F],
    gammas: &[F],
    prover_data: &ProverOnlyCircuitData<F, C, D>,
    common_data: &CommonCircuitData<F, C, D>,
) -> Vec<PolynomialValues<F>> {
    let n = common_data.degree();
    let routed = common_data.config.num_routed_wires;
    // column-major u64 buffers: the routed wires are the first columns of the witness matrix, sigmas[i][j] is transposed
    let wires: Vec<u64> = (0..routed).flat_map(|j| (0..n).map(move |i| witness.get_wire(i, j).to_noncanonical_u64())).collect();
    let sigmas: Vec<u64> = (0..routed).flat_map(|j| (0..n).map(move |i| prover_data.sigmas[i][j].to_noncanonical_u64())).collect();
    let k_is: Vec<u64> = common_data.k_is.iter().map(|k| k.to_canonical_u64()).collect();
    let b: Vec<u64> = betas.iter().map(|x| x.to_canonical_u64()).collect();
    let g: Vec<u64> = gammas.iter().map(|x| x.to_canonical_u64()).collect();
    let cols = betas.len() * (1 + common_data.num_partial_products);
    let mut out = vec![0u64; cols * n];
    let rc = CTX.with(|c| unsafe {
        sys::b200zkp_partial_products_and_zs(*c, wires.as_ptr(), sigmas.as_ptr(), log2_strict(n) as u32, routed as u32,
                                             common_data.quotient_degree_factor as u32, k_is.as_ptr(), b.as_ptr(), g.as_ptr(),
                                             betas.len() as u32, out.as_mut_ptr())
    });
    assert_eq!(rc, 0, "b200zkp_partial_products_and_zs failed");
    out.chunks(n).map(|c| PolynomialValues::new(c.iter().map(|&x| F::from_canonical_u64(x)).collect())).collect()
}

/// tail of compute_quotient_polys + the chunking in prove(): quotient values on the coset 7 <w>, natural order, one
/// vector per challenge -> `all_quotient_poly_chunks` for PolynomialBatch::from_coeffs
fn quotient_poly_chunks<F: RichField>(quotient_values: Vec<Vec<F>>, degree: usize) -> Vec<PolynomialCoeffs<F>> {
    let len = quotient_values[0].len();
    let mut flat: Vec<u64> = quotient_values.iter().flat_map(|v| v.iter().map(|x| x.to_noncanonical_u64())).collect();
    let rc = CTX.with(|c| unsafe {
        sys::b200zkp_coset_intt(*c, flat.as_mut_ptr(), log2_strict(len) as u32, quotient_values.len() as u32,
                                F::coset_shift().to_canonical_u64())
    });
    assert_eq!(rc, 0, "b200zkp_coset_intt failed");
    flat.chunks(degree).map(|c| PolynomialCoeffs::new(c.iter().map(|&x| F::from_canonical_u64(x)).collect())).collect()
}

/// The whole prove() with every polynomial resident in HBM, in plonky2's transcript order (the sequence
/// intmax_zkp_core_b200/prover.py::prove runs and tests/test_gpu_prove.py / tests/test_gpu_zk.py check word for word).
/// With config.zero_knowledge the wires, Z + partial products and quotient commitments are salted: the salt key is drawn
/// from the OS once per proof, each salt is generated on the device with nonce = le32(PlonkOracle index) || 0^8.
/// `wires_dev`: the 135 x n column-major witness matrix already on the device; `cs`: the constants + sigmas handle that
/// CircuitBuilder::build committed with b200zkp_batch_from_device, `sigmas_dev` its sigma columns.  Sketch only: the
/// device allocations, the vanishing descriptor and the FRI query loop are those of prover.py / fri.py.
#[allow(dead_code)]
fn prove_gpu<F: RichField + Extendable<D>, C: GenericConfig<D, F = F>, const D: usize>(
    ctx: *mut sys::b200zkp_ctx,
    cs: *mut sys::b200zkp_batch,
    sigmas_dev: *const u64,
    wires_dev: *const u64,
    public_inputs: &[F],
    circuit_digest: &[F; 4],
    common_data: &CommonCircuitData<F, C, D>,
    challenger: &mut crate::iop::challenger::Challenger<F, C::Hasher>,
) {
    let n_log = common_data.degree_bits() as u32;
    let n = 1u64 << n_log;
    let cfg = &common_data.config.fri_config;
    let nc = common_data.config.num_challenges;
    let zk = common_data.config.zero_knowledge;
    // the salt key: secret, from the OS, fresh for every proof (never reused, never logged)
    let mut salt_key = [0u8; 32];
    if zk {
        OsRng.fill_bytes(&mut salt_key);
    }
    let lde_size = n << cfg.rate_bits;
    let salt_dev: *mut u64 = std::ptr::null_mut(); // (device buffer of SALT_SIZE * lde_size words per blinded commitment)
    // PolynomialBatch::from_values / from_coeffs with blinding = zk && oracle.blinding (PlonkOracle index `oracle`)
    let commit = |input: *const u64, k: usize, is_coeffs: bool, oracle: u32| {
        let mut salt: *const u64 = std::ptr::null();
        if zk {
            let mut nonce = [0u8; 12];
            nonce[..4].copy_from_slice(&oracle.to_le_bytes());
            assert_eq!(unsafe { sys::b200zkp_dev_random_field(ctx, salt_key.as_ptr(), nonce.as_ptr(), 0,
                                                               sys::B200ZKP_SALT_SIZE as u64 * lde_size, salt_dev) }, 0);
            salt = salt_dev;
        }
        let mut b = std::ptr::null_mut();
        assert_eq!(unsafe { sys::b200zkp_batch_from_device(ctx, input, is_coeffs as i32, n_log, k as u32, cfg.rate_bits as u32,
                                                            cfg.cap_height as u32, salt, &mut b) }, 0);
        b
    };
    // 1. circuit digest, public inputs hash
    challenger.observe_elements(circuit_digest);
    challenger.observe_hash::<C::InnerHasher>(C::InnerHasher::hash_no_pad(public_inputs));
    // 2. wires
    let wires = commit(wires_dev, common_data.config.num_wires, false, 1);
    // observe_cap(b200zkp_batch_cap(wires)); betas = get_n_challenges(nc); gammas = get_n_challenges(nc)
    // 3. Z + partial products: b200zkp_dev_partial_products_and_zs(ctx, wires_dev, n, sigmas_dev, n, ...) into zpp_dev
    let zpp_dev: *const u64 = std::ptr::null(); // (device buffer of nc * (1 + num_partial_products) columns)
    let zpp = commit(zpp_dev, nc * (1 + common_data.num_partial_products), false, 2);
    // observe_cap(zpp); alphas = get_n_challenges(nc)
    // 4. quotient: b200zkp_dev_quotient_values on the LDE pointers of cs / wires / zpp (b200zkp_batch_device_ptrs),
    //    b200zkp_dev_coset_intt(shift 7) into chunks_dev, then (the salt columns come last in a blinded LDE: the quotient
    //    kernel is given the first k columns only)
    let chunks_dev: *const u64 = std::ptr::null();
    let quotient = commit(chunks_dev, nc * common_data.quotient_degree_factor, true, 3);
    // observe_cap(quotient)
    // 5. zeta = get_extension_challenge(); ensure!(zeta.exp_power_of_2(degree_bits) != ONE)
    // 6. OpeningSet::new + to_fri_openings in one call: every polynomial of the four oracles at zeta, the Zs at g zeta
    let oracles = [cs, wires, zpp, quotient];
    let mut counts = [0u32; 2];
    let (mut po, mut pi) = (Vec::new(), Vec::new());
    for (o, &b) in oracles.iter().enumerate() {
        let mut shape = [0u32; 5];
        unsafe { sys::b200zkp_batch_shape(b, shape.as_mut_ptr()) };
        for i in 0..shape[1] { po.push(o as u32); pi.push(i); }
        counts[0] += shape[1];
    }
    for i in 0..nc as u32 { po.push(2); pi.push(i); }
    counts[1] = nc as u32;
    let points = [0u64; 4]; // (zeta, g * zeta) as (re, im) pairs
    let mut openings = vec![0u64; 2 * po.len()];
    assert_eq!(unsafe { sys::b200zkp_batch_openings(ctx, oracles.as_ptr(), 4, 2, points.as_ptr(), counts.as_ptr(), po.as_ptr(),
                                                    pi.as_ptr(), openings.as_mut_ptr()) }, 0);
    // challenger.observe_extension_elements per batch, then
    // 7. PolynomialBatch::prove_openings(get_fri_instance(zeta), [cs, wires, zpp, quotient]) through b200zkp_fri_begin (oracle_gpu.rs);
    //    with fri_params.hiding the query rounds open whole salted leaves (k + 4 words) of the blinded oracles
    let _ = (n, wires, zpp, quotient);
}
