// UNCOMPILED SOURCE (see ../../README.md).  The `extern "C"` block is GENERATED from include/pcdgpu.h by
// tools/gen_rust_sys.py: one declaration per exported function, same order, same names.
// Encodings (include/pcdgpu.h): field element = 5 x u64 little-endian Montgomery limbs (ark-ff Fp320 / BigInteger320);
// MSM scalar = 5 x u64 plain (`into_repr()`); affine point = x || y, infinity = all zero; every function returns 0 or
// a negative PCDGPU_E_* code and never unwinds.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct pcdgpu_ctx { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_bases { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_r1cs { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_pk { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_gm17_pk { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_csr { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_groth16_pvk { _p: [u8; 0] }
#[repr(C)] pub struct pcdgpu_gm17_pvk { _p: [u8; 0] }

pub const PCDGPU_OK: c_int = 0;
pub const PCDGPU_E_ARG: c_int = -1;
pub const PCDGPU_E_NODEVICE: c_int = -2;
pub const PCDGPU_E_CUDA: c_int = -3;
pub const PCDGPU_E_DOMAIN: c_int = -4;
pub const PCDGPU_E_NOMEM: c_int = -5;
pub const PCDGPU_FIELD_R4: c_int = 0;
pub const PCDGPU_FIELD_Q4: c_int = 1;
pub const PCDGPU_MNT4_298: c_int = 0;
pub const PCDGPU_MNT6_298: c_int = 1;
pub const PCDGPU_MNT4_G1: c_int = 0;
pub const PCDGPU_MNT4_G2: c_int = 1;
pub const PCDGPU_MNT6_G1: c_int = 2;
pub const PCDGPU_MNT6_G2: c_int = 3;
pub const PCDGPU_COMM_ID_BYTES: usize = 128;
pub const PCDGPU_PROF_CLASSES: usize = 11;

#[link(name = "pcdgpu")]
extern "C" {
    pub fn pcdgpu_strerror(code: c_int) -> *const c_char;
    pub fn pcdgpu_last_error(ctx: *const pcdgpu_ctx) -> *const c_char;
    pub fn pcdgpu_affine_bytes(curve: c_int) -> usize;
    pub fn pcdgpu_ctx_create(device: c_int, out: *mut *mut pcdgpu_ctx) -> c_int;
    pub fn pcdgpu_ctx_destroy(ctx: *mut pcdgpu_ctx);
    pub fn pcdgpu_sync(ctx: *mut pcdgpu_ctx) -> c_int;
    pub fn pcdgpu_set_stream(ctx: *mut pcdgpu_ctx, stream: *mut c_void) -> c_int;
    pub fn pcdgpu_set_concurrency(ctx: *mut pcdgpu_ctx, on: c_int) -> c_int;
    pub fn pcdgpu_set_msm_window(ctx: *mut pcdgpu_ctx, c: c_int) -> c_int;
    pub fn pcdgpu_set_proof_graphs(ctx: *mut pcdgpu_ctx, on: c_int) -> c_int;
    pub fn pcdgpu_proof_graph_stats(ctx: *mut pcdgpu_ctx, captured: *mut u64, replayed: *mut u64) -> c_int;
    pub fn pcdgpu_ntt(ctx: *mut pcdgpu_ctx, field: c_int, data: *mut c_void, log_n: u32, inverse: c_int, coset: c_int) -> c_int;
    pub fn pcdgpu_ntt_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_data: *mut c_void, log_n: u32, inverse: c_int, coset: c_int) -> c_int;
    pub fn pcdgpu_domain_size(field: c_int, min_size: usize, pow7: *mut c_int, pow2: *mut c_int) -> usize;
    pub fn pcdgpu_ntt_general(ctx: *mut pcdgpu_ctx, field: c_int, data: *mut c_void, pow7: c_int, pow2: c_int, inverse: c_int, coset: c_int) -> c_int;
    pub fn pcdgpu_msm(ctx: *mut pcdgpu_ctx, curve: c_int, bases: *const c_void, scalars: *const c_void, n: usize, out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_msm_dev(ctx: *mut pcdgpu_ctx, curve: c_int, d_bases: *const c_void, d_scalars: *const c_void, scalars_mont: c_int, n: usize, d_out_xyzz: *mut c_void) -> c_int;
    pub fn pcdgpu_bases_upload(ctx: *mut pcdgpu_ctx, curve: c_int, bases: *const c_void, n: usize, precompute: c_int, out: *mut *mut pcdgpu_bases) -> c_int;
    pub fn pcdgpu_bases_free(b: *mut pcdgpu_bases);
    pub fn pcdgpu_msm_bases(ctx: *mut pcdgpu_ctx, b: *const pcdgpu_bases, offset: usize, scalars: *const c_void, n: usize, out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_msm_bases_dev(ctx: *mut pcdgpu_ctx, b: *const pcdgpu_bases, offset: usize, d_scalars: *const c_void, scalars_mont: c_int, n: usize, d_out_xyzz: *mut c_void) -> c_int;
    pub fn pcdgpu_xyzz_sum(ctx: *mut pcdgpu_ctx, curve: c_int, xyzz: *const c_void, n: usize, out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_xyzz_download(ctx: *mut pcdgpu_ctx, curve: c_int, d_xyzz: *const c_void, out_xyzz: *mut c_void) -> c_int;
    pub fn pcdgpu_fixed_base_mul(ctx: *mut pcdgpu_ctx, curve: c_int, base: *const c_void, scalars: *const c_void, n: usize, out: *mut c_void) -> c_int;
    pub fn pcdgpu_fixed_base_mul_dev(ctx: *mut pcdgpu_ctx, curve: c_int, base_host: *const c_void, d_scalars: *const c_void, n: usize, d_out: *mut c_void) -> c_int;
    pub fn pcdgpu_r1cs_upload(ctx: *mut pcdgpu_ctx, pairing: c_int, num_constraints: usize, num_inputs: usize, num_witness: usize, a_ptr: *const u32, a_col: *const u32, a_val: *const c_void, b_ptr: *const u32, b_col: *const u32, b_val: *const c_void, c_ptr: *const u32, c_col: *const u32, c_val: *const c_void, out: *mut *mut pcdgpu_r1cs) -> c_int;
    pub fn pcdgpu_r1cs_free(r: *mut pcdgpu_r1cs);
    pub fn pcdgpu_r1cs_domain_size(r: *const pcdgpu_r1cs) -> usize;
    pub fn pcdgpu_witness_map(ctx: *mut pcdgpu_ctx, r: *const pcdgpu_r1cs, z: *const c_void, h: *mut c_void) -> c_int;
    pub fn pcdgpu_qap_vector_dev(ctx: *mut pcdgpu_ctx, r: *const pcdgpu_r1cs, which: c_int, d_z: *const c_void, d_out: *mut c_void) -> c_int;
    pub fn pcdgpu_qap_combine_dev(ctx: *mut pcdgpu_ctx, r: *const pcdgpu_r1cs, d_a: *mut c_void, d_b: *const c_void, d_c: *const c_void) -> c_int;
    pub fn pcdgpu_pk_upload(ctx: *mut pcdgpu_ctx, pairing: c_int, num_vars: usize, num_inputs: usize, h_len: usize, alpha_g1: *const c_void, beta_g1: *const c_void, delta_g1: *const c_void, beta_g2: *const c_void, delta_g2: *const c_void, a_query: *const c_void, b_g1_query: *const c_void, b_g2_query: *const c_void, h_query: *const c_void, l_query: *const c_void, precompute: c_int, out: *mut *mut pcdgpu_pk) -> c_int;
    pub fn pcdgpu_pk_free(pk: *mut pcdgpu_pk);
    pub fn pcdgpu_groth16_prove(ctx: *mut pcdgpu_ctx, pk: *const pcdgpu_pk, r1cs: *const pcdgpu_r1cs, z: *const c_void, r: *const c_void, s: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_groth16_prove_dev(ctx: *mut pcdgpu_ctx, pk: *const pcdgpu_pk, r1cs: *const pcdgpu_r1cs, d_z: *const c_void, r: *const c_void, s: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_sap_domain_size(pairing: c_int, m: usize, num_inputs: usize) -> usize;
    pub fn pcdgpu_sap_witness_map(ctx: *mut pcdgpu_ctx, r: *const pcdgpu_r1cs, z: *const c_void, d1: *const c_void, d2: *const c_void, full: *mut c_void, h: *mut c_void) -> c_int;
    pub fn pcdgpu_gm17_pk_upload(ctx: *mut pcdgpu_ctx, pairing: c_int, num_sap_vars: usize, num_inputs: usize, h_len: usize, a_query: *const c_void, b_query: *const c_void, c_query_1: *const c_void, c_query_2: *const c_void, g_gamma2_z_t: *const c_void, g_gamma_z: *const c_void, h_gamma_z: *const c_void, g_ab_gamma_z: *const c_void, g_gamma2_z2: *const c_void, precompute: c_int, out: *mut *mut pcdgpu_gm17_pk) -> c_int;
    pub fn pcdgpu_gm17_pk_free(pk: *mut pcdgpu_gm17_pk);
    pub fn pcdgpu_gm17_prove(ctx: *mut pcdgpu_ctx, pk: *const pcdgpu_gm17_pk, r1cs: *const pcdgpu_r1cs, z: *const c_void, d1: *const c_void, d2: *const c_void, r: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_gm17_prove_dev(ctx: *mut pcdgpu_ctx, pk: *const pcdgpu_gm17_pk, r1cs: *const pcdgpu_r1cs, d_z: *const c_void, d1: *const c_void, d2: *const c_void, r: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_poly_divide_linear(ctx: *mut pcdgpu_ctx, field: c_int, coeffs: *const c_void, n: usize, z: *const c_void, quotient: *mut c_void, eval: *mut c_void) -> c_int;
    pub fn pcdgpu_poly_mul(ctx: *mut pcdgpu_ctx, field: c_int, a: *const c_void, na: usize, b: *const c_void, nb: usize, out: *mut c_void) -> c_int;
    pub fn pcdgpu_kzg_commit(ctx: *mut pcdgpu_ctx, powers_of_g: *const pcdgpu_bases, coeffs: *const c_void, n: usize, powers_of_gamma_g: *const pcdgpu_bases, rand_coeffs: *const c_void, n_rand: usize, out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_kzg_open(ctx: *mut pcdgpu_ctx, powers_of_g: *const pcdgpu_bases, coeffs: *const c_void, n: usize, powers_of_gamma_g: *const pcdgpu_bases, rand_coeffs: *const c_void, n_rand: usize, z: *const c_void, out_w_affine: *mut c_void, out_value: *mut c_void, out_random_v: *mut c_void) -> c_int;
    pub fn pcdgpu_dev_alloc(ctx: *mut pcdgpu_ctx, bytes: usize, d_out: *mut *mut c_void) -> c_int;
    pub fn pcdgpu_dev_free(ctx: *mut pcdgpu_ctx, d: *mut c_void) -> c_int;
    pub fn pcdgpu_dev_upload(ctx: *mut pcdgpu_ctx, d_dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
    pub fn pcdgpu_dev_download(ctx: *mut pcdgpu_ctx, dst: *mut c_void, d_src: *const c_void, bytes: usize) -> c_int;
    pub fn pcdgpu_dev_copy(ctx: *mut pcdgpu_ctx, d_dst: *mut c_void, d_src: *const c_void, bytes: usize) -> c_int;
    pub fn pcdgpu_dev_zero(ctx: *mut pcdgpu_ctx, d: *mut c_void, bytes: usize) -> c_int;
    pub fn pcdgpu_vec_binary_dev(ctx: *mut pcdgpu_ctx, field: c_int, op: c_int, d_out: *mut c_void, d_a: *const c_void, d_b: *const c_void, n: usize) -> c_int;
    pub fn pcdgpu_vec_scalar_dev(ctx: *mut pcdgpu_ctx, field: c_int, op: c_int, d_out: *mut c_void, d_a: *const c_void, scalar: *const c_void, n: usize) -> c_int;
    pub fn pcdgpu_vec_axpy_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_y: *mut c_void, scalar: *const c_void, d_x: *const c_void, n: usize) -> c_int;
    pub fn pcdgpu_vec_inverse_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_data: *mut c_void, n: usize) -> c_int;
    pub fn pcdgpu_vec_powers_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_out: *mut c_void, base: *const c_void, scale: *const c_void, n: usize) -> c_int;
    pub fn pcdgpu_vec_gather_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_out: *mut c_void, d_src: *const c_void, d_index: *const u32, n: usize) -> c_int;
    pub fn pcdgpu_poly_eval_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_coeffs: *const c_void, n: usize, z: *const c_void, out: *mut c_void) -> c_int;
    pub fn pcdgpu_poly_divide_vanishing_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_p: *const c_void, n: usize, domain_n: usize, d_q: *mut c_void, d_r: *mut c_void) -> c_int;
    pub fn pcdgpu_poly_divide_linear_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_p: *const c_void, n: usize, z: *const c_void, d_q: *mut c_void, out_eval: *mut c_void) -> c_int;
    pub fn pcdgpu_ntt_general_dev(ctx: *mut pcdgpu_ctx, field: c_int, d_data: *mut c_void, pow7: c_int, pow2: c_int, inverse: c_int, coset: c_int) -> c_int;
    pub fn pcdgpu_csr_upload(ctx: *mut pcdgpu_ctx, field: c_int, m: usize, ncols: usize, row_ptr: *const u32, col: *const u32, val: *const c_void, out: *mut *mut pcdgpu_csr) -> c_int;
    pub fn pcdgpu_csr_free(c: *mut pcdgpu_csr);
    pub fn pcdgpu_csr_matvec_dev(ctx: *mut pcdgpu_ctx, c: *const pcdgpu_csr, d_x: *const c_void, d_out: *mut c_void) -> c_int;
    pub fn pcdgpu_kzg_commit_dev(ctx: *mut pcdgpu_ctx, powers_of_g: *const pcdgpu_bases, shift: usize, d_coeffs: *const c_void, n: usize, powers_of_gamma_g: *const pcdgpu_bases, d_rand: *const c_void, n_rand: usize, out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_set_msm_side_by_side(ctx: *mut pcdgpu_ctx, on: c_int) -> c_int;
    pub fn pcdgpu_groth16_assemble_begin_dev(ctx: *mut pcdgpu_ctx, pairing: c_int, r: *const c_void, s: *const c_void, world: c_int, d_partials_ab: *const c_void, d_partials_g2: *const c_void) -> c_int;
    pub fn pcdgpu_groth16_assemble_finish_dev(ctx: *mut pcdgpu_ctx, pairing: c_int, world: c_int, d_partials_hl: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_comm_unique_id(out_id: *mut c_void) -> c_int;
    pub fn pcdgpu_comm_init(ctx: *mut pcdgpu_ctx, id: *const c_void, rank: c_int, world: c_int) -> c_int;
    pub fn pcdgpu_comm_info(ctx: *const pcdgpu_ctx, rank: *mut c_int, world: *mut c_int) -> c_int;
    pub fn pcdgpu_comm_destroy(ctx: *mut pcdgpu_ctx);
    pub fn pcdgpu_pk_upload_sharded(ctx: *mut pcdgpu_ctx, pairing: c_int, num_vars: usize, num_inputs: usize, h_len: usize, alpha_g1: *const c_void, beta_g1: *const c_void, delta_g1: *const c_void, beta_g2: *const c_void, delta_g2: *const c_void, a_query: *const c_void, b_g1_query: *const c_void, b_g2_query: *const c_void, h_query: *const c_void, l_query: *const c_void, precompute: c_int, out: *mut *mut pcdgpu_pk) -> c_int;
    pub fn pcdgpu_groth16_prove_sharded(ctx: *mut pcdgpu_ctx, pk: *const pcdgpu_pk, r1cs: *const pcdgpu_r1cs, z: *const c_void, r: *const c_void, s: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_groth16_prove_sharded_dev(ctx: *mut pcdgpu_ctx, pk: *const pcdgpu_pk, r1cs: *const pcdgpu_r1cs, d_z: *const c_void, r: *const c_void, s: *const c_void, out_proof: *mut c_void) -> c_int;
    pub fn pcdgpu_msm_bases_sharded(ctx: *mut pcdgpu_ctx, slice: *const pcdgpu_bases, scalars: *const c_void, n: usize, out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_msm_bases_sharded_dev(ctx: *mut pcdgpu_ctx, slice: *const pcdgpu_bases, d_scalars: *const c_void, scalars_mont: c_int, n: usize, d_out_affine: *mut c_void) -> c_int;
    pub fn pcdgpu_serialize_proof(ctx: *mut pcdgpu_ctx, pairing: c_int, proof_affine: *const c_void, out: *mut u8, out_len: *mut usize) -> c_int;
    pub fn pcdgpu_pairing(ctx: *mut pcdgpu_ctx, pairing: c_int, g1: *const c_void, g2: *const c_void, n: usize, out_gt: *mut c_void) -> c_int;
    pub fn pcdgpu_groth16_pvk_create(ctx: *mut pcdgpu_ctx, pairing: c_int, alpha_g1: *const c_void, beta_g2: *const c_void, gamma_g2: *const c_void, delta_g2: *const c_void, gamma_abc_g1: *const c_void, num_inputs: usize, out: *mut *mut pcdgpu_groth16_pvk) -> c_int;
    pub fn pcdgpu_groth16_pvk_free(pvk: *mut pcdgpu_groth16_pvk);
    pub fn pcdgpu_groth16_verify_batch(ctx: *mut pcdgpu_ctx, pvk: *const pcdgpu_groth16_pvk, proofs: *const c_void, inputs: *const c_void, n: usize, out_ok: *mut u8) -> c_int;
    pub fn pcdgpu_gm17_pvk_create(ctx: *mut pcdgpu_ctx, pairing: c_int, h_g2: *const c_void, g_alpha_g1: *const c_void, h_beta_g2: *const c_void, g_gamma_g1: *const c_void, h_gamma_g2: *const c_void, query: *const c_void, num_inputs: usize, out: *mut *mut pcdgpu_gm17_pvk) -> c_int;
    pub fn pcdgpu_gm17_pvk_free(pvk: *mut pcdgpu_gm17_pvk);
    pub fn pcdgpu_gm17_verify_batch(ctx: *mut pcdgpu_ctx, pvk: *const pcdgpu_gm17_pvk, proofs: *const c_void, inputs: *const c_void, n: usize, out_ok: *mut u8) -> c_int;
    pub fn pcdgpu_deserialize_proofs(ctx: *mut pcdgpu_ctx, pairing: c_int, bytes: *const u8, n: usize, out_affine: *mut c_void, out_ok: *mut u8) -> c_int;
    pub fn pcdgpu_groth16_verify_batch_serialized(ctx: *mut pcdgpu_ctx, pvk: *const pcdgpu_groth16_pvk, bytes: *const u8, inputs: *const c_void, n: usize, out_ok: *mut u8) -> c_int;
    pub fn pcdgpu_gm17_verify_batch_serialized(ctx: *mut pcdgpu_ctx, pvk: *const pcdgpu_gm17_pvk, bytes: *const u8, inputs: *const c_void, n: usize, out_ok: *mut u8) -> c_int;
    pub fn pcdgpu_profile_enable(ctx: *mut pcdgpu_ctx, on: c_int) -> c_int;
    pub fn pcdgpu_profile_read(ctx: *mut pcdgpu_ctx, ms: *mut f64, units: *mut f64, spans: *mut u64, launches: *mut u64) -> c_int;
    pub fn pcdgpu_profile_timeline(ctx: *mut pcdgpu_ctx, t0_ms: *mut f64, t1_ms: *mut f64, cls: *mut c_int, cap: usize, count: *mut usize) -> c_int;
    pub fn pcdgpu_bench_imad(ctx: *mut pcdgpu_ctx, modmul: c_int, iters: c_int, out_ops_per_s: *mut f64, out_ms: *mut f64) -> c_int;
}
