/* pcdgpu.h -- C ABI of libpcdgpu.so: the B200 (sm_100a) prover backend for the Groth16 proving
 * step of arkworks-rs/pcd on the MNT4-298 / MNT6-298 cycle.
 *
 * This is the drop-in boundary (SURVEY.md 8b): a Rust shim implementing ark-snark's `SNARK`
 * trait binds exactly these entry points (INTEGRATION.md shows the `extern "C"` block).  The
 * reference reaches the replaced code through
 *     IC::MainSNARK::prove / IC::HelpSNARK::prove   /root/reference/src/ec_cycle_pcd/mod.rs:171,179
 *     tiny default-circuit proves                   /root/reference/src/ec_cycle_pcd/data_structures.rs:139-143,343-350
 * and the arithmetic itself lives in the un-vendored arkworks crates named per function below.
 *
 * Conventions
 *   - every function returns 0 (PCDGPU_OK) or a negative PCDGPU_E_* code; nothing throws or aborts
 *     across the boundary; pcdgpu_strerror() names a code, pcdgpu_last_error() gives detail.
 *   - the caller owns every host buffer; device objects are opaque handles with explicit free.
 *   - one context = one GPU + one stream set; a context must not be used from two host threads at
 *     once (the prover entry points refuse a second concurrent call with PCDGPU_E_ARG).  There is NO
 *     CPU fallback: without a usable sm_100 device ctx_create fails.
 *   - encodings are arkworks' in-memory ones so the shim copies, never converts:
 *       field element  : 40 bytes, five little-endian u64 limbs of a*R mod p, R = 2^320
 *                        (ark-ff Fp320 / BigInteger320)
 *       MSM scalar     : 40 bytes, five little-endian u64 limbs of the plain integer
 *                        (`into_repr()`); *_mont variants take Montgomery-form elements instead
 *       affine point   : x || y (G1: 80 B; MNT4 G2 over Fq2: 160 B = x.c0 x.c1 y.c0 y.c1;
 *                        MNT6 G2 over Fq3: 240 B); the point at infinity is x = y = 0
 *       xyzz point     : X || Y || ZZ || ZZZ (x = X/ZZ, y = Y/ZZZ; infinity: ZZ = 0) -- only used
 *                        for partial sums exchanged between GPUs
 *   - functions with the _dev suffix take DEVICE pointers on the context's GPU and are
 *     asynchronous on the context's stream (pcdgpu_sync() waits) -- except the provers
 *     (*_prove_dev, *_prove_sharded_dev), whose proof lands in a HOST buffer: they return when it
 *     is there; the others take HOST pointers and return when the result is in the host buffer.
 */
#ifndef PCDGPU_H
#define PCDGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pcdgpu_ctx pcdgpu_ctx;
typedef struct pcdgpu_bases pcdgpu_bases; /* device-resident MSM base vector             */
typedef struct pcdgpu_r1cs pcdgpu_r1cs;   /* device-resident CSR matrices A, B, C        */
typedef struct pcdgpu_pk pcdgpu_pk;       /* device-resident Groth16 proving key         */

enum {
  PCDGPU_OK = 0,
  PCDGPU_E_ARG = -1,       /* bad argument (null pointer, unknown id, size out of range)  */
  PCDGPU_E_NODEVICE = -2,  /* no usable CUDA device (there is no CPU fallback)            */
  PCDGPU_E_CUDA = -3,      /* a CUDA call failed; see pcdgpu_last_error()                 */
  PCDGPU_E_DOMAIN = -4,    /* evaluation domain larger than the field's 2-adicity allows  */
  PCDGPU_E_NOMEM = -5
};

/* scalar fields (ark-mnt4-298 Fr / ark-mnt6-298 Fr) */
enum { PCDGPU_FIELD_R4 = 0, PCDGPU_FIELD_Q4 = 1 };
/* pairings: MNT4-298 has Fr = r4, G1 over q4, G2 over Fq2; MNT6-298 has Fr = q4, G1 over r4, G2 over Fq3 */
enum { PCDGPU_MNT4_298 = 0, PCDGPU_MNT6_298 = 1 };
/* groups */
enum { PCDGPU_MNT4_G1 = 0, PCDGPU_MNT4_G2 = 1, PCDGPU_MNT6_G1 = 2, PCDGPU_MNT6_G2 = 3 };

const char* pcdgpu_strerror(int code);
const char* pcdgpu_last_error(const pcdgpu_ctx* ctx);
/* bytes of an affine point of `curve` (80 / 160 / 80 / 240) */
size_t pcdgpu_affine_bytes(int curve);

/* ---- context ------------------------------------------------------------------------------- */
int pcdgpu_ctx_create(int device, pcdgpu_ctx** out);
void pcdgpu_ctx_destroy(pcdgpu_ctx* ctx);
int pcdgpu_sync(pcdgpu_ctx* ctx);
/* use a caller-owned CUDA stream (e.g. torch's current stream) instead of the context's own;
 * stream = the cudaStream_t value; 0 restores the context's stream */
int pcdgpu_set_stream(pcdgpu_ctx* ctx, void* stream);
/* on (default): the five MSMs of a proof run on separate internal streams and overlap; off: every
 * kernel runs on the context's stream in program order (used for per-kernel timing) */
int pcdgpu_set_concurrency(pcdgpu_ctx* ctx, int on);
/* MSM window override (0 = automatic); exposed for benchmarking */
int pcdgpu_set_msm_window(pcdgpu_ctx* ctx, int c);
/* Proof graphs (default OFF): when on, pcdgpu_groth16_prove[_dev] captures the launch sequence of a proof into a CUDA
 * graph the second time it sees the same (key, constraint system, device assignment address) and replays it afterwards
 * -- one launch instead of 150 - 250 on up to seven streams.  Results are identical (tests/test_gpu_graphs.py).
 * MEASURED on B200 inside the PCD step (tools/probe_step.py): replay is SLOWER than eager enqueueing -- main proof
 * (2^18) 7.58 vs 6.75 ms, helper (2^16) 4.31 vs 4.24 ms, default-circuit proofs 1.27 - 1.34 vs 1.21 - 1.25 ms: the
 * eager path's stream priorities and enqueue order (witness map first, accumulation grids gated) schedule the lanes
 * better than the graph's dependency-only order, and a 250-node launch costs about what the staggered enqueue did.
 * Kept as an option for hosts whose enqueue rate is the bound.
 * stats: graphs captured / proofs replayed from a graph since the context exists. */
int pcdgpu_set_proof_graphs(pcdgpu_ctx* ctx, int on);
int pcdgpu_proof_graph_stats(pcdgpu_ctx* ctx, uint64_t* captured, uint64_t* replayed);

/* ---- radix-2 (coset) NTT --------------------------------------------------------------------
 * Replaces ark-poly EvaluationDomain::{fft,ifft,coset_fft,coset_ifft}_in_place on
 * Radix2EvaluationDomain (natural order in and out; omega_n = TWO_ADIC_ROOT^(2^(s-log_n)); coset
 * shift by GENERATOR = 10 (r4) / 17 (q4); ifft includes the 1/n scale).  data: 2^log_n elements,
 * transformed in place.  log_n <= 34 (r4) / 17 (q4), else PCDGPU_E_DOMAIN. */
int pcdgpu_ntt(pcdgpu_ctx* ctx, int field, void* data, uint32_t log_n, int inverse, int coset);
int pcdgpu_ntt_dev(pcdgpu_ctx* ctx, int field, void* d_data, uint32_t log_n, int inverse, int coset);
/* ark-poly GeneralEvaluationDomain::new(min_size): radix-2 when log2 fits the field's 2-adicity, otherwise
 * (q4 only: its multiplicative group has a subgroup of order 7^2) the smallest 7^a 2^b >= min_size
 * (MixedRadixEvaluationDomain).  Returns the size (0: none) and its exponents. */
size_t pcdgpu_domain_size(int field, size_t min_size, int* pow7, int* pow2);
/* the four transforms on the domain 7^pow7 * 2^pow2 (pow7 = 0: same as pcdgpu_ntt) */
int pcdgpu_ntt_general(pcdgpu_ctx* ctx, int field, void* data, int pow7, int pow2, int inverse, int coset);

/* ---- variable-base MSM ----------------------------------------------------------------------
 * Replaces ark-ec VariableBaseMSM::multi_scalar_mul(bases, scalars): sum_i scalars[i] * bases[i]
 * over min(n_bases, n_scalars) pairs.  out_affine: one affine point (arkworks returns a
 * projective point whose representation is algorithm dependent; callers compare / serialize
 * after into_affine(), which is what is returned here). */
int pcdgpu_msm(pcdgpu_ctx* ctx, int curve, const void* bases, const void* scalars, size_t n, void* out_affine);
/* device pointers; scalars_mont != 0: scalars are Montgomery-form field elements (converted on
 * the fly).  d_out_xyzz: one xyzz point in device memory (not normalised). */
int pcdgpu_msm_dev(pcdgpu_ctx* ctx, int curve, const void* d_bases, const void* d_scalars, int scalars_mont,
                   size_t n, void* d_out_xyzz);
/* Resident base vectors (proving-key queries, KZG powers): uploaded once, reused by every MSM.
 * precompute != 0 additionally stores 2^(c*j) * P for every window j so that all windows share
 * one bucket set (no window-combination doubling chain; costs ~ceil(299/c) x the memory). */
int pcdgpu_bases_upload(pcdgpu_ctx* ctx, int curve, const void* bases, size_t n, int precompute, pcdgpu_bases** out);
void pcdgpu_bases_free(pcdgpu_bases* b);
int pcdgpu_msm_bases(pcdgpu_ctx* ctx, const pcdgpu_bases* b, size_t offset, const void* scalars, size_t n,
                     void* out_affine);
int pcdgpu_msm_bases_dev(pcdgpu_ctx* ctx, const pcdgpu_bases* b, size_t offset, const void* d_scalars,
                         int scalars_mont, size_t n, void* d_out_xyzz);
/* sum of n xyzz partial sums (host buffers), normalised to affine: the gather step of a
 * point-range sharded MSM (SURVEY.md 8e) */
int pcdgpu_xyzz_sum(pcdgpu_ctx* ctx, int curve, const void* xyzz, size_t n, void* out_affine);
/* copy an xyzz point from device to host (partials for the gather) */
int pcdgpu_xyzz_download(pcdgpu_ctx* ctx, int curve, const void* d_xyzz, void* out_xyzz);

/* ---- fixed-base batch multiplication --------------------------------------------------------
 * out[i] = scalars[i] * base (affine).  Replaces ark-ec FixedBaseMSM::multi_scalar_mul as used by
 * the Groth16 generator; here it builds proving keys and synthetic point sets. */
int pcdgpu_fixed_base_mul(pcdgpu_ctx* ctx, int curve, const void* base, const void* scalars, size_t n, void* out);
int pcdgpu_fixed_base_mul_dev(pcdgpu_ctx* ctx, int curve, const void* base_host, const void* d_scalars, size_t n,
                              void* d_out);

/* ---- R1CS -> QAP witness map ----------------------------------------------------------------
 * Replaces ark-relations ConstraintSystem::to_matrices consumers + ark-groth16
 * R1CStoQAP::witness_map.  Matrices are CSR: row_ptr[m + 1] (u32), col[nnz] (u32, instance
 * variables first, column 0 is the constant 1), val[nnz] (field elements). */
int pcdgpu_r1cs_upload(pcdgpu_ctx* ctx, int pairing, size_t num_constraints, size_t num_inputs, size_t num_witness,
                       const uint32_t* a_ptr, const uint32_t* a_col, const void* a_val, const uint32_t* b_ptr,
                       const uint32_t* b_col, const void* b_val, const uint32_t* c_ptr, const uint32_t* c_col,
                       const void* c_val, pcdgpu_r1cs** out);
void pcdgpu_r1cs_free(pcdgpu_r1cs* r);
/* domain size n = |GeneralEvaluationDomain::new(num_constraints + num_inputs)| of an uploaded system */
size_t pcdgpu_r1cs_domain_size(const pcdgpu_r1cs* r);
/* z: num_inputs + num_witness elements (instance || witness, z[0] = 1); h: n elements */
int pcdgpu_witness_map(pcdgpu_ctx* ctx, const pcdgpu_r1cs* r, const void* z, void* h);
/* The same map in two stages, for spreading its three independent vectors over the GPUs of a box (the a, b, c
 * chains of R1CStoQAP::witness_map never interact before the pointwise step; a single NTT is not split):
 *   stage 1 (any GPU holding the matrices): d_out = coset_fft(ifft(M z)), which = 0: A (with the instance rows),
 *            1: B, 2: C; n = pcdgpu_r1cs_domain_size elements, device memory, asynchronous on the context's stream
 *   stage 2 (one GPU, after the vectors were copied to it): d_a <- coset_ifft((a * b - c) / Z) = h */
int pcdgpu_qap_vector_dev(pcdgpu_ctx* ctx, const pcdgpu_r1cs* r, int which, const void* d_z, void* d_out);
int pcdgpu_qap_combine_dev(pcdgpu_ctx* ctx, const pcdgpu_r1cs* r, void* d_a, const void* d_b, const void* d_c);

/* ---- Groth16 --------------------------------------------------------------------------------
 * Replaces ark-groth16 create_proof_with_reduction (Groth16::prove).  The key is uploaded once
 * (ProvingKey {vk.alpha_g1, beta_g1, delta_g1, vk.beta_g2, vk.delta_g2, a_query, b_g1_query,
 * b_g2_query, h_query, l_query}); r and s are inputs so that the RNG and its draw order stay on the
 * Rust side.  out_proof: A (G1 affine) || B (G2 affine) || C (G1 affine) = 320 B (MNT4) / 400 B
 * (MNT6); pcdgpu_serialize_proof() gives ark-serialize's compressed bytes (152 / 190). */
int pcdgpu_pk_upload(pcdgpu_ctx* ctx, int pairing, size_t num_vars, size_t num_inputs, size_t h_len,
                     const void* alpha_g1, const void* beta_g1, const void* delta_g1, const void* beta_g2,
                     const void* delta_g2, const void* a_query, const void* b_g1_query, const void* b_g2_query,
                     const void* h_query, const void* l_query, int precompute, pcdgpu_pk** out);
void pcdgpu_pk_free(pcdgpu_pk* pk);
int pcdgpu_groth16_prove(pcdgpu_ctx* ctx, const pcdgpu_pk* pk, const pcdgpu_r1cs* r1cs, const void* z, const void* r,
                         const void* s, void* out_proof);
/* same with z already in device memory (Montgomery elements) */
int pcdgpu_groth16_prove_dev(pcdgpu_ctx* ctx, const pcdgpu_pk* pk, const pcdgpu_r1cs* r1cs, const void* d_z,
                             const void* r, const void* s, void* out_proof);
/* ---- GM17 (ark-gm17: R1CStoSAP::witness_map + create_proof) --------------------------------------------
 * Replaces `GM17::<E>::prove` as the reference binds it (/root/reference/tests/mnt4_gm17.rs:27-28,
 * tests/mnt4_mix_groth16gm17.rs, tests/mnt4_mix_gm17groth16.rs), reached through IC::MainSNARK::prove /
 * IC::HelpSNARK::prove (/root/reference/src/ec_cycle_pcd/mod.rs:171,179).  The R1CS handle is the one of
 * pcdgpu_r1cs_upload; the SAP (2m + 2(ni - 1) + 1 rows, m + ni - 1 extra variables) is derived on the GPU.
 * d1, d2, r: plain-integer scalars drawn by the caller in this order (create_random_proof), like r, s above.
 * Query vectors are ark-gm17's ProvingKey fields: a_query, b_query (G2), c_query_2 hold one point per SAP
 * variable (num_sap_vars = num_inputs + num_witness + m + num_inputs - 1), c_query_1 one per non-input SAP
 * variable, g_gamma2_z_t h_len = n + 1 points (n = pcdgpu_sap_domain_size).  Proof layout = Groth16's. */
typedef struct pcdgpu_gm17_pk pcdgpu_gm17_pk;
/* size of GeneralEvaluationDomain::new(2m + 2(num_inputs - 1) + 1) over the pairing's scalar field; 0 if none */
size_t pcdgpu_sap_domain_size(int pairing, size_t m, size_t num_inputs);
/* R1CStoSAP::witness_map: full = the SAP assignment (num_sap_vars elements), h = n + 1 coefficients */
int pcdgpu_sap_witness_map(pcdgpu_ctx* ctx, const pcdgpu_r1cs* r, const void* z, const void* d1, const void* d2,
                           void* full, void* h);
int pcdgpu_gm17_pk_upload(pcdgpu_ctx* ctx, int pairing, size_t num_sap_vars, size_t num_inputs, size_t h_len,
                          const void* a_query, const void* b_query, const void* c_query_1, const void* c_query_2,
                          const void* g_gamma2_z_t, const void* g_gamma_z, const void* h_gamma_z,
                          const void* g_ab_gamma_z, const void* g_gamma2_z2, int precompute, pcdgpu_gm17_pk** out);
void pcdgpu_gm17_pk_free(pcdgpu_gm17_pk* pk);
int pcdgpu_gm17_prove(pcdgpu_ctx* ctx, const pcdgpu_gm17_pk* pk, const pcdgpu_r1cs* r1cs, const void* z, const void* d1,
                      const void* d2, const void* r, void* out_proof);
/* same with z already in device memory (Montgomery elements) */
int pcdgpu_gm17_prove_dev(pcdgpu_ctx* ctx, const pcdgpu_gm17_pk* pk, const pcdgpu_r1cs* r1cs, const void* d_z,
                          const void* d1, const void* d2, const void* r, void* out_proof);

/* ---- dense polynomials and KZG10 (ark-poly DensePolynomial, ark-poly-commit kzg10::KZG10::{commit, open}) -----
 * The operations ark-marlin's prover spends its time in when the reference runs MarlinSNARK over MarlinKZG10
 * (/root/reference/tests/mnt4_marlin.rs:68-94), reached through IC::MainSNARK::prove / IC::HelpSNARK::prove
 * (/root/reference/src/ec_cycle_pcd/mod.rs:171,179).  Coefficient vectors are Montgomery elements, lowest degree
 * first; the committer key's `powers_of_g` / `powers_of_gamma_g` are resident pcdgpu_bases over G1. */
/* quotient (n - 1 coefficients) and value of p / (X - z): q = (p - p(z)) / (X - z), eval = p(z); z Montgomery */
int pcdgpu_poly_divide_linear(pcdgpu_ctx* ctx, int field, const void* coeffs, size_t n, const void* z, void* quotient,
                              void* eval);
/* DensePolynomial mul: out = a * b (na + nb - 1 coefficients) through GeneralEvaluationDomain::new(na + nb - 1) */
int pcdgpu_poly_mul(pcdgpu_ctx* ctx, int field, const void* a, size_t na, const void* b, size_t nb, void* out);
/* KZG10::commit: MSM(powers_of_g, coeffs) + MSM(powers_of_gamma_g, rand_coeffs) (the hiding part is skipped when
 * n_rand == 0); one affine G1 point.  The blinding polynomial is drawn by the caller (the RNG stays on its side). */
int pcdgpu_kzg_commit(pcdgpu_ctx* ctx, const pcdgpu_bases* powers_of_g, const void* coeffs, size_t n,
                      const pcdgpu_bases* powers_of_gamma_g, const void* rand_coeffs, size_t n_rand, void* out_affine);
/* KZG10::open: w = commit((p - p(z)) / (X - z)) [+ hiding witness over powers_of_gamma_g]; out_value = p(z)
 * (may be NULL), out_random_v = r(z) (Proof.random_v; written when n_rand > 0) */
int pcdgpu_kzg_open(pcdgpu_ctx* ctx, const pcdgpu_bases* powers_of_g, const void* coeffs, size_t n,
                    const pcdgpu_bases* powers_of_gamma_g, const void* rand_coeffs, size_t n_rand, const void* z,
                    void* out_w_affine, void* out_value, void* out_random_v);

/* ---- device-resident polynomials: what ark-marlin's AHP prover does between its FFTs and its commitments ------------
 * Replaces, under `MarlinSNARK::prove` as the reference binds it (/root/reference/tests/mnt4_marlin.rs:72-75, reached
 * through /root/reference/src/ec_cycle_pcd/mod.rs:171,179): ark-poly `DensePolynomial` / `EvaluationsOnDomain`
 * arithmetic (add, sub, pointwise mul, scalar mul, `evaluate`, `divide_by_vanishing_poly`, division by X - z),
 * ark-ff `batch_inversion`, `EvaluationDomain::elements`, the sparse matrix products of ark-marlin's
 * prover_first_round / prover_second_round, and `KZG10::commit` over powers_of_g[shift..] (MarlinKZG10's shifted
 * commitments).  Vectors live in device memory (Montgomery elements, 40 B each) between calls so that a prover round is
 * a sequence of kernels on the context's stream with no host copies; scalars (challenges) are 40-byte HOST values
 * passed by value into the kernels.  The AHP round logic and the Fiat-Shamir sponge are host code above these calls
 * (pcd_b200/marlin.py mirrors ark-marlin's; INTEGRATION.md shows where the Rust side would call them). */
typedef struct pcdgpu_csr pcdgpu_csr; /* device-resident sparse matrix (CSR) */
int pcdgpu_dev_alloc(pcdgpu_ctx* ctx, size_t bytes, void** d_out); /* stream-ordered (cudaMallocAsync) */
int pcdgpu_dev_free(pcdgpu_ctx* ctx, void* d);
int pcdgpu_dev_upload(pcdgpu_ctx* ctx, void* d_dst, const void* src, size_t bytes);   /* returns when copied */
int pcdgpu_dev_download(pcdgpu_ctx* ctx, void* dst, const void* d_src, size_t bytes); /* returns when copied */
int pcdgpu_dev_copy(pcdgpu_ctx* ctx, void* d_dst, const void* d_src, size_t bytes);
int pcdgpu_dev_zero(pcdgpu_ctx* ctx, void* d, size_t bytes);
enum { PCDGPU_VEC_ADD = 0, PCDGPU_VEC_SUB = 1, PCDGPU_VEC_MUL = 2, PCDGPU_VEC_RSUB = 3 /* b - a */ };
/* out[i] = a[i] op b[i]; out may alias a or b */
int pcdgpu_vec_binary_dev(pcdgpu_ctx* ctx, int field, int op, void* d_out, const void* d_a, const void* d_b, size_t n);
/* out[i] = a[i] op scalar */
int pcdgpu_vec_scalar_dev(pcdgpu_ctx* ctx, int field, int op, void* d_out, const void* d_a, const void* scalar, size_t n);
/* y[i] += scalar * x[i] */
int pcdgpu_vec_axpy_dev(pcdgpu_ctx* ctx, int field, void* d_y, const void* scalar, const void* d_x, size_t n);
/* ark-ff batch_inversion in place (zeros stay zero) */
int pcdgpu_vec_inverse_dev(pcdgpu_ctx* ctx, int field, void* d_data, size_t n);
/* out[i] = scale * base^i (EvaluationDomain::elements with base = group_gen, scale = 1) */
int pcdgpu_vec_powers_dev(pcdgpu_ctx* ctx, int field, void* d_out, const void* base, const void* scale, size_t n);
/* out[i] = src[index[i]], index 0xffffffff gives 0 (d_index: device u32) */
int pcdgpu_vec_gather_dev(pcdgpu_ctx* ctx, int field, void* d_out, const void* d_src, const uint32_t* d_index, size_t n);
/* DensePolynomial::evaluate: out (host) = p(z) */
int pcdgpu_poly_eval_dev(pcdgpu_ctx* ctx, int field, const void* d_coeffs, size_t n, const void* z, void* out);
/* DensePolynomial::divide_by_vanishing_poly for the domain of size domain_n: p = q (X^N - 1) + r; q: n - N coefficients
 * (untouched when n <= N), r: N coefficients */
int pcdgpu_poly_divide_vanishing_dev(pcdgpu_ctx* ctx, int field, const void* d_p, size_t n, size_t domain_n, void* d_q,
                                     void* d_r);
/* (p - p(z)) / (X - z) on device coefficients; out_eval (host, may be NULL: then the call stays asynchronous) = p(z) */
int pcdgpu_poly_divide_linear_dev(pcdgpu_ctx* ctx, int field, const void* d_p, size_t n, const void* z, void* d_q,
                                  void* out_eval);
/* pcdgpu_ntt_general on device memory */
int pcdgpu_ntt_general_dev(pcdgpu_ctx* ctx, int field, void* d_data, int pow7, int pow2, int inverse, int coset);
/* sparse matrix (CSR: row_ptr[m + 1], col[nnz] < ncols, val[nnz] Montgomery) resident on the GPU; out[row] = M[row] . x */
int pcdgpu_csr_upload(pcdgpu_ctx* ctx, int field, size_t m, size_t ncols, const uint32_t* row_ptr, const uint32_t* col,
                      const void* val, pcdgpu_csr** out);
void pcdgpu_csr_free(pcdgpu_csr* c);
int pcdgpu_csr_matvec_dev(pcdgpu_ctx* ctx, const pcdgpu_csr* c, const void* d_x, void* d_out);
/* KZG10::commit of device-resident coefficients over powers_of_g[shift .. shift + n) (+ the blinding polynomial over
 * powers_of_gamma_g[0 .. n_rand)); out_affine: host */
int pcdgpu_kzg_commit_dev(pcdgpu_ctx* ctx, const pcdgpu_bases* powers_of_g, size_t shift, const void* d_coeffs, size_t n,
                          const pcdgpu_bases* powers_of_gamma_g, const void* d_rand, size_t n_rand, void* out_affine);

/* Launch heuristics for callers that run several MSMs side by side on contexts of their own (the multi-GPU prover):
 * on != 0 selects, for bases uploaded and MSMs launched through this context afterwards, the window and occupancy
 * rules the single-GPU prover uses for its five concurrent MSMs (one bit smaller window from 2^18 points up, two
 * accumulate CTAs per SM) instead of the lone-MSM rules.  Results do not depend on it. */
int pcdgpu_set_msm_side_by_side(pcdgpu_ctx* ctx, int on);

/* The last step of a Groth16 proof computed by several GPUs (MSM point ranges split per GPU, SURVEY.md 8e): every
 * rank computes xyzz partial sums of the five MSMs over its slice of each query (pcdgpu_msm_bases_dev; the rank that
 * holds the constant points delta, query[0], alpha / beta adds them to its slices with scalars r or s, 1, 1 and
 * -(r s)), the partials are gathered, and one GPU adds them and assembles the proof in two steps so that the
 * double-scalar multiplication runs while the MSM over h is still going:
 *   begin  (asynchronous): d_partials_ab = world x 2 xyzz G1 points, rank-major, (a, b_g1) per rank; d_partials_g2 =
 *          world x 1 (b_g2).  Normalises A and B and computes s g_a + r g1_b.
 *   finish (synchronous, same context): d_partials_hl = world x 2 (h, l) per rank; writes A || B || C (affine).
 * The result is bit-identical to pcdgpu_groth16_prove for any number of GPUs (affine points are canonical). */
int pcdgpu_groth16_assemble_begin_dev(pcdgpu_ctx* ctx, int pairing, const void* r, const void* s, int world,
                                      const void* d_partials_ab, const void* d_partials_g2);
int pcdgpu_groth16_assemble_finish_dev(pcdgpu_ctx* ctx, int pairing, int world, const void* d_partials_hl,
                                       void* out_proof);

/* ---- multi-GPU inside the library (SURVEY.md 8e) ------------------------------------------------------------
 * One proof / one MSM over the GPUs of a box, one process (or host thread) and one context per GPU, driven through the
 * C ABI alone: MSM point ranges are split per GPU and the per-GPU partial sums are combined with ONE gather of
 * projective points per exchange (NCCL all-gather over NVLink; libnccl.so.2 is resolved at run time, single-GPU users
 * never load it).
 *   rank 0: pcdgpu_comm_unique_id(id), ships the PCDGPU_COMM_ID_BYTES bytes to the other ranks by any means;
 *   every rank: pcdgpu_comm_init(ctx, id, rank, world)                         (collective; world 1 needs no id)
 *               pcdgpu_pk_upload_sharded(... the WHOLE host key ...)           (uploads this rank's slice of each query)
 *               pcdgpu_groth16_prove_sharded(ctx, pk, r1cs, z, r, s, out)      (collective; same inputs on every rank;
 *                                                                               every rank receives the proof)
 * The proof is bit-identical to pcdgpu_groth16_prove for any number of ranks (affine points are canonical). */
#define PCDGPU_COMM_ID_BYTES 128
int pcdgpu_comm_unique_id(void* out_id);
int pcdgpu_comm_init(pcdgpu_ctx* ctx, const void* id, int rank, int world);
int pcdgpu_comm_info(const pcdgpu_ctx* ctx, int* rank, int* world);
void pcdgpu_comm_destroy(pcdgpu_ctx* ctx);
int pcdgpu_pk_upload_sharded(pcdgpu_ctx* ctx, int pairing, size_t num_vars, size_t num_inputs, size_t h_len,
                             const void* alpha_g1, const void* beta_g1, const void* delta_g1, const void* beta_g2,
                             const void* delta_g2, const void* a_query, const void* b_g1_query, const void* b_g2_query,
                             const void* h_query, const void* l_query, int precompute, pcdgpu_pk** out);
int pcdgpu_groth16_prove_sharded(pcdgpu_ctx* ctx, const pcdgpu_pk* pk, const pcdgpu_r1cs* r1cs, const void* z,
                                 const void* r, const void* s, void* out_proof);
int pcdgpu_groth16_prove_sharded_dev(pcdgpu_ctx* ctx, const pcdgpu_pk* pk, const pcdgpu_r1cs* r1cs, const void* d_z,
                                     const void* r, const void* s, void* out_proof);
/* one MSM sharded by point range: `slice` = this rank's points (pcdgpu_bases_upload of the slice), scalars = this
 * rank's scalars; every rank receives the affine sum.  Collective. */
int pcdgpu_msm_bases_sharded(pcdgpu_ctx* ctx, const pcdgpu_bases* slice, const void* scalars, size_t n, void* out_affine);
int pcdgpu_msm_bases_sharded_dev(pcdgpu_ctx* ctx, const pcdgpu_bases* slice, const void* d_scalars, int scalars_mont,
                                 size_t n, void* d_out_affine);

/* ark-serialize CanonicalSerialize of the proof (compressed points: x with flag bits 7 = "y is the
 * larger root", 6 = infinity on the last byte): 152 B (MNT4) / 190 B (MNT6).  out: >= 190 bytes. */
int pcdgpu_serialize_proof(pcdgpu_ctx* ctx, int pairing, const void* proof_affine, uint8_t* out, size_t* out_len);

/* ---- pairings and proof verification (ark-ec PairingEngine::pairing, ark-groth16 / ark-gm17 verifier.rs) -------
 * Reduced ate pairings of MNT4-298 (GT = Fq4 = Fq2[v]/(v^2 - u), 160 B) and MNT6-298 (GT = Fq6 = Fq3[v]/(v^2 - u),
 * 240 B); GT bytes are arkworks' in-memory QuadExtField {c0, c1}, Montgomery limbs.  One GPU thread per pair / proof:
 * a single call takes milliseconds, throughput comes from large batches.  These calls take the same
 * one-caller-at-a-time guard as the provers.
 * Input rules of the verifiers: a proof with a coordinate >= p or a point off its curve gets out_ok = 0 (not an
 * error).  Membership of B in the prime-order subgroup of G2 is NOT checked -- arkworks' verify does not check it
 * either, its deserialization does: callers that take proofs from untrusted bytes pass the bytes to
 * pcdgpu_deserialize_proofs or pcdgpu_*_verify_batch_serialized below, which check it. */
/* out_gt[i] = e(g1[i], g2[i]); a point at infinity (x = y = 0) gives 1 */
int pcdgpu_pairing(pcdgpu_ctx* ctx, int pairing, const void* g1, const void* g2, size_t n, void* out_gt);
/* ark-groth16 prepare_verifying_key of VerifyingKey {alpha_g1, beta_g2, gamma_g2, delta_g2, gamma_abc_g1[num_inputs]}
 * (num_inputs counts the constant: gamma_abc_g1.len()).  Runs on the GPU: line coefficients of -gamma and -delta and
 * e(alpha, beta).  A key point off its curve or with a coordinate >= p: PCDGPU_E_ARG. */
typedef struct pcdgpu_groth16_pvk pcdgpu_groth16_pvk;
int pcdgpu_groth16_pvk_create(pcdgpu_ctx* ctx, int pairing, const void* alpha_g1, const void* beta_g2,
                              const void* gamma_g2, const void* delta_g2, const void* gamma_abc_g1, size_t num_inputs,
                              pcdgpu_groth16_pvk** out);
void pcdgpu_groth16_pvk_free(pcdgpu_groth16_pvk* pvk);
/* verify_with_processed_vk for n proofs: proofs = n x (A || B || C) in pcdgpu_groth16_prove's layout, inputs =
 * n x (num_inputs - 1) Montgomery Fr elements (ark's &[E::Fr]; may be NULL when num_inputs = 1); out_ok[i] = 1 / 0.
 * n = 0 returns PCDGPU_OK. */
int pcdgpu_groth16_verify_batch(pcdgpu_ctx* ctx, const pcdgpu_groth16_pvk* pvk, const void* proofs, const void* inputs,
                                size_t n, uint8_t* out_ok);
/* the same for GM17: VerifyingKey {h_g2, g_alpha_g1, h_beta_g2, g_gamma_g1, h_gamma_g2, query[num_inputs]}; both of
 * ark-gm17's pairing equations are checked per proof */
typedef struct pcdgpu_gm17_pvk pcdgpu_gm17_pvk;
int pcdgpu_gm17_pvk_create(pcdgpu_ctx* ctx, int pairing, const void* h_g2, const void* g_alpha_g1,
                           const void* h_beta_g2, const void* g_gamma_g1, const void* h_gamma_g2, const void* query,
                           size_t num_inputs, pcdgpu_gm17_pvk** out);
void pcdgpu_gm17_pvk_free(pcdgpu_gm17_pvk* pvk);
int pcdgpu_gm17_verify_batch(pcdgpu_ctx* ctx, const pcdgpu_gm17_pvk* pvk, const void* proofs, const void* inputs,
                             size_t n, uint8_t* out_ok);

/* ---- proofs from bytes (ark-serialize CanonicalDeserialize for Proof {a, b, c}, checked) -------------------------
 * bytes = n x pcdgpu_serialize_proof's encoding (152 B MNT4 / 190 B MNT6, rows back to back).  A point is valid when
 * every coordinate chunk (flag bits masked) is < p, not both flag bits are set, and either the infinity flag is set
 * (the point is infinity, whatever x is) or x^3 + a x + b has a square root (the one flag bit 7 selects); B must also
 * satisfy [r]B = O (G2 subgroup membership; both G1 groups have cofactor 1).  One GPU thread per proof.
 * out_affine = n x (A || B || C) in pcdgpu_groth16_prove's layout, all zero for an invalid proof; out_ok[i] = 1 / 0.
 * An invalid proof is a verdict, not an error.  n = 0 returns PCDGPU_OK; an unknown pairing or a null pointer with
 * n > 0: PCDGPU_E_ARG. */
int pcdgpu_deserialize_proofs(pcdgpu_ctx* ctx, int pairing, const uint8_t* bytes, size_t n, void* out_affine,
                              uint8_t* out_ok);
/* deserialize and verify in one call, the proofs staying on the device in between: out_ok[i] = the bytes are a valid
 * proof && it verifies (pcdgpu_*_verify_batch's rules for inputs and n) */
int pcdgpu_groth16_verify_batch_serialized(pcdgpu_ctx* ctx, const pcdgpu_groth16_pvk* pvk, const uint8_t* bytes,
                                           const void* inputs, size_t n, uint8_t* out_ok);
int pcdgpu_gm17_verify_batch_serialized(pcdgpu_ctx* ctx, const pcdgpu_gm17_pvk* pvk, const uint8_t* bytes,
                                        const void* inputs, size_t n, uint8_t* out_ok);

/* ---- profiling ----------------------------------------------------------------------------------
 * CUDA-event spans around the library's kernel groups, on the context's stream.  Classes (array
 * index): 0 MSM digit/sort, 1 the accumulate kernel of a large G1 MSM, 2 same G2 over Fq2, 3 MSM bucket reduction,
 * 4 MSM window Horner, 5 NTT (all passes of a transform), 6 CSR mat-vec + QAP combine, 7 proof
 * assembly, 8 the accumulate kernel of a large G2 MSM over Fq3, 9 the whole accumulation phase of MSMs below 2^14
 * points (any curve), 10 what follows the accumulate kernel of a large MSM: part fold + heavy-bucket kernels.
 * read() synchronises, returns per class the summed milliseconds, algorithmic units
 * (bucket entries, butterflies, matrix rows, ...) and span count since the last read / enable, the
 * number of kernels launched, and resets.  Arrays hold PCDGPU_PROF_CLASSES entries. */
#define PCDGPU_PROF_CLASSES 11
int pcdgpu_profile_enable(pcdgpu_ctx* ctx, int on);
int pcdgpu_profile_read(pcdgpu_ctx* ctx, double* ms, double* units, uint64_t* spans, uint64_t* launches);
/* start / end (ms after the first span's start) and class of every span recorded since the last read:
 * the timeline of a proof whose MSMs overlap on the context's internal streams.  Does not reset. */
int pcdgpu_profile_timeline(pcdgpu_ctx* ctx, double* t0_ms, double* t1_ms, int* cls, size_t cap, size_t* count);

/* ---- measurement helpers ----------------------------------------------------------------------
 * Integer-pipe microbenchmark: every thread runs `iters` rounds of 8 independent
 * mad.wide-style chains; returns achieved 32x32->64 multiply-adds per second (the IMAD roof of
 * SURVEY.md 8d) and, with modmul != 0, Montgomery products per second of fp.cuh's operator*. */
int pcdgpu_bench_imad(pcdgpu_ctx* ctx, int modmul, int iters, double* out_ops_per_s, double* out_ms);

#ifdef __cplusplus
}
#endif
#endif /* PCDGPU_H */
