// pcdgpu_snark.hpp -- C++ host mirror of the reference's SNARK interface for the Groth16 and GM17 proving paths,
// on top of the C ABI (pcdgpu.h).  Header only.
//
// The reference binds its SNARKs through ark-snark's traits (re-exported by ark-crypto-primitives):
//     trait SNARK<F> { type ProvingKey; type VerifyingKey; type Proof; type ProcessedVerifyingKey; type Error;
//                      fn circuit_specific_setup(circuit, rng) -> Result<(PK, VK), Error>;
//                      fn prove(pk, circuit, rng) -> Result<Proof, Error>;
//                      fn verify(vk, x, proof) -> Result<bool, Error>; ... }
// used at /root/reference/src/ec_cycle_pcd/mod.rs:69,71,78,171,179,239 with
// MainSNARK = Groth16<MNT4_298>, HelpSNARK = Groth16<MNT6_298> (/root/reference/tests/mnt4_groth16.rs:23-30).
// The Rust toolchain is absent from the build environment, so this mirror is C++ (the reference is
// compiled code); INTEGRATION.md holds the Rust shim a maintainer would add.  Names and argument meaning
// follow ark-groth16 / ark-relations: ProvingKey, VerifyingKey parts, Proof {a, b, c},
// ConstraintMatrices (rows of (coeff, column); instance variables first, column 0 = constant 1),
// Groth16::prove draws r then s from the caller's rng (create_random_proof) and calls
// create_proof_with_reduction.  Setup and verification stay with the CPU implementation on the other side
// of the boundary (SURVEY.md 3.3 / 3.4) and report Error::Unsupported here.
//
// Error behaviour: like the Rust `Result`, every operation returns a Result<T>; nothing throws.
#ifndef PCDGPU_SNARK_HPP
#define PCDGPU_SNARK_HPP

#include <array>
#include <cstdint>
#include <cstring>
#include <string>
#include <utility>
#include <map>
#include <vector>

#include "pcdgpu.h"

namespace pcdgpu {

// ---- Result / Error (ark-relations SynthesisError + backend errors) --------------------------------
enum class ErrorKind { None, Unsupported, AssignmentMissing, MalformedKey, DomainTooLarge, Backend, InvalidData };
struct Error {
  ErrorKind kind = ErrorKind::None;
  int code = 0;          // PCDGPU_E_* for Backend errors
  std::string message;
};
template <class T>
struct Result {
  T value{};
  Error error;
  bool is_ok() const { return error.kind == ErrorKind::None; }
  explicit operator bool() const { return is_ok(); }
};

// ---- curve cycle configuration (ark-mnt4-298 / ark-mnt6-298) ------------------------------------------
using Fr = std::array<uint64_t, 5>;  // BigInteger320 limbs; Montgomery form for field elements
struct MNT4_298 {
  static constexpr int PAIRING = PCDGPU_MNT4_298;
  static constexpr size_t G1_LIMBS = 10, G2_LIMBS = 20, PROOF_BYTES = 152;
};
struct MNT6_298 {
  static constexpr int PAIRING = PCDGPU_MNT6_298;
  static constexpr size_t G1_LIMBS = 10, G2_LIMBS = 30, PROOF_BYTES = 190;
};
template <class E> using G1Affine = std::array<uint64_t, E::G1_LIMBS>;  // x || y, infinity = zeros
template <class E> using G2Affine = std::array<uint64_t, E::G2_LIMBS>;

// ---- ark-relations ------------------------------------------------------------------------------------
// ConstraintMatrices<F>: a, b, c as rows of (coefficient, column index)
struct ConstraintMatrices {
  size_t num_instance_variables = 0;  // includes the constant 1
  size_t num_witness_variables = 0;
  size_t num_constraints = 0;
  std::vector<std::vector<std::pair<Fr, size_t>>> a, b, c;
};
// What synthesis (`ConstraintSynthesizer::generate_constraints` + `finalize`) leaves behind: the matrices
// and the two assignment vectors.  Circuits stay on the CPU; this is the object that crosses the boundary.
struct SynthesizedCircuit {
  ConstraintMatrices matrices;
  std::vector<Fr> instance_assignment;  // instance_assignment[0] = 1
  std::vector<Fr> witness_assignment;
};

// ---- ark-groth16 data structures ------------------------------------------------------------------------
template <class E>
struct VerifyingKey {
  G1Affine<E> alpha_g1{};
  G2Affine<E> beta_g2{}, gamma_g2{}, delta_g2{};
  std::vector<G1Affine<E>> gamma_abc_g1;
};
template <class E>
struct ProvingKey {
  VerifyingKey<E> vk;
  G1Affine<E> beta_g1{}, delta_g1{};
  std::vector<G1Affine<E>> a_query, b_g1_query, h_query, l_query;
  std::vector<G2Affine<E>> b_g2_query;
};
template <class E>
struct Proof {
  G1Affine<E> a{};
  G2Affine<E> b{};
  G1Affine<E> c{};
};

// one GPU context per host thread AND device (the ABI's rule: a context is never shared between host threads); shared
// by every Groth16<E> / GM17<E> call of that thread on that device, destroyed when the thread ends
class Backend {
  struct PerThread {
    std::map<int, pcdgpu_ctx*> by_device;
    ~PerThread() {
      for (auto& kv : by_device) pcdgpu_ctx_destroy(kv.second);
    }
  };

 public:
  static Result<pcdgpu_ctx*> get(int device = 0) {
    thread_local PerThread mine;
    Result<pcdgpu_ctx*> r;
    auto it = mine.by_device.find(device);
    if (it == mine.by_device.end()) {
      pcdgpu_ctx* ctx = nullptr;
      int rc = pcdgpu_ctx_create(device, &ctx);
      if (rc != PCDGPU_OK) {
        r.error = {ErrorKind::Backend, rc, pcdgpu_strerror(rc)};  // no CPU fallback: the error surfaces
        return r;
      }
      it = mine.by_device.emplace(device, ctx).first;
    }
    r.value = it->second;
    return r;
  }
};

// ---- Groth16<E>: SNARK + CircuitSpecificSetupSNARK --------------------------------------------------------
template <class E>
class Groth16 {
 public:
  using ProvingKeyT = ProvingKey<E>;
  using VerifyingKeyT = VerifyingKey<E>;
  using ProofT = Proof<E>;

  // Device-resident key + matrices; built once per circuit shape and reused by every prove()
  // (upstream rebuilds the matrices and re-reads the key on every call).
  struct Index {
    pcdgpu_pk* pk = nullptr;
    pcdgpu_r1cs* r1cs = nullptr;
    size_t num_vars = 0;
    ~Index() {
      if (pk) pcdgpu_pk_free(pk);
      if (r1cs) pcdgpu_r1cs_free(r1cs);
    }
    Index() = default;
    Index(const Index&) = delete;
    Index& operator=(const Index&) = delete;
  };

  // SNARK::circuit_specific_setup / verify: CPU side of the boundary
  template <class C, class R>
  static Result<std::pair<ProvingKeyT, VerifyingKeyT>> circuit_specific_setup(const C&, R&) {
    Result<std::pair<ProvingKeyT, VerifyingKeyT>> r;
    r.error = {ErrorKind::Unsupported, 0, "Groth16 setup stays with the CPU generator (ark-groth16 generate_random_parameters)"};
    return r;
  }
  static Result<bool> verify(const VerifyingKeyT&, const std::vector<Fr>&, const ProofT&) {
    Result<bool> r;
    r.error = {ErrorKind::Unsupported, 0, "verification (one pairing check) stays on the CPU"};
    return r;
  }

  static Result<bool> index(const ProvingKeyT& pk, const ConstraintMatrices& m, Index* out, bool precompute = true) {
    return upload(pk, m, out, precompute, false, 0, nullptr, 0, 1);
  }

  // ONE proof over the GPUs of a box (include/pcdgpu.h, multi-GPU section; PCD chains, whose proofs depend on each
  // other and cannot be spread over GPUs as independent jobs).  Called by `world` host threads (or processes), thread
  // `rank` on CUDA device `device`; comm_id = the PCDGPU_COMM_ID_BYTES bytes rank 0 got from pcdgpu_comm_unique_id
  // (ignored for world 1).  Collective: every rank calls index_sharded, then create_proof_sharded with the SAME
  // circuit, r and s, and every rank receives the proof -- bit-identical to create_proof_with_reduction's.
  static Result<bool> index_sharded(const ProvingKeyT& pk, const ConstraintMatrices& m, Index* out, int device,
                                    const void* comm_id, int rank, int world, bool precompute = true) {
    return upload(pk, m, out, precompute, true, device, comm_id, rank, world);
  }
  static Result<ProofT> create_proof_sharded(const Index& idx, const SynthesizedCircuit& circuit, const Fr& r, const Fr& s,
                                             int device) {
    return prove_impl(idx, circuit, r, s, device, true);
  }

 private:
  static Result<bool> upload(const ProvingKeyT& pk, const ConstraintMatrices& m, Index* out, bool precompute, bool sharded,
                             int device, const void* comm_id, int rank, int world) {
    Result<bool> res;
    auto ctx = Backend::get(device);
    if (!ctx) { res.error = ctx.error; return res; }
    if (sharded) {
      int have_rank = 0, have_world = 0;
      int rc = pcdgpu_comm_info(ctx.value, &have_rank, &have_world);
      if (rc == PCDGPU_OK && !(have_world == world && have_rank == rank))
        rc = pcdgpu_comm_init(ctx.value, comm_id, rank, world);
      if (rc != PCDGPU_OK) {
        res.error = {ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
        return res;
      }
    }
    const size_t nv = m.num_instance_variables + m.num_witness_variables;
    if (pk.a_query.size() != nv || pk.b_g1_query.size() != nv || pk.b_g2_query.size() != nv ||
        pk.l_query.size() != m.num_witness_variables) {
      res.error = {ErrorKind::MalformedKey, 0, "query lengths do not match the constraint system"};
      return res;
    }
    std::vector<uint32_t> ptr[3], col[3];
    std::vector<Fr> val[3];
    const std::vector<std::vector<std::pair<Fr, size_t>>>* mats[3] = {&m.a, &m.b, &m.c};
    for (int k = 0; k < 3; k++) {
      ptr[k].push_back(0);
      for (const auto& row : *mats[k]) {
        for (const auto& e : row) {
          val[k].push_back(e.first);
          col[k].push_back((uint32_t)e.second);
        }
        ptr[k].push_back((uint32_t)col[k].size());
      }
      ptr[k].resize(m.num_constraints + 1, (uint32_t)col[k].size());
    }
    int rc = pcdgpu_r1cs_upload(ctx.value, E::PAIRING, m.num_constraints, m.num_instance_variables,
                                m.num_witness_variables, ptr[0].data(), col[0].data(), val[0].data(), ptr[1].data(),
                                col[1].data(), val[1].data(), ptr[2].data(), col[2].data(), val[2].data(), &out->r1cs);
    if (rc == PCDGPU_OK)
      rc = (sharded ? pcdgpu_pk_upload_sharded : pcdgpu_pk_upload)(
          ctx.value, E::PAIRING, nv, m.num_instance_variables, pk.h_query.size(), pk.vk.alpha_g1.data(),
          pk.beta_g1.data(), pk.delta_g1.data(), pk.vk.beta_g2.data(), pk.vk.delta_g2.data(), pk.a_query.data(),
          pk.b_g1_query.data(), pk.b_g2_query.data(), pk.h_query.data(), pk.l_query.data(), precompute ? 1 : 0, &out->pk);
    if (rc != PCDGPU_OK) {
      res.error = {ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
      return res;
    }
    out->num_vars = nv;
    res.value = true;
    return res;
  }

 public:

  // ark-groth16 create_proof_with_reduction(circuit, pk, r, s); r, s as plain integers (into_repr)
  static Result<ProofT> create_proof_with_reduction(const Index& idx, const SynthesizedCircuit& circuit, const Fr& r,
                                                    const Fr& s) {
    return prove_impl(idx, circuit, r, s, 0, false);
  }

 private:
  static Result<ProofT> prove_impl(const Index& idx, const SynthesizedCircuit& circuit, const Fr& r, const Fr& s, int device,
                                   bool sharded) {
    Result<ProofT> res;
    auto ctx = Backend::get(device);
    if (!ctx) { res.error = ctx.error; return res; }
    std::vector<Fr> z(circuit.instance_assignment);
    z.insert(z.end(), circuit.witness_assignment.begin(), circuit.witness_assignment.end());
    if (z.size() != idx.num_vars || z.empty()) {
      res.error = {ErrorKind::AssignmentMissing, 0, "assignment length does not match the indexed circuit"};
      return res;
    }
    std::vector<uint64_t> out(2 * E::G1_LIMBS + E::G2_LIMBS);
    int rc = (sharded ? pcdgpu_groth16_prove_sharded : pcdgpu_groth16_prove)(ctx.value, idx.pk, idx.r1cs, z.data(), r.data(),
                                                                             s.data(), out.data());
    if (rc != PCDGPU_OK) {
      res.error = {rc == PCDGPU_E_DOMAIN ? ErrorKind::DomainTooLarge : ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
      return res;
    }
    std::memcpy(res.value.a.data(), out.data(), 8 * E::G1_LIMBS);
    std::memcpy(res.value.b.data(), out.data() + E::G1_LIMBS, 8 * E::G2_LIMBS);
    std::memcpy(res.value.c.data(), out.data() + E::G1_LIMBS + E::G2_LIMBS, 8 * E::G1_LIMBS);
    return res;
  }

 public:

  // SNARK::prove(pk, circuit, rng): r = Fr::rand(rng), then s = Fr::rand(rng) (create_random_proof's order).
  // Rng: any type with `Fr next_scalar(int pairing)` returning a uniform scalar as plain-integer limbs.
  template <class Rng>
  static Result<ProofT> prove(const Index& idx, const SynthesizedCircuit& circuit, Rng& rng) {
    Fr r = rng.next_scalar(E::PAIRING);
    Fr s = rng.next_scalar(E::PAIRING);
    return create_proof_with_reduction(idx, circuit, r, s);
  }

  // CanonicalSerialize for Proof<E>: a || b || c compressed
  static Result<std::vector<uint8_t>> serialize(const ProofT& p) {
    Result<std::vector<uint8_t>> res;
    auto ctx = Backend::get();
    if (!ctx) { res.error = ctx.error; return res; }
    std::vector<uint64_t> in(2 * E::G1_LIMBS + E::G2_LIMBS);
    std::memcpy(in.data(), p.a.data(), 8 * E::G1_LIMBS);
    std::memcpy(in.data() + E::G1_LIMBS, p.b.data(), 8 * E::G2_LIMBS);
    std::memcpy(in.data() + E::G1_LIMBS + E::G2_LIMBS, p.c.data(), 8 * E::G1_LIMBS);
    res.value.resize(192);
    size_t len = 0;
    int rc = pcdgpu_serialize_proof(ctx.value, E::PAIRING, in.data(), res.value.data(), &len);
    if (rc != PCDGPU_OK) {
      res.error = {ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
      return res;
    }
    res.value.resize(len);
    return res;
  }

  // CanonicalDeserialize for Proof<E> (checked, on the GPU): bytes that are not a valid proof give
  // ErrorKind::InvalidData (ark's SerializationError::InvalidData)
  static Result<ProofT> deserialize(const std::vector<uint8_t>& bytes) {
    Result<ProofT> res;
    if (bytes.size() != E::PROOF_BYTES) {
      res.error = {ErrorKind::InvalidData, 0, "a compressed proof has the wrong length"};
      return res;
    }
    auto ctx = Backend::get();
    if (!ctx) { res.error = ctx.error; return res; }
    std::vector<uint64_t> out(2 * E::G1_LIMBS + E::G2_LIMBS);
    uint8_t ok = 0;
    int rc = pcdgpu_deserialize_proofs(ctx.value, E::PAIRING, bytes.data(), 1, out.data(), &ok);
    if (rc != PCDGPU_OK) {
      res.error = {ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
      return res;
    }
    if (!ok) {
      res.error = {ErrorKind::InvalidData, 0, "invalid proof encoding"};
      return res;
    }
    std::memcpy(res.value.a.data(), out.data(), 8 * E::G1_LIMBS);
    std::memcpy(res.value.b.data(), out.data() + E::G1_LIMBS, 8 * E::G2_LIMBS);
    std::memcpy(res.value.c.data(), out.data() + E::G1_LIMBS + E::G2_LIMBS, 8 * E::G1_LIMBS);
    return res;
  }
};

// ---- ark-gm17 data structures and GM17<E>: SNARK + CircuitSpecificSetupSNARK -------------------------------
// Bound by the reference as MainSNARK / HelpSNARK at /root/reference/tests/mnt4_gm17.rs:27-28 and in the two
// mixed configurations (tests/mnt4_mix_groth16gm17.rs, tests/mnt4_mix_gm17groth16.rs).
template <class E>
struct GM17VerifyingKey {
  G2Affine<E> h_g2{}, h_beta_g2{}, h_gamma_g2{};
  G1Affine<E> g_alpha_g1{}, g_gamma_g1{};
  std::vector<G1Affine<E>> query;
};
template <class E>
struct GM17ProvingKey {
  GM17VerifyingKey<E> vk;
  std::vector<G1Affine<E>> a_query, c_query_1, c_query_2, g_gamma2_z_t;
  std::vector<G2Affine<E>> b_query;
  G1Affine<E> g_gamma_z{}, g_ab_gamma_z{}, g_gamma2_z2{};
  G2Affine<E> h_gamma_z{};
};

template <class E>
class GM17 {
 public:
  using ProvingKeyT = GM17ProvingKey<E>;
  using VerifyingKeyT = GM17VerifyingKey<E>;
  using ProofT = Proof<E>;  // ark-gm17 Proof { a: G1, b: G2, c: G1 }

  struct Index {
    pcdgpu_gm17_pk* pk = nullptr;
    pcdgpu_r1cs* r1cs = nullptr;
    size_t num_vars = 0;
    ~Index() {
      if (pk) pcdgpu_gm17_pk_free(pk);
      if (r1cs) pcdgpu_r1cs_free(r1cs);
    }
    Index() = default;
    Index(const Index&) = delete;
    Index& operator=(const Index&) = delete;
  };

  template <class C, class R>
  static Result<std::pair<ProvingKeyT, VerifyingKeyT>> circuit_specific_setup(const C&, R&) {
    Result<std::pair<ProvingKeyT, VerifyingKeyT>> r;
    r.error = {ErrorKind::Unsupported, 0, "GM17 setup stays with the CPU generator (ark-gm17 generate_random_parameters)"};
    return r;
  }
  static Result<bool> verify(const VerifyingKeyT&, const std::vector<Fr>&, const ProofT&) {
    Result<bool> r;
    r.error = {ErrorKind::Unsupported, 0, "verification (pairing checks) stays on the CPU"};
    return r;
  }

  static Result<bool> index(const ProvingKeyT& pk, const ConstraintMatrices& m, Index* out, bool precompute = true) {
    Result<bool> res;
    auto ctx = Backend::get();
    if (!ctx) { res.error = ctx.error; return res; }
    const size_t ni = m.num_instance_variables, nv = ni + m.num_witness_variables;
    const size_t nsap = nv + m.num_constraints + ni - 1;
    const size_t n = pcdgpu_sap_domain_size(E::PAIRING, m.num_constraints, ni);
    if (n == 0) {
      res.error = {ErrorKind::DomainTooLarge, PCDGPU_E_DOMAIN, "no evaluation domain large enough for the SAP"};
      return res;
    }
    if (ni < 1 || pk.a_query.size() != nsap || pk.b_query.size() != nsap || pk.c_query_2.size() != nsap ||
        pk.c_query_1.size() != nsap - ni || pk.g_gamma2_z_t.size() != n + 1) {
      res.error = {ErrorKind::MalformedKey, 0, "query lengths do not match the square arithmetic program"};
      return res;
    }
    std::vector<uint32_t> ptr[3], col[3];
    std::vector<Fr> val[3];
    const std::vector<std::vector<std::pair<Fr, size_t>>>* mats[3] = {&m.a, &m.b, &m.c};
    for (int k = 0; k < 3; k++) {
      ptr[k].push_back(0);
      for (const auto& row : *mats[k]) {
        for (const auto& e : row) {
          val[k].push_back(e.first);
          col[k].push_back((uint32_t)e.second);
        }
        ptr[k].push_back((uint32_t)col[k].size());
      }
      ptr[k].resize(m.num_constraints + 1, (uint32_t)col[k].size());
    }
    int rc = pcdgpu_r1cs_upload(ctx.value, E::PAIRING, m.num_constraints, ni, m.num_witness_variables, ptr[0].data(),
                                col[0].data(), val[0].data(), ptr[1].data(), col[1].data(), val[1].data(), ptr[2].data(),
                                col[2].data(), val[2].data(), &out->r1cs);
    if (rc == PCDGPU_OK)
      rc = pcdgpu_gm17_pk_upload(ctx.value, E::PAIRING, nsap, ni, n + 1, pk.a_query.data(), pk.b_query.data(),
                                 pk.c_query_1.data(), pk.c_query_2.data(), pk.g_gamma2_z_t.data(), pk.g_gamma_z.data(),
                                 pk.h_gamma_z.data(), pk.g_ab_gamma_z.data(), pk.g_gamma2_z2.data(), precompute ? 1 : 0,
                                 &out->pk);
    if (rc != PCDGPU_OK) {
      res.error = {ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
      return res;
    }
    out->num_vars = nv;
    res.value = true;
    return res;
  }

  // ark-gm17 create_proof(circuit, pk, d1, d2, r); d1, d2, r as plain integers (into_repr)
  static Result<ProofT> create_proof(const Index& idx, const SynthesizedCircuit& circuit, const Fr& d1, const Fr& d2,
                                     const Fr& r) {
    Result<ProofT> res;
    auto ctx = Backend::get();
    if (!ctx) { res.error = ctx.error; return res; }
    std::vector<Fr> z(circuit.instance_assignment);
    z.insert(z.end(), circuit.witness_assignment.begin(), circuit.witness_assignment.end());
    if (z.size() != idx.num_vars || z.empty()) {
      res.error = {ErrorKind::AssignmentMissing, 0, "assignment length does not match the indexed circuit"};
      return res;
    }
    std::vector<uint64_t> out(2 * E::G1_LIMBS + E::G2_LIMBS);
    int rc = pcdgpu_gm17_prove(ctx.value, idx.pk, idx.r1cs, z.data(), d1.data(), d2.data(), r.data(), out.data());
    if (rc != PCDGPU_OK) {
      res.error = {rc == PCDGPU_E_DOMAIN ? ErrorKind::DomainTooLarge : ErrorKind::Backend, rc, pcdgpu_last_error(ctx.value)};
      return res;
    }
    std::memcpy(res.value.a.data(), out.data(), 8 * E::G1_LIMBS);
    std::memcpy(res.value.b.data(), out.data() + E::G1_LIMBS, 8 * E::G2_LIMBS);
    std::memcpy(res.value.c.data(), out.data() + E::G1_LIMBS + E::G2_LIMBS, 8 * E::G1_LIMBS);
    return res;
  }

  // SNARK::prove(pk, circuit, rng): d1, d2, r = Fr::rand(rng) in this order (create_random_proof)
  template <class Rng>
  static Result<ProofT> prove(const Index& idx, const SynthesizedCircuit& circuit, Rng& rng) {
    Fr d1 = rng.next_scalar(E::PAIRING);
    Fr d2 = rng.next_scalar(E::PAIRING);
    Fr r = rng.next_scalar(E::PAIRING);
    return create_proof(idx, circuit, d1, d2, r);
  }

  static Result<std::vector<uint8_t>> serialize(const ProofT& p) { return Groth16<E>::serialize(p); }
  static Result<ProofT> deserialize(const std::vector<uint8_t>& bytes) { return Groth16<E>::deserialize(bytes); }
};

}  // namespace pcdgpu
#endif  // PCDGPU_SNARK_HPP
