// pairing.cu -- batched MNT4-298 / MNT6-298 pairings and Groth16 / GM17 proof verification on the GPU.
//
// Replaces ark-ec PairingEngine::pairing, ark-groth16 prepare_verifying_key / verify_with_processed_vk and ark-gm17
// verify_proof for callers that check many proofs.  One thread per pair or per proof: each runs the whole
// dependency chain of pairing.cuh (input checks, the public-input combination, one multi-Miller loop per pairing
// equation, the final exponentiation).  Throughput comes from the batch; a single proof is one long chain.
//
// Processed keys live on the device: the line coefficients of the key's G2 points (prepared once, read by every
// thread of a batch from the same addresses) and the key's G1 query; e(alpha, beta) is computed by the same code
// when the key is processed and travels to the kernels as a parameter.
#include <cstring>

#include "common.cuh"
#include "deserialize.cuh"

#define PAIR_CHECK_ARG(ctx, cond, msg)      \
  do {                                      \
    if (!(cond)) {                          \
      if (ctx) (ctx)->set_error("%s", msg); \
      return PCDGPU_E_ARG;                  \
    }                                       \
  } while (0)

static const int PAIR_BLOCK = 64;

template <class PP>
__global__ void __launch_bounds__(PAIR_BLOCK) pairing_kernel(const AffinePoint<typename PP::B>* __restrict__ g1,
                                                             const AffinePoint<typename PP::E>* __restrict__ g2,
                                                             size_t n, GT<PP>* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = pairing<PP>(g1[i], g2[i]);
}

// bad = 1 when a key point is off its curve or has a non-canonical coordinate
template <class PP>
__global__ void vk_check_kernel(const AffinePoint<typename PP::B>* g1, size_t n1, const AffinePoint<typename PP::E>* g2,
                                int n2, u32* bad) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n1 && !valid_point<typename PP::G1>(g1[i])) *bad = 1;
  if (i < (size_t)n2 && !valid_point<typename PP::G2>(g2[i])) *bad = 1;
}

struct PrepSpec {
  int n;
  int idx[3];  // G2 point of the key
  int neg[3];  // prepare -Q
};
template <class PP>
__global__ void vk_prepare_kernel(const AffinePoint<typename PP::E>* g2, PrepSpec spec, Line<typename PP::E>* lines) {
  const int j = threadIdx.x;
  if (j >= spec.n) return;
  AffinePoint<typename PP::E> q = g2[spec.idx[j]];
  if (q.is_inf()) return;  // no lines: the pair contributes 1 (the key keeps a null pointer)
  prepare_lines<PP>(spec.neg[j] ? q.neg() : q, lines + (size_t)j * num_lines<PP>());
}

template <class PP>
__global__ void __launch_bounds__(PAIR_BLOCK) groth16_verify_kernel(Groth16Pvk<PP> vk, const char* __restrict__ proofs,
                                                                    const typename PP::Fr* __restrict__ x, size_t n,
                                                                    unsigned char* __restrict__ ok, bool gated) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (gated && !ok[i])) return;
  const char* p = proofs + i * (2 * sizeof(A1) + sizeof(A2));
  ok[i] = groth16_verify_one<PP>(vk, *reinterpret_cast<const A1*>(p), *reinterpret_cast<const A2*>(p + sizeof(A1)),
                                 *reinterpret_cast<const A1*>(p + sizeof(A1) + sizeof(A2)),
                                 x + i * (size_t)(vk.num_inputs - 1));
}

template <class PP>
__global__ void __launch_bounds__(PAIR_BLOCK) gm17_verify_kernel(GM17Pvk<PP> vk, const char* __restrict__ proofs,
                                                                 const typename PP::Fr* __restrict__ x, size_t n,
                                                                 unsigned char* __restrict__ ok, bool gated) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (gated && !ok[i])) return;
  const char* p = proofs + i * (2 * sizeof(A1) + sizeof(A2));
  ok[i] = gm17_verify_one<PP>(vk, *reinterpret_cast<const A1*>(p), *reinterpret_cast<const A2*>(p + sizeof(A1)),
                              *reinterpret_cast<const A1*>(p + sizeof(A1) + sizeof(A2)),
                              x + i * (size_t)(vk.num_inputs - 1));
}

static unsigned grid_of(size_t n) { return (unsigned)((n + PAIR_BLOCK - 1) / PAIR_BLOCK); }

// A processed key of either scheme.  Groth16: G1 {alpha}, G2 {beta, gamma, delta}, lines of -gamma, -delta.
// GM17: G1 {g_alpha, g_gamma}, G2 {h, h_beta, h_gamma}, lines of -h_gamma, -h, h_gamma.
struct VkCommon {
  int pairing = 0, device = 0;
  size_t num_inputs = 0;
  void* d_mem = nullptr;
  const void* lines[3] = {nullptr, nullptr, nullptr};
  const void* query = nullptr;
  unsigned char g1[2][80];
  unsigned char g2[3][240];
  unsigned char e_ab[240];
};
struct pcdgpu_groth16_pvk : VkCommon {};
struct pcdgpu_gm17_pvk : VkCommon {};

static bool all_zero(const void* p, size_t n) {
  const unsigned char* b = (const unsigned char*)p;
  for (size_t i = 0; i < n; i++)
    if (b[i]) return false;
  return true;
}

// Uploads the key's points, checks them, prepares the lines of spec and computes e(g1[0], g2[pair_g2]).
template <class PP>
static int vk_process(pcdgpu_ctx* ctx, VkCommon* v, int n1, int n2, const PrepSpec& spec, int pair_g2,
                      const void* query) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  typedef Line<typename PP::E> L;
  const size_t nl = num_lines<PP>();
  const size_t off_q = 3 * nl * sizeof(L);
  const size_t off_g1 = off_q + v->num_inputs * sizeof(A1);
  const size_t off_g2 = off_g1 + 2 * sizeof(A1);
  const size_t off_gt = off_g2 + 3 * sizeof(A2);
  const size_t off_bad = off_gt + sizeof(GT<PP>);
  const size_t bytes = off_bad + 16;
  if (cudaMalloc(&v->d_mem, bytes) != cudaSuccess) {
    ctx->set_error("cudaMalloc(%zu) for a verifying key", bytes);
    return PCDGPU_E_NOMEM;
  }
  char* d = (char*)v->d_mem;
  cudaStream_t st = ctx->stream;
  PCD_CUDA(ctx, cudaMemsetAsync(d + off_bad, 0, 16, st));
  PCD_CUDA(ctx, cudaMemcpyAsync(d + off_q, query, v->num_inputs * sizeof(A1), cudaMemcpyHostToDevice, st));
  for (int i = 0; i < n1; i++)
    PCD_CUDA(ctx, cudaMemcpyAsync(d + off_g1 + i * sizeof(A1), v->g1[i], sizeof(A1), cudaMemcpyHostToDevice, st));
  for (int i = 0; i < n2; i++)
    PCD_CUDA(ctx, cudaMemcpyAsync(d + off_g2 + i * sizeof(A2), v->g2[i], sizeof(A2), cudaMemcpyHostToDevice, st));
  // the query and the fixed points in one pass (they are contiguous)
  vk_check_kernel<PP><<<grid_of(v->num_inputs + n1), PAIR_BLOCK, 0, st>>>((const A1*)(d + off_q), v->num_inputs + n1,
                                                                          (const A2*)(d + off_g2), n2, (u32*)(d + off_bad));
  vk_prepare_kernel<PP><<<1, 32, 0, st>>>((const A2*)(d + off_g2), spec, (L*)d);
  pairing_kernel<PP><<<1, 1, 0, st>>>((const A1*)(d + off_g1), (const A2*)(d + off_g2 + pair_g2 * sizeof(A2)), 1,
                                      (GT<PP>*)(d + off_gt));
  PCD_CUDA(ctx, cudaGetLastError());
  u32 bad = 0;
  PCD_CUDA(ctx, cudaMemcpyAsync(v->e_ab, d + off_gt, sizeof(GT<PP>), cudaMemcpyDeviceToHost, st));
  PCD_CUDA(ctx, cudaMemcpyAsync(&bad, d + off_bad, 4, cudaMemcpyDeviceToHost, st));
  PCD_CUDA(ctx, cudaStreamSynchronize(st));
  PAIR_CHECK_ARG(ctx, !bad, "a verifying-key point is off its curve or has a coordinate >= p");
  for (int j = 0; j < spec.n; j++)
    v->lines[j] = all_zero(v->g2[spec.idx[j]], sizeof(A2)) ? nullptr : d + j * nl * sizeof(L);
  v->query = d + off_q;
  return 0;
}

template <class PP>
static Groth16Pvk<PP> groth16_view(const VkCommon* v) {
  typedef Line<typename PP::E> L;
  Groth16Pvk<PP> k;
  k.neg_gamma = (const L*)v->lines[0];
  k.neg_delta = (const L*)v->lines[1];
  k.abc = (const AffinePoint<typename PP::B>*)v->query;
  k.num_inputs = (int)v->num_inputs;
  memcpy((void*)&k.e_ab, v->e_ab, sizeof(GT<PP>));
  return k;
}
template <class PP>
static GM17Pvk<PP> gm17_view(const VkCommon* v) {
  typedef Line<typename PP::E> L;
  typedef AffinePoint<typename PP::B> A1;
  GM17Pvk<PP> k;
  k.neg_h_gamma = (const L*)v->lines[0];
  k.neg_h = (const L*)v->lines[1];
  k.h_gamma = (const L*)v->lines[2];
  k.query = (const A1*)v->query;
  k.num_inputs = (int)v->num_inputs;
  memcpy((void*)&k.g_alpha, v->g1[0], sizeof(A1));
  memcpy((void*)&k.g_gamma, v->g1[1], sizeof(A1));
  memcpy((void*)&k.h_beta, v->g2[1], sizeof(AffinePoint<typename PP::E>));
  memcpy((void*)&k.e_ab, v->e_ab, sizeof(GT<PP>));
  return k;
}

static void vk_free(VkCommon* v) {
  if (!v) return;
  if (v->d_mem) {
    cudaSetDevice(v->device);
    cudaFree(v->d_mem);
  }
}

// Stages n proofs (and their inputs) and runs the scheme's kernel; out_ok on the host when it returns.  serialized:
// the proofs are compressed bytes, deserialized on the device into the rows the verifier reads; a proof whose bytes
// are invalid keeps verdict 0 (the verify kernel skips it).
static int verify_batch(pcdgpu_ctx* ctx, const VkCommon* v, bool gm17, const void* proofs, const void* inputs, size_t n,
                        uint8_t* out_ok, bool serialized = false) {
  PAIR_CHECK_ARG(ctx, v && (n == 0 || (proofs && out_ok && (v->num_inputs == 1 || inputs))), "null pointer");
  if (n == 0) return PCDGPU_OK;
  PAIR_CHECK_ARG(ctx, v->device == ctx->device, "the key was processed on another device");
  PCD_CUDA(ctx, cudaSetDevice(ctx->device));
  InProofGuard guard(ctx);
  PAIR_CHECK_ARG(ctx, guard.ok, "the context is running a call on another host thread (one context per thread)");
  const bool m4 = v->pairing == PCDGPU_MNT4_298;
  const size_t proof_bytes = m4 ? 320 : 400;
  const size_t ser_bytes = serialized ? n * (m4 ? 152 : 190) : 0;
  const size_t ok_bytes = (n + 255) & ~(size_t)255;
  const size_t x_bytes = n * (v->num_inputs - 1) * 40;
  void *dp, *dx, *dok;
  PCD_TRY(ctx->scratch(SLOT_IO, n * proof_bytes, &dp));
  PCD_TRY(ctx->scratch(SLOT_IO2, x_bytes + 16, &dx));
  PCD_TRY(ctx->scratch(SLOT_MISC, ok_bytes + ser_bytes, &dok));
  cudaStream_t st = ctx->stream;
  if (serialized) {
    unsigned char* dser = (unsigned char*)dok + ok_bytes;
    PCD_CUDA(ctx, cudaMemcpyAsync(dser, proofs, ser_bytes, cudaMemcpyHostToDevice, st));
    PCD_TRY(pcd_deserialize_proofs_dev(ctx, v->pairing, dser, n, dp, (unsigned char*)dok));
  } else {
    PCD_CUDA(ctx, cudaMemcpyAsync(dp, proofs, n * proof_bytes, cudaMemcpyHostToDevice, st));
  }
  if (x_bytes) PCD_CUDA(ctx, cudaMemcpyAsync(dx, inputs, x_bytes, cudaMemcpyHostToDevice, st));
  if (m4 && !gm17)
    groth16_verify_kernel<PairMnt4><<<grid_of(n), PAIR_BLOCK, 0, st>>>(groth16_view<PairMnt4>(v), (const char*)dp,
                                                                      (const FpR4*)dx, n, (unsigned char*)dok,
                                                                      serialized);
  else if (!gm17)
    groth16_verify_kernel<PairMnt6><<<grid_of(n), PAIR_BLOCK, 0, st>>>(groth16_view<PairMnt6>(v), (const char*)dp,
                                                                      (const FpQ4*)dx, n, (unsigned char*)dok,
                                                                      serialized);
  else if (m4)
    gm17_verify_kernel<PairMnt4><<<grid_of(n), PAIR_BLOCK, 0, st>>>(gm17_view<PairMnt4>(v), (const char*)dp,
                                                                   (const FpR4*)dx, n, (unsigned char*)dok,
                                                                   serialized);
  else
    gm17_verify_kernel<PairMnt6><<<grid_of(n), PAIR_BLOCK, 0, st>>>(gm17_view<PairMnt6>(v), (const char*)dp,
                                                                   (const FpQ4*)dx, n, (unsigned char*)dok,
                                                                   serialized);
  PCD_CUDA(ctx, cudaGetLastError());
  PCD_CUDA(ctx, cudaMemcpyAsync(out_ok, dok, n, cudaMemcpyDeviceToHost, st));
  PCD_CUDA(ctx, cudaStreamSynchronize(st));
  return PCDGPU_OK;
}

extern "C" {

int pcdgpu_pairing(pcdgpu_ctx* ctx, int pairing, const void* g1, const void* g2, size_t n, void* out_gt) {
  if (!ctx) return PCDGPU_E_ARG;
  PAIR_CHECK_ARG(ctx, pairing == PCDGPU_MNT4_298 || pairing == PCDGPU_MNT6_298, "unknown pairing id");
  PAIR_CHECK_ARG(ctx, n == 0 || (g1 && g2 && out_gt), "null pointer");
  if (n == 0) return PCDGPU_OK;
  PCD_CUDA(ctx, cudaSetDevice(ctx->device));
  InProofGuard guard(ctx);
  PAIR_CHECK_ARG(ctx, guard.ok, "the context is running a call on another host thread (one context per thread)");
  const bool m4 = pairing == PCDGPU_MNT4_298;
  const size_t b1 = 80, b2 = m4 ? 160 : 240, bt = m4 ? 160 : 240;
  void *d1, *d2, *dt;
  PCD_TRY(ctx->scratch(SLOT_IO, n * b1, &d1));
  PCD_TRY(ctx->scratch(SLOT_IO2, n * b2, &d2));
  PCD_TRY(ctx->scratch(SLOT_MISC, n * bt, &dt));
  cudaStream_t st = ctx->stream;
  PCD_CUDA(ctx, cudaMemcpyAsync(d1, g1, n * b1, cudaMemcpyHostToDevice, st));
  PCD_CUDA(ctx, cudaMemcpyAsync(d2, g2, n * b2, cudaMemcpyHostToDevice, st));
  if (m4)
    pairing_kernel<PairMnt4><<<grid_of(n), PAIR_BLOCK, 0, st>>>((const AffinePoint<FpQ4>*)d1, (const AffinePoint<Fq2>*)d2,
                                                               n, (GT<PairMnt4>*)dt);
  else
    pairing_kernel<PairMnt6><<<grid_of(n), PAIR_BLOCK, 0, st>>>((const AffinePoint<FpR4>*)d1, (const AffinePoint<Fq3>*)d2,
                                                               n, (GT<PairMnt6>*)dt);
  PCD_CUDA(ctx, cudaGetLastError());
  PCD_CUDA(ctx, cudaMemcpyAsync(out_gt, dt, n * bt, cudaMemcpyDeviceToHost, st));
  PCD_CUDA(ctx, cudaStreamSynchronize(st));
  return PCDGPU_OK;
}

int pcdgpu_groth16_pvk_create(pcdgpu_ctx* ctx, int pairing, const void* alpha_g1, const void* beta_g2,
                              const void* gamma_g2, const void* delta_g2, const void* gamma_abc_g1, size_t num_inputs,
                              pcdgpu_groth16_pvk** out) {
  if (!ctx) return PCDGPU_E_ARG;
  PAIR_CHECK_ARG(ctx, pairing == PCDGPU_MNT4_298 || pairing == PCDGPU_MNT6_298, "unknown pairing id");
  PAIR_CHECK_ARG(ctx, out && alpha_g1 && beta_g2 && gamma_g2 && delta_g2 && gamma_abc_g1, "null pointer");
  PAIR_CHECK_ARG(ctx, num_inputs >= 1, "gamma_abc_g1 holds at least the constant's point");
  PCD_CUDA(ctx, cudaSetDevice(ctx->device));
  InProofGuard guard(ctx);
  PAIR_CHECK_ARG(ctx, guard.ok, "the context is running a call on another host thread (one context per thread)");
  const size_t b2 = pairing == PCDGPU_MNT4_298 ? 160 : 240;
  pcdgpu_groth16_pvk* v = new pcdgpu_groth16_pvk();
  v->pairing = pairing;
  v->device = ctx->device;
  v->num_inputs = num_inputs;
  memcpy(v->g1[0], alpha_g1, 80);
  memset(v->g1[1], 0, 80);
  memcpy(v->g2[0], beta_g2, b2);
  memcpy(v->g2[1], gamma_g2, b2);
  memcpy(v->g2[2], delta_g2, b2);
  PrepSpec spec = {2, {1, 2, 0}, {1, 1, 0}};
  int rc = pairing == PCDGPU_MNT4_298 ? vk_process<PairMnt4>(ctx, v, 1, 3, spec, 0, gamma_abc_g1)
                                      : vk_process<PairMnt6>(ctx, v, 1, 3, spec, 0, gamma_abc_g1);
  if (rc) {
    vk_free(v);
    delete v;
    return rc;
  }
  *out = v;
  return PCDGPU_OK;
}

void pcdgpu_groth16_pvk_free(pcdgpu_groth16_pvk* v) {
  vk_free(v);
  delete v;
}

int pcdgpu_groth16_verify_batch(pcdgpu_ctx* ctx, const pcdgpu_groth16_pvk* pvk, const void* proofs, const void* inputs,
                                size_t n, uint8_t* out_ok) {
  if (!ctx) return PCDGPU_E_ARG;
  return verify_batch(ctx, pvk, false, proofs, inputs, n, out_ok);
}

int pcdgpu_gm17_pvk_create(pcdgpu_ctx* ctx, int pairing, const void* h_g2, const void* g_alpha_g1,
                           const void* h_beta_g2, const void* g_gamma_g1, const void* h_gamma_g2, const void* query,
                           size_t num_inputs, pcdgpu_gm17_pvk** out) {
  if (!ctx) return PCDGPU_E_ARG;
  PAIR_CHECK_ARG(ctx, pairing == PCDGPU_MNT4_298 || pairing == PCDGPU_MNT6_298, "unknown pairing id");
  PAIR_CHECK_ARG(ctx, out && h_g2 && g_alpha_g1 && h_beta_g2 && g_gamma_g1 && h_gamma_g2 && query, "null pointer");
  PAIR_CHECK_ARG(ctx, num_inputs >= 1, "query holds at least the constant's point");
  PCD_CUDA(ctx, cudaSetDevice(ctx->device));
  InProofGuard guard(ctx);
  PAIR_CHECK_ARG(ctx, guard.ok, "the context is running a call on another host thread (one context per thread)");
  const size_t b2 = pairing == PCDGPU_MNT4_298 ? 160 : 240;
  pcdgpu_gm17_pvk* v = new pcdgpu_gm17_pvk();
  v->pairing = pairing;
  v->device = ctx->device;
  v->num_inputs = num_inputs;
  memcpy(v->g1[0], g_alpha_g1, 80);
  memcpy(v->g1[1], g_gamma_g1, 80);
  memcpy(v->g2[0], h_g2, b2);
  memcpy(v->g2[1], h_beta_g2, b2);
  memcpy(v->g2[2], h_gamma_g2, b2);
  PrepSpec spec = {3, {2, 0, 2}, {1, 1, 0}};
  int rc = pairing == PCDGPU_MNT4_298 ? vk_process<PairMnt4>(ctx, v, 2, 3, spec, 1, query)
                                      : vk_process<PairMnt6>(ctx, v, 2, 3, spec, 1, query);
  if (rc) {
    vk_free(v);
    delete v;
    return rc;
  }
  *out = v;
  return PCDGPU_OK;
}

void pcdgpu_gm17_pvk_free(pcdgpu_gm17_pvk* v) {
  vk_free(v);
  delete v;
}

int pcdgpu_gm17_verify_batch(pcdgpu_ctx* ctx, const pcdgpu_gm17_pvk* pvk, const void* proofs, const void* inputs,
                             size_t n, uint8_t* out_ok) {
  if (!ctx) return PCDGPU_E_ARG;
  return verify_batch(ctx, pvk, true, proofs, inputs, n, out_ok);
}

int pcdgpu_groth16_verify_batch_serialized(pcdgpu_ctx* ctx, const pcdgpu_groth16_pvk* pvk, const uint8_t* bytes,
                                           const void* inputs, size_t n, uint8_t* out_ok) {
  if (!ctx) return PCDGPU_E_ARG;
  return verify_batch(ctx, pvk, false, bytes, inputs, n, out_ok, true);
}

int pcdgpu_gm17_verify_batch_serialized(pcdgpu_ctx* ctx, const pcdgpu_gm17_pvk* pvk, const uint8_t* bytes,
                                        const void* inputs, size_t n, uint8_t* out_ok) {
  if (!ctx) return PCDGPU_E_ARG;
  return verify_batch(ctx, pvk, true, bytes, inputs, n, out_ok, true);
}

}  // extern "C"
