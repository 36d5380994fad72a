// deserialize.cu -- batched checked deserialization of compressed Groth16 / GM17 proofs (deserialize.cuh).
//
// Replaces ark-serialize's CanonicalDeserialize for Proof {a, b, c} for callers that receive many proofs.  One thread
// per proof: byte checks, three decompressions (a square root each) and the G2 subgroup check [r]B = O, which is most
// of the work.  The rows land in pcdgpu_groth16_prove's layout (A || B || C affine Montgomery limbs), so that the
// verifiers of pairing.cu read them where they are.
#include "common.cuh"
#include "deserialize.cuh"

static const int DESER_BLOCK = 64;

template <class PP>
__global__ void __launch_bounds__(DESER_BLOCK) deserialize_kernel(const unsigned char* __restrict__ bytes, size_t n,
                                                                  char* __restrict__ rows,
                                                                  unsigned char* __restrict__ ok) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t nb = 2 * compressed_bytes<typename PP::G1>() + compressed_bytes<typename PP::G2>();
  A1 a, c;
  A2 b;
  ok[i] = deserialize_proof<PP>(bytes + i * nb, &a, &b, &c);
  char* r = rows + i * (2 * sizeof(A1) + sizeof(A2));
  *reinterpret_cast<A1*>(r) = a;
  *reinterpret_cast<A2*>(r + sizeof(A1)) = b;
  *reinterpret_cast<A1*>(r + sizeof(A1) + sizeof(A2)) = c;
}

int pcd_deserialize_proofs_dev(pcdgpu_ctx* ctx, int pairing, const void* d_bytes, size_t n, void* d_rows,
                               uint8_t* d_ok) {
  const unsigned grid = (unsigned)((n + DESER_BLOCK - 1) / DESER_BLOCK);
  if (pairing == PCDGPU_MNT4_298)
    deserialize_kernel<PairMnt4><<<grid, DESER_BLOCK, 0, ctx->stream>>>((const unsigned char*)d_bytes, n,
                                                                         (char*)d_rows, d_ok);
  else
    deserialize_kernel<PairMnt6><<<grid, DESER_BLOCK, 0, ctx->stream>>>((const unsigned char*)d_bytes, n,
                                                                         (char*)d_rows, d_ok);
  PCD_CUDA(ctx, cudaGetLastError());
  return PCDGPU_OK;
}

extern "C" int pcdgpu_deserialize_proofs(pcdgpu_ctx* ctx, int pairing, const uint8_t* bytes, size_t n,
                                         void* out_affine, uint8_t* out_ok) {
  if (!ctx) return PCDGPU_E_ARG;
  if (pairing != PCDGPU_MNT4_298 && pairing != PCDGPU_MNT6_298) {
    ctx->set_error("unknown pairing id");
    return PCDGPU_E_ARG;
  }
  if (n != 0 && !(bytes && out_affine && out_ok)) {
    ctx->set_error("null pointer");
    return PCDGPU_E_ARG;
  }
  if (n == 0) return PCDGPU_OK;
  PCD_CUDA(ctx, cudaSetDevice(ctx->device));
  InProofGuard guard(ctx);
  if (!guard.ok) {
    ctx->set_error("the context is running a call on another host thread (one context per thread)");
    return PCDGPU_E_ARG;
  }
  const bool m4 = pairing == PCDGPU_MNT4_298;
  const size_t nb = m4 ? 152 : 190, row = m4 ? 320 : 400;
  const size_t ok_bytes = (n + 255) & ~(size_t)255;
  void *drows, *dmisc;
  PCD_TRY(ctx->scratch(SLOT_IO, n * row, &drows));
  PCD_TRY(ctx->scratch(SLOT_MISC, ok_bytes + n * nb, &dmisc));
  uint8_t* dok = (uint8_t*)dmisc;
  cudaStream_t st = ctx->stream;
  PCD_CUDA(ctx, cudaMemcpyAsync(dok + ok_bytes, bytes, n * nb, cudaMemcpyHostToDevice, st));
  PCD_TRY(pcd_deserialize_proofs_dev(ctx, pairing, dok + ok_bytes, n, drows, dok));
  PCD_CUDA(ctx, cudaMemcpyAsync(out_affine, drows, n * row, cudaMemcpyDeviceToHost, st));
  PCD_CUDA(ctx, cudaMemcpyAsync(out_ok, dok, n, cudaMemcpyDeviceToHost, st));
  PCD_CUDA(ctx, cudaStreamSynchronize(st));
  return PCDGPU_OK;
}
