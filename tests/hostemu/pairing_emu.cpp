// CPU build of pcd_b200/csrc/pairing.cuh with the emulated PTX carry primitives (tests/hostemu/hostemu_prims.h).
// TEST INFRASTRUCTURE ONLY: compiled by tests/test_pairing_cpu.py into tests/hostemu/_build/libpairingemu.so and
// driven through ctypes, so that the device towers, Miller loop, final exponentiation and the per-proof verification
// are compared with oracle/pairing_oracle.py without a GPU, and their base-field products can be counted.
#define PCDGPU_HOSTEMU 1
#include "pairing.cuh"

#include <cstring>
#include <vector>

template <class T> static T ld(const void* p) { T r; memcpy((void*)&r, p, sizeof(T)); return r; }
template <class T> static void st(void* p, const T& a) { memcpy(p, (const void*)&a, sizeof(T)); }

template <class PP>
static void gt_op(int op, const void* a, const void* b, void* out) {
  typedef GT<PP> G;
  G x = ld<G>(a), y = ld<G>(b), r;
  switch (op) {
    case 0: r = G::mul(x, y); break;
    case 1: r = G::sqr(x); break;
    case 2: r = G::inverse(x); break;
    case 3: r = G::frobenius(x); break;
    case 4: r = x.conj(); break;
    case 5: r = final_exponentiation<PP>(x); break;
    default: r = G::one();
  }
  st(out, r);
}
extern "C" void emu_gt_op(int pairing, int op, const void* a, const void* b, void* out) {
  if (pairing == 0) gt_op<PairMnt4>(op, a, b, out); else gt_op<PairMnt6>(op, a, b, out);
}

template <class PP>
static void pairing_n(const char* g1, const char* g2, size_t n, char* out) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  for (size_t i = 0; i < n; i++)
    st(out + i * sizeof(GT<PP>), pairing<PP>(ld<A1>(g1 + i * sizeof(A1)), ld<A2>(g2 + i * sizeof(A2))));
}
extern "C" void emu_pairing(int pairing, const void* g1, const void* g2, size_t n, void* out) {
  if (pairing == 0) pairing_n<PairMnt4>((const char*)g1, (const char*)g2, n, (char*)out);
  else pairing_n<PairMnt6>((const char*)g1, (const char*)g2, n, (char*)out);
}

// base-field products since the last call (this thread)
extern "C" unsigned long long emu_products() {
  unsigned long long v = pcd_emu_products;
  pcd_emu_products = 0;
  return v;
}

template <class PP>
static std::vector<Line<typename PP::E>> lines_of(AffinePoint<typename PP::E> q, bool neg) {
  std::vector<Line<typename PP::E>> v(num_lines<PP>());
  prepare_lines<PP>(neg ? q.neg() : q, v.data());
  return v;
}

// vk: alpha_g1 || beta_g2 || gamma_g2 || delta_g2 || gamma_abc_g1[num_inputs]; proofs: n x (A || B || C);
// x: n x (num_inputs - 1) Montgomery elements; out_ok: n bytes
template <class PP>
static void g16(const char* vk, int num_inputs, const char* proofs, const char* x, size_t n, unsigned char* ok) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  A1 alpha = ld<A1>(vk);
  A2 beta = ld<A2>(vk + sizeof(A1)), gamma = ld<A2>(vk + sizeof(A1) + sizeof(A2)),
     delta = ld<A2>(vk + sizeof(A1) + 2 * sizeof(A2));
  auto lg = lines_of<PP>(gamma, true), ld_ = lines_of<PP>(delta, true);
  Groth16Pvk<PP> pvk;
  pvk.neg_gamma = lg.data();
  pvk.neg_delta = ld_.data();
  pvk.abc = reinterpret_cast<const A1*>(vk + sizeof(A1) + 3 * sizeof(A2));
  pvk.num_inputs = num_inputs;
  pvk.e_ab = pairing<PP>(alpha, beta);
  const size_t pb = 2 * sizeof(A1) + sizeof(A2);
  for (size_t i = 0; i < n; i++) {
    const char* p = proofs + i * pb;
    ok[i] = groth16_verify_one<PP>(pvk, ld<A1>(p), ld<A2>(p + sizeof(A1)), ld<A1>(p + sizeof(A1) + sizeof(A2)),
                                   reinterpret_cast<const typename PP::Fr*>(x) + i * (num_inputs - 1));
  }
}
extern "C" void emu_groth16_verify(int pairing, const void* vk, int num_inputs, const void* proofs, const void* x,
                                   size_t n, unsigned char* ok) {
  if (pairing == 0) g16<PairMnt4>((const char*)vk, num_inputs, (const char*)proofs, (const char*)x, n, ok);
  else g16<PairMnt6>((const char*)vk, num_inputs, (const char*)proofs, (const char*)x, n, ok);
}

// vk: h_g2 || g_alpha_g1 || h_beta_g2 || g_gamma_g1 || h_gamma_g2 || query[num_inputs]
template <class PP>
static void gm17(const char* vk, int num_inputs, const char* proofs, const char* x, size_t n, unsigned char* ok) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  const char* p = vk;
  A2 h = ld<A2>(p); p += sizeof(A2);
  A1 ga = ld<A1>(p); p += sizeof(A1);
  A2 hb = ld<A2>(p); p += sizeof(A2);
  A1 gg = ld<A1>(p); p += sizeof(A1);
  A2 hg = ld<A2>(p); p += sizeof(A2);
  auto l1 = lines_of<PP>(hg, true), l2 = lines_of<PP>(h, true), l3 = lines_of<PP>(hg, false);
  GM17Pvk<PP> pvk;
  pvk.neg_h_gamma = l1.data();
  pvk.neg_h = l2.data();
  pvk.h_gamma = l3.data();
  pvk.query = reinterpret_cast<const A1*>(p);
  pvk.num_inputs = num_inputs;
  pvk.g_alpha = ga;
  pvk.g_gamma = gg;
  pvk.h_beta = hb;
  pvk.e_ab = pairing<PP>(ga, hb);
  const size_t pb = 2 * sizeof(A1) + sizeof(A2);
  for (size_t i = 0; i < n; i++) {
    const char* q = proofs + i * pb;
    ok[i] = gm17_verify_one<PP>(pvk, ld<A1>(q), ld<A2>(q + sizeof(A1)), ld<A1>(q + sizeof(A1) + sizeof(A2)),
                                reinterpret_cast<const typename PP::Fr*>(x) + i * (num_inputs - 1));
  }
}
extern "C" void emu_gm17_verify(int pairing, const void* vk, int num_inputs, const void* proofs, const void* x,
                                size_t n, unsigned char* ok) {
  if (pairing == 0) gm17<PairMnt4>((const char*)vk, num_inputs, (const char*)proofs, (const char*)x, n, ok);
  else gm17<PairMnt6>((const char*)vk, num_inputs, (const char*)proofs, (const char*)x, n, ok);
}
