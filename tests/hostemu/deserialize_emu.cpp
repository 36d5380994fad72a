// CPU build of pcd_b200/csrc/deserialize.cuh with the emulated PTX carry primitives (tests/hostemu/hostemu_prims.h).
// TEST INFRASTRUCTURE ONLY: compiled by tests/test_deserialize_cpu.py into tests/hostemu/_build/libdeserializeemu.so
// and driven through ctypes, so that the device square roots, point decompression, subgroup check and proof
// deserialization are compared with oracle/deserialize_oracle.py without a GPU, and their base-field products counted.
#define PCDGPU_HOSTEMU 1
#include "deserialize.cuh"

#include <cstring>

template <class T> static T ld(const void* p) { T r; memcpy((void*)&r, p, sizeof(T)); return r; }
template <class T> static void st(void* p, const T& a) { memcpy(p, (const void*)&a, sizeof(T)); }

// field: 0 Fq of MNT4 (q4), 1 Fq of MNT6 (r4), 2 Fq2, 3 Fq3; n Montgomery elements in, roots out (0 when none)
template <class F>
static void sqrt_n(const char* a, size_t n, char* out, unsigned char* ok) {
  for (size_t i = 0; i < n; i++) {
    F y = F::zero();
    ok[i] = field_sqrt<F>(ld<F>(a + i * sizeof(F)), &y);
    st(out + i * sizeof(F), ok[i] ? y : F::zero());
  }
}
extern "C" void emu_sqrt(int field, const void* a, size_t n, void* out, unsigned char* ok) {
  const char* ac = (const char*)a;
  char* oc = (char*)out;
  if (field == 0) sqrt_n<FpQ4>(ac, n, oc, ok);
  else if (field == 1) sqrt_n<FpR4>(ac, n, oc, ok);
  else if (field == 2) sqrt_n<Fq2>(ac, n, oc, ok);
  else sqrt_n<Fq3>(ac, n, oc, ok);
}

// curve ids of include/pcdgpu.h; compressed points in, affine points out (zero when invalid).  subgroup: also check
// [r]P = O (what the proof deserializer does for G2)
template <class C>
static void points_n(const unsigned char* in, size_t n, char* out, unsigned char* ok, int subgroup) {
  typedef AffinePoint<typename C::F> A;
  for (size_t i = 0; i < n; i++) {
    A p = A::inf();
    bool v = decompress<C>(in + i * compressed_bytes<C>(), &p) && (!subgroup || in_prime_subgroup<C>(p));
    ok[i] = v;
    st(out + i * sizeof(A), v ? p : A::inf());
  }
}
extern "C" void emu_deserialize_points(int curve, const unsigned char* in, size_t n, void* out, unsigned char* ok,
                                       int subgroup) {
  char* oc = (char*)out;
  if (curve == 0) points_n<CurveMnt4G1>(in, n, oc, ok, subgroup);
  else if (curve == 1) points_n<CurveMnt4G2>(in, n, oc, ok, subgroup);
  else if (curve == 2) points_n<CurveMnt6G1>(in, n, oc, ok, subgroup);
  else points_n<CurveMnt6G2>(in, n, oc, ok, subgroup);
}

// [r]P = O for n affine points of a G2 curve (1 or 3)
template <class C>
static void subgroup_n(const char* pts, size_t n, unsigned char* ok) {
  for (size_t i = 0; i < n; i++) ok[i] = in_prime_subgroup<C>(ld<AffinePoint<typename C::F>>(pts + i * sizeof(AffinePoint<typename C::F>)));
}
extern "C" void emu_subgroup(int curve, const void* pts, size_t n, unsigned char* ok) {
  if (curve == 1) subgroup_n<CurveMnt4G2>((const char*)pts, n, ok);
  else subgroup_n<CurveMnt6G2>((const char*)pts, n, ok);
}

// n proofs of compressed bytes -> n x (A || B || C) affine limbs (zero rows when invalid) and verdicts
template <class PP>
static void proofs_n(const unsigned char* in, size_t n, char* out, unsigned char* ok) {
  typedef AffinePoint<typename PP::B> A1;
  typedef AffinePoint<typename PP::E> A2;
  const size_t nb = 2 * compressed_bytes<typename PP::G1>() + compressed_bytes<typename PP::G2>();
  const size_t pb = 2 * sizeof(A1) + sizeof(A2);
  for (size_t i = 0; i < n; i++) {
    A1 a, c;
    A2 b;
    ok[i] = deserialize_proof<PP>(in + i * nb, &a, &b, &c);
    st(out + i * pb, a);
    st(out + i * pb + sizeof(A1), b);
    st(out + i * pb + sizeof(A1) + sizeof(A2), c);
  }
}
extern "C" void emu_deserialize_proofs(int pairing, const unsigned char* in, size_t n, void* out, unsigned char* ok) {
  if (pairing == 0) proofs_n<PairMnt4>(in, n, (char*)out, ok);
  else proofs_n<PairMnt6>(in, n, (char*)out, ok);
}

// base-field products since the last call (this thread)
extern "C" unsigned long long emu_products() {
  unsigned long long v = pcd_emu_products;
  pcd_emu_products = 0;
  return v;
}
