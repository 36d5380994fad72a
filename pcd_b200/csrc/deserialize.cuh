// deserialize.cuh -- ark-serialize's checked CanonicalDeserialize of compressed MNT4-298 / MNT6-298 points and of
// Groth16 / GM17 proofs (SURVEY.md B.5; oracle/deserialize_oracle.py restates the rules):
//
//   * x = 1 / 2 / 3 chunks of 38 bytes (c0, c1, c2), little-endian; flags in the top two bits of the last byte:
//     bit 7 "y is the lexicographically larger root", bit 6 "infinity"; both set is invalid.
//   * every chunk (flags masked) must be < p; with the infinity flag the point is infinity, whatever x is;
//   * otherwise y = sqrt(x^3 + a x + b), re-checked by squaring (so what the root routine returns on a non-square does
//     not matter), negated as the flag says;
//   * G2: [r]B = O (ark-ec 0.3's is_in_correct_subgroup_assuming_on_curve).  Both G1 curves have cofactor 1.
//
// Square roots are Tonelli-Shanks in every field (constants from tools/gen_constants.py).  The subgroup check is a
// double-and-add over the bits of r with XYZZ's exception-complete mixed addition: an intermediate multiple of a point
// outside the subgroup can equal +-B, and madd handles both (doubling, infinity).
#pragma once
#include "pairing.cuh"

template <class F> struct SqrtConsts;
template <> struct SqrtConsts<FpQ4> { typedef SqrtConstsQ4 K; };
template <> struct SqrtConsts<FpR4> { typedef SqrtConstsR4 K; };
template <> struct SqrtConsts<Fq2> { typedef SqrtConstsFq2 K; };
template <> struct SqrtConsts<Fq3> { typedef SqrtConstsFq3 K; };

// a square root of a (Tonelli-Shanks); false when a is not a square.  a = 0 gives 0.
template <class F>
PCD_NOINLINE bool field_sqrt(F a, F* out) {
  typedef typename SqrtConsts<F>::K K;
  const F one = F::one();
  if (a.is_zero()) {
    *out = a;
    return true;
  }
  F w = a;  // a^e, e = (t - 1) / 2, square and multiply from the top bit
#pragma unroll 1
  for (int b = K::E_BITS - 2; b >= 0; b--) {
    w = w.sqr();
    if ((K::e(b >> 5) >> (b & 31)) & 1u) w = w * a;
  }
  F x = a * w;  // a^((t + 1) / 2)
  F t = x * w;  // a^t, of order 2^k with k < v while a is a square
  F z;
  u32* zw = reinterpret_cast<u32*>(&z);
#pragma unroll 1
  for (int i = 0; i < F::WORDS; i++) zw[i] = K::zt(i);
  int v = K::S;
#pragma unroll 1
  while (!(t == one)) {
    int k = 0;
    F t2 = t;
#pragma unroll 1
    while (!(t2 == one)) {
      t2 = t2.sqr();
      if (++k == v) return false;  // t has order 2^v: a is not a square
    }
    F c = z;
#pragma unroll 1
    for (int j = 0; j < v - k - 1; j++) c = c.sqr();
    z = c.sqr();
    t = t * z;
    x = x * c;
    v = k;
  }
  *out = x;
  return true;
}

// 38 bytes -> the plain integer; false when it is not < p.  The flag bits of the last chunk are masked by the caller.
template <class B>
PCD_HD bool parse_coeff(const unsigned char* in, bool last, B* out) {
  B v;
#pragma unroll
  for (int i = 0; i < FP_LIMBS; i++) v.l[i] = 0;
#pragma unroll 1
  for (int i = 0; i < 38; i++) v.l[i >> 2] |= (u32)in[i] << ((i & 3) * 8);
  if (last) v.l[9] &= ~(0xC0u << 8);  // byte 37 = bits 8..15 of limb 9
  if (!base_canonical(v)) return false;
  *out = v.to_mont();
  return true;
}

template <class C>
PCD_HD constexpr int compressed_bytes() { return 38 * (C::F::WORDS / FP_LIMBS); }

// compressed bytes -> affine point on C (not yet checked for subgroup membership); false when invalid
template <class C>
PCD_HD bool decompress(const unsigned char* in, AffinePoint<typename C::F>* out) {
  typedef typename C::F F;
  typedef typename BaseOf<F>::T B;
  constexpr int D = F::WORDS / FP_LIMBS;
  const u32 flags = in[38 * D - 1] & 0xC0u;
  F x;
  B* xc = reinterpret_cast<B*>(&x);
  for (int i = 0; i < D; i++)
    if (!parse_coeff(in + 38 * i, i == D - 1, xc + i)) return false;
  if (flags == 0xC0u) return false;
  if (flags & 0x40u) {
    *out = AffinePoint<F>::inf();
    return true;
  }
  const F rhs = curve_rhs<C>(x);
  F y;
  if (!field_sqrt<F>(rhs, &y) || !(y.sqr() == rhs)) return false;
  if (y.lexicographically_largest() != ((flags & 0x80u) != 0)) y = y.neg();
  out->x = x;
  out->y = y;
  return true;
}

// bits of the scalar field's modulus r (the order of the prime subgroup)
template <class SP>
PCD_HD constexpr int modulus_bits() {
  int i = FP_LIMBS - 1;
  while (SP::mod(i) == 0) i--;
  int b = 0;
  while (SP::mod(i) >> b) b++;
  return 32 * i + b;
}

// [r]Q == O, Q on the curve
template <class C>
PCD_HD bool in_prime_subgroup(const AffinePoint<typename C::F>& q) {
  typedef typename C::ScalarParams SP;
  typedef XYZZ<C> P;
  if (q.is_inf()) return true;
  P acc = P::from_affine(q);
#pragma unroll 1
  for (int b = modulus_bits<SP>() - 2; b >= 0; b--) {
    acc = acc.dbl();
    if ((SP::mod(b >> 5) >> (b & 31)) & 1u) acc.madd(q);
  }
  return acc.is_inf();
}

// one proof A || B || C in compressed bytes -> affine points (all zero when invalid); returns the verdict
template <class PP>
PCD_HD bool deserialize_proof(const unsigned char* in, AffinePoint<typename PP::B>* a, AffinePoint<typename PP::E>* b,
                              AffinePoint<typename PP::B>* c) {
  typedef typename PP::G1 G1;
  typedef typename PP::G2 G2;
  const int n1 = compressed_bytes<G1>(), n2 = compressed_bytes<G2>();
  // the G1 points and the byte checks first: the subgroup check is most of the work
  bool ok = decompress<G1>(in, a) && decompress<G1>(in + n1 + n2, c) && decompress<G2>(in + n1, b) &&
            in_prime_subgroup<G2>(*b);
  if (!ok) {
    *a = AffinePoint<typename PP::B>::inf();
    *b = AffinePoint<typename PP::E>::inf();
    *c = AffinePoint<typename PP::B>::inf();
  }
  return ok;
}

#if defined(__CUDACC__)
// deserialize.cu: n compressed proofs at d_bytes -> n rows (A || B || C) at d_rows and verdicts at d_ok, enqueued on
// the context's stream
struct pcdgpu_ctx;
int pcd_deserialize_proofs_dev(pcdgpu_ctx* ctx, int pairing, const void* d_bytes, size_t n, void* d_rows,
                               unsigned char* d_ok);
#endif
