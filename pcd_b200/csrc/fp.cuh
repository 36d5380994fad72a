// fp.cuh -- 298-bit prime field arithmetic, Montgomery form, ten 32-bit limbs (R = 2^320).
//
// Replaces ark-ff's Fp320 (5 x u64 CIOS) on the GPU; the in-memory bytes are identical (little
// endian limbs of a*R mod p), so buffers cross the ABI without conversion.  Reached from the
// reference through every field op below IC::MainSNARK::prove / IC::HelpSNARK::prove
// (/root/reference/src/ec_cycle_pcd/mod.rs:171,179).
//
// The product is a row-wise Montgomery multiplication with the accumulator split into an
// "even" and an "odd" half so that every row is two long mad.lo.cc/madc.hi.cc chains, which
// ptxas turns into IMAD.WIDE.U32.X: 2*10*10 wide multiply-adds + 10 for the per-row quotient.
// All values are kept fully reduced (< p) so that results are canonical bytes.
#pragma once
#include "constants.cuh"

#define FP_LIMBS 10

// The modulus limbs and -p^-1 mod 2^32 of r4 as the Montgomery REDUCTION rows see them: read from constant memory, so
// that ptxas cannot see their values.  r4 has p[0] = 1 and -p^-1 = 0xffffffff; given those as immediates ptxas
// rewrites the quotient digit as a negation and the rows' mad.lo.cc / madc.hi.cc pairs no longer fuse into
// IMAD.WIDE.U32.X: every pair becomes IMAD.X + IMAD.HI.U32.X, two instructions on the fmaheavy pipe instead of one
// (cuobjdump, round 2: ntt_pass_kernel<FpR4> 81 IMAD.WIDE.X + 80 IMAD.X + 80 IMAD.HI.X per product against 161 + 0 + 0
// for q4) -- a third more multiply issue slots on every kernel over r4 (the main proof's NTTs, MNT6 G1 and G2).
#if defined(__CUDACC__)
static __constant__ u32 pcd_modc_r4[FP_LIMBS + 2] = {
    ParamsR4::mod(0), ParamsR4::mod(1), ParamsR4::mod(2), ParamsR4::mod(3), ParamsR4::mod(4), ParamsR4::mod(5),
    ParamsR4::mod(6), ParamsR4::mod(7), ParamsR4::mod(8), ParamsR4::mod(9), ParamsR4::INV, 0};
#endif
template <class P>
PCD_HD u32 fp_mod_opaque(int i) {  // i = FP_LIMBS: -p^-1 mod 2^32
#if defined(__CUDA_ARCH__)
  if (P::ID == 0) return pcd_modc_r4[i];
#endif
  return i < FP_LIMBS ? P::mod(i) : P::INV;
}

#if defined(PCDGPU_HOSTEMU)
// base-field products executed by this host thread: the work model of the pairing code (tests/hostemu)
inline thread_local unsigned long long pcd_emu_products = 0;
#endif

template <class P>
struct Fp {
  u32 l[FP_LIMBS];
  typedef P Params;
  static constexpr int WORDS = FP_LIMBS;  // u32 words per element

  PCD_HD static Fp zero() {
    Fp r;
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) r.l[i] = 0;
    return r;
  }
  PCD_HD static Fp one() {
    Fp r;
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) r.l[i] = P::one(i);
    return r;
  }
  PCD_HD static Fp r2() {
    Fp r;
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) r.l[i] = P::r2(i);
    return r;
  }
  PCD_HD bool is_zero() const {
    u32 t = 0;
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) t |= l[i];
    return t == 0;
  }
  PCD_HD bool operator==(const Fp& o) const {
    u32 t = 0;
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) t |= l[i] ^ o.l[i];
    return t == 0;
  }
  PCD_HD bool operator!=(const Fp& o) const { return !(*this == o); }

  // r = (a >= p) ? a - p : a, for a < 2p.
  PCD_HD static void reduce_once(u32* a) {
    u32 t[FP_LIMBS];
    t[0] = prims::sub_cc(a[0], P::mod(0));
#pragma unroll
    for (int i = 1; i < FP_LIMBS; i++) t[i] = prims::subc_cc(a[i], P::mod(i));
    u32 borrow = prims::subc(0, 0);  // 0xffffffff if a < p
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) a[i] = borrow ? a[i] : t[i];
  }

  PCD_HD friend Fp operator+(const Fp& a, const Fp& b) {
    Fp r;
    r.l[0] = prims::add_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < FP_LIMBS - 1; i++) r.l[i] = prims::addc_cc(a.l[i], b.l[i]);
    r.l[FP_LIMBS - 1] = prims::addc(a.l[FP_LIMBS - 1], b.l[FP_LIMBS - 1]);  // 2p < 2^320: no carry out
    reduce_once(r.l);
    return r;
  }
  PCD_HD friend Fp operator-(const Fp& a, const Fp& b) {
    Fp r;
    r.l[0] = prims::sub_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < FP_LIMBS; i++) r.l[i] = prims::subc_cc(a.l[i], b.l[i]);
    u32 borrow = prims::subc(0, 0);
    u32 t[FP_LIMBS];
    t[0] = prims::add_cc(r.l[0], P::mod(0));
#pragma unroll
    for (int i = 1; i < FP_LIMBS - 1; i++) t[i] = prims::addc_cc(r.l[i], P::mod(i));
    t[FP_LIMBS - 1] = prims::addc(r.l[FP_LIMBS - 1], P::mod(FP_LIMBS - 1));
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) r.l[i] = borrow ? t[i] : r.l[i];
    return r;
  }
  PCD_HD Fp neg() const {
    if (is_zero()) return *this;
    Fp r;
    r.l[0] = prims::sub_cc(P::mod(0), l[0]);
#pragma unroll
    for (int i = 1; i < FP_LIMBS - 1; i++) r.l[i] = prims::subc_cc(P::mod(i), l[i]);
    r.l[FP_LIMBS - 1] = prims::subc(P::mod(FP_LIMBS - 1), l[FP_LIMBS - 1]);
    return r;
  }
  PCD_HD Fp dbl() const { return *this + *this; }

  // ---- Montgomery product -------------------------------------------------------------------
  // acc[j], acc[j+1] = a[j] * bi   for j = 0, 2, ... n-2
  PCD_HD static void mul_n(u32* acc, const u32* a, u32 bi, int n = FP_LIMBS) {
#pragma unroll
    for (int j = 0; j < n; j += 2) {
      acc[j] = prims::mul_lo(a[j], bi);
      acc[j + 1] = prims::mul_hi(a[j], bi);
    }
  }
  // acc += sum_j a[j] * bi * 2^(32 j), j = 0, 2, ... n-2; one carry chain, carry left in CC.
  PCD_HD static void cmad_n(u32* acc, const u32* a, u32 bi, int n = FP_LIMBS) {
    acc[0] = prims::mad_lo_cc(a[0], bi, acc[0]);
    acc[1] = prims::madc_hi_cc(a[0], bi, acc[1]);
#pragma unroll
    for (int j = 2; j < n; j += 2) {
      acc[j] = prims::madc_lo_cc(a[j], bi, acc[j]);
      acc[j + 1] = prims::madc_hi_cc(a[j], bi, acc[j + 1]);
    }
  }
  // same with the modulus (compile-time limbs, offset off = 0 or 1)
  template <int OFF>
  PCD_HD static void cmad_mod(u32* acc, u32 m) {
    acc[0] = prims::mad_lo_cc(fp_mod_opaque<P>(OFF), m, acc[0]);
    acc[1] = prims::madc_hi_cc(fp_mod_opaque<P>(OFF), m, acc[1]);
#pragma unroll
    for (int j = 2; j < FP_LIMBS; j += 2) {
      acc[j] = prims::madc_lo_cc(fp_mod_opaque<P>(OFF + j), m, acc[j]);
      acc[j + 1] = prims::madc_hi_cc(fp_mod_opaque<P>(OFF + j), m, acc[j + 1]);
    }
  }
  // odd = (odd >> 64) + sum_j a[j] * bi * 2^(32 j) + CC, j = 0, 2, ... (a already offset by one)
  PCD_HD static void madc_n_rshift(u32* odd, const u32* a, u32 bi) {
#pragma unroll
    for (int j = 0; j < FP_LIMBS - 2; j += 2) {
      odd[j] = prims::madc_lo_cc(a[j], bi, odd[j + 2]);
      odd[j + 1] = prims::madc_hi_cc(a[j], bi, odd[j + 3]);
    }
    odd[FP_LIMBS - 2] = prims::madc_lo_cc(a[FP_LIMBS - 2], bi, 0);
    odd[FP_LIMBS - 1] = prims::madc_hi(a[FP_LIMBS - 2], bi, 0);
  }
  // One row: T = (T + a*bi + m*p) / 2^32 with T = even + odd*2^32 on entry (roles swap per row).
  PCD_HD static void mont_row(u32* even, u32* odd, const u32* a, u32 bi, bool first) {
    if (first) {
      mul_n(odd, a + 1, bi);
      mul_n(even, a, bi);
    } else {
      even[0] = prims::add_cc(even[0], odd[1]);
      madc_n_rshift(odd, a + 1, bi);
      cmad_n(even, a, bi);
      odd[FP_LIMBS - 1] = prims::addc(odd[FP_LIMBS - 1], 0);
    }
    u32 m = prims::mul_lo(even[0], fp_mod_opaque<P>(FP_LIMBS));
    cmad_mod<1>(odd, m);
    cmad_mod<0>(even, m);
    odd[FP_LIMBS - 1] = prims::addc(odd[FP_LIMBS - 1], 0);
  }

  PCD_HD friend Fp operator*(const Fp& a, const Fp& b) {
#if defined(PCDGPU_HOSTEMU)
    ++pcd_emu_products;
#endif
    return mul_cc(a, b);
  }
  // carry-chain product (IMAD.WIDE.U32.X rows)
  PCD_HD static Fp mul_cc(const Fp& a, const Fp& b) {
    u32 even[FP_LIMBS], odd[FP_LIMBS];
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i += 2) {
      mont_row(even, odd, a.l, b.l[i], i == 0);
      mont_row(odd, even, a.l, b.l[i + 1], false);
    }
    // T = even + (odd >> 32) (odd[0] is zero by construction)
    Fp r;
    r.l[0] = prims::add_cc(even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < FP_LIMBS - 1; i++) r.l[i] = prims::addc_cc(even[i], odd[i + 1]);
    r.l[FP_LIMBS - 1] = prims::addc(even[FP_LIMBS - 1], 0);
    reduce_once(r.l);
    return r;
  }
  PCD_HD Fp sqr() const { return (*this) * (*this); }
  // Out-of-line product for the extension-field code (Fq2/Fq3 points would otherwise inline
  // 40-80 copies of the 260-instruction product per group addition).
  PCD_NOINLINE static Fp mul_ni(Fp a, Fp b) { return a * b; }

  // multiply by a small compile-time constant with additions only
  template <u32 K>
  PCD_HD Fp mul_small() const {
    static_assert(K >= 1 && K < 256, "small constant");
    Fp acc = *this;
    bool started = false;
    Fp r = *this;
#pragma unroll
    for (int bit = 7; bit >= 0; bit--) {
      if (started) r = r.dbl();
      if ((K >> bit) & 1) {
        if (started) r = r + acc;
        else started = true;
      }
    }
    return r;
  }

  // limb i of p - 2 (exponent of the Fermat inverse)
  PCD_HD static constexpr u32 pm2(int i) {
    u64 borrow = 2;
    u32 out = 0;
    for (int k = 0; k <= i; k++) {
      u64 v = P::mod(k);
      out = (u32)(v - borrow);
      borrow = (v < borrow) ? 1 : 0;
    }
    return out;
  }
  // a^-1 = a^(p-2) (Fermat): ~450 dependent products.  Kept as the independent cross-check of inverse() in
  // tests/hostemu; the product path uses the binary Euclid below.
  PCD_HD Fp inverse_fermat() const {
    Fp r = one();
    bool started = false;
    for (int i = FP_LIMBS - 1; i >= 0; i--) {
      u32 e = 0;
#pragma unroll
      for (int k = 0; k < FP_LIMBS; k++)
        if (k == i) e = pm2(k);
      for (int b = 31; b >= 0; b--) {
        if (started) r = r.sqr();
        if ((e >> b) & 1) {
          r = started ? r * (*this) : *this;
          started = true;
        }
      }
    }
    return r;
  }
  // ---- inversion by the binary extended Euclidean algorithm -------------------------------------------------
  // Invariants: x1 * A = u, x2 * A = v (mod p) with A the integer held in the limbs (the Montgomery representative
  // a R); u and v lose a bit per step (< 2 * 298 halvings in all), every step is shifts and additions on ten limbs --
  // about a tenth of the ~450 dependent Montgomery products of Fermat's a^(p-2), which is what the single-thread
  // normalisations at the end of every MSM and proof used to wait for (0.3 - 0.4 ms each on B200).
  // The result (a R)^-1 is brought back to Montgomery form a^-1 R with two products by R^2.  Zero maps to zero.
  PCD_HD static void shr1(u32* a) {
#pragma unroll
    for (int i = 0; i < FP_LIMBS - 1; i++) a[i] = (a[i] >> 1) | (a[i + 1] << 31);
    a[FP_LIMBS - 1] >>= 1;
  }
  // x <- x / 2 mod p (x < p; p odd, x + p < 2^320)
  PCD_HD static void halve_mod(u32* x) {
    if (x[0] & 1) {
      x[0] = prims::add_cc(x[0], P::mod(0));
#pragma unroll
      for (int i = 1; i < FP_LIMBS - 1; i++) x[i] = prims::addc_cc(x[i], P::mod(i));
      x[FP_LIMBS - 1] = prims::addc(x[FP_LIMBS - 1], P::mod(FP_LIMBS - 1));
    }
    shr1(x);
  }
  // a >= b as integers
  PCD_HD static bool geq(const u32* a, const u32* b) {
    prims::sub_cc(a[0], b[0]);
#pragma unroll
    for (int i = 1; i < FP_LIMBS; i++) prims::subc_cc(a[i], b[i]);
    return prims::subc(0, 0) == 0;  // no borrow
  }
  PCD_HD static void sub_raw(u32* a, const u32* b) {  // a -= b, a >= b
    a[0] = prims::sub_cc(a[0], b[0]);
#pragma unroll
    for (int i = 1; i < FP_LIMBS - 1; i++) a[i] = prims::subc_cc(a[i], b[i]);
    a[FP_LIMBS - 1] = prims::subc(a[FP_LIMBS - 1], b[FP_LIMBS - 1]);
  }
  PCD_HD static bool is_one_raw(const u32* a) {
    u32 t = a[0] ^ 1u;
#pragma unroll
    for (int i = 1; i < FP_LIMBS; i++) t |= a[i];
    return t == 0;
  }
  PCD_HD Fp inverse() const {
    if (is_zero()) return *this;
    u32 u[FP_LIMBS], v[FP_LIMBS];
    Fp x1 = zero(), x2 = zero();
    x1.l[0] = 1;
#pragma unroll
    for (int i = 0; i < FP_LIMBS; i++) {
      u[i] = l[i];
      v[i] = P::mod(i);
    }
    while (!is_one_raw(u) && !is_one_raw(v)) {
      while (!(u[0] & 1)) {
        shr1(u);
        halve_mod(x1.l);
      }
      while (!(v[0] & 1)) {
        shr1(v);
        halve_mod(x2.l);
      }
      if (geq(u, v)) {
        sub_raw(u, v);
        x1 = x1 - x2;
      } else {
        sub_raw(v, u);
        x2 = x2 - x1;
      }
    }
    Fp r = is_one_raw(u) ? x1 : x2;  // (a R)^-1 as a plain integer
    return (r * r2()) * r2();         // -> a^-1 (plain) -> a^-1 R
  }
  // generic power by a 64-bit exponent
  PCD_HD Fp pow64(u64 e) const {
    Fp r = one();
    Fp base = *this;
    while (e) {
      if (e & 1) r = r * base;
      e >>= 1;
      if (e) base = base.sqr();
    }
    return r;
  }
  // leave / enter Montgomery form
  PCD_HD Fp from_mont() const {
    Fp o = zero();
    o.l[0] = 1;
    return (*this) * o;
  }
  PCD_HD Fp to_mont() const { return (*this) * r2(); }
  PCD_HD static Fp from_u32(u32 v) {
    Fp o = zero();
    o.l[0] = v;
    return o.to_mont();
  }
  // canonical-integer comparison helper for serialization flags: is this (Montgomery) element's
  // plain integer value > (p-1)/2 ?
  PCD_HD bool lexicographically_largest() const {
    Fp v = from_mont();
    Fp n = neg().from_mont();
    // compare v > n
#pragma unroll
    for (int i = FP_LIMBS - 1; i >= 0; i--) {
      if (v.l[i] != n.l[i]) return v.l[i] > n.l[i];
    }
    return false;
  }
};

typedef Fp<ParamsR4> FpR4;
typedef Fp<ParamsQ4> FpQ4;
