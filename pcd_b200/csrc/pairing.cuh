// pairing.cuh -- reduced ate pairings of MNT4-298 and MNT6-298 (ark-ec models/mnt4, models/mnt6) and the pieces of
// Groth16 / GM17 verification that run per proof.
//
//   GT of MNT4: Fq4 = Fq2[v]/(v^2 - u), u^2 = 17      GT of MNT6: Fq6 = Fq3[v]/(v^2 - u), u^3 = 5
// Memory layout = arkworks' QuadExtField {c0, c1}: 160 B / 240 B of Montgomery limbs.  Under w = v, w^2 = u the
// coefficient i of half h is the coefficient of w^(2 i + h) of Fq[w]/(w^k - nr) (oracle/pairing_oracle.py).
//
// Miller loop: on the twist, Jacobian coordinates (x' = X/Z^2, y' = Y/Z^3), loop count |T| = |t - 1|.  The line
// through the untwisted points A, A' with twist slope L, evaluated at P = (xP, yP) in G1 and scaled by u^2, is
//     u^2 yP  +  v (L x'_A - y'_A - xP u L)
// (untwisting is (x', y') -> (x'/u, y'/(u v))).  Each step stores it as three twist-field coefficients
//     a0 = u^2 s,  a1 = s (L x'_A - y'_A),  a2 = s u L      line(P) = yP a0 + v (a1 - xP a2)
// with s in the twist field chosen to clear the denominators.  Factors in the twist field and vertical lines lie in
// Fq^(k/2) and vanish in the final exponentiation, whose easy part contains q^(k/2) - 1.  A negative T is applied as
// the conjugate before the final exponentiation: conj = ^q^(k/2), and q^(k/2) = -1 modulo Phi_k(q).
//
// Final exponentiation: easy part f^(q^2 - 1) (MNT4) / f^((q^3 - 1)(q + 1)) (MNT6), then the hard part
// g^(Phi_k(q)/r) = g^q g^w0 (conjugate of g for negative w0: g is unitary after the easy part).
//
// Every product of two twist-field elements is a Karatsuba over out-of-line base products (Fp::mul_ni), and the
// products, squares and steps of this file are out-of-line themselves: one copy of each per kernel.
#pragma once
#include "ec.cuh"

// multiplication by u (the generator of the twist field over Fq) -- u^2 = 17 / u^3 = 5
PCD_HD Fq2 mul_by_u(const Fq2& a) { Fq2 r; r.c0 = a.c1.template mul_small<17>(); r.c1 = a.c0; return r; }
PCD_HD Fq3 mul_by_u(const Fq3& a) { Fq3 r; r.c0 = a.c2.template mul_small<5>(); r.c1 = a.c0; r.c2 = a.c1; return r; }
template <class E>
PCD_HD E scale(const E& a, const typename E::Base& s) {  // a * s, s in Fq
  typedef typename E::Base B;
  E r;
  const B* ai = reinterpret_cast<const B*>(&a);
  B* ri = reinterpret_cast<B*>(&r);
#pragma unroll
  for (int i = 0; i < E::WORDS / B::WORDS; i++) ri[i] = B::mul_ni(ai[i], s);
  return r;
}

struct PairMnt4 {
  typedef FpQ4 B; typedef Fq2 E; typedef CurveMnt4G1 G1; typedef CurveMnt4G2 G2; typedef PairingConstsMnt4 K;
  typedef FpR4 Fr;
};
struct PairMnt6 {
  typedef FpR4 B; typedef Fq3 E; typedef CurveMnt6G1 G1; typedef CurveMnt6G2 G2; typedef PairingConstsMnt6 K;
  typedef FpQ4 Fr;
};

template <class PP>
struct GT {
  typedef typename PP::E E;
  typedef typename PP::B B;
  static constexpr int D = PP::K::K / 2;  // degree of the twist field
  E c0, c1;

  PCD_HD static GT one() { GT r; r.c0 = E::one(); r.c1 = E::zero(); return r; }
  PCD_HD bool operator==(const GT& o) const { return c0 == o.c0 && c1 == o.c1; }
  PCD_HD GT conj() const { GT r; r.c0 = c0; r.c1 = c1.neg(); return r; }
  // Karatsuba: 3 twist-field products
  PCD_NOINLINE static GT mul(GT a, GT b) {
    E v0 = a.c0 * b.c0;
    E v1 = a.c1 * b.c1;
    GT r;
    r.c1 = (a.c0 + a.c1) * (b.c0 + b.c1) - v0 - v1;
    r.c0 = v0 + mul_by_u(v1);
    return r;
  }
  // complex squaring: 2 twist-field products
  PCD_NOINLINE static GT sqr(GT a) {
    E ab = a.c0 * a.c1;
    E t = (a.c0 + a.c1) * (a.c0 + mul_by_u(a.c1));
    GT r;
    r.c0 = t - ab - mul_by_u(ab);
    r.c1 = ab.dbl();
    return r;
  }
  PCD_NOINLINE static GT inverse(GT a) {  // zero stays zero (Fp::inverse(0) = 0)
    E n = (a.c0 * a.c0 - mul_by_u(a.c1 * a.c1)).inverse();
    GT r;
    r.c0 = a.c0 * n;
    r.c1 = (a.c1 * n).neg();
    return r;
  }
  // a^q: the coefficient of w^j times gamma^j (PairingConsts::frob)
  PCD_NOINLINE static GT frobenius(GT a) {
    GT r;
    const B* ai = reinterpret_cast<const B*>(&a);
    B* ri = reinterpret_cast<B*>(&r);
    for (int h = 0; h < 2; h++)
      for (int i = 0; i < D; i++) {
        B g;
#pragma unroll
        for (int l = 0; l < FP_LIMBS; l++) g.l[l] = PP::K::frob((2 * i + h) * FP_LIMBS + l);
        ri[h * D + i] = B::mul_ni(ai[h * D + i], g);
      }
    return r;
  }
};

template <class E>
struct Line {
  E a0, a1, a2;
};

template <class PP>
PCD_HD GT<PP> line_at(const Line<typename PP::E>& l, const AffinePoint<typename PP::B>& p) {
  GT<PP> r;
  r.c0 = scale(l.a0, p.y);
  r.c1 = l.a1 - scale(l.a2, p.x);
  return r;
}

template <class PP>
struct TwistJac {
  typedef typename PP::E E;
  E x, y, z;
  struct Step;
  PCD_HD static TwistJac from_affine(const AffinePoint<E>& q) { TwistJac r; r.x = q.x; r.y = q.y; r.z = E::one(); return r; }
};
template <class PP>
struct TwistJac<PP>::Step {
  TwistJac r;
  Line<typename PP::E> l;
};

// R <- 2R and the tangent at R (dbl-2009-l with a != 0; s = 2 Y Z^3)
template <class PP>
PCD_NOINLINE typename TwistJac<PP>::Step dbl_step(TwistJac<PP> R) {
  typedef typename PP::E E;
  E XX = R.x.sqr(), YY = R.y.sqr(), ZZ = R.z.sqr();
  E M = XX.dbl() + XX + PP::G2::mul_a(ZZ.sqr());
  E S = (R.x * YY).dbl().dbl();
  E Z3 = (R.y * R.z).dbl();
  typename TwistJac<PP>::Step o;
  o.l.a0 = mul_by_u(mul_by_u(Z3 * ZZ));
  o.l.a1 = M * R.x - YY.dbl();
  o.l.a2 = mul_by_u(M * ZZ);
  o.r.x = M.sqr() - S.dbl();
  o.r.y = M * (S - o.r.x) - YY.sqr().dbl().dbl().dbl();
  o.r.z = Z3;
  return o;
}

// R <- R + Q (Q affine) and the line through Q and R (s = Z H)
template <class PP>
PCD_NOINLINE typename TwistJac<PP>::Step add_step(TwistJac<PP> R, AffinePoint<typename PP::E> q) {
  typedef typename PP::E E;
  E ZZ = R.z.sqr();
  E H = q.x * ZZ - R.x;
  E Rr = q.y * (R.z * ZZ) - R.y;
  E Z3 = R.z * H;
  typename TwistJac<PP>::Step o;
  o.l.a0 = mul_by_u(mul_by_u(Z3));
  o.l.a1 = Rr * q.x - q.y * Z3;
  o.l.a2 = mul_by_u(Rr);
  E HH = H.sqr();
  E HHH = H * HH;
  E V = R.x * HH;
  o.r.x = Rr.sqr() - HHH - V.dbl();
  o.r.y = Rr * (V - o.r.x) - R.y * HHH;
  o.r.z = Z3;
  return o;
}

template <class PP>
PCD_HD bool ate_bit(int b) { return (PP::K::ate(b >> 5) >> (b & 31)) & 1u; }

// lines of one G2 point, in the order the Miller loop consumes them: (ATE_BITS - 1) + (popcount - 1)
template <class PP>
PCD_HD constexpr int num_lines() {
  int n = 0;
  for (int b = PP::K::ATE_BITS - 2; b >= 0; b--) n += 1 + (int)((PP::K::ate(b >> 5) >> (b & 31)) & 1u);
  return n;
}

// ark-ec G2Prepared: every line coefficient of the Miller loop of q (q != infinity)
template <class PP>
PCD_HD void prepare_lines(const AffinePoint<typename PP::E>& q, Line<typename PP::E>* out) {
  TwistJac<PP> R = TwistJac<PP>::from_affine(q);
  int li = 0;
#pragma unroll 1
  for (int b = PP::K::ATE_BITS - 2; b >= 0; b--) {
    typename TwistJac<PP>::Step s = dbl_step<PP>(R);
    R = s.r;
    out[li++] = s.l;
    if (ate_bit<PP>(b)) {
      s = add_step<PP>(R, q);
      R = s.r;
      out[li++] = s.l;
    }
  }
}

// Multi-Miller loop over NF pairs whose G2 point is stepped here (fresh) and NP pairs with prepared lines (read from
// memory every thread shares).  Pairs with a point at infinity are left out by the caller (they contribute 1).
template <class PP, int NF, int NP>
struct MillerArgs {
  int nf = 0, np = 0;
  AffinePoint<typename PP::E> fq[NF > 0 ? NF : 1];
  AffinePoint<typename PP::B> fp[NF > 0 ? NF : 1];
  const Line<typename PP::E>* pre[NP > 0 ? NP : 1];
  AffinePoint<typename PP::B> pp[NP > 0 ? NP : 1];
  PCD_HD void fresh(const AffinePoint<typename PP::B>& p, const AffinePoint<typename PP::E>& q) {
    if (p.is_inf() || q.is_inf()) return;
    fp[nf] = p; fq[nf] = q; nf++;
  }
  PCD_HD void prepared(const AffinePoint<typename PP::B>& p, const Line<typename PP::E>* lines) {
    if (p.is_inf() || lines == nullptr) return;
    pp[np] = p; pre[np] = lines; np++;
  }
};

template <class PP, int NF, int NP>
PCD_HD GT<PP> miller_loop(const MillerArgs<PP, NF, NP>& a) {
  typedef GT<PP> G;
  G f = G::one();
  TwistJac<PP> R[NF > 0 ? NF : 1];
#pragma unroll 1
  for (int j = 0; j < a.nf; j++) R[j] = TwistJac<PP>::from_affine(a.fq[j]);
  int li = 0;
#pragma unroll 1
  for (int b = PP::K::ATE_BITS - 2; b >= 0; b--) {
    f = G::sqr(f);
#pragma unroll 1
    for (int j = 0; j < a.nf; j++) {
      typename TwistJac<PP>::Step s = dbl_step<PP>(R[j]);
      R[j] = s.r;
      f = G::mul(f, line_at<PP>(s.l, a.fp[j]));
    }
#pragma unroll 1
    for (int j = 0; j < a.np; j++) f = G::mul(f, line_at<PP>(a.pre[j][li], a.pp[j]));
    li++;
    if (ate_bit<PP>(b)) {
#pragma unroll 1
      for (int j = 0; j < a.nf; j++) {
        typename TwistJac<PP>::Step s = add_step<PP>(R[j], a.fq[j]);
        R[j] = s.r;
        f = G::mul(f, line_at<PP>(s.l, a.fp[j]));
      }
#pragma unroll 1
      for (int j = 0; j < a.np; j++) f = G::mul(f, line_at<PP>(a.pre[j][li], a.pp[j]));
      li++;
    }
  }
  return PP::K::ATE_IS_NEG ? f.conj() : f;
}

template <class PP>
PCD_HD GT<PP> pow_w0(GT<PP> g) {  // g^|w0|, square and multiply from the top bit
  GT<PP> r = g;
#pragma unroll 1
  for (int b = PP::K::W0_BITS - 2; b >= 0; b--) {
    r = GT<PP>::sqr(r);
    if ((PP::K::w0(b >> 5) >> (b & 31)) & 1u) r = GT<PP>::mul(r, g);
  }
  return r;
}

template <class PP>
PCD_HD GT<PP> final_exponentiation(const GT<PP>& f) {
  typedef GT<PP> G;
  G g = G::mul(f.conj(), G::inverse(f));               // f^(q^(k/2) - 1)
  if (PP::K::K == 6) g = G::mul(G::frobenius(g), g);   // ^(q + 1)
  G gw = pow_w0<PP>(PP::K::W0_IS_NEG ? g.conj() : g);  // g^w0
  return G::mul(G::frobenius(g), gw);
}

template <class PP>
PCD_HD GT<PP> pairing(const AffinePoint<typename PP::B>& p, const AffinePoint<typename PP::E>& q) {
  MillerArgs<PP, 1, 0> a;
  a.fresh(p, q);
  return final_exponentiation<PP>(miller_loop<PP>(a));
}

// ---- input checks (ark-serialize's: canonical coordinates, on the curve; G2 subgroup membership is checked by the
// deserialization of deserialize.cuh, not here) ----
template <class B>
PCD_HD bool base_canonical(const B& x) {
  for (int i = FP_LIMBS - 1; i >= 0; i--)
    if (x.l[i] != B::Params::mod(i)) return x.l[i] < B::Params::mod(i);
  return false;
}
template <class F> struct BaseOf { typedef typename F::Base T; };
template <class P> struct BaseOf<Fp<P>> { typedef Fp<P> T; };
// x^3 + a x + b on C
template <class C>
PCD_HD typename C::F curve_rhs(const typename C::F& x) {
  typedef typename C::F F;
  F b;
  u32* bw = reinterpret_cast<u32*>(&b);
  for (int i = 0; i < F::WORDS; i++) bw[i] = C::Gen::coeff_b(i);
  return (x.sqr() + C::mul_a(F::one())) * x + b;
}
template <class C>
PCD_HD bool valid_point(const AffinePoint<typename C::F>& p) {
  typedef typename C::F F;
  typedef typename BaseOf<F>::T B;
  const B* c = reinterpret_cast<const B*>(&p);
  for (int i = 0; i < 2 * F::WORDS / FP_LIMBS; i++)
    if (!base_canonical(c[i])) return false;
  if (p.is_inf()) return true;
  return p.y.sqr() == curve_rhs<C>(p.x);
}

// gamma_abc[0] + sum_i x_i gamma_abc[i + 1] (x: Montgomery scalar-field elements), affine
template <class PP>
PCD_HD AffinePoint<typename PP::B> input_combination(const AffinePoint<typename PP::B>* abc, const typename PP::Fr* x,
                                                     int num_inputs) {
  typedef XYZZ<typename PP::G1> P1;
  P1 acc = P1::from_affine(abc[0]);
#pragma unroll 1
  for (int i = 0; i + 1 < num_inputs; i++) {
    typename PP::Fr k = x[i].from_mont();
    acc.add(P1::mul(P1::from_affine(abc[i + 1]), k.l, FP_LIMBS));
  }
  return acc.to_affine();
}

// ---- one verification (ark-groth16 / ark-gm17 verifier.rs) -------------------------------------------------------
// Processed keys: G2 points that every proof pairs with are prepared once (Line arrays of num_lines<PP>() entries).
template <class PP>
struct Groth16Pvk {
  const Line<typename PP::E>* neg_gamma;  // lines of -gamma_g2
  const Line<typename PP::E>* neg_delta;  // lines of -delta_g2
  const AffinePoint<typename PP::B>* abc;  // gamma_abc_g1
  int num_inputs;
  GT<PP> e_ab;  // e(alpha_g1, beta_g2)
};
template <class PP>
struct GM17Pvk {
  const Line<typename PP::E>* neg_h_gamma;  // lines of -h_gamma_g2
  const Line<typename PP::E>* neg_h;        // lines of -h_g2
  const Line<typename PP::E>* h_gamma;      // lines of h_gamma_g2
  const AffinePoint<typename PP::B>* query;
  int num_inputs;
  AffinePoint<typename PP::B> g_alpha, g_gamma;
  AffinePoint<typename PP::E> h_beta;
  GT<PP> e_ab;  // e(g_alpha_g1, h_beta_g2)
};

// e(A, B) = e(alpha, beta) e(IC, gamma) e(C, delta)
template <class PP>
PCD_HD bool groth16_verify_one(const Groth16Pvk<PP>& vk, const AffinePoint<typename PP::B>& A,
                               const AffinePoint<typename PP::E>& B, const AffinePoint<typename PP::B>& C,
                               const typename PP::Fr* x) {
  if (!valid_point<typename PP::G1>(A) || !valid_point<typename PP::G2>(B) || !valid_point<typename PP::G1>(C))
    return false;
  MillerArgs<PP, 1, 2> m;
  m.fresh(A, B);
  m.prepared(input_combination<PP>(vk.abc, x, vk.num_inputs), vk.neg_gamma);
  m.prepared(C, vk.neg_delta);
  return final_exponentiation<PP>(miller_loop<PP>(m)) == vk.e_ab;
}

// e(A + g_alpha, B + h_beta) = e(g_alpha, h_beta) e(g_psi, h_gamma) e(C, h)  and  e(A, h_gamma) = e(g_gamma, B)
template <class PP>
PCD_HD bool gm17_verify_one(const GM17Pvk<PP>& vk, const AffinePoint<typename PP::B>& A,
                            const AffinePoint<typename PP::E>& B, const AffinePoint<typename PP::B>& C,
                            const typename PP::Fr* x) {
  typedef XYZZ<typename PP::G1> P1;
  typedef XYZZ<typename PP::G2> P2;
  if (!valid_point<typename PP::G1>(A) || !valid_point<typename PP::G2>(B) || !valid_point<typename PP::G1>(C))
    return false;
  P1 a = P1::from_affine(A);
  a.madd(vk.g_alpha);
  P2 b = P2::from_affine(B);
  b.madd(vk.h_beta);
  MillerArgs<PP, 1, 2> m;
  m.fresh(a.to_affine(), b.to_affine());
  m.prepared(input_combination<PP>(vk.query, x, vk.num_inputs), vk.neg_h_gamma);
  m.prepared(C, vk.neg_h);
  if (!(final_exponentiation<PP>(miller_loop<PP>(m)) == vk.e_ab)) return false;
  MillerArgs<PP, 1, 2> m2;
  m2.fresh(vk.g_gamma.neg(), B);
  m2.prepared(A, vk.h_gamma);
  return final_exponentiation<PP>(miller_loop<PP>(m2)) == GT<PP>::one();
}
