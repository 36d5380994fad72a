"""CPU oracle for the MNT4-298 / MNT6-298 pairings and for Groth16 / GM17 verification.

TEST INFRASTRUCTURE ONLY, like the rest of ``oracle/``: the product path never imports it.

The pairing is the textbook reduced ate pairing, written independently of the device code:

  * Fq4 = Fq[w]/(w^4 - 17) over q4 and Fq6 = Fq[w]/(w^6 - 5) over r4, plain polynomial arithmetic.  They are
    isomorphic to the device towers Fq2[v]/(v^2 - u) (u^2 = 17) and Fq3[v]/(v^2 - u) (u^3 = 5) by w = v, w^2 = u:
    coefficient i of tower half h (c0: h = 0, c1: h = 1) is the coefficient of w^(2 i + h).
  * G2 points of the twists (pcd_oracle._build_curves: a' = a w^4, b' = b w^6) are untwisted to E(Fq^k) by
    (x', y') -> (x' / w^2, y' / w^3).
  * Affine Miller loop f_{|T|, Q}(P) with T = t - 1, vertical lines dropped (they lie in Fq^(k/2) and die in the final
    exponentiation), inverted for negative T, then f^((q^k - 1) / r).

Every constant is derived here from q and r and asserted in ``self_check()``.  GT bytes follow arkworks' in-memory
``QuadExtField {c0, c1}`` over the twist field (Montgomery limbs); parity of those bytes with arkworks is unpinned, the
accept / reject verdict of a verifier does not depend on it.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence

import pcd_oracle as o


# ----------------------------------------------------------------------------------------------
# Fq^k = Fq[w]/(w^k - nr): elements are tuples of k ints, lowest degree first.
# ----------------------------------------------------------------------------------------------
class FpK:
    def __init__(self, p: int, k: int, nr: int):
        self.p, self.k, self.nr = p, k, nr
        self.zero = (0,) * k
        self.one = (1,) + (0,) * (k - 1)

    def add(self, a, b):
        return tuple((x + y) % self.p for x, y in zip(a, b))

    def sub(self, a, b):
        return tuple((x - y) % self.p for x, y in zip(a, b))

    def neg(self, a):
        return tuple((-x) % self.p for x in a)

    def mul(self, a, b):
        k, p = self.k, self.p
        c = [0] * (2 * k - 1)
        for i, x in enumerate(a):
            if x:
                for j, y in enumerate(b):
                    c[i + j] += x * y
        return tuple((c[i] + (self.nr * c[i + k] if i + k < 2 * k - 1 else 0)) % p for i in range(k))

    def sqr(self, a):
        return self.mul(a, a)

    def scalar(self, a, s: int):
        return tuple(x * s % self.p for x in a)

    def embed(self, c: int):
        return (c % self.p,) + (0,) * (self.k - 1)

    def is_zero(self, a):
        return all(x % self.p == 0 for x in a)

    def eq(self, a, b):
        return self.is_zero(self.sub(a, b))

    def inv(self, a):
        """Extended Euclid on polynomials over Fq against the (irreducible) modulus w^k - nr."""
        p, k = self.p, self.k

        def trim(f):
            f = list(f)
            while f and f[-1] % p == 0:
                f.pop()
            return f

        def divmod_(f, g):
            f = [x % p for x in f]
            q = [0] * max(len(f) - len(g) + 1, 1)
            li = pow(g[-1], -1, p)
            while len(f) >= len(g) and f:
                c = f[-1] * li % p
                d = len(f) - len(g)
                q[d] = c
                for i, y in enumerate(g):
                    f[d + i] = (f[d + i] - c * y) % p
                f = trim(f)
            return trim(q), f

        def psub(f, g):
            n = max(len(f), len(g))
            return trim([((f[i] if i < len(f) else 0) - (g[i] if i < len(g) else 0)) % p for i in range(n)])

        def pmul(f, g):
            if not f or not g:
                return []
            c = [0] * (len(f) + len(g) - 1)
            for i, x in enumerate(f):
                for j, y in enumerate(g):
                    c[i + j] = (c[i + j] + x * y) % p
            return trim(c)

        r0, r1 = trim([(-self.nr) % p] + [0] * (k - 1) + [1]), trim(a)
        if not r1:
            raise ZeroDivisionError("inverse of zero")
        s0, s1 = [], [1]
        while len(r1) > 1:
            q, r = divmod_(r0, r1)
            r0, r1 = r1, r
            s0, s1 = s1, psub(s0, pmul(q, s1))
        c = pow(r1[0], -1, p)
        s = [x * c % p for x in s1] + [0] * k
        return tuple(s[:k])

    def pow(self, a, e: int):
        if e < 0:
            return self.pow(self.inv(a), -e)
        r = self.one
        for bit in bin(e)[2:]:
            r = self.sqr(r)
            if bit == "1":
                r = self.mul(r, a)
        return r

    def frobenius(self, a, consts):
        return tuple(x * c % self.p for x, c in zip(a, consts))


@dataclass(frozen=True)
class PairingParams:
    name: str
    q: int  # base field of G1
    r: int  # group order
    k: int
    nr: int
    pairing: o.Pairing
    F: FpK

    @property
    def t(self) -> int:
        return self.q + 1 - self.r

    @property
    def ate_loop_count(self) -> int:  # T = t - 1 (signed)
        return self.t - 1

    @property
    def final_exponent(self) -> int:
        return (self.q ** self.k - 1) // self.r

    @property
    def hard_exponent(self) -> int:  # Phi_k(q) / r
        q = self.q
        return ((q * q + 1) if self.k == 4 else (q * q - q + 1)) // self.r

    @property
    def w0(self) -> int:  # Phi_k(q) / r = q + w0
        return self.hard_exponent - self.q

    @property
    def frobenius_coeffs(self) -> List[int]:  # w^q = gamma w, gamma = nr^((q - 1) / k); coefficient j of w^j: gamma^j
        g = pow(self.nr, (self.q - 1) // self.k, self.q)
        return [pow(g, j, self.q) for j in range(self.k)]


MNT4P = PairingParams("mnt4_298", o.Q4, o.R4, 4, o.FQ2_NONRESIDUE, o.MNT4, FpK(o.Q4, 4, o.FQ2_NONRESIDUE))
MNT6P = PairingParams("mnt6_298", o.R4, o.Q4, 6, o.FQ3_NONRESIDUE, o.MNT6, FpK(o.R4, 6, o.FQ3_NONRESIDUE))
PARAMS = {0: MNT4P, 1: MNT6P}


def tower_to_poly(P: PairingParams, c0, c1):
    """Tower element c0 + c1 v (c0, c1 tuples over the twist field) -> coefficients of w."""
    e = P.k // 2
    out = [0] * P.k
    for i in range(e):
        out[2 * i] = c0[i] % P.q
        out[2 * i + 1] = c1[i] % P.q
    return tuple(out)


def poly_to_tower(P: PairingParams, a):
    e = P.k // 2
    return tuple(a[2 * i] for i in range(e)), tuple(a[2 * i + 1] for i in range(e))


def twist_to_poly(P: PairingParams, c) -> tuple:
    """Twist-field element (coefficients of u = w^2) as an element of Fq^k."""
    out = [0] * P.k
    for i, x in enumerate(c):
        out[2 * i] = x % P.q
    return tuple(out)


def untwist(P: PairingParams, Q):
    F = P.F
    x, y = Q
    w = (0, 1) + (0,) * (P.k - 2)
    w2, w3 = F.sqr(w), F.mul(F.sqr(w), w)
    return F.mul(twist_to_poly(P, x), F.inv(w2)), F.mul(twist_to_poly(P, y), F.inv(w3))


def miller_loop(P: PairingParams, Pg1, Qg2):
    """f_{T, Q}(P) (up to factors in Fq^(k/2)); 1 if either point is infinity."""
    F = P.F
    if Pg1 is None or Qg2 is None:
        return F.one
    xp, yp = F.embed(Pg1[0]), F.embed(Pg1[1])
    xq, yq = untwist(P, Qg2)
    a = F.embed(P.pairing.g1.a)
    T = abs(P.ate_loop_count)

    def line(xa, ya, lam):  # y_P - y_A - lam (x_P - x_A)
        return F.sub(F.sub(yp, ya), F.mul(lam, F.sub(xp, xa)))

    f = F.one
    xr, yr = xq, yq
    for bit in bin(T)[3:]:
        lam = F.mul(F.add(F.scalar(F.sqr(xr), 3), a), F.inv(F.scalar(yr, 2)))
        f = F.mul(F.sqr(f), line(xr, yr, lam))
        x3 = F.sub(F.sqr(lam), F.scalar(xr, 2))
        yr = F.sub(F.mul(lam, F.sub(xr, x3)), yr)
        xr = x3
        if bit == "1":
            lam = F.mul(F.sub(yq, yr), F.inv(F.sub(xq, xr)))
            f = F.mul(f, line(xr, yr, lam))
            x3 = F.sub(F.sub(F.sqr(lam), xr), xq)
            yr = F.sub(F.mul(lam, F.sub(xr, x3)), yr)
            xr = x3
    if P.ate_loop_count < 0:
        f = F.inv(f)
    return f


def final_exponentiation(P: PairingParams, f):
    return P.F.pow(f, P.final_exponent)


def pairing(P: PairingParams, Pg1, Qg2):
    return final_exponentiation(P, miller_loop(P, Pg1, Qg2))


def multi_pairing(P: PairingParams, pairs):
    F = P.F
    f = F.one
    for a, b in pairs:
        f = F.mul(f, miller_loop(P, a, b))
    return final_exponentiation(P, f)


def gt_to_limbs(P: PairingParams, g):
    """GT element -> u64 limbs of arkworks' QuadExtField {c0, c1} (Montgomery coefficients)."""
    import numpy as np
    fp = o.FQ4 if P.q == o.Q4 else o.FR4
    c0, c1 = poly_to_tower(P, g)
    b = b"".join(o.fp_to_mont_bytes(x, fp) for x in c0 + c1)
    return np.frombuffer(b, dtype="<u8").copy()


# ----------------------------------------------------------------------------------------------
# Verifying keys and verifiers (ark-groth16 / ark-gm17 verifier.rs)
# ----------------------------------------------------------------------------------------------
@dataclass
class Groth16VK:
    pairing: o.Pairing
    alpha_g1: tuple
    beta_g2: tuple
    gamma_g2: tuple
    delta_g2: tuple
    gamma_abc_g1: list


def groth16_vk(pairing: o.Pairing, t: dict, num_inputs: int, gamma: int) -> Groth16VK:
    """The verifying key of a known-trapdoor proving key (t = groth16_setup_scalars): gamma_g2 = [gamma]H,
    gamma_abc_g1[j] = [(beta At_j + alpha Bt_j + Ct_j) / gamma]G.  The proving key does not depend on gamma, so any
    nonzero gamma gives a valid key for it."""
    G1, G2 = pairing.g1, pairing.g2
    p = pairing.fr.p
    gi = pow(gamma, -1, p)
    g1, g2 = o.generator(G1), o.generator(G2)
    abc = [G1.mul(g1, (t["beta"] * t["At"][j] + t["alpha"] * t["Bt"][j] + t["Ct"][j]) * gi % p) for j in range(num_inputs)]
    return Groth16VK(pairing, G1.mul(g1, t["alpha"]), G2.mul(g2, t["beta"]), G2.mul(g2, gamma), G2.mul(g2, t["delta"]),
                     abc)


@dataclass
class GM17VK:
    pairing: o.Pairing
    h_g2: tuple
    g_alpha_g1: tuple
    h_beta_g2: tuple
    g_gamma_g1: tuple
    h_gamma_g2: tuple
    query: list


def gm17_vk(pairing: o.Pairing, t: dict, num_inputs: int) -> GM17VK:
    """The verifying key of a known-trapdoor GM17 key (t = gm17_setup_scalars; GM17PK carries the same fields)."""
    G1, G2 = pairing.g1, pairing.g2
    g, h = o.generator(G1), o.generator(G2)
    return GM17VK(pairing, h, G1.mul(g, t["alpha"]), G2.mul(h, t["beta"]), G1.mul(g, t["gamma"]), G2.mul(h, t["gamma"]),
                  [G1.mul(g, t["vk_sc"][j]) for j in range(num_inputs)])


def _params_of(pairing: o.Pairing) -> PairingParams:
    return MNT4P if pairing is o.MNT4 else MNT6P


def _input_combination(G1, query, x: Sequence[int]):
    return G1.sum([query[0]] + [G1.mul(q, xi) for q, xi in zip(query[1:], x)])


def groth16_verify(vk: Groth16VK, x: Sequence[int], proof) -> bool:
    """e(A, B) = e(alpha, beta) e(IC, gamma) e(C, delta) with IC = gamma_abc[0] + sum x_i gamma_abc[i + 1]."""
    if len(x) + 1 != len(vk.gamma_abc_g1):
        raise ValueError("wrong number of public inputs")
    P = _params_of(vk.pairing)
    G1, G2 = vk.pairing.g1, vk.pairing.g2
    A, B, C = proof
    ic = _input_combination(G1, vk.gamma_abc_g1, x)
    lhs = multi_pairing(P, [(A, B), (ic, G2.neg(vk.gamma_g2)), (C, G2.neg(vk.delta_g2))])
    return P.F.eq(lhs, pairing(P, vk.alpha_g1, vk.beta_g2))


def gm17_verify(pk, x: Sequence[int], proof) -> bool:
    """ark-gm17 verify_proof: test 1 e(A + g_alpha, B + h_beta) = e(g_alpha, h_beta) e(g_psi, h_gamma) e(C, h);
    test 2 e(A, h_gamma) = e(g_gamma, B).  pk: a GM17VK or a GM17PK (its vk part)."""
    query = pk.query if isinstance(pk, GM17VK) else pk.vk_query
    if len(x) + 1 != len(query):
        raise ValueError("wrong number of public inputs")
    P = _params_of(pk.pairing)
    G1, G2 = pk.pairing.g1, pk.pairing.g2
    A, B, C = proof
    psi = _input_combination(G1, query, x)
    t1 = multi_pairing(P, [(G1.add(A, pk.g_alpha_g1), G2.add(B, pk.h_beta_g2)), (psi, G2.neg(pk.h_gamma_g2)),
                           (C, G2.neg(pk.h_g2))])
    if not P.F.eq(t1, pairing(P, pk.g_alpha_g1, pk.h_beta_g2)):
        return False
    t2 = multi_pairing(P, [(A, pk.h_gamma_g2), (G1.neg(pk.g_gamma_g1), B)])
    return P.F.eq(t2, P.F.one)


# ----------------------------------------------------------------------------------------------
# Proof simulators: valid proofs from the trapdoor, two or three fixed-base multiplications each.
# They return discrete logs; the caller multiplies the generators (c_oracle / GPU fixed-base mul).
# ----------------------------------------------------------------------------------------------
def groth16_simulated_logs(t: dict, x: Sequence[int], a: int, b: int, p: int):
    """(a, b, c) with c = (a b - alpha beta - sum_i x_i (beta At_i + alpha Bt_i + Ct_i)) / delta, x_0 = 1:
    A = [a]G, B = [b]H, C = [c]G verify against groth16_vk(pk, ...) for any gamma."""
    xs = [1] + list(x)
    s = sum(xi * (t["beta"] * t["At"][i] + t["alpha"] * t["Bt"][i] + t["Ct"][i]) for i, xi in enumerate(xs))
    return a, b, (a * b - t["alpha"] * t["beta"] - s) % p * pow(t["delta"], -1, p) % p


def gm17_simulated_logs(t: dict, x: Sequence[int], a: int, p: int):
    """(a, c) with c = (a + alpha)(a + beta) - alpha beta - gamma psi, psi = sum_i x_i vk_sc_i (x_0 = 1):
    A = [a]G, B = [a]H, C = [c]G."""
    psi = (t["vk_sc"][0] + sum(xi * v for xi, v in zip(x, t["vk_sc"][1:]))) % p
    return a, ((a + t["alpha"]) * (a + t["beta"]) - t["alpha"] * t["beta"] - t["gamma"] * psi) % p


def self_check() -> None:
    for P in (MNT4P, MNT6P):
        q, r, k = P.q, P.r, P.k
        assert (q ** k - 1) % r == 0 and all((q ** i - 1) % r for i in range(1, k)), "embedding degree"
        assert P.hard_exponent * r == ((q * q + 1) if k == 4 else (q * q - q + 1))
        assert P.ate_loop_count % r == q % r, "T = t - 1 = q mod r"
        assert (q - 1) % k == 0
        # w^k - nr irreducible: nr is not a square (k = 4, q = 1 mod 4) / neither square nor cube (k = 6, q = 1 mod 6)
        assert pow(P.nr, (q - 1) // 2, q) == q - 1
        if k == 6:
            assert pow(P.nr, (q - 1) // 3, q) != 1
        else:
            assert q % 4 == 1
        g = P.frobenius_coeffs
        assert pow(g[1], k, q) == 1 and g[1] != 1
        F = P.F
        a = tuple(range(3, 3 + k))
        assert F.eq(F.frobenius(a, g), F.pow(a, q)), "Frobenius coefficients"
        assert F.eq(F.mul(a, F.inv(a)), F.one)
    assert MNT4P.ate_loop_count == 689871209842287392837045615510547309923794944
    assert MNT6P.ate_loop_count == -689871209842287392837045615510547309923794944
    assert MNT4P.w0 > 0 and str(MNT4P.w0).endswith("945")
    assert MNT6P.w0 < 0 and str(-MNT6P.w0).endswith("944")


self_check()
