"""CPU oracle for ark-serialize's checked ``CanonicalDeserialize`` of compressed points and of ``Proof {a, b, c}``.

TEST INFRASTRUCTURE ONLY, like the rest of ``oracle/``: the product path never imports it.  It is the inverse of
``pcd_oracle.serialize_point`` / ``serialize_proof`` and restates SURVEY.md B.5 plus the checks of ark-ec 0.3's
``SWModelParameters`` deserialization [RECALL, like all of B.5]:

  * x is 1 / 2 / 3 chunks of 38 bytes (c0, c1, c2), little-endian; the flags sit in the top two bits of the last
    chunk's last byte: bit 7 "y is the lexicographically larger of {y, -y}" (highest coefficient compared first), bit 6
    "infinity".  Both bits set is invalid.
  * Every chunk, with the flags masked on the last one, must be < p (so bits 298 - 301 of any chunk are invalid).
  * Infinity flag: the point is infinity whatever the (canonical) x is [RECALL: ark-ec 0.3 reads x and the flags,
    then returns zero() without looking at x].
  * Otherwise y is a square root of x^3 + a x + b (invalid if there is none), the one the flag selects.
  * Subgroup membership (``is_in_correct_subgroup_assuming_on_curve``): [r]P = O.  Both G1 curves have cofactor 1, so
    a point on the curve is in the group; the test asserts it rather than trusting it.

An invalid encoding raises ``InvalidData`` (ark's ``SerializationError::InvalidData``).

The square root is ``pcd_oracle.field_sqrt`` (Tonelli-Shanks, checked against y^2 here anyway); ``sqrt_constants``
gives the Tonelli-Shanks constants the device code uses, derived and checked from the field order alone.
"""
from __future__ import annotations

import pcd_oracle as o

FLAG_Y = 0x80
FLAG_INF = 0x40
CHUNK = 38


class InvalidData(ValueError):
    pass


def rhs(curve, x):
    F = curve.F
    return F.add(F.add(F.mul(F.sqr(x), x), F.mul(curve.a, x)), curve.b)


def deserialize_point(curve, data: bytes):
    """compressed point -> (x, y) or None (infinity); raises InvalidData"""
    F = curve.F
    d = F.degree
    if len(data) != CHUNK * d:
        raise InvalidData("a compressed point of %s is %d bytes" % (curve.name, CHUNK * d))
    flags = data[-1] & (FLAG_Y | FLAG_INF)
    cs = []
    for i in range(d):
        chunk = bytearray(data[CHUNK * i:CHUNK * (i + 1)])
        if i == d - 1:
            chunk[-1] &= 0x3F
        v = int.from_bytes(chunk, "little")
        if v >= F.p:
            raise InvalidData("coordinate chunk %d is not < p" % i)
        cs.append(v)
    if flags == FLAG_Y | FLAG_INF:
        raise InvalidData("both flags set")
    if flags & FLAG_INF:
        return None
    x = F.from_coeffs(tuple(cs)) if d > 1 else cs[0]
    r = rhs(curve, x)
    y = o.field_sqrt(F, r)
    if y is None or not F.eq(F.sqr(y), r):
        raise InvalidData("x^3 + a x + b is not a square")
    if o._lex_larger(F, y) != bool(flags & FLAG_Y):
        y = F.neg(y)
    P = (x, y)
    if curve.cofactor != 1 and curve.mul(P, curve.order) is not None:
        raise InvalidData("point is not in the prime-order subgroup")
    return P


def point_bytes(curve) -> int:
    return CHUNK * curve.F.degree


def deserialize_proof(pairing, data: bytes):
    """Groth16 / GM17 ``Proof {a, b, c}`` (152 / 190 bytes) -> (A, B, C); raises InvalidData"""
    n1, n2 = point_bytes(pairing.g1), point_bytes(pairing.g2)
    if len(data) != 2 * n1 + n2:
        raise InvalidData("a proof over %s is %d bytes" % (pairing.name, 2 * n1 + n2))
    return (deserialize_point(pairing.g1, data[:n1]), deserialize_point(pairing.g2, data[n1:n1 + n2]),
            deserialize_point(pairing.g1, data[n1 + n2:]))


def is_square(F, a) -> bool:
    return F.is_zero(a) or F.eq(F.pow(a, (F.order - 1) // 2), F.one)


def sqrt_constants(F):
    """Tonelli-Shanks constants of F: (s, t, z) with |F*| = 2^s t, t odd, and z^t for the first non-residue z of
    field_sqrt's search order; z^t has order exactly 2^s (checked)."""
    q1 = F.order - 1
    s = (q1 & -q1).bit_length() - 1
    t = q1 >> s
    k = 2
    while True:
        z = F.from_coeffs(tuple([k] + [1] * (F.degree - 1))) if F.degree > 1 else F.from_int(k)
        if not is_square(F, z):
            break
        k += 1
    zt = F.pow(z, t)
    assert t % 2 == 1 and (t << s) == q1
    assert F.eq(F.pow(zt, 1 << (s - 1)), F.neg(F.one))
    return s, t, zt


def off_subgroup_point(curve, start: int = 1):
    """a point on the curve (a twist) outside its prime-order subgroup: pcd_oracle._find_point without cofactor
    clearing, from `start` on"""
    i = start
    while True:
        P = o._find_point(curve, i)
        if curve.mul(P, curve.order) is not None:
            return P
        i = (P[0] if curve.F.degree == 1 else P[0][0]) + 1
