"""Compressed proof bytes and their tamperings for the deserialization tests (test infrastructure): rows of affine
limbs <-> oracle points <-> ark-serialize bytes, and byte-level corruptions of one point, each of a kind the checked
deserializer must reject."""
import numpy as np

import codec
import deserialize_oracle as do
import pcd_oracle as o
import synth

PROOF_BYTES = {0: 152, 1: 190}


def limbs_point(curve_id, limbs):
    """affine Montgomery limbs -> oracle point (None for all zero)"""
    limbs = np.ascontiguousarray(limbs, dtype=np.uint64)
    if not limbs.any():
        return None
    F, fp = synth.CURVES[curve_id].F, synth.COORD_FP[curve_id]
    cs = [o.fp_from_mont_bytes(limbs[5 * i:5 * i + 5].tobytes(), fp) for i in range(len(limbs) // 5)]
    d = F.degree
    if d == 1:
        return cs[0], cs[1]
    return tuple(cs[:d]), tuple(cs[d:])


def split(pid, row):
    """(A, B, C) limb slices of one proof row"""
    a1, a2 = codec.POINT_LIMBS[codec.G1_OF[pid]], codec.POINT_LIMBS[codec.G2_OF[pid]]
    return row[:a1], row[a1:a1 + a2], row[a1 + a2:]


def proof_bytes(pid, row) -> bytes:
    """oracle serialization of one (A || B || C) limb row"""
    A, B, C = split(pid, row)
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    return o.serialize_proof(synth.PAIRINGS[pid], (limbs_point(g1, A), limbs_point(g2, B), limbs_point(g1, C)))


def proof_row(pid, proof):
    """oracle (A, B, C) -> limb row"""
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    return np.concatenate([synth.point_limbs(g1, proof[0]), synth.point_limbs(g2, proof[1]),
                           synth.point_limbs(g1, proof[2])])


def point_offsets(pid):
    """(byte offset, curve id) of A, B, C in a compressed proof"""
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    n1, n2 = do.point_bytes(synth.CURVES[g1]), do.point_bytes(synth.CURVES[g2])
    return [(0, g1), (n1, g2), (n1 + n2, g1)]


def _chunk_set(data, off, chunk, value):
    """replace coefficient chunk `chunk` of the point at `off` by value < 2^298 (flags kept on the last chunk)"""
    b = bytearray(data)
    lo = off + 38 * chunk
    flags = b[lo + 37] & 0xC0
    b[lo:lo + 38] = value.to_bytes(38, "little")
    b[lo + 37] |= flags
    return bytes(b)


def nonsquare_x(curve_id):
    """compressed bytes (no flags) of an x whose x^3 + a x + b is not a square"""
    curve = synth.CURVES[curve_id]
    F = curve.F
    i = 1
    while True:
        x = F.from_int(i) if F.degree == 1 else F.from_coeffs(tuple([i, 1] + [0] * (F.degree - 2)))
        if not do.is_square(F, do.rhs(curve, x)):
            return b"".join(o.serialize_fp(c) for c in F.coeffs(x))
        i += 1


_OFF_SUBGROUP = {}


def off_subgroup_bytes(curve_id, k=0):
    """compressed bytes of the k-th twist point outside the prime-order subgroup (asserted [r]P != O)"""
    if (curve_id, k) not in _OFF_SUBGROUP:
        curve = synth.CURVES[curve_id]
        start = 1
        for _ in range(k + 1):
            P = do.off_subgroup_point(curve, start)
            start = P[0][0] + 1
        assert curve.mul(P, curve.order) is not None and curve.is_on_curve(P)
        _OFF_SUBGROUP[(curve_id, k)] = o.serialize_point(curve, P)
    return _OFF_SUBGROUP[(curve_id, k)]


def tamper_point(data, off, curve_id, kind, chunk=0):
    """one corruption of the point at byte `off`; every kind but "inf" makes the encoding invalid"""
    curve = synth.CURVES[curve_id]
    n = do.point_bytes(curve)
    last = off + n - 1
    if kind == "subgroup":
        return data[:off] + off_subgroup_bytes(curve_id, chunk) + data[off + n:]
    chunk %= curve.F.degree
    if kind == "x=p":
        return _chunk_set(data, off, chunk, curve.F.p)
    if kind.startswith("bit"):  # bit 298 .. 301 of one chunk
        b = bytearray(data)
        bit = int(kind[3:])
        b[off + 38 * chunk + bit // 8] |= 1 << (bit % 8)
        return bytes(b)
    if kind == "flags":
        b = bytearray(data)
        b[last] |= 0xC0
        return bytes(b)
    if kind == "nonsquare":
        return data[:off] + nonsquare_x(curve_id) + data[off + n:]
    if kind == "inf":  # infinity flag over a non-zero canonical x: valid, the point is infinity
        b = bytearray(data)
        b[last] = (b[last] & 0x3F) | 0x40
        return bytes(b)
    raise ValueError(kind)


REJECTIONS = ["x=p", "bit298", "bit299", "bit300", "bit301", "flags", "nonsquare"]
