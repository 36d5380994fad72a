"""Checked deserialization of compressed points and proofs without a GPU: the oracle (oracle/deserialize_oracle.py)
against serialization and every rejection rule, and the device header pcd_b200/csrc/deserialize.cuh, compiled for the
CPU with the emulated carry primitives (tests/hostemu/deserialize_emu.cpp), against the oracle byte for byte."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import codec
import deserialize_helpers as dh
import deserialize_oracle as do
import pcd_oracle as o
import synth
import verify_helpers as vh

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "hostemu", "_build", "libdeserializeemu.so")
CURVES = (0, 1, 2, 3)
G2S = (1, 3)
#: emu field ids: Fq of MNT4, Fq of MNT6, Fq2, Fq3
FIELDS = {0: (o.FQ4_F, o.FQ4), 1: (o.FR4_F, o.FR4), 2: (o.FQ2_F, o.FQ4), 3: (o.FQ3_F, o.FR4)}


@pytest.fixture(scope="module")
def emu():
    src = os.path.join(HERE, "hostemu", "deserialize_emu.cpp")
    csrc = os.path.join(ROOT, "pcd_b200", "csrc")
    deps = [src, os.path.join(HERE, "hostemu", "hostemu_prims.h")] + [
        os.path.join(csrc, f) for f in ("deserialize.cuh", "pairing.cuh", "fp.cuh", "fpx.cuh", "ec.cuh", "prims.cuh",
                                        "constants.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-I", csrc, "-I",
                               os.path.join(HERE, "hostemu"), src, "-o", SO])
    lib = ctypes.CDLL(SO)
    lib.emu_products.restype = ctypes.c_ulonglong
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _emu_points(emu, curve_id, blobs, subgroup=True):
    data = np.frombuffer(b"".join(blobs), dtype=np.uint8).copy()
    out = np.zeros((len(blobs), codec.POINT_LIMBS[curve_id]), dtype=np.uint64)
    ok = np.zeros(len(blobs), dtype=np.uint8)
    emu.emu_deserialize_points(curve_id, _p(data), ctypes.c_size_t(len(blobs)), _p(out), _p(ok), int(subgroup))
    return out, ok


def _oracle(curve, blob):
    try:
        return True, do.deserialize_point(curve, blob)
    except do.InvalidData:
        return False, None


def test_g1_cofactors_are_one():
    """G1 points need no subgroup check: both G1 curves have prime order (cofactor 1); the G2 twists do not"""
    assert o.MNT4_G1.cofactor == 1 and o.MNT6_G1.cofactor == 1
    assert o.MNT4_G2.cofactor > 1 and o.MNT6_G2.cofactor > 1


@pytest.mark.parametrize("curve_id", CURVES)
def test_round_trip(emu, curve_id):
    """deserialize(serialize(P)) == P for 200 random subgroup points, their negations (the other y flag) and
    infinity, in the oracle and in the device header"""
    curve = synth.CURVES[curve_id]
    limbs = synth.random_points(200, curve_id, 40 + curve_id)
    pts = [dh.limbs_point(curve_id, r) for r in limbs]
    pts = pts + [curve.neg(P) for P in pts[:100]] + [None]
    blobs = [o.serialize_point(curve, P) for P in pts]
    flags = {b[-1] & 0xC0 for b in blobs}
    assert flags == {0x00, 0x80, 0x40}
    for P, b in zip(pts, blobs):
        assert do.deserialize_point(curve, b) == P
    out, ok = _emu_points(emu, curve_id, blobs)
    assert ok.all()
    assert np.array_equal(out, np.stack([synth.point_limbs(curve_id, P) for P in pts]))


def _rejection_cases(curve_id):
    curve = synth.CURVES[curve_id]
    g = o.serialize_point(curve, o.generator(curve))
    cases = []
    for chunk in range(curve.F.degree):
        for kind in ("x=p", "bit298", "bit299", "bit300", "bit301"):
            cases.append(("%s/c%d" % (kind, chunk), dh.tamper_point(g, 0, curve_id, kind, chunk)))
    cases.append(("flags", dh.tamper_point(g, 0, curve_id, "flags")))
    cases.append(("flags-inf", o.serialize_point(curve, None)[:-1] + bytes([0xC0])))
    cases.append(("nonsquare", dh.tamper_point(g, 0, curve_id, "nonsquare")))
    if curve_id in G2S:
        for k in range(3):
            cases.append(("subgroup%d" % k, dh.tamper_point(g, 0, curve_id, "subgroup", k)))
    return cases


@pytest.mark.parametrize("curve_id", CURVES)
def test_rejections(emu, curve_id):
    """every kind of invalid encoding is rejected by the oracle and by the device header (zero point, verdict 0);
    the infinity flag over any canonical x is infinity"""
    curve = synth.CURVES[curve_id]
    cases = _rejection_cases(curve_id)
    for name, blob in cases:
        assert not _oracle(curve, blob)[0], name
    out, ok = _emu_points(emu, curve_id, [b for _, b in cases])
    assert ok.tolist() == [0] * len(cases), [n for (n, _), v in zip(cases, ok) if v]
    assert not out.any()
    g = o.serialize_point(curve, o.generator(curve))
    inf = dh.tamper_point(g, 0, curve_id, "inf")
    assert do.deserialize_point(curve, inf) is None
    out, ok = _emu_points(emu, curve_id, [inf])
    assert ok.tolist() == [1] and not out.any()


@pytest.mark.parametrize("field", sorted(FIELDS))
def test_sqrt(emu, field):
    """500 random elements (squares and non-squares) and 100 squares: y^2 = a, or rejection exactly when a is not a
    square"""
    F, fp = FIELDS[field]
    rng = o.SplitMix64(500 + field)
    d = F.degree
    draw = (lambda: rng.field(fp.p)) if d == 1 else (lambda: tuple(rng.field(fp.p) for _ in range(d)))
    vals = [draw() for _ in range(500)]
    vals += [F.sqr(draw()) for _ in range(100)] + [F.zero]
    coeffs = lambda v: F.coeffs(v) if d > 1 else (v,)
    a = np.stack([synth.mont_limbs(coeffs(v), fp).reshape(-1) for v in vals])
    out = np.zeros_like(a)
    ok = np.zeros(len(vals), dtype=np.uint8)
    emu.emu_sqrt(field, _p(a), ctypes.c_size_t(len(vals)), _p(out), _p(ok))
    squares = [do.is_square(F, v) for v in vals]
    assert ok.astype(bool).tolist() == squares
    assert 150 < sum(squares[:500]) < 350
    for i, v in enumerate(vals):
        if ok[i]:
            y = [o.fp_from_mont_bytes(out[i, 5 * j:5 * j + 5].tobytes(), fp) for j in range(d)]
            y = tuple(y) if d > 1 else y[0]
            assert F.eq(F.sqr(y), v), i
        else:
            assert not out[i].any()


@pytest.mark.parametrize("pid", (0, 1))
def test_proofs_match_oracle(emu, pid):
    """compressed proofs, valid and tampered at every point: the device header's rows and verdicts equal the oracle's;
    reports the base-field products of one proof's deserialization (decompression and subgroup check apart)"""
    inst = synth.make_instance(pid, 8, num_inputs=2)
    proofs, _ = vh.simulated(inst, 12, 77 + pid)
    blobs = [dh.proof_bytes(pid, r) for r in proofs]
    rows = [b for b in blobs]
    kinds = dh.REJECTIONS + ["inf"]
    for i, kind in enumerate(kinds):
        for j, (off, curve_id) in enumerate(dh.point_offsets(pid)):
            rows.append(dh.tamper_point(blobs[(i + j) % len(blobs)], off, curve_id, kind, i))
    rows.append(dh.tamper_point(blobs[0], dh.point_offsets(pid)[1][0], codec.G2_OF[pid], "subgroup"))
    pairing = synth.PAIRINGS[pid]
    want_rows, want_ok = [], []
    for b in rows:
        try:
            want_rows.append(dh.proof_row(pid, do.deserialize_proof(pairing, b)))
            want_ok.append(1)
        except do.InvalidData:
            want_rows.append(np.zeros(proofs.shape[1], dtype=np.uint64))
            want_ok.append(0)
    assert want_ok[:len(blobs)] == [1] * len(blobs)
    assert np.array_equal(np.stack(want_rows[:len(blobs)]), proofs)
    assert want_ok.count(1) == len(blobs) + 3  # the infinity flags
    data = np.frombuffer(b"".join(rows), dtype=np.uint8).copy()
    out = np.zeros((len(rows), proofs.shape[1]), dtype=np.uint64)
    ok = np.zeros(len(rows), dtype=np.uint8)
    emu.emu_deserialize_proofs(pid, _p(data), ctypes.c_size_t(len(rows)), _p(out), _p(ok))
    assert ok.tolist() == want_ok
    assert np.array_equal(out, np.stack(want_rows))
    # work model: products of one valid proof, split into the three decompressions and the subgroup check of B
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    n1 = do.point_bytes(synth.CURVES[g1])
    emu.emu_products()
    emu.emu_deserialize_proofs(pid, _p(data), ctypes.c_size_t(1), _p(out), _p(ok))
    total = emu.emu_products()
    _emu_points(emu, g1, [blobs[0][:n1], blobs[0][-n1:]], subgroup=False)
    _emu_points(emu, g2, [blobs[0][n1:-n1]], subgroup=False)
    decomp = emu.emu_products()
    b = np.ascontiguousarray(dh.split(pid, proofs[0])[1])
    emu.emu_subgroup(g2, _p(b), ctypes.c_size_t(1), _p(ok))
    sub = emu.emu_products()
    assert decomp + sub == total
    print("base-field products of one proof's deserialization (%s): %d = decompression %d + G2 subgroup check %d" % (
        "mnt4" if pid == 0 else "mnt6", total, decomp, sub))
