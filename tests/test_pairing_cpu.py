"""The MNT4-298 / MNT6-298 pairings and Groth16 / GM17 verification without a GPU: the oracle
(oracle/pairing_oracle.py) against its algebraic definition, and the device header pcd_b200/csrc/pairing.cuh,
compiled for the CPU with the emulated carry primitives (tests/hostemu/pairing_emu.cpp), against the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import codec
import pairing_oracle as po
import pcd_oracle as o
import synth
import verify_helpers as vh

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "hostemu", "_build", "libpairingemu.so")
PIDS = (0, 1)


@pytest.fixture(scope="module")
def emu():
    src = os.path.join(HERE, "hostemu", "pairing_emu.cpp")
    csrc = os.path.join(ROOT, "pcd_b200", "csrc")
    deps = [src, os.path.join(HERE, "hostemu", "hostemu_prims.h")] + [
        os.path.join(csrc, f) for f in ("pairing.cuh", "fp.cuh", "fpx.cuh", "ec.cuh", "prims.cuh", "constants.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-I", csrc, "-I",
                               os.path.join(HERE, "hostemu"), src, "-o", SO])
    lib = ctypes.CDLL(SO)
    lib.emu_products.restype = ctypes.c_ulonglong
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _gens(P):
    return o.generator(P.pairing.g1), o.generator(P.pairing.g2)


# ---- oracle ------------------------------------------------------------------------------------------------------
def test_derived_constants():
    for P in (po.MNT4P, po.MNT6P):
        q, r = P.q, P.r
        assert P.ate_loop_count == q + 1 - r - 1
        assert (q ** P.k - 1) // r == P.final_exponent and (q ** P.k - 1) % r == 0
        assert P.hard_exponent == q + P.w0
        g = P.frobenius_coeffs
        assert g[1] == pow(P.nr, (q - 1) // P.k, q)
        a = tuple(range(11, 11 + P.k))
        assert P.F.eq(P.F.frobenius(a, g), P.F.pow(a, q))
    assert po.MNT4P.ate_loop_count == -po.MNT6P.ate_loop_count == 689871209842287392837045615510547309923794944
    assert str(po.MNT4P.w0).endswith("945") and str(po.MNT6P.w0).endswith("944") and po.MNT6P.w0 < 0


@pytest.mark.parametrize("pid", PIDS)
def test_oracle_bilinear_nondegenerate(pid):
    P = po.PARAMS[pid]
    G1, G2 = P.pairing.g1, P.pairing.g2
    g, h = _gens(P)
    F = P.F
    e = po.pairing(P, g, h)
    assert not F.eq(e, F.one)
    assert F.eq(F.pow(e, P.r), F.one)
    rng = o.SplitMix64(100 + pid)
    for _ in range(2):
        a, b = rng.field(P.r), rng.field(P.r)
        assert F.eq(po.pairing(P, G1.mul(g, a), G2.mul(h, b)), F.pow(e, a * b))
    assert F.eq(po.pairing(P, None, h), F.one) and F.eq(po.pairing(P, g, None), F.one)


@pytest.mark.parametrize("pid", PIDS)
def test_oracle_verifiers(pid):
    inst = synth.make_instance(pid, 8, num_inputs=3)
    pairing, t = synth.PAIRINGS[pid], inst["trapdoor"]
    p = pairing.fr.p
    G1, G2 = pairing.g1, pairing.g2
    g, h = o.generator(G1), o.generator(G2)
    vk = po.groth16_vk(pairing, t, inst["num_inputs"], 12345)
    x = inst["z_int"][1:inst["num_inputs"]]
    a, b, c = po.groth16_simulated_logs(t, x, 777, 999, p)
    proof = (G1.mul(g, a), G2.mul(h, b), G1.mul(g, c))
    assert po.groth16_verify(vk, x, proof)
    assert not po.groth16_verify(vk, [x[0] + 1] + list(x[1:]), proof)
    assert not po.groth16_verify(vk, x, (G1.add(proof[0], g), proof[1], proof[2]))
    gi = synth.make_gm17_instance(pid, 8, num_inputs=3)
    gvk = po.gm17_vk(pairing, gi["trapdoor"], gi["num_inputs"])
    x = gi["z_int"][1:gi["num_inputs"]]
    a, c = po.gm17_simulated_logs(gi["trapdoor"], x, 4242, p)
    proof = (G1.mul(g, a), G2.mul(h, a), G1.mul(g, c))
    assert po.gm17_verify(gvk, x, proof)
    assert not po.gm17_verify(gvk, x, (proof[0], G2.mul(h, a + 1), proof[2]))
    assert not po.gm17_verify(gvk, x, (proof[0], proof[1], G1.neg(proof[2])))


# ---- device header on the CPU --------------------------------------------------------------------------------------
@pytest.mark.parametrize("pid", PIDS)
def test_emu_tower_arithmetic(emu, pid):
    P = po.PARAMS[pid]
    F = P.F
    rng = o.SplitMix64(7 + pid)
    out = np.zeros(P.k * 5, dtype=np.uint64)
    for _ in range(4):
        x = tuple(rng.field(P.q) for _ in range(P.k))
        y = tuple(rng.field(P.q) for _ in range(P.k))
        xl, yl = po.gt_to_limbs(P, x), po.gt_to_limbs(P, y)
        for op, want in ((0, F.mul(x, y)), (1, F.sqr(x)), (2, F.inv(x)), (3, F.pow(x, P.q)),
                         (4, F.pow(x, P.q ** (P.k // 2)))):
            emu.emu_gt_op(pid, op, _p(xl), _p(yl), _p(out))
            assert np.array_equal(out, po.gt_to_limbs(P, want)), op


@pytest.mark.parametrize("pid", PIDS)
def test_emu_pairing_bytes_match_oracle(emu, pid):
    P = po.PARAMS[pid]
    G1, G2 = P.pairing.g1, P.pairing.g2
    g, h = _gens(P)
    c1, c2 = codec.G1_OF[pid], codec.G2_OF[pid]
    rng = o.SplitMix64(31 + pid)
    pairs = [(G1.mul(g, rng.field(P.r)), G2.mul(h, rng.field(P.r))) for _ in range(8)]
    pairs += [(None, h), (g, None), (None, None)]
    a = np.stack([synth.point_limbs(c1, p) for p, _ in pairs])
    b = np.stack([synth.point_limbs(c2, q) for _, q in pairs])
    out = np.zeros((len(pairs), P.k * 5), dtype=np.uint64)
    emu.emu_pairing(pid, _p(a), _p(b), ctypes.c_size_t(len(pairs)), _p(out))
    for i, (p, q) in enumerate(pairs):
        assert np.array_equal(out[i], po.gt_to_limbs(P, po.pairing(P, p, q))), i


def _vk_bytes(vk, gm17):
    keys = ["h_g2", "g_alpha_g1", "h_beta_g2", "g_gamma_g1", "h_gamma_g2", "query"] if gm17 else \
        ["alpha_g1", "beta_g2", "gamma_g2", "delta_g2", "gamma_abc_g1"]
    return np.ascontiguousarray(np.concatenate([np.asarray(vk[k]).reshape(-1) for k in keys]))


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_emu_verify(emu, pid, gm17):
    """per-proof verification of pairing.cuh: simulated proofs accepted, every tampering rejected; reports the
    base-field products of one verification (the work model of the GPU kernels)"""
    inst = (synth.make_gm17_instance if gm17 else synth.make_instance)(pid, 8, num_inputs=3)
    vk = _vk_bytes(vh.gm17_vk(inst) if gm17 else vh.groth16_vk(inst), gm17)
    proofs, inputs = vh.simulated(inst, 3, 5 + pid, gm17)
    rows, xs = [proofs[0], proofs[1]], [inputs[0], inputs[1]]
    for kind in vh.TAMPERINGS:
        pr, x = vh.tamper(pid, proofs[2], inputs[2], kind, other=proofs[0])
        rows.append(pr)
        xs.append(x)
    rows, xs = np.ascontiguousarray(np.stack(rows)), np.ascontiguousarray(np.stack(xs))
    ok = np.zeros(len(rows), dtype=np.uint8)
    fn = emu.emu_gm17_verify if gm17 else emu.emu_groth16_verify
    emu.emu_products()
    fn(pid, _p(vk), inst["num_inputs"], _p(rows[:1]), _p(xs[:1]), ctypes.c_size_t(1), _p(ok))
    one = emu.emu_products()
    fn(pid, _p(vk), inst["num_inputs"], _p(rows[:2]), _p(xs[:2]), ctypes.c_size_t(2), _p(ok))
    per_proof = emu.emu_products() - one  # the key's processing cancels
    fn(pid, _p(vk), inst["num_inputs"], _p(rows), _p(xs), ctypes.c_size_t(len(rows)), _p(ok))
    assert ok.tolist() == [1, 1] + [0] * len(vh.TAMPERINGS), ok.tolist()
    print("base-field products of one verification (%s, %s, 2 public inputs): %d" % (
        "mnt4" if pid == 0 else "mnt6", "gm17" if gm17 else "groth16", per_proof))
