"""Degenerate Groth16 / GM17 proofs without a GPU: the references every GPU comparison of test_gpu_edge_proofs.py
relies on.  For every target of edge_proofs (randomness 0, 1, p - 1, recoding boundaries of the double-scalar chain,
points at infinity, doublings and cancellations in proof assembly) the C++ oracle's prover equals the proof built
from discrete logs, the Python pairing oracle and the device header pairing.cuh built for the CPU accept it, and
its bytes round-trip through the device deserializer built for the CPU.  Degenerate simulated proofs (zero logs,
public inputs 0 / 1 / p - 1, an input combination at infinity, GM17's A + g_alpha = O) are accepted and a
one-point tampering of each is rejected."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import c_oracle as co
import codec
import deserialize_helpers as dh
import deserialize_oracle as do
import edge_proofs as ep
import pairing_oracle as po
import pcd_oracle as o
import synth
import verify_helpers as vh

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "pcd_b200", "csrc")
PIDS = (0, 1)
M = 24  # constraints of the synthetic instances


def _emu_lib(name, headers):
    src = os.path.join(HERE, "hostemu", name + ".cpp")
    so = os.path.join(HERE, "hostemu", "_build", "lib%s.so" % name.replace("_", ""))
    deps = [src, os.path.join(HERE, "hostemu", "hostemu_prims.h")] + [os.path.join(CSRC, f) for f in headers]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-I", CSRC, "-I",
                               os.path.join(HERE, "hostemu"), src, "-o", so])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def pemu():
    return _emu_lib("pairing_emu", ("pairing.cuh", "fp.cuh", "fpx.cuh", "ec.cuh", "prims.cuh", "constants.cuh"))


@pytest.fixture(scope="module")
def demu():
    return _emu_lib("deserialize_emu", ("deserialize.cuh", "pairing.cuh", "fp.cuh", "fpx.cuh", "ec.cuh", "prims.cuh",
                                        "constants.cuh"))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


_INST = {}


def instance(pid, gm17):
    """the synth instance of the prover matrix (the same seeds as test_gpu_edge_proofs.py) and its targets"""
    key = (pid, gm17)
    if key not in _INST:
        _INST[key] = ep.make_instance(pid, M, seed=(3100 if gm17 else 3000) + 10 * pid, gm17=gm17)
    return _INST[key]


def _vk_bytes(vk, gm17):
    keys = ["h_g2", "g_alpha_g1", "h_beta_g2", "g_gamma_g1", "h_gamma_g2", "query"] if gm17 else \
        ["alpha_g1", "beta_g2", "gamma_g2", "delta_g2", "gamma_abc_g1"]
    return np.ascontiguousarray(np.concatenate([np.asarray(vk[k]).reshape(-1) for k in keys]))


def emu_verify(emu, inst, rows, xs, gm17):
    vk = _vk_bytes(vh.gm17_vk(inst) if gm17 else vh.groth16_vk(inst), gm17)
    rows, xs = np.ascontiguousarray(np.stack(rows)), np.ascontiguousarray(np.stack(xs))
    ok = np.zeros(len(rows), dtype=np.uint8)
    fn = emu.emu_gm17_verify if gm17 else emu.emu_groth16_verify
    fn(inst["pairing"], _p(vk), inst["num_inputs"], _p(rows), _p(xs), ctypes.c_size_t(len(rows)), _p(ok))
    return ok.tolist()


def oracle_verify(inst, x, row, gm17):
    pid = inst["pairing"]
    pairing = synth.PAIRINGS[pid]
    proof = tuple(dh.limbs_point(c, v) for c, v in zip((codec.G1_OF[pid], codec.G2_OF[pid], codec.G1_OF[pid]),
                                                           dh.split(pid, row)))
    if gm17:
        return po.gm17_verify(po.gm17_vk(pairing, inst["trapdoor"], inst["num_inputs"]), x, proof)
    return po.groth16_verify(po.groth16_vk(pairing, inst["trapdoor"], inst["num_inputs"], vh_gamma(pid)), x, proof)


def vh_gamma(pid):
    """the gamma of verify_helpers.groth16_vk, so that both verifiers see one key"""
    return o.SplitMix64(vh.GAMMA_SEED).field(synth.PAIRINGS[pid].fr.p) or 1


def tamper_c(pid, row):
    """C + G: changes e(C, delta) (Groth16) / e(C, h) (GM17) whatever the other points are"""
    g1 = codec.G1_OF[pid]
    a1, a2 = vh.widths(pid)
    out = row.copy()
    out[a1 + a2:] = co.msm(g1, np.stack([row[a1 + a2:], synth.generator_limbs(g1)]), codec.ints_to_limbs([1, 1]), 1)
    return out


def zero_pattern(pid, row):
    return tuple(not v.any() for v in dh.split(pid, row))


def prove_oracle(inst, rand, gm17):
    args = (inst["pairing"], inst["pk"], inst["A"], inst["B"], inst["C"], inst["m"], inst["num_inputs"],
            inst["num_witness"], inst["z"])
    lim = [codec.int_to_limbs(v) for v in rand]
    return co.gm17_prove(*args, *lim, threads=4) if gm17 else co.groth16_prove(*args, *lim, threads=4)


def trapdoor(inst, rand, gm17):
    return synth.gm17_trapdoor_proof(inst, *rand) if gm17 else synth.trapdoor_proof(inst, *rand)


def expected_zeros(inst, rand, gm17):
    """(A = O, B = O, C = O) from the discrete logs"""
    if gm17:
        e = ep.gm17_terms(ep.gm17_logs(inst), *rand)
        return e["A"] == 0, e["A"] == 0, e["C"] == 0
    e = ep.groth16_terms(ep.groth16_logs(inst), *rand)
    return e["A"] == 0, e["B"] == 0, e["C"] == 0


# ---- the constructors ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pid", PIDS)
def test_constructors(pid):
    """every target exists on both schemes and hits what it names; identity-R1CS assignments satisfy it"""
    _, g16 = instance(pid, False)
    _, gm = instance(pid, True)
    names16, names_gm = {t[0] for t in g16}, {t[0] for t in gm}
    for n in ("r=s=0", "r=0", "s=0", "r=s=1", "r=s=p-1", "r=2,s=p-2", "A=O", "B=O", "A=B=O", "C=O",
              "last addition doubles", "small-path last addition doubles", "chain join doubles", "chain join cancels",
              "first addition doubles", "first addition cancels"):
        assert n in names16, n
    for n in ("d1=d2=r=0", "r=0", "d2=0", "d1=d2=r=1", "d1=d2=r=p-1", "A=B=O", "C=O", "last addition doubles",
              "first addition cancels", "first addition doubles"):
        assert n in names_gm, n
    p = codec.FIELD_P[pid]
    b = ep.boundary_scalars(p)
    assert {7, 8, 9, 15, 16, 17} <= set(b) and all(0 < v < p for v in b)
    assert sum(1 for n in names16 if n.startswith("chain r=")) == len(b)
    for v in (2, 5, 12345, p - 1):
        assert pow(ep.sqrt_mod(v * v, p), 2, p) == v * v % p
    r1cs = ep.identity_r1cs(pid, 10)
    for z in ep.identity_assignments(pid, r1cs.num_vars).values():
        assert r1cs.is_satisfied(z)


# ---- provers: C++ oracle == discrete logs; both verifiers accept; bytes round-trip ----------------------------------------
def _check_prover_targets(pemu, demu, inst, targets, gm17, oracle_verifier=True):
    pid = inst["pairing"]
    x = list(inst["z_int"][1:inst["num_inputs"]])
    xl = vh.public_inputs(inst)
    rows = []
    for name, *rand in targets:
        ref = prove_oracle(inst, rand, gm17)
        assert np.array_equal(ref, trapdoor(inst, rand, gm17)), name
        assert zero_pattern(pid, ref) == expected_zeros(inst, rand, gm17), name
        rows.append(ref)
        if oracle_verifier and not name.startswith("chain"):
            assert oracle_verify(inst, x, ref, gm17), name
    n = len(rows)
    assert emu_verify(pemu, inst, rows + [tamper_c(pid, r) for r in rows], [xl] * (2 * n), gm17) == [1] * n + [0] * n
    # compressed bytes, points at infinity included, back through the device deserializer and the oracle
    blobs = [dh.proof_bytes(pid, r) for r in rows]
    data = np.frombuffer(b"".join(blobs), dtype=np.uint8).copy()
    out = np.zeros((n, rows[0].shape[0]), dtype=np.uint64)
    ok = np.zeros(n, dtype=np.uint8)
    demu.emu_deserialize_proofs(pid, _p(data), ctypes.c_size_t(n), _p(out), _p(ok))
    assert ok.tolist() == [1] * n
    assert np.array_equal(out, np.stack(rows))
    for b, r in zip(blobs, rows):
        assert np.array_equal(dh.proof_row(pid, do.deserialize_proof(synth.PAIRINGS[pid], b)), r)
    return rows


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_prover_targets(pemu, demu, pid, gm17):
    inst, targets = instance(pid, gm17)
    rows = _check_prover_targets(pemu, demu, inst, targets, gm17)
    pats = {zero_pattern(pid, r) for r in rows}
    want = {(True, True, False), (False, False, True)}  # A (= B in GM17) at infinity; C at infinity
    if not gm17:
        want |= {(True, False, False), (False, True, False)}
    assert want <= pats, pats


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_identity_r1cs(pemu, demu, pid, gm17):
    """x_i * 1 = x_i for every variable, with the witness all 0, all 1, all p - 1 or one repeated value"""
    p = codec.FIELD_P[pid]
    nv = 32
    rg, sg = ep.generic(p)
    for name, z in ep.identity_assignments(pid, nv).items():
        inst = ep.identity_instance(pid, z, gm17, num_witness=nv - 2)
        rands = [(0, 0, 0), (rg, sg, rg), (1, 1, 1)] if gm17 else [(0, 0), (rg, sg), (p - 1, p - 1)]
        _check_prover_targets(pemu, demu, inst, [(name,) + r for r in rands], gm17, oracle_verifier=name == "zeros")


# ---- simulated degenerate proofs -------------------------------------------------------------------------------------
def simulated_rows(inst, gm17):
    """[(name, row, x ints)] of the degenerate simulated proofs of edge_proofs"""
    pid = inst["pairing"]
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    out = []
    if gm17:
        for name, x, a, c in ep.gm17_simulated_edges(inst):
            out.append((name, np.concatenate([vh._mul(g1, [a])[0], vh._mul(g2, [a])[0], vh._mul(g1, [c])[0]]), x))
    else:
        for name, x, a, b, c in ep.groth16_simulated_edges(inst):
            out.append((name, np.concatenate([vh._mul(g1, [a])[0], vh._mul(g2, [b])[0], vh._mul(g1, [c])[0]]), x))
    return out


def x_limbs(inst, x):
    return synth.mont_limbs(x, synth.PAIRINGS[inst["pairing"]].fr).reshape(-1, 5)


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_simulated_edges(pemu, pid, gm17):
    inst, _ = instance(pid, gm17)
    for key_inst in (inst, ep.key_with_zero_constant(inst, gm17)):
        sims = simulated_rows(key_inst, gm17)
        names = {n for n, _, _ in sims}
        assert {"a=0", "x=0", "x=1", "x=p-1", "input combination O"} <= names
        assert ({"A+g_alpha=O", "B+h_beta=O"} if gm17 else {"b=0", "c=0"}) <= names
        for name, row, x in sims:
            assert oracle_verify(key_inst, x, row, gm17), name
            assert not oracle_verify(key_inst, x, tamper_c(pid, row), gm17), name
        rows = [r for _, r, _ in sims]
        xs = [x_limbs(key_inst, x) for _, _, x in sims]
        n = len(rows)
        assert emu_verify(pemu, key_inst, rows + [tamper_c(pid, r) for r in rows], xs + xs, gm17) == [1] * n + [0] * n
    vk = vh.gm17_vk(ep.key_with_zero_constant(inst, True)) if gm17 else \
        vh.groth16_vk(ep.key_with_zero_constant(inst, False))
    assert not np.asarray(vk["query" if gm17 else "gamma_abc_g1"])[0].any()
