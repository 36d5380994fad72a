"""Degenerate Groth16 / GM17 proofs end to end on the GPU, against the proofs built from discrete logs and the C++
oracle (pinned to each other by test_edge_proofs_cpu.py): randomness 0, 1, p - 1 and the recoding boundaries of the
double-scalar chain, proof points at infinity, doublings and cancellations in every addition of proof assembly
(edge_proofs.py).  The small-proof path (<= 2^17 variables: s g_a and r g1_b as MSMs of their own) runs on synth
instances and identity-R1CS assignments, the chain path (wec_multi_mul_kernel) on GPU-built instances above 2^17
variables, and the assembly entry points on chosen xyzz partial sums.  The verifier sees every one of these proofs,
and degenerate simulated ones, beside generic and tampered proofs, as limbs and as compressed bytes."""
import ctypes

import numpy as np
import pytest

import c_oracle as co
import codec
import deserialize_helpers as dh
import edge_proofs as ep
import synth
import test_edge_proofs_cpu as cpu
import test_gpu_poly_dev as tpd
import verify_helpers as vh

pytestmark = pytest.mark.gpu
PIDS = (0, 1)
M = 1000  # constraints of the small-path instances


@pytest.fixture(scope="module")
def ctx():
    import pcd_b200
    c = pcd_b200.Context(0)
    yield c
    c.close()


_INST = {}


def small_instance(pid, gm17):
    if (pid, gm17) not in _INST:
        _INST[(pid, gm17)] = ep.make_instance(pid, M, seed=(5100 if gm17 else 5000) + 10 * pid, gm17=gm17)
    return _INST[(pid, gm17)]


def _index(ctx, inst, gm17, precompute):
    import pcd_b200
    cm = pcd_b200.ConstraintMatrices(inst["pairing"], inst["num_inputs"], inst["num_witness"], inst["A"], inst["B"],
                                     inst["C"])
    if gm17:
        g = pcd_b200.GM17(ctx, inst["pairing"])
        return g, g.index(pcd_b200.GM17ProvingKey(pairing=inst["pairing"], **inst["pk"]), cm, precompute)
    g = pcd_b200.Groth16(ctx, inst["pairing"])
    return g, g.index(pcd_b200.ProvingKey(pairing=inst["pairing"], **inst["pk"]), cm, precompute)


def _limbs(rand):
    return [codec.int_to_limbs(v) for v in rand]


def _prove(g, idx, z, rand, gm17):
    return (g.create_proof(idx, z, *_limbs(rand)) if gm17 else
            g.create_proof_with_reduction(idx, z, *_limbs(rand))).affine_limbs()


def _prove_dev(g, idx, d_z, rand):
    return g.create_proof_dev(idx, d_z, *_limbs(rand)).affine_limbs()


def _device(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).to("cuda:0")


def _run_matrix(ctx, inst, cases, gm17, expect, oracle=True):
    """every (name, randomness) of cases through the host and device entry points, with and without window tables
    and with serialised lanes, against expect(randomness); byte for byte against the C++ oracle when asked"""
    pid = inst["pairing"]
    d_z = _device(inst["z"])
    for pre in (False, True):
        g, idx = _index(ctx, inst, gm17, pre)
        for name, *rand in cases:
            want = expect(rand)
            got = _prove(g, idx, inst["z"], rand, gm17)
            assert np.array_equal(got, want), (name, pre)
            assert np.array_equal(_prove_dev(g, idx, d_z.data_ptr(), rand), want), (name, pre, "dev")
            assert g.ctx.serialize_proof(pid, got) == dh.proof_bytes(pid, want), name
            if oracle and not pre:
                assert np.array_equal(got, cpu.prove_oracle(inst, rand, gm17)), name
        if pre:
            ctx.set_concurrency(False)
            try:
                for name, *rand in cases:
                    assert np.array_equal(_prove(g, idx, inst["z"], rand, gm17), expect(rand)), (name, "serial")
            finally:
                ctx.set_concurrency(True)
            if not gm17:  # proof graphs: one key, a sequence of edge (r, s) replayed from one captured graph
                ctx.set_proof_graphs(True)
                try:
                    cap0, rep0 = ctx.proof_graph_stats()
                    for name, *rand in cases:
                        assert np.array_equal(_prove_dev(g, idx, d_z.data_ptr(), rand), expect(rand)), (name, "graph")
                    cap1, rep1 = ctx.proof_graph_stats()
                    assert cap1 - cap0 >= 1 and rep1 - rep0 >= len(cases) - 2
                finally:
                    ctx.set_proof_graphs(False)
        idx.close()


# ---- prover: small-proof path --------------------------------------------------------------------------------------
@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_prover_targets_small_path(ctx, pid, gm17):
    inst, targets = small_instance(pid, gm17)
    assert inst["num_inputs"] + inst["num_witness"] <= 1 << 17
    _run_matrix(ctx, inst, targets, gm17, lambda rand: cpu.trapdoor(inst, rand, gm17))


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_identity_r1cs(ctx, pid, gm17):
    """x_i * 1 = x_i per variable: witnesses all 0 (every MSM over the assignment is O), all 1, all p - 1, repeated"""
    p = codec.FIELD_P[pid]
    nv = 600
    rg, sg = ep.generic(p)
    for name, z in ep.identity_assignments(pid, nv).items():
        inst = ep.identity_instance(pid, z, gm17, num_witness=nv - 2)
        rands = [(0, 0, 0), (rg, sg, rg), (p - 1, p - 1, p - 1)] if gm17 else [(0, 0), (0, sg), (rg, sg), (p - 1, p - 1)]
        _run_matrix(ctx, inst, [(name,) + r for r in rands], gm17, lambda rand: cpu.trapdoor(inst, rand, gm17))


# ---- prover: the double-scalar chain (> 2^17 variables) ---------------------------------------------------------------
_LARGE = {}


def large_instance(ctx, pid):
    """MNT4: radix-2 domain 2^18; MNT6: 2^17 + 1 constraints on the mixed-radix domain 49 * 2^12"""
    if pid not in _LARGE:
        from pcd_b200 import synthetic
        inst = synthetic.make_groth16_instance(ctx, 0, 18, seed=6000) if pid == 0 else \
            synthetic.make_groth16_instance(ctx, 1, 0, seed=6001, num_constraints=(1 << 17) + 1)
        _LARGE[pid] = inst
    return _LARGE[pid]


@pytest.mark.parametrize("pid", PIDS)
def test_prover_targets_chain_path(ctx, pid):
    from pcd_b200 import synthetic
    inst = large_instance(ctx, pid)
    assert inst["num_inputs"] + inst["num_witness"] > 1 << 17
    p = inst["p"]
    targets = ep.groth16_targets(ep.groth16_logs_from_expected(inst["expected_logs"], p))
    assert len(targets) >= 25
    expect = lambda rand: synthetic.expected_proof(ctx, inst, *rand, mul=co.fixed_base_mul)
    _run_matrix(ctx, dict(inst, pairing=pid), targets, False, expect, oracle=False)


def test_gm17_a_inf_from_expected_logs(ctx):
    """GM17 on a GPU-built instance: A = B = O solved from expected_logs alone"""
    from pcd_b200 import synthetic
    inst = synthetic.make_gm17_instance(ctx, 1, 3000, seed=6100)
    p = inst["p"]
    a = ep.gm17_a_inf_from_expected(inst["expected_logs"], p)
    rg = ep.generic(p)[0]
    cases = [("A=B=O", (a - rg) % p, 5, rg), ("A=B=O, r=0", a, 0, 0)]
    for _, *rand in cases:
        assert inst["expected_logs"](*rand)[0] == 0
    expect = lambda rand: synthetic.expected_gm17_proof(ctx, inst, *rand, mul=co.fixed_base_mul)
    _run_matrix(ctx, dict(inst, pairing=1), cases, True, expect, oracle=False)


# ---- the assembly entry points as a unit ----------------------------------------------------------------------------
def _msm(curve, pts, ks):
    order = codec.CURVE_ORDER[curve]
    return co.msm(curve, np.stack(pts), codec.ints_to_limbs([k % order for k in ks]), 1)


def _assembly_cases(pid, world):
    """[(name, ga parts, g1b parts, g2 parts, h parts, l parts, r, s)], one affine point per rank each"""
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    p = codec.FIELD_P[pid]
    P1 = synth.random_points(4 * world, g1, 700 + 10 * pid + world)
    P2 = synth.random_points(world, g2, 750 + 10 * pid + world)
    O1, O2 = np.zeros(10, np.uint64), np.zeros(codec.POINT_LIMBS[g2], np.uint64)
    ga, g1b, h, l = (list(P1[k * world:(k + 1) * world]) for k in range(4))
    g2p = list(P2)
    rg, sg = ep.generic(p)
    ones = [1] * world
    out = [("all O", [O1] * world, [O1] * world, [O2] * world, [O1] * world, [O1] * world, rg, sg),
           ("generic", ga, g1b, g2p, h, l, rg, sg)]
    if world >= 2:
        pm = lambda pts, c: [pts[0], tpd._neg(c, pts[0])] + ([O1 if c == g1 else O2] * (world - 2))
        out.append(("P and -P", pm(ga, g1), pm(g1b, g1), pm(g2p, g2), pm(h, g1), pm(l, g1), rg, sg))
    out.append(("equal partials", [ga[0]] * world, [g1b[0]] * world, [g2p[0]] * world, [h[0]] * world,
                [l[0]] * world, rg, sg))
    bnd = ep.boundary_scalars(p)
    for i, v in enumerate(bnd):
        out.append(("chain r=%#x" % v, ga, g1b, g2p, h, l, v, bnd[-1 - i]))
    out.append(("r=s=0", ga, g1b, g2p, h, l, 0, 0))
    out.append(("r=s=p-1", ga, g1b, g2p, h, l, p - 1, p - 1))
    sum_a = _msm(g1, ga, ones)
    for name, k in (("join doubles", sg * pow(rg, -1, p)), ("join cancels", -sg * pow(rg, -1, p))):
        out.append((name, ga, [_msm(g1, [sum_a], [k])] + [O1] * (world - 1), g2p, h, l, rg, sg))
    sum_b, sum_l, sum_h = _msm(g1, g1b, ones), _msm(g1, l, ones), _msm(g1, h, ones)
    # C = h + l + T with T = s A + r g1_b: h chosen so that C = O, or so that the last addition doubles
    for name, sign in (("C=O", -1), ("last addition doubles", 1)):
        h0 = _msm(g1, [sum_a, sum_b, sum_l], [sign * sg, sign * rg, -1])
        out.append((name, ga, g1b, g2p, [h0] + [O1] * (world - 1), l, rg, sg))
    for name, k in (("first addition doubles", 1), ("first addition cancels", -1)):
        out.append((name, ga, g1b, g2p, h, [_msm(g1, [sum_h], [k])] + [O1] * (world - 1), rg, sg))
    return out


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("world", [1, 2, 3])
def test_assemble_entry_points(ctx, pid, world):
    """pcdgpu_groth16_assemble_begin_dev / _finish_dev on xyzz partials of `world` ranks (Z != 1 on every rank but
    the first): A = sum g_a, B = sum g2_b, C = sum h + sum l + [s] A + [r] sum g1_b"""
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    lib = ctx.lib
    a1, a2 = codec.POINT_LIMBS[g1], codec.POINT_LIMBS[g2]
    for name, ga, g1b, g2p, h, l, r, s in _assembly_cases(pid, world):
        lam = lambda k: 1 if k == 0 else 12345 + 77 * k
        ab = np.concatenate([np.concatenate([tpd._xyzz(g1, ga[k], lam(k)), tpd._xyzz(g1, g1b[k], lam(k) + 1)])
                             for k in range(world)])
        pg2 = np.concatenate([tpd._xyzz(g2, g2p[k], lam(k) + 2) for k in range(world)])
        hl = np.concatenate([np.concatenate([tpd._xyzz(g1, h[k], lam(k) + 3), tpd._xyzz(g1, l[k], lam(k) + 4)])
                             for k in range(world)])
        d_ab, d_g2, d_hl = _device(ab), _device(pg2), _device(hl)
        rl, sl = codec.int_to_limbs(r), codec.int_to_limbs(s)
        out = np.zeros(2 * a1 + a2, dtype=np.uint64)
        ctx._check(lib.pcdgpu_groth16_assemble_begin_dev(ctx.h, pid, rl.ctypes.data, sl.ctypes.data, world,
                                                         d_ab.data_ptr(), d_g2.data_ptr()))
        ctx._check(lib.pcdgpu_groth16_assemble_finish_dev(ctx.h, pid, world, d_hl.data_ptr(), out.ctypes.data))
        ones = [1] * world
        A = _msm(g1, ga, ones)
        B = _msm(g2, g2p, ones)
        C = _msm(g1, [A, _msm(g1, g1b, ones), _msm(g1, h, ones), _msm(g1, l, ones)], [s, r, 1, 1])
        assert np.array_equal(out[:a1], A), (name, "A")
        assert np.array_equal(out[a1:a1 + a2], B), (name, "B")
        assert np.array_equal(out[a1 + a2:], C), (name, "C")
        if name == "C=O" or name == "all O":
            assert not C.any()


# ---- verifier ----------------------------------------------------------------------------------------------------------
def _vk(ctx, inst, gm17):
    import pcd_b200
    if gm17:
        return pcd_b200.GM17(ctx, inst["pairing"]), pcd_b200.GM17VerifyingKey(**vh.gm17_vk(inst))
    return pcd_b200.Groth16(ctx, inst["pairing"]), pcd_b200.VerifyingKey(**vh.groth16_vk(inst))


BYTE_VALID_TAMPERINGS = ["A+G", "2B", "-C", "input", "swapB", "B=O"]


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_verifier(ctx, pid, gm17):
    """GPU edge proofs, degenerate simulated proofs, generic proofs and tamperings of each in one batch: the expected
    mask from limbs and from compressed bytes; deserialize_batch returns the prover's rows"""
    inst, targets = small_instance(pid, gm17)
    g, idx = _index(ctx, inst, gm17, False)
    x = vh.public_inputs(inst)
    rows, xs, want = [], [], []
    for name, *rand in targets:
        got = _prove(g, idx, inst["z"], rand, gm17)
        assert np.array_equal(got, cpu.trapdoor(inst, rand, gm17)), name
        rows += [got, cpu.tamper_c(pid, got)]
        xs += [x, x]
        want += [True, False]
    idx.close()
    for _, row, xi in cpu.simulated_rows(inst, gm17):
        xl = cpu.x_limbs(inst, xi)
        rows += [row, cpu.tamper_c(pid, row)]
        xs += [xl, xl]
        want += [True, False]
    gen, gx = vh.simulated(inst, 4, 321 + pid, gm17)
    for i, kind in enumerate(BYTE_VALID_TAMPERINGS):
        pr, xx = vh.tamper(pid, gen[i % 4], gx[i % 4], kind, other=gen[(i + 1) % 4])
        rows += [gen[i % 4], pr]
        xs += [gx[i % 4], xx]
        want += [True, False]
    perm = np.random.Generator(np.random.Philox(17 + pid)).permutation(len(rows))
    rows = np.ascontiguousarray(np.stack(rows)[perm])
    xs = np.ascontiguousarray(np.stack(xs)[perm])
    want = np.array(want)[perm]
    v, vk = _vk(ctx, inst, gm17)
    pvk = v.process_vk(vk)
    assert np.array_equal(v.verify_batch(pvk, xs, rows), want)
    blobs = [ctx.serialize_proof(pid, r) for r in rows]
    assert blobs == [dh.proof_bytes(pid, r) for r in rows]
    back, ok = v.deserialize_batch(blobs)
    assert ok.all() and np.array_equal(back, rows)
    assert np.array_equal(v.verify_batch_serialized(pvk, xs, blobs), want)
    pvk.close()


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_key_with_constant_at_infinity(ctx, pid, gm17):
    """process_vk of a key whose gamma_abc_g1[0] (GM17: query[0]) is O, and verification against it"""
    inst, _ = small_instance(pid, gm17)
    key_inst = ep.key_with_zero_constant(inst, gm17)
    v, vk = _vk(ctx, key_inst, gm17)
    assert not np.asarray(vk.query if gm17 else vk.gamma_abc_g1)[0].any()
    pvk = v.process_vk(vk)
    sims = cpu.simulated_rows(key_inst, gm17)
    rows = np.stack([r for _, r, _ in sims] + [cpu.tamper_c(pid, r) for _, r, _ in sims])
    xs = np.stack([cpu.x_limbs(key_inst, xi) for _, _, xi in sims] * 2)
    n = len(sims)
    assert v.verify_batch(pvk, xs, rows).tolist() == [True] * n + [False] * n
    assert v.verify_batch_serialized(pvk, xs, [ctx.serialize_proof(pid, r) for r in rows]).tolist() == \
        [True] * n + [False] * n
    pvk.close()
