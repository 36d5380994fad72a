"""Verifying keys and simulated proofs for the verification tests (test infrastructure): keys from the known
trapdoors of synth.make_instance / make_gm17_instance, and valid proofs with known verdicts from their discrete logs
(pairing_oracle's simulators), multiplied out by the C++ oracle's fixed-base multiplication."""
import numpy as np

import c_oracle as co
import codec
import pairing_oracle as po
import pcd_oracle as o
import synth

GAMMA_SEED = 0x6A77A  # gamma is drawn from its own generator: the instance's draws stay as they are


def _mul(curve, logs):
    return co.fixed_base_mul(curve, synth.generator_limbs(curve), codec.ints_to_limbs([x % _order(curve) for x in logs]))


def _order(curve):
    return synth.CURVES[curve].order


def groth16_vk(inst, gamma=None):
    """dict of VerifyingKey fields (limbs) for inst's key; gamma defaults to a draw of GAMMA_SEED"""
    pid, t, ni = inst["pairing"], inst["trapdoor"], inst["num_inputs"]
    p = synth.PAIRINGS[pid].fr.p
    if gamma is None:
        gamma = o.SplitMix64(GAMMA_SEED).field(p) or 1
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    gi = pow(gamma, -1, p)
    abc = [(t["beta"] * t["At"][j] + t["alpha"] * t["Bt"][j] + t["Ct"][j]) * gi % p for j in range(ni)]
    return dict(pairing=pid, alpha_g1=_mul(g1, [t["alpha"]])[0], beta_g2=_mul(g2, [t["beta"]])[0],
                gamma_g2=_mul(g2, [gamma])[0], delta_g2=_mul(g2, [t["delta"]])[0], gamma_abc_g1=_mul(g1, abc))


def gm17_vk(inst):
    pid, t, ni = inst["pairing"], inst["trapdoor"], inst["num_inputs"]
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    return dict(pairing=pid, h_g2=synth.generator_limbs(g2), g_alpha_g1=_mul(g1, [t["alpha"]])[0],
                h_beta_g2=_mul(g2, [t["beta"]])[0], g_gamma_g1=_mul(g1, [t["gamma"]])[0],
                h_gamma_g2=_mul(g2, [t["gamma"]])[0], query=_mul(g1, t["vk_sc"][:ni]))


def public_inputs(inst):
    """the instance's public inputs x = z[1 : num_inputs] as Montgomery limbs, (num_inputs - 1, 5)"""
    fp = synth.PAIRINGS[inst["pairing"]].fr
    return synth.mont_limbs(inst["z_int"][1:inst["num_inputs"]], fp).reshape(-1, 5)


def simulated(inst, n, seed, gm17=False):
    """n valid proofs for random public inputs: (proofs (n, A || B || C limbs), inputs (n, num_inputs - 1, 5))"""
    pid, t, ni = inst["pairing"], inst["trapdoor"], inst["num_inputs"]
    fr = synth.PAIRINGS[pid].fr
    p = fr.p
    rng = o.SplitMix64(seed)
    xs = [[rng.field(p) for _ in range(ni - 1)] for _ in range(n)]
    a_l, b_l, c_l = [], [], []
    for x in xs:
        if gm17:
            a, c = po.gm17_simulated_logs(t, x, rng.field(p), p)
            b = a
        else:
            a, b, c = po.groth16_simulated_logs(t, x, rng.field(p), rng.field(p), p)
        a_l.append(a)
        b_l.append(b)
        c_l.append(c)
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    proofs = np.concatenate([_mul(g1, a_l), _mul(g2, b_l), _mul(g1, c_l)], axis=1)
    inputs = synth.mont_limbs([v for x in xs for v in x], fr).reshape(n, ni - 1, 5) if ni > 1 else \
        np.zeros((n, 0, 5), dtype=np.uint64)
    return np.ascontiguousarray(proofs), np.ascontiguousarray(inputs)


def widths(pid):
    a1 = codec.POINT_LIMBS[codec.G1_OF[pid]]
    a2 = codec.POINT_LIMBS[codec.G2_OF[pid]]
    return a1, a2


def tamper(pid, proofs, inputs, kind, other=None):
    """one proof (row) changed in one way; returns (proof, inputs)"""
    a1, a2 = widths(pid)
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    pr, x = proofs.copy(), inputs.copy()
    A, B, C = pr[:a1], pr[a1:a1 + a2], pr[a1 + a2:]
    fp = synth.COORD_FP[g1]
    if kind == "A+G":
        pr[:a1] = co.msm(g1, np.stack([A, synth.generator_limbs(g1)]), codec.ints_to_limbs([1, 1]), 1)
    elif kind == "2B":
        pr[a1:a1 + a2] = co.fixed_base_mul(g2, B, codec.ints_to_limbs([2]), 1)[0]
    elif kind == "-C":
        pr[a1 + a2:] = co.fixed_base_mul(g1, C, codec.ints_to_limbs([_order(g1) - 1]), 1)[0]
    elif kind == "input":
        x[0] = synth.mont_limbs([(o.fp_from_mont_bytes(x[0].tobytes(), synth.PAIRINGS[pid].fr) + 1)],
                                synth.PAIRINGS[pid].fr)[0]
    elif kind == "swapB":
        pr[a1:a1 + a2] = other[a1:a1 + a2]
    elif kind == "B=O":
        pr[a1:a1 + a2] = 0
    elif kind == "offcurve":
        y = o.fp_from_mont_bytes(A[5:10].tobytes(), fp)
        pr[5:10] = synth.mont_limbs([(y + 1) % fp.p], fp)[0]
    elif kind == ">=p":
        v = o.fp_from_mont_bytes(A[0:5].tobytes(), fp) * fp.R % fp.p + fp.p  # same residue, not canonical
        if v < 1 << 320:
            pr[0:5] = codec.int_to_limbs(v)
        else:
            pr[0:5] = codec.int_to_limbs(fp.p)
    else:
        raise ValueError(kind)
    return pr, x


TAMPERINGS = ["A+G", "2B", "-C", "input", "swapB", "B=O", "offcurve", ">=p"]
