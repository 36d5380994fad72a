"""Seeded synthetic inputs for the parity tests (SURVEY.md 8d): curve points, witness-like scalars,
satisfiable R1CS and Groth16 keys with a known trapdoor.  Test infrastructure: built on the two
oracles (Python big-int for the scalar side, C++ for the point multiplications)."""
import numpy as np

import c_oracle as co
import codec
import pcd_oracle as o

PAIRINGS = {0: o.MNT4, 1: o.MNT6}
CURVES = {0: o.MNT4_G1, 1: o.MNT4_G2, 2: o.MNT6_G1, 3: o.MNT6_G2}
COORD_FP = {0: o.FQ4, 1: o.FQ4, 2: o.FR4, 3: o.FR4}


def point_limbs(curve_id, P):
    curve, fp = CURVES[curve_id], COORD_FP[curve_id]
    F = curve.F
    if P is None:
        return np.zeros(codec.POINT_LIMBS[curve_id], dtype=np.uint64)
    b = b"".join(o.fp_to_mont_bytes(c, fp) for c in F.coeffs(P[0])) + \
        b"".join(o.fp_to_mont_bytes(c, fp) for c in F.coeffs(P[1]))
    return np.frombuffer(b, dtype="<u8").copy()


def generator_limbs(curve_id):
    return point_limbs(curve_id, o.generator(CURVES[curve_id]))


def coeff_b_limbs(curve_id):
    curve, fp = CURVES[curve_id], COORD_FP[curve_id]
    b = b"".join(o.fp_to_mont_bytes(c, fp) for c in curve.F.coeffs(curve.b))
    return np.frombuffer(b, dtype="<u8").copy()


def random_scalars(n, curve_id, seed, dist="U"):
    """(n, 5) plain-integer scalars below the group order.  dist U: uniform; W: witness-like
    (55 % zero-or-one, 45 % uniform), as real R1CS assignments are."""
    f = codec.SCALAR_FIELD[curve_id]
    s = codec.random_field_elems(n, f, seed)
    if dist == "W":
        rng = np.random.Generator(np.random.Philox(seed + 1))
        u = rng.random(n)
        s[u < 0.55] = 0
        s[u < 0.30, 0] = 1
    return s


def random_points(n, curve_id, seed, threads=0):
    """n points k_i * G (k_i uniform), via the C++ oracle's double-and-add."""
    k = codec.random_field_elems(n, codec.SCALAR_FIELD[curve_id], seed + 7)
    return co.fixed_base_mul(curve_id, generator_limbs(curve_id), k, threads)


def r1cs_to_csr(r1cs):
    fp = r1cs.fp

    def one(rows):
        ptr, col, val = [0], [], []
        for r in rows:
            for c, j in r:
                col.append(j)
                val.append(o.fp_to_mont_bytes(c, fp))
            ptr.append(len(col))
        v = np.frombuffer(b"".join(val), dtype="<u8").copy().reshape(-1, 5) if val else np.zeros((0, 5), np.uint64)
        return np.array(ptr, dtype=np.uint32), np.array(col, dtype=np.uint32), v

    return one(r1cs.A), one(r1cs.B), one(r1cs.C)


def mont_limbs(vals, fp):
    return np.frombuffer(b"".join(o.fp_to_mont_bytes(v, fp) for v in vals), dtype="<u8").copy().reshape(-1, 5)


def make_instance(pairing_id, m, seed=20261017, bitlike=0.3, num_inputs=2, r1cs_z=None):
    """Satisfiable R1CS + assignment + Groth16 key with known trapdoor.  Returns a dict with the CSR
    matrices, z (Montgomery limbs), the key as numpy arrays (PK_FIELDS), and the python-side objects
    needed for the trapdoor check.  r1cs_z = (R1CS, assignment) replaces the synthetic system (m, bitlike
    and num_inputs are then ignored)."""
    pairing = PAIRINGS[pairing_id]
    fp = pairing.fr
    r1cs, z = r1cs_z or o.synthetic_r1cs(fp, m, num_inputs=num_inputs, seed=seed, bitlike=bitlike)
    m = r1cs.num_constraints
    t = o.groth16_setup_scalars(pairing, r1cs, seed=seed + 100)
    g1, g2 = codec.G1_OF[pairing_id], codec.G2_OF[pairing_id]
    G1, G2 = generator_limbs(g1), generator_limbs(g2)
    sc = lambda vals: codec.ints_to_limbs(vals)
    pk = {
        "alpha_g1": co.fixed_base_mul(g1, G1, sc([t["alpha"]]))[0],
        "beta_g1": co.fixed_base_mul(g1, G1, sc([t["beta"]]))[0],
        "delta_g1": co.fixed_base_mul(g1, G1, sc([t["delta"]]))[0],
        "beta_g2": co.fixed_base_mul(g2, G2, sc([t["beta"]]))[0],
        "delta_g2": co.fixed_base_mul(g2, G2, sc([t["delta"]]))[0],
        "a_query": co.fixed_base_mul(g1, G1, sc(t["At"])),
        "b_g1_query": co.fixed_base_mul(g1, G1, sc(t["Bt"])),
        "b_g2_query": co.fixed_base_mul(g2, G2, sc(t["Bt"])),
        "h_query": co.fixed_base_mul(g1, G1, sc(t["h_sc"])),
        "l_query": co.fixed_base_mul(g1, G1, sc(t["l_sc"])),
    }
    A, B, C = r1cs_to_csr(r1cs)
    return dict(pairing=pairing_id, r1cs=r1cs, z_int=z, z=mont_limbs(z, fp), A=A, B=B, C=C, pk=pk, trapdoor=t,
                m=m, num_inputs=r1cs.num_inputs, num_witness=r1cs.num_witness)


def trapdoor_proof(inst, r, s):
    """The proof every correct prover must output, from its discrete logs (SURVEY.md 7.3): returns
    affine limbs A || B || C computed as [a_log]G1, [b_log]G2, [c_log]G1 by the C++ oracle."""
    t, r1cs, z = inst["trapdoor"], inst["r1cs"], inst["z_int"]
    pid = inst["pairing"]
    p = PAIRINGS[pid].fr.p
    az = sum(zi * x for zi, x in zip(z, t["At"])) % p
    bz = sum(zi * x for zi, x in zip(z, t["Bt"])) % p
    cz = sum(zi * x for zi, x in zip(z, t["Ct"])) % p
    a_log = (t["alpha"] + az + r * t["delta"]) % p
    b_log = (t["beta"] + bz + s * t["delta"]) % p
    dinv = pow(t["delta"], -1, p)
    ni = r1cs.num_inputs
    l_part = sum(z[ni + j] * t["l_sc"][j] for j in range(r1cs.num_witness)) % p
    h_part = (az * bz - cz) % p * dinv % p
    c_log = (l_part + h_part + s * a_log + r * b_log - r * s % p * t["delta"]) % p
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    A = co.fixed_base_mul(g1, generator_limbs(g1), codec.ints_to_limbs([a_log]), 1)[0]
    B = co.fixed_base_mul(g2, generator_limbs(g2), codec.ints_to_limbs([b_log]), 1)[0]
    Cc = co.fixed_base_mul(g1, generator_limbs(g1), codec.ints_to_limbs([c_log]), 1)[0]
    return np.concatenate([A, B, Cc])


def make_gm17_instance(pairing_id, m, seed=20261017, bitlike=0.3, num_inputs=2, r1cs_z=None):
    """Satisfiable R1CS + assignment + GM17 key with known trapdoor (c_oracle.GM17_PK_FIELDS as numpy arrays);
    r1cs_z as in make_instance."""
    pairing = PAIRINGS[pairing_id]
    fp = pairing.fr
    p = fp.p
    r1cs, z = r1cs_z or o.synthetic_r1cs(fp, m, num_inputs=num_inputs, seed=seed, bitlike=bitlike)
    m = r1cs.num_constraints
    t = o.gm17_setup_scalars(pairing, r1cs, seed=seed + 100)
    g1, g2 = codec.G1_OF[pairing_id], codec.G2_OF[pairing_id]
    G1, G2 = generator_limbs(g1), generator_limbs(g2)
    sc = lambda vals: codec.ints_to_limbs(vals)
    gam, zt, ab = t["gamma"], t["zt"], (t["alpha"] + t["beta"]) % p
    pk = {
        "a_query": co.fixed_base_mul(g1, G1, sc(t["a_sc"])),
        "b_query": co.fixed_base_mul(g2, G2, sc(t["a_sc"])),
        "c_query_1": co.fixed_base_mul(g1, G1, sc(t["c1_sc"])),
        "c_query_2": co.fixed_base_mul(g1, G1, sc(t["c2_sc"])),
        "g_gamma2_z_t": co.fixed_base_mul(g1, G1, sc(t["gzt_sc"])),
        "g_gamma_z": co.fixed_base_mul(g1, G1, sc([gam * zt % p]))[0],
        "h_gamma_z": co.fixed_base_mul(g2, G2, sc([gam * zt % p]))[0],
        "g_ab_gamma_z": co.fixed_base_mul(g1, G1, sc([ab * gam % p * zt % p]))[0],
        "g_gamma2_z2": co.fixed_base_mul(g1, G1, sc([gam * gam % p * zt % p * zt % p]))[0],
    }
    A, B, C = r1cs_to_csr(r1cs)
    return dict(pairing=pairing_id, r1cs=r1cs, z_int=z, z=mont_limbs(z, fp), A=A, B=B, C=C, pk=pk, trapdoor=t,
                m=m, num_inputs=r1cs.num_inputs, num_witness=r1cs.num_witness)


def gm17_trapdoor_proof(inst, d1, d2, r):
    """The GM17 proof every correct prover must output for this randomness, from the verification equations in
    the exponent (oracle gm17_trapdoor_check): a = gamma (u + (r + d1) Z), b = a, c = (a + alpha)(a + beta) -
    alpha beta - gamma psi.  Affine limbs A || B || C."""
    t, r1cs, z = inst["trapdoor"], inst["r1cs"], inst["z_int"]
    pid = inst["pairing"]
    p = PAIRINGS[pid].fr.p
    full = o.sap_extend_assignment(r1cs, z)
    u = sum(x * y for x, y in zip(full, t["At"])) % p
    a_log = t["gamma"] * ((u + (r + d1) * t["zt"]) % p) % p
    psi = sum(z[i] * t["vk_sc"][i] for i in range(r1cs.num_inputs)) % p
    c_log = ((a_log + t["alpha"]) * (a_log + t["beta"]) - t["alpha"] * t["beta"] - t["gamma"] * psi) % p
    g1, g2 = codec.G1_OF[pid], codec.G2_OF[pid]
    A = co.fixed_base_mul(g1, generator_limbs(g1), codec.ints_to_limbs([a_log]), 1)[0]
    B = co.fixed_base_mul(g2, generator_limbs(g2), codec.ints_to_limbs([a_log]), 1)[0]
    Cc = co.fixed_base_mul(g1, generator_limbs(g1), codec.ints_to_limbs([c_log]), 1)[0]
    return np.concatenate([A, B, Cc])
