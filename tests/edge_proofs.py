"""Degenerate Groth16 / GM17 proofs with known discrete logs (test infrastructure).

Every constructor works in the exponent, from the trapdoor of an instance (synth.make_instance /
make_gm17_instance, or pcd_b200.synthetic's `expected_logs`), and solves for the randomness that hits a named
target: a proof point at infinity, a doubling or a cancellation in one addition of proof assembly, or a digit
pattern of the signed 4-bit recoding in the double-scalar chain (wec_multi_mul_kernel).  It returns the
randomness and asserts that the target holds for the discrete logs of every proof term, so a change of seed
cannot quietly turn an edge case into a generic one.  A target without a solution for an instance (a quadratic
without a root) moves to the next seed; nothing is skipped.

Groth16 (ark-groth16 prover.rs; the GPU assembles C the same way):
  a0 = alpha + sum z At, b0 = beta + sum z Bt, g_a = a0 + r delta (= A), g1_b = b0 + s delta (= B),
  T = s g_a + r g1_b (one double-scalar chain above 2^17 variables), l' = l - r s delta,
  C = h + l' + T, summed in this order.
GM17 (ark-gm17; gm17.cu): with a = r + d1, u = sum full At, Z = Z(tau), c = sum full Ct,
  A = B = gamma (u + a Z), C2' = 2 gamma^2 Z u, G' = gamma^2 ((u + d1 Z)^2 - c) (d2 cancels between h and its
  extra pair), C1' = gamma^2 sum_aux full Ct + (alpha + beta) gamma (sum_aux full At + a Z) + (r^2 + 2 r d1) gamma^2 Z^2,
  C = G' + C1' + [r] C2', summed in this order.
"""
import pairing_oracle as po
import pcd_oracle as o
import synth


# ---- field helpers ------------------------------------------------------------------------------------------------
def _inv(x, p):
    assert x % p, "division by zero while solving a target"
    return pow(x, -1, p)


def sqrt_mod(a, p):
    """a square root of a mod p (Tonelli-Shanks), or None"""
    a %= p
    if a == 0:
        return 0
    if pow(a, (p - 1) // 2, p) != 1:
        return None
    q, e = p - 1, 0
    while q % 2 == 0:
        q, e = q // 2, e + 1
    z = 2
    while pow(z, (p - 1) // 2, p) == 1:
        z += 1
    m, c, t, x = e, pow(z, q, p), pow(a, q, p), pow(a, (q + 1) // 2, p)
    while t != 1:
        i, t2 = 0, t
        while t2 != 1:
            t2, i = t2 * t2 % p, i + 1
        b = pow(c, 1 << (m - i - 1), p)
        m, c, t, x = i, b * b % p, t * b * b % p, x * b % p
    assert x * x % p == a
    return x


def quadratic_roots(a, b, c, p):
    """roots of a x^2 + b x + c mod p (a != 0)"""
    d = sqrt_mod(b * b - 4 * a * c, p)
    if d is None:
        return []
    i2a = _inv(2 * a, p)
    return sorted({(-b + d) * i2a % p, (-b - d) * i2a % p})


def generic(p, k=0):
    """two fixed generic scalars (the free variable of a target)"""
    return pow(3, 200 + k, p), pow(7, 190 + k, p)


def boundary_scalars(p):
    """scalars at the edges of the chain's signed 4-bit recoding (digits -7 .. 8, carry on 9 .. 15): 7, 8, 9, 15,
    16, 17, powers of two, every nibble 8 (no carry anywhere) and every nibble 9 (a carry into every window), as
    long as they stay below p"""
    vals = [7, 8, 9, 15, 16, 17, 1 << 64, 1 << 200, 1 << 296, 1 << 297]
    for nib in (8, 9, 15):
        k = (p.bit_length() + 3) // 4
        while int(("%x" % nib) * k, 16) >= p:
            k -= 1
        vals.append(int(("%x" % nib) * k, 16))
    return [v for v in vals if v < p]


# ---- Groth16 --------------------------------------------------------------------------------------------------------
def groth16_logs(inst):
    """the prover's term logs of a synth instance: dict(p, a0, b0, delta, h, l, hl)"""
    t, z, r1cs = inst["trapdoor"], inst["z_int"], inst["r1cs"]
    p = synth.PAIRINGS[inst["pairing"]].fr.p
    az = sum(zi * x for zi, x in zip(z, t["At"])) % p
    bz = sum(zi * x for zi, x in zip(z, t["Bt"])) % p
    cz = sum(zi * x for zi, x in zip(z, t["Ct"])) % p
    ni = r1cs.num_inputs
    l_part = sum(z[ni + j] * t["l_sc"][j] for j in range(r1cs.num_witness)) % p
    h_part = (az * bz - cz) % p * _inv(t["delta"], p) % p
    return dict(p=p, a0=(t["alpha"] + az) % p, b0=(t["beta"] + bz) % p, delta=t["delta"], h=h_part, l=l_part,
                hl=(h_part + l_part) % p)


def groth16_logs_from_expected(expected_logs, p):
    """the same from pcd_b200.synthetic's expected_logs(r, s) -> (A, B, C): a0, b0, delta and h + l only"""
    a0, b0, hl = expected_logs(0, 0)
    delta = (expected_logs(1, 0)[0] - a0) % p
    return dict(p=p, a0=a0, b0=b0, delta=delta, h=None, l=None, hl=hl)


def groth16_terms(L, r, s):
    """discrete logs of every term of proof assembly for randomness (r, s)"""
    p, d = L["p"], L["delta"]
    A = (L["a0"] + r * d) % p
    B = (L["b0"] + s * d) % p
    T = (s * A + r * B) % p
    rsd = r * s % p * d % p
    out = dict(A=A, B=B, sga=s * A % p, rg1b=r * B % p, T=T, hl_prime=(L["hl"] - rsd) % p,
               C=(L["hl"] - rsd + T) % p)
    if L["h"] is not None:
        out.update(h=L["h"], lp=(L["l"] - rsd) % p)
    return out


def groth16_targets(L):
    """[(name, r, s)]: every Groth16 target the logs L allow (h and l separately: synth instances only).  Each one
    is asserted in the exponent."""
    p, a0, b0, d, hl = L["p"], L["a0"], L["b0"], L["delta"], L["hl"]
    rg, sg = generic(p)
    out = []

    def add(name, r, s, check):
        r, s = r % p, s % p
        e = groth16_terms(L, r, s)
        assert check(e), (name, r, s)
        out.append((name, r, s))

    add("r=s=0", 0, 0, lambda e: True)
    add("r=0", 0, sg, lambda e: e["rg1b"] == 0)
    add("s=0", rg, 0, lambda e: e["sga"] == 0)
    add("r=s=1", 1, 1, lambda e: True)
    add("r=s=p-1", p - 1, p - 1, lambda e: True)
    add("r=2,s=p-2", 2, p - 2, lambda e: True)
    bnd = boundary_scalars(p)
    for i, v in enumerate(bnd):
        add("chain r=%#x" % v, v, bnd[-1 - i], lambda e: True)
    ra = -a0 * _inv(d, p)
    sb = -b0 * _inv(d, p)
    add("A=O", ra, sg, lambda e: e["A"] == 0 and e["B"] and e["C"])
    add("B=O", rg, sb, lambda e: e["B"] == 0 and e["A"] and e["C"])
    add("A=B=O", ra, sb, lambda e: e["A"] == 0 and e["B"] == 0 and e["T"] == 0)
    # C = hl - r s delta + s a0 + r b0 + 2 r s delta = hl + r b0 + s (a0 + r delta)
    add("C=O", rg, (-hl - rg * b0) * _inv(a0 + rg * d, p), lambda e: e["C"] == 0 and e["A"] and e["B"])
    # T = h + l': s a0 + r b0 + 2 r s delta = hl - r s delta
    add("last addition doubles", rg, (hl - rg * b0) * _inv(a0 + 3 * rg * d, p),
        lambda e: e["T"] == e["hl_prime"] and e["T"])
    # h + l' + s g_a = r g1_b: the last addition of the four-term sum of small proofs doubles
    add("small-path last addition doubles", rg, (rg * b0 - hl) * _inv(a0 - rg * d, p),
        lambda e: (e["hl_prime"] + e["sga"]) % p == e["rg1b"] and e["rg1b"])
    add("chain join doubles", rg, rg * b0 * _inv(a0, p), lambda e: e["sga"] == e["rg1b"] and e["sga"])
    add("chain join cancels", rg, -rg * b0 * _inv(a0 + 2 * rg * d, p),
        lambda e: (e["sga"] + e["rg1b"]) % p == 0 and e["sga"] and e["T"] == 0)
    if L["h"] is not None:
        add("first addition doubles", rg, (L["l"] - L["h"]) * _inv(d * rg, p), lambda e: e["lp"] == e["h"] and e["h"])
        add("first addition cancels", rg, (L["l"] + L["h"]) * _inv(d * rg, p),
            lambda e: (e["lp"] + e["h"]) % p == 0 and e["h"])
    return out


# ---- GM17 -----------------------------------------------------------------------------------------------------------
def gm17_logs(inst):
    """the prover's term logs of a synth GM17 instance"""
    t, r1cs, z = inst["trapdoor"], inst["r1cs"], inst["z_int"]
    p = synth.PAIRINGS[inst["pairing"]].fr.p
    ni = r1cs.num_inputs
    full = o.sap_extend_assignment(r1cs, z)
    u = sum(x * y for x, y in zip(full, t["At"])) % p
    c = sum(x * y for x, y in zip(full, t["Ct"])) % p
    aux = sum(full[ni + j] * v for j, v in enumerate(t["c1_sc"])) % p
    psi = sum(z[i] * t["vk_sc"][i] for i in range(ni)) % p
    return dict(p=p, alpha=t["alpha"], beta=t["beta"], gamma=t["gamma"], Z=t["zt"], u=u, c=c, aux=aux, psi=psi)


def gm17_terms(L, d1, d2, r):
    p, g, Z, u = L["p"], L["gamma"], L["Z"], L["u"]
    a = (r + d1) % p
    A = g * (u + a * Z) % p
    g2 = g * g % p
    Gp = g2 * ((u + d1 * Z) ** 2 - L["c"]) % p
    C1 = (L["aux"] + (r * r + 2 * r * d1) * g2 * Z * Z + a * (L["alpha"] + L["beta"]) * g * Z) % p
    rC2 = 2 * r * g2 * Z * u % p
    C = ((A + L["alpha"]) * (A + L["beta"]) - L["alpha"] * L["beta"] - g * L["psi"]) % p
    assert (Gp + C1 + rC2) % p == C, "the term decomposition disagrees with the verification equation"
    return dict(A=A, Gp=Gp, C1=C1, rC2=rC2, C=C)


def gm17_c_of(L, a):
    """C's log as a function of a = r + d1 alone"""
    p = L["p"]
    A = L["gamma"] * (L["u"] + a * L["Z"]) % p
    return ((A + L["alpha"]) * (A + L["beta"]) - L["alpha"] * L["beta"] - L["gamma"] * L["psi"]) % p


def gm17_targets(L):
    """[(name, d1, d2, r)], each asserted in the exponent.  d2 does not reach the proof (it cancels between h and
    the extra pair of the g_gamma2_z_t MSM), so the assembly targets are solved through r and d1."""
    p, g, Z, u = L["p"], L["gamma"], L["Z"], L["u"]
    g2 = g * g % p
    rg, dg = generic(p)
    out = []

    def add(name, d1, d2, r, check):
        d1, d2, r = d1 % p, d2 % p, r % p
        e = gm17_terms(L, d1, d2, r)
        assert check(e), (name, d1, d2, r)
        out.append((name, d1, d2, r))

    add("d1=d2=r=0", 0, 0, 0, lambda e: True)
    add("r=0", dg, rg, 0, lambda e: e["rC2"] == 0)
    add("d2=0", dg, 0, rg, lambda e: True)
    add("d1=d2=r=1", 1, 1, 1, lambda e: True)
    add("d1=d2=r=p-1", p - 1, p - 1, p - 1, lambda e: True)
    for v in boundary_scalars(p):
        add("chain r=%#x" % v, dg, rg, v, lambda e: e["rC2"])
    a_inf = -u * _inv(Z, p)
    add("A=B=O", a_inf - rg, dg, rg, lambda e: e["A"] == 0 and e["C"])
    roots = quadratic_roots(1, L["alpha"] + L["beta"], -g * L["psi"], p)  # C = A^2 + (alpha + beta) A - gamma psi
    assert roots, "no root: the instance must move to the next seed"
    a_c = (roots[0] * _inv(g, p) - u) * _inv(Z, p)
    add("C=O", a_c - rg, dg, rg, lambda e: e["C"] == 0 and e["A"])
    a = dg  # a generic r + d1; r solved from it
    # G' + C1' = [r] C2'  <=>  C = 2 [r] C2' = 4 r gamma^2 Z u
    r_last = gm17_c_of(L, a) * _inv(4 * g2 * Z * u, p)
    add("last addition doubles", a - r_last, dg, r_last, lambda e: (e["Gp"] + e["C1"]) % p == e["rC2"] and e["rC2"])
    # G' + C1' = O  <=>  C = [r] C2'
    r_fc = gm17_c_of(L, a) * _inv(2 * g2 * Z * u, p)
    add("first addition cancels", a - r_fc, dg, r_fc, lambda e: (e["Gp"] + e["C1"]) % p == 0 and e["Gp"])
    # G' = C1'  <=>  2 G' + [r] C2' = C, quadratic in r for a fixed a: G' = gamma^2 ((w - r Z)^2 - c), w = u + a Z
    for k in range(64):
        a = (dg + k) % p
        w = (u + a * Z) % p
        rts = quadratic_roots(2 * g2 * Z * Z, -4 * g2 * w * Z + 2 * g2 * Z * u, 2 * g2 * (w * w - L["c"]) - gm17_c_of(L, a), p)
        if rts:
            break
    assert rts, "no root for 64 values of r + d1"
    add("first addition doubles", a - rts[0], dg, rts[0], lambda e: e["Gp"] == e["C1"] and e["Gp"])
    return out


def gm17_a_inf_from_expected(expected_logs, p):
    """r + d1 making A = B = O, from pcd_b200.synthetic's GM17 expected_logs alone"""
    a0 = expected_logs(0, 0, 0)[0]
    step = (expected_logs(0, 0, 1)[0] - a0) % p  # gamma Z
    return -a0 * _inv(step, p) % p


# ---- instances ------------------------------------------------------------------------------------------------------
def identity_r1cs(pairing_id, num_witness, num_inputs=2):
    """one constraint x_i * 1 = x_i per variable: every assignment satisfies it"""
    fp = synth.PAIRINGS[pairing_id].fr
    nv = num_inputs + num_witness
    return o.R1CS(fp, num_inputs, num_witness, [[(1, i)] for i in range(nv)], [[(1, 0)] for _ in range(nv)],
                  [[(1, i)] for i in range(nv)])


def identity_assignments(pairing_id, nv):
    """{name: z} with z[0] = 1 and every other variable at one value"""
    p = synth.PAIRINGS[pairing_id].fr.p
    vals = {"zeros": 0, "ones": 1, "p-1": p - 1, "repeated": pow(5, 111, p)}
    return {k: [1] + [v] * (nv - 1) for k, v in vals.items()}


def make_instance(pairing_id, m, seed, gm17=False, num_inputs=3, bitlike=0.4):
    """a synth instance on which every target of the scheme has a solution (the next seed otherwise)"""
    for k in range(16):
        mk = synth.make_gm17_instance if gm17 else synth.make_instance
        inst = mk(pairing_id, m, seed=seed + k, bitlike=bitlike, num_inputs=num_inputs)
        try:
            targets = gm17_targets(gm17_logs(inst)) if gm17 else groth16_targets(groth16_logs(inst))
        except AssertionError as e:
            if "no root" in str(e) or "division by zero" in str(e):
                continue
            raise
        return inst, targets
    raise AssertionError("no seed gives every target")


def identity_instance(pairing_id, z, gm17=False, num_witness=30, num_inputs=2, seed=4321):
    r1cs = identity_r1cs(pairing_id, num_witness, num_inputs)
    assert r1cs.is_satisfied(z)
    mk = synth.make_gm17_instance if gm17 else synth.make_instance
    return mk(pairing_id, r1cs.num_constraints, seed=seed, r1cs_z=(r1cs, z))


# ---- simulated proofs for the verifier --------------------------------------------------------------------------------
def _combination_zero(coeffs, x_rest, p):
    """x_1 such that coeffs[0] + x_1 coeffs[1] + sum x_rest coeffs[2:] = 0"""
    s = (coeffs[0] + sum(x * c for x, c in zip(x_rest, coeffs[2:]))) % p
    return -s * _inv(coeffs[1], p) % p


def groth16_simulated_edges(inst):
    """[(name, x, a, b, c)]: valid degenerate proofs (logs) for inst's verifying key (verify_helpers.groth16_vk)"""
    t, ni = inst["trapdoor"], inst["num_inputs"]
    p = synth.PAIRINGS[inst["pairing"]].fr.p
    assert ni >= 3
    x0 = list(inst["z_int"][1:ni])
    rg, sg = generic(p, 5)
    abc = [(t["beta"] * t["At"][j] + t["alpha"] * t["Bt"][j] + t["Ct"][j]) % p for j in range(ni)]
    ab = (t["alpha"] * t["beta"] + sum(xi * c for xi, c in zip([1] + x0, abc))) % p  # c = 0 <=> a b = ab
    cases = [("a=0", x0, 0, sg), ("b=0", x0, rg, 0), ("a=b=0", x0, 0, 0), ("c=0", x0, rg, ab * _inv(rg, p)),
             ("x=0", [0] * (ni - 1), rg, sg), ("x=1", [1] * (ni - 1), rg, sg), ("x=p-1", [p - 1] * (ni - 1), rg, sg),
             ("x mixed 0 1 p-1", ([0, 1, p - 1] * ni)[:ni - 1], rg, sg)]
    x_ic = [_combination_zero(abc, [7] * (ni - 2), p)] + [7] * (ni - 2)
    cases.append(("input combination O", x_ic, rg, sg))
    out = []
    for name, x, a, b in cases:
        a_, b_, c = po.groth16_simulated_logs(t, x, a, b, p)
        if name == "input combination O":
            assert sum(xi * cc for xi, cc in zip([1] + x, abc)) % p == 0
        if name == "c=0":
            assert c == 0
        out.append((name, x, a_, b_, c))
    return out


def gm17_simulated_edges(inst):
    """[(name, x, a, c)] (B = [a] H): valid degenerate GM17 proofs for inst's verifying key"""
    t, ni = inst["trapdoor"], inst["num_inputs"]
    p = synth.PAIRINGS[inst["pairing"]].fr.p
    assert ni >= 3
    x0 = list(inst["z_int"][1:ni])
    ag = generic(p, 9)[0]
    cases = [("a=0", x0, 0), ("A+g_alpha=O", x0, -t["alpha"] % p), ("B+h_beta=O", x0, -t["beta"] % p),
             ("x=0", [0] * (ni - 1), ag), ("x=1", [1] * (ni - 1), ag), ("x=p-1", [p - 1] * (ni - 1), ag),
             ("input combination O", [_combination_zero(t["vk_sc"], [7] * (ni - 2), p)] + [7] * (ni - 2), ag)]
    roots = quadratic_roots(1, t["alpha"] + t["beta"], -t["gamma"] * (
        t["vk_sc"][0] + sum(xi * v for xi, v in zip(x0, t["vk_sc"][1:]))), p)
    if roots:
        cases.append(("c=0", x0, roots[0]))
    out = []
    for name, x, a in cases:
        a_, c = po.gm17_simulated_logs(t, x, a, p)
        if name == "input combination O":
            assert (t["vk_sc"][0] + sum(xi * v for xi, v in zip(x, t["vk_sc"][1:]))) % p == 0
        if name == "c=0":
            assert c == 0
        out.append((name, x, a_, c))
    return out


def key_with_zero_constant(inst, gm17=False):
    """a copy of inst's trapdoor whose verifying key has gamma_abc_g1[0] = O (GM17: query[0] = O): the constant's C
    polynomial is changed so that its combination vanishes; the simulators then give valid proofs for that key"""
    t = dict(inst["trapdoor"])
    p = synth.PAIRINGS[inst["pairing"]].fr.p
    if gm17:
        t["vk_sc"] = [0] + list(t["vk_sc"][1:])
    else:
        Ct = list(t["Ct"])
        Ct[0] = -(t["beta"] * t["At"][0] + t["alpha"] * t["Bt"][0]) % p
        t["Ct"] = Ct
    return dict(inst, trapdoor=t)
