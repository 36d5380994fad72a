"""Host-side mirror of the reference's SNARK interface for the Groth16 proving path.

In the reference, `ECCyclePCD::prove` calls `IC::MainSNARK::prove(&pk.main_pk, main_circuit, rng)` and
`IC::HelpSNARK::prove(&pk.help_pk, help_circuit, rng)` (/root/reference/src/ec_cycle_pcd/mod.rs:171,179)
with `MainSNARK = Groth16<MNT4_298>` / `HelpSNARK = Groth16<MNT6_298>`
(/root/reference/tests/mnt4_groth16.rs:23-30).  Constraint synthesis stays on the CPU side of the
boundary; what crosses it is ark-relations' `ConstraintMatrices` (CSR rows of (coeff, col)), the
full assignment z = instance || witness, the `ProvingKey` and the two field elements r, s drawn by
the caller's RNG (r first, then s: ark-groth16 prover.rs `create_random_proof`).  Names and argument
meaning follow ark-groth16 / ark-snark; everything numeric happens in libpcdgpu.so.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Callable, Optional, Tuple

import numpy as np

from . import lib as L

CSR = Tuple[np.ndarray, np.ndarray, np.ndarray]  # (row_ptr u32[m+1], col u32[nnz], val u64[nnz,5] Montgomery)


def _scalar(a) -> np.ndarray:
    """one scalar as five u64 limbs (the C side reads exactly 40 bytes)"""
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1)
    if a.size != 5:
        raise ValueError("a scalar is five 64-bit limbs, got %d" % a.size)
    return a


@dataclass
class ConstraintMatrices:
    """ark-relations `ConstraintMatrices`: instance variables first (column 0 is the constant 1)."""

    pairing: int
    num_instance_variables: int
    num_witness_variables: int
    a: CSR
    b: CSR
    c: CSR

    @property
    def num_constraints(self) -> int:
        return len(self.a[0]) - 1


@dataclass
class ProvingKey:
    """ark-groth16 `ProvingKey<E>` (vk.alpha_g1, vk.beta_g2, vk.delta_g2 flattened in)."""

    pairing: int
    alpha_g1: np.ndarray
    beta_g1: np.ndarray
    delta_g1: np.ndarray
    beta_g2: np.ndarray
    delta_g2: np.ndarray
    a_query: np.ndarray
    b_g1_query: np.ndarray
    b_g2_query: np.ndarray
    h_query: np.ndarray
    l_query: np.ndarray


@dataclass
class Proof:
    """ark-groth16 `Proof<E>`: a in G1, b in G2, c in G1 (affine limbs, Montgomery coordinates)."""

    pairing: int
    a: np.ndarray
    b: np.ndarray
    c: np.ndarray

    def affine_limbs(self) -> np.ndarray:
        return np.concatenate([self.a, self.b, self.c])


class ProverIndex:
    """Device-resident proving key + constraint matrices (uploaded once per circuit shape)."""

    def __init__(self, ctx: L.Context, pk: ProvingKey, cm: ConstraintMatrices, precompute: bool = False,
                 sharded: bool = False):
        """sharded: the context has a communicator (Context.comm_init): upload only this rank's slice of every query
        (pcdgpu_pk_upload_sharded); proofs then go through Groth16.create_proof_sharded on every rank."""
        self.sharded = sharded
        if pk.pairing != cm.pairing:
            raise ValueError("proving key and constraint matrices are over different pairings")
        self.ctx, self.pairing = ctx, pk.pairing
        self.num_inputs = cm.num_instance_variables
        self.num_witness = cm.num_witness_variables
        self.num_vars = self.num_inputs + self.num_witness
        g1, g2 = L.G1_OF[pk.pairing], L.G2_OF[pk.pairing]
        lib = ctx.lib
        keep = []

        def arr(a, dt, width=None):
            a = np.ascontiguousarray(a, dtype=dt)
            if width:
                a = a.reshape(-1, width)
            keep.append(a)
            return ctypes.c_void_p(a.ctypes.data)

        m = cm.num_constraints
        args = []
        for (ptr, col, val) in (cm.a, cm.b, cm.c):
            args += [arr(ptr, np.uint32), arr(col, np.uint32), arr(val, np.uint64)]
        h = ctypes.c_void_p()
        ctx._check(lib.pcdgpu_r1cs_upload(ctx.h, pk.pairing, m, self.num_inputs, self.num_witness, *args,
                                          ctypes.byref(h)))
        self.r1cs = h
        self.domain_size = lib.pcdgpu_r1cs_domain_size(h)
        a_q = np.ascontiguousarray(pk.a_query, dtype=np.uint64).reshape(-1, L.AFFINE_LIMBS[g1])
        if a_q.shape[0] != self.num_vars:
            raise ValueError("a_query has %d points for %d variables" % (a_q.shape[0], self.num_vars))
        h_q = np.ascontiguousarray(pk.h_query, dtype=np.uint64).reshape(-1, L.AFFINE_LIMBS[g1])
        # every query goes to C as a raw pointer and is read num_vars (num_witness) points deep: check the lengths here
        for name, q, limbs_, want in (("b_g1_query", pk.b_g1_query, L.AFFINE_LIMBS[g1], self.num_vars),
                                      ("b_g2_query", pk.b_g2_query, L.AFFINE_LIMBS[g2], self.num_vars),
                                      ("l_query", pk.l_query, L.AFFINE_LIMBS[g1], self.num_witness)):
            got = np.asarray(q).size // limbs_ if np.asarray(q).size % limbs_ == 0 else -1
            if got != want:
                raise ValueError("%s has %d points, expected %d" % (name, got, want))
        for name, pt, limbs_ in (("alpha_g1", pk.alpha_g1, L.AFFINE_LIMBS[g1]), ("beta_g1", pk.beta_g1, L.AFFINE_LIMBS[g1]),
                                 ("delta_g1", pk.delta_g1, L.AFFINE_LIMBS[g1]), ("beta_g2", pk.beta_g2, L.AFFINE_LIMBS[g2]),
                                 ("delta_g2", pk.delta_g2, L.AFFINE_LIMBS[g2])):
            if np.asarray(pt).size != limbs_:
                raise ValueError("%s is not one affine point" % name)
        pkh = ctypes.c_void_p()
        ctx._check((lib.pcdgpu_pk_upload_sharded if sharded else lib.pcdgpu_pk_upload)(
            ctx.h, pk.pairing, self.num_vars, self.num_inputs, h_q.shape[0],
            arr(pk.alpha_g1, np.uint64), arr(pk.beta_g1, np.uint64), arr(pk.delta_g1, np.uint64),
            arr(pk.beta_g2, np.uint64), arr(pk.delta_g2, np.uint64), arr(a_q, np.uint64),
            arr(pk.b_g1_query, np.uint64), arr(pk.b_g2_query, np.uint64), arr(h_q, np.uint64),
            arr(pk.l_query, np.uint64), int(precompute), ctypes.byref(pkh)))
        self.pk = pkh

    def close(self):
        if getattr(self, "pk", None) and self.ctx.h:
            self.ctx.lib.pcdgpu_pk_free(self.pk)
            self.ctx.lib.pcdgpu_r1cs_free(self.r1cs)
        self.pk = None
        self.r1cs = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- verification (ark-groth16 / ark-gm17 verifier.rs) ------------------------------------------------------------
@dataclass
class VerifyingKey:
    """ark-groth16 `VerifyingKey<E>`; gamma_abc_g1 has one point per public input plus the constant's."""

    pairing: int
    alpha_g1: np.ndarray
    beta_g2: np.ndarray
    gamma_g2: np.ndarray
    delta_g2: np.ndarray
    gamma_abc_g1: np.ndarray


@dataclass
class GM17VerifyingKey:
    """ark-gm17 `VerifyingKey<E>`; query has one point per public input plus the constant's."""

    pairing: int
    h_g2: np.ndarray
    g_alpha_g1: np.ndarray
    h_beta_g2: np.ndarray
    g_gamma_g1: np.ndarray
    h_gamma_g2: np.ndarray
    query: np.ndarray


class PreparedVerifyingKey:
    """A verifying key processed on the GPU (pcdgpu_groth16_pvk / pcdgpu_gm17_pvk): the line coefficients of its G2
    points and e(alpha, beta) stay in device memory."""

    def __init__(self, ctx: L.Context, pairing: int, gm17: bool, handle, num_inputs: int):
        self.ctx, self.pairing, self.gm17, self.h, self.num_inputs = ctx, pairing, gm17, handle, num_inputs

    def close(self):
        if getattr(self, "h", None):
            free = self.ctx.lib.pcdgpu_gm17_pvk_free if self.gm17 else self.ctx.lib.pcdgpu_groth16_pvk_free
            free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _points(a, curve) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, L.AFFINE_LIMBS[curve])


def _verify_batch(ctx: L.Context, pvk: PreparedVerifyingKey, gm17: bool, xs, proofs, serialized=False) -> np.ndarray:
    if pvk.gm17 != gm17:
        raise ValueError("the prepared key belongs to the other proof system")
    width = L.AFFINE_LIMBS[L.G1_OF[pvk.pairing]] * 2 + L.AFFINE_LIMBS[L.G2_OF[pvk.pairing]]
    if serialized:
        pr = _proof_rows(pvk.pairing, proofs)
    elif isinstance(proofs, np.ndarray):
        pr = np.ascontiguousarray(proofs, dtype=np.uint64).reshape(-1, width)
    else:
        pr = np.ascontiguousarray([p.affine_limbs() for p in proofs], dtype=np.uint64).reshape(-1, width)
    n = pr.shape[0]
    ni = pvk.num_inputs - 1
    x = np.ascontiguousarray(xs, dtype=np.uint64).reshape(n, -1) if n else np.zeros((0, 5), dtype=np.uint64)
    if n and x.shape[1] != 5 * ni:
        # ark: SynthesisError::MalformedVerifyingKey for a public-input count the key does not have
        raise L.PcdGpuError(-1, "the key takes %d public inputs, got %d" % (ni, x.shape[1] // 5))
    ok = np.zeros(n, dtype=np.uint8)
    if n == 0:
        return ok.astype(bool)
    lib = ctx.lib
    if serialized:
        fn = lib.pcdgpu_gm17_verify_batch_serialized if gm17 else lib.pcdgpu_groth16_verify_batch_serialized
    else:
        fn = lib.pcdgpu_gm17_verify_batch if gm17 else lib.pcdgpu_groth16_verify_batch
    ctx._check(fn(ctx.h, pvk.h, L._p(pr), L._p(x) if ni else None, n, L._p(ok)))
    return ok.astype(bool)


def _proof_rows(pairing: int, data) -> np.ndarray:
    """compressed proofs as one (n, PROOF_BYTES[pairing]) uint8 array: a 2-D array, or a sequence of bytes objects"""
    width = L.PROOF_BYTES[pairing]
    if isinstance(data, np.ndarray):
        rows = np.ascontiguousarray(data, dtype=np.uint8)
        if rows.ndim != 2 or rows.shape[1] != width:
            raise ValueError("compressed proofs over this pairing are rows of %d bytes, got shape %s" % (
                width, rows.shape))
        return rows
    data = [bytes(b) for b in data]
    for b in data:
        if len(b) != width:
            raise ValueError("a compressed proof over this pairing is %d bytes, got %d" % (width, len(b)))
    return np.frombuffer(b"".join(data), dtype=np.uint8).reshape(-1, width).copy()


def _process_vk(ctx: L.Context, pairing: int, gm17: bool, vk) -> PreparedVerifyingKey:
    """ark-groth16 / ark-gm17 prepare_verifying_key, on the GPU (a key point off its curve: PcdGpuError -1)"""
    g1, g2 = L.G1_OF[pairing], L.G2_OF[pairing]
    if gm17:
        pts = [_points(vk.h_g2, g2), _points(vk.g_alpha_g1, g1), _points(vk.h_beta_g2, g2),
               _points(vk.g_gamma_g1, g1), _points(vk.h_gamma_g2, g2), _points(vk.query, g1)]
        create = ctx.lib.pcdgpu_gm17_pvk_create
    else:
        pts = [_points(vk.alpha_g1, g1), _points(vk.beta_g2, g2), _points(vk.gamma_g2, g2), _points(vk.delta_g2, g2),
               _points(vk.gamma_abc_g1, g1)]
        create = ctx.lib.pcdgpu_groth16_pvk_create
    if vk.pairing != pairing:
        raise ValueError("verifying key of another pairing")
    h = ctypes.c_void_p()
    ctx._check(create(ctx.h, pairing, *[L._p(a) for a in pts], pts[-1].shape[0], ctypes.byref(h)))
    return PreparedVerifyingKey(ctx, pairing, gm17, h, pts[-1].shape[0])


class _Verifier:
    """verify / verify_with_processed_vk / verify_batch shared by Groth16 and GM17 (GM17 sets _GM17)"""

    _GM17 = False

    def process_vk(self, vk) -> PreparedVerifyingKey:
        return _process_vk(self.ctx, self.pairing, self._GM17, vk)

    def verify_batch(self, pvk: PreparedVerifyingKey, xs, proofs) -> np.ndarray:
        """one verdict per proof: xs = n x (num_inputs - 1) Montgomery Fr elements, proofs = Proof objects or an
        (n, A || B || C) limb array"""
        return _verify_batch(self.ctx, pvk, self._GM17, xs, proofs)

    def verify_with_processed_vk(self, pvk: PreparedVerifyingKey, x, proof: Proof) -> bool:
        x = np.ascontiguousarray(x, dtype=np.uint64).reshape(1, -1)
        return bool(_verify_batch(self.ctx, pvk, self._GM17, x, [proof])[0])

    def verify(self, vk, x, proof: Proof) -> bool:
        pvk = self.process_vk(vk)
        try:
            return self.verify_with_processed_vk(pvk, x, proof)
        finally:
            pvk.close()

    def deserialize_batch(self, data):
        """ark-serialize CanonicalDeserialize (checked) of n compressed proofs, on the GPU: data = an (n, 152 / 190)
        uint8 array or a sequence of bytes.  Returns ((n, A || B || C) affine limbs, zero rows for invalid proofs;
        (n,) bool mask of valid proofs)."""
        rows = _proof_rows(self.pairing, data)
        return self.ctx.deserialize_proofs(self.pairing, rows)

    def deserialize(self, data: bytes) -> Proof:
        """one compressed proof -> Proof; ValueError when the bytes are not a valid proof (ark's
        SerializationError::InvalidData): a coordinate >= p, both flags, no square root, B outside the subgroup"""
        limbs, ok = self.deserialize_batch([data])
        if not ok[0]:
            raise ValueError("invalid proof encoding")
        g1, g2 = L.AFFINE_LIMBS[L.G1_OF[self.pairing]], L.AFFINE_LIMBS[L.G2_OF[self.pairing]]
        row = limbs[0]
        return Proof(self.pairing, row[:g1].copy(), row[g1:g1 + g2].copy(), row[g1 + g2:].copy())

    def verify_batch_serialized(self, pvk: PreparedVerifyingKey, xs, data) -> np.ndarray:
        """verify_batch for compressed proofs (deserialize_batch's input): one verdict per proof, true when the bytes
        deserialize to a valid proof and it verifies; the proofs stay on the GPU in between"""
        return _verify_batch(self.ctx, pvk, self._GM17, xs, data, serialized=True)


class Groth16(_Verifier):
    """`Groth16<E>` as the reference binds it (SNARK + CircuitSpecificSetupSNARK): `prove` and its building
    blocks, `process_vk` and verification run on the GPU.  Setup stays with the CPU implementation on the
    Rust side of the boundary (SURVEY.md 3.3, 3.4)."""

    def __init__(self, ctx: L.Context, pairing: int):
        self.ctx, self.pairing = ctx, pairing

    def index(self, pk: ProvingKey, cm: ConstraintMatrices, precompute: bool = False, sharded: bool = False) -> ProverIndex:
        return ProverIndex(self.ctx, pk, cm, precompute, sharded)

    def witness_map(self, index: ProverIndex, z: np.ndarray) -> np.ndarray:
        """R1CStoQAP::witness_map: the n coefficients of h."""
        z = np.ascontiguousarray(z, dtype=np.uint64).reshape(-1, 5)
        if z.shape[0] != index.num_vars:
            raise ValueError("assignment has %d elements for %d variables" % (z.shape[0], index.num_vars))
        h = np.zeros((index.domain_size, 5), dtype=np.uint64)
        self.ctx._check(self.ctx.lib.pcdgpu_witness_map(self.ctx.h, index.r1cs, ctypes.c_void_p(z.ctypes.data),
                                                        ctypes.c_void_p(h.ctypes.data)))
        return h

    def create_proof_with_reduction(self, index: ProverIndex, z: np.ndarray, r: np.ndarray, s: np.ndarray) -> Proof:
        """ark-groth16 `create_proof_with_reduction(circuit, pk, r, s)`; r, s plain-integer limbs."""
        z = np.ascontiguousarray(z, dtype=np.uint64).reshape(-1, 5)
        if z.shape[0] != index.num_vars:
            raise ValueError("assignment has %d elements for %d variables" % (z.shape[0], index.num_vars))
        r = _scalar(r)
        s = _scalar(s)
        g1, g2 = L.AFFINE_LIMBS[L.G1_OF[self.pairing]], L.AFFINE_LIMBS[L.G2_OF[self.pairing]]
        out = np.zeros(2 * g1 + g2, dtype=np.uint64)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        self.ctx._check(self.ctx.lib.pcdgpu_groth16_prove(self.ctx.h, index.pk, index.r1cs, vp(z), vp(r), vp(s),
                                                          vp(out)))
        return Proof(self.pairing, out[:g1].copy(), out[g1:g1 + g2].copy(), out[g1 + g2:].copy())

    def create_proof_dev(self, index: ProverIndex, d_z: int, r: np.ndarray, s: np.ndarray) -> Proof:
        """same with the assignment already resident on the GPU (device pointer)."""
        r = _scalar(r)
        s = _scalar(s)
        g1, g2 = L.AFFINE_LIMBS[L.G1_OF[self.pairing]], L.AFFINE_LIMBS[L.G2_OF[self.pairing]]
        out = np.zeros(2 * g1 + g2, dtype=np.uint64)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        self.ctx._check(self.ctx.lib.pcdgpu_groth16_prove_dev(self.ctx.h, index.pk, index.r1cs, ctypes.c_void_p(d_z),
                                                              vp(r), vp(s), vp(out)))
        return Proof(self.pairing, out[:g1].copy(), out[g1:g1 + g2].copy(), out[g1 + g2:].copy())

    def create_proof_sharded_dev(self, index: ProverIndex, d_z: int, r: np.ndarray, s: np.ndarray) -> Proof:
        """One proof over the GPUs of the context's communicator (collective: every rank calls it with the same
        inputs over its slice of the key, index = g.index(..., sharded=True); every rank receives the proof)."""
        r = _scalar(r)
        s = _scalar(s)
        g1, g2 = L.AFFINE_LIMBS[L.G1_OF[self.pairing]], L.AFFINE_LIMBS[L.G2_OF[self.pairing]]
        out = np.zeros(2 * g1 + g2, dtype=np.uint64)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        self.ctx._check(self.ctx.lib.pcdgpu_groth16_prove_sharded_dev(self.ctx.h, index.pk, index.r1cs,
                                                                      ctypes.c_void_p(d_z), vp(r), vp(s), vp(out)))
        return Proof(self.pairing, out[:g1].copy(), out[g1:g1 + g2].copy(), out[g1 + g2:].copy())

    def prove(self, index: ProverIndex, z: np.ndarray, rng: Callable[[int], np.ndarray]) -> Proof:
        """`SNARK::prove(pk, circuit, rng)`: draws r, then s (`create_random_proof`), then proves.
        rng(field_id) returns one uniformly random scalar as five plain-integer u64 limbs."""
        f = L.SCALAR_FIELD_OF[self.pairing]
        r = rng(f)
        s = rng(f)
        return self.create_proof_with_reduction(index, z, r, s)

    def serialize(self, proof: Proof) -> bytes:
        """ark-serialize canonical (compressed) bytes: 152 B (MNT4-298) / 190 B (MNT6-298)."""
        return self.ctx.serialize_proof(self.pairing, proof.affine_limbs())


# ---- GM17 ------------------------------------------------------------------------------------------------
@dataclass
class GM17ProvingKey:
    """ark-gm17 `ProvingKey<E>` (the fields the prover reads; vk is not needed to prove)."""

    pairing: int
    a_query: np.ndarray        # G1, one per SAP variable
    b_query: np.ndarray        # G2, one per SAP variable
    c_query_1: np.ndarray      # G1, non-input SAP variables
    c_query_2: np.ndarray      # G1, one per SAP variable
    g_gamma_z: np.ndarray      # G1
    h_gamma_z: np.ndarray      # G2
    g_ab_gamma_z: np.ndarray   # G1
    g_gamma2_z2: np.ndarray    # G1
    g_gamma2_z_t: np.ndarray   # G1, SAP domain size + 1


class GM17ProverIndex:
    """Device-resident GM17 proving key + the R1CS matrices the SAP is derived from."""

    def __init__(self, ctx: L.Context, pk: GM17ProvingKey, cm: ConstraintMatrices, precompute: bool = False):
        if pk.pairing != cm.pairing:
            raise ValueError("proving key and constraint matrices are over different pairings")
        self.ctx, self.pairing = ctx, pk.pairing
        self.num_inputs = cm.num_instance_variables
        self.num_witness = cm.num_witness_variables
        self.num_vars = self.num_inputs + self.num_witness
        m = cm.num_constraints
        self.num_sap_vars = self.num_vars + m + self.num_inputs - 1
        g1 = L.G1_OF[pk.pairing]
        lib = ctx.lib
        keep = []

        def arr(a, dt, width=None):
            a = np.ascontiguousarray(a, dtype=dt)
            if width:
                a = a.reshape(-1, width)
            keep.append(a)
            return ctypes.c_void_p(a.ctypes.data)

        args = []
        for (ptr, col, val) in (cm.a, cm.b, cm.c):
            args += [arr(ptr, np.uint32), arr(col, np.uint32), arr(val, np.uint64)]
        h = ctypes.c_void_p()
        ctx._check(lib.pcdgpu_r1cs_upload(ctx.h, pk.pairing, m, self.num_inputs, self.num_witness, *args,
                                          ctypes.byref(h)))
        self.r1cs = h
        self.domain_size = lib.pcdgpu_sap_domain_size(pk.pairing, m, self.num_inputs)
        if not self.domain_size:
            lib.pcdgpu_r1cs_free(h)
            raise L.PcdGpuError(-6, "no evaluation domain large enough for the SAP")
        a_q = np.ascontiguousarray(pk.a_query, dtype=np.uint64).reshape(-1, L.AFFINE_LIMBS[g1])
        if a_q.shape[0] != self.num_sap_vars:
            lib.pcdgpu_r1cs_free(h)
            raise ValueError("a_query has %d points for %d SAP variables" % (a_q.shape[0], self.num_sap_vars))
        t_q = np.ascontiguousarray(pk.g_gamma2_z_t, dtype=np.uint64).reshape(-1, L.AFFINE_LIMBS[g1])
        pkh = ctypes.c_void_p()
        ctx._check(lib.pcdgpu_gm17_pk_upload(
            ctx.h, pk.pairing, self.num_sap_vars, self.num_inputs, t_q.shape[0], arr(a_q, np.uint64),
            arr(pk.b_query, np.uint64), arr(pk.c_query_1, np.uint64), arr(pk.c_query_2, np.uint64), arr(t_q, np.uint64),
            arr(pk.g_gamma_z, np.uint64), arr(pk.h_gamma_z, np.uint64), arr(pk.g_ab_gamma_z, np.uint64),
            arr(pk.g_gamma2_z2, np.uint64), int(precompute), ctypes.byref(pkh)))
        self.pk = pkh

    def close(self):
        if getattr(self, "pk", None) and self.ctx.h:
            self.ctx.lib.pcdgpu_gm17_pk_free(self.pk)
            self.ctx.lib.pcdgpu_r1cs_free(self.r1cs)
        self.pk = None
        self.r1cs = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GM17(_Verifier):
    """`GM17<E>` as the reference binds it (/root/reference/tests/mnt4_gm17.rs:27-28): `prove` and its building
    blocks, `process_vk` and verification on the GPU; setup stays with the CPU implementation on the Rust side of
    the boundary."""

    _GM17 = True

    def __init__(self, ctx: L.Context, pairing: int):
        self.ctx, self.pairing = ctx, pairing

    def index(self, pk: GM17ProvingKey, cm: ConstraintMatrices, precompute: bool = False) -> GM17ProverIndex:
        return GM17ProverIndex(self.ctx, pk, cm, precompute)

    def witness_map(self, index: GM17ProverIndex, z: np.ndarray, d1: np.ndarray, d2: np.ndarray):
        """R1CStoSAP::witness_map -> (full SAP assignment, the n + 1 coefficients of H); d1, d2 plain-integer limbs."""
        z = np.ascontiguousarray(z, dtype=np.uint64).reshape(-1, 5)
        if z.shape[0] != index.num_vars:
            raise ValueError("assignment has %d elements for %d variables" % (z.shape[0], index.num_vars))
        d1 = np.ascontiguousarray(d1, dtype=np.uint64)
        d2 = np.ascontiguousarray(d2, dtype=np.uint64)
        full = np.zeros((index.num_sap_vars, 5), dtype=np.uint64)
        h = np.zeros((index.domain_size + 1, 5), dtype=np.uint64)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        self.ctx._check(self.ctx.lib.pcdgpu_sap_witness_map(self.ctx.h, index.r1cs, vp(z), vp(d1), vp(d2), vp(full), vp(h)))
        return full, h

    def create_proof(self, index: GM17ProverIndex, z: np.ndarray, d1: np.ndarray, d2: np.ndarray, r: np.ndarray) -> Proof:
        """ark-gm17 `create_proof(circuit, pk, d1, d2, r)`; d1, d2, r plain-integer limbs."""
        z = np.ascontiguousarray(z, dtype=np.uint64).reshape(-1, 5)
        if z.shape[0] != index.num_vars:
            raise ValueError("assignment has %d elements for %d variables" % (z.shape[0], index.num_vars))
        d1, d2, r = (_scalar(x) for x in (d1, d2, r))
        g1, g2 = L.AFFINE_LIMBS[L.G1_OF[self.pairing]], L.AFFINE_LIMBS[L.G2_OF[self.pairing]]
        out = np.zeros(2 * g1 + g2, dtype=np.uint64)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        self.ctx._check(self.ctx.lib.pcdgpu_gm17_prove(self.ctx.h, index.pk, index.r1cs, vp(z), vp(d1), vp(d2), vp(r),
                                                       vp(out)))
        return Proof(self.pairing, out[:g1].copy(), out[g1:g1 + g2].copy(), out[g1 + g2:].copy())

    def create_proof_dev(self, index: GM17ProverIndex, d_z: int, d1: np.ndarray, d2: np.ndarray, r: np.ndarray) -> Proof:
        d1, d2, r = (_scalar(x) for x in (d1, d2, r))
        g1, g2 = L.AFFINE_LIMBS[L.G1_OF[self.pairing]], L.AFFINE_LIMBS[L.G2_OF[self.pairing]]
        out = np.zeros(2 * g1 + g2, dtype=np.uint64)
        vp = lambda a: ctypes.c_void_p(a.ctypes.data)
        self.ctx._check(self.ctx.lib.pcdgpu_gm17_prove_dev(self.ctx.h, index.pk, index.r1cs, ctypes.c_void_p(d_z), vp(d1),
                                                           vp(d2), vp(r), vp(out)))
        return Proof(self.pairing, out[:g1].copy(), out[g1:g1 + g2].copy(), out[g1 + g2:].copy())

    def prove(self, index: GM17ProverIndex, z: np.ndarray, rng: Callable[[int], np.ndarray]) -> Proof:
        """`SNARK::prove(pk, circuit, rng)`: draws d1, d2, r in this order (`create_random_proof`), then proves."""
        f = L.SCALAR_FIELD_OF[self.pairing]
        d1 = rng(f)
        d2 = rng(f)
        r = rng(f)
        return self.create_proof(index, z, d1, d2, r)

    def serialize(self, proof: Proof) -> bytes:
        """ark-serialize canonical (compressed) bytes of `Proof {a, b, c}`: 152 B (MNT4-298) / 190 B (MNT6-298)."""
        return self.ctx.serialize_proof(self.pairing, proof.affine_limbs())

