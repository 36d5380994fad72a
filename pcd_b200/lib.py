"""ctypes binding of libpcdgpu.so (include/pcdgpu.h) -- the only way this package computes anything.

There is no CPU fallback: if the shared library is missing or no sm_100 GPU is usable, loading /
context creation raises.  Buffers are numpy arrays in the ABI encodings (uint64 little-endian
limbs); `*_dev` methods take raw device pointers (e.g. ``torch_tensor.data_ptr()``).
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# PCDGPU_LIB selects another build of the SAME library (A/B runs of kernel variants); there is no non-CUDA build
LIB_PATH = os.environ.get("PCDGPU_LIB") or os.path.join(HERE, "libpcdgpu.so")

# ids (include/pcdgpu.h)
FIELD_R4, FIELD_Q4 = 0, 1
MNT4_298, MNT6_298 = 0, 1
MNT4_G1, MNT4_G2, MNT6_G1, MNT6_G2 = 0, 1, 2, 3
G1_OF = {MNT4_298: MNT4_G1, MNT6_298: MNT6_G1}
G2_OF = {MNT4_298: MNT4_G2, MNT6_298: MNT6_G2}
SCALAR_FIELD_OF = {MNT4_298: FIELD_R4, MNT6_298: FIELD_Q4}
#: u64 limbs of an affine point / an xyzz point per curve
AFFINE_LIMBS = {0: 10, 1: 20, 2: 10, 3: 30}
XYZZ_LIMBS = {0: 20, 1: 40, 2: 20, 3: 60}
TWO_ADICITY = {FIELD_R4: 34, FIELD_Q4: 17}

EXPORTS = [
    "pcdgpu_strerror", "pcdgpu_last_error", "pcdgpu_affine_bytes", "pcdgpu_ctx_create", "pcdgpu_ctx_destroy",
    "pcdgpu_sync", "pcdgpu_set_stream", "pcdgpu_set_concurrency", "pcdgpu_set_msm_window", "pcdgpu_set_proof_graphs", "pcdgpu_proof_graph_stats", "pcdgpu_ntt", "pcdgpu_ntt_dev", "pcdgpu_domain_size", "pcdgpu_ntt_general", "pcdgpu_msm",
    "pcdgpu_msm_dev", "pcdgpu_bases_upload", "pcdgpu_bases_free", "pcdgpu_msm_bases", "pcdgpu_msm_bases_dev",
    "pcdgpu_xyzz_sum", "pcdgpu_xyzz_download", "pcdgpu_fixed_base_mul", "pcdgpu_fixed_base_mul_dev",
    "pcdgpu_r1cs_upload", "pcdgpu_r1cs_free", "pcdgpu_r1cs_domain_size", "pcdgpu_witness_map", "pcdgpu_pk_upload",
    "pcdgpu_pk_free", "pcdgpu_groth16_prove", "pcdgpu_groth16_prove_dev", "pcdgpu_serialize_proof",
    "pcdgpu_profile_enable", "pcdgpu_profile_read", "pcdgpu_profile_timeline", "pcdgpu_bench_imad",
    "pcdgpu_sap_domain_size", "pcdgpu_sap_witness_map", "pcdgpu_gm17_pk_upload", "pcdgpu_gm17_pk_free",
    "pcdgpu_gm17_prove", "pcdgpu_gm17_prove_dev",
    "pcdgpu_poly_divide_linear", "pcdgpu_poly_mul", "pcdgpu_kzg_commit", "pcdgpu_kzg_open",
    "pcdgpu_qap_vector_dev", "pcdgpu_qap_combine_dev", "pcdgpu_set_msm_side_by_side", "pcdgpu_groth16_assemble_begin_dev", "pcdgpu_groth16_assemble_finish_dev",
    "pcdgpu_comm_unique_id", "pcdgpu_comm_init", "pcdgpu_comm_info", "pcdgpu_comm_destroy", "pcdgpu_pk_upload_sharded",
    "pcdgpu_groth16_prove_sharded", "pcdgpu_groth16_prove_sharded_dev", "pcdgpu_msm_bases_sharded",
    "pcdgpu_msm_bases_sharded_dev",
    "pcdgpu_dev_alloc", "pcdgpu_dev_free", "pcdgpu_dev_upload", "pcdgpu_dev_download", "pcdgpu_dev_copy", "pcdgpu_dev_zero",
    "pcdgpu_vec_binary_dev", "pcdgpu_vec_scalar_dev", "pcdgpu_vec_axpy_dev", "pcdgpu_vec_inverse_dev",
    "pcdgpu_vec_powers_dev", "pcdgpu_vec_gather_dev", "pcdgpu_poly_eval_dev", "pcdgpu_poly_divide_vanishing_dev",
    "pcdgpu_poly_divide_linear_dev", "pcdgpu_ntt_general_dev", "pcdgpu_csr_upload", "pcdgpu_csr_free",
    "pcdgpu_csr_matvec_dev", "pcdgpu_kzg_commit_dev",
    "pcdgpu_pairing", "pcdgpu_groth16_pvk_create", "pcdgpu_groth16_pvk_free", "pcdgpu_groth16_verify_batch",
    "pcdgpu_gm17_pvk_create", "pcdgpu_gm17_pvk_free", "pcdgpu_gm17_verify_batch",
    "pcdgpu_deserialize_proofs", "pcdgpu_groth16_verify_batch_serialized", "pcdgpu_gm17_verify_batch_serialized",
]
#: u64 limbs of a GT element per pairing (arkworks' QuadExtField over Fq2 / Fq3)
GT_LIMBS = {MNT4_298: 20, MNT6_298: 30}
#: bytes of a compressed proof (pcdgpu_serialize_proof) per pairing
PROOF_BYTES = {MNT4_298: 152, MNT6_298: 190}
COMM_ID_BYTES = 128


class PcdGpuError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        super().__init__("libpcdgpu error %d%s" % (code, (": " + detail) if detail else ""))


_lib = None


def load():
    """Load libpcdgpu.so; raises (never falls back) when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or `make -C pcd_b200/csrc`); pcd_b200 has no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, ci = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    lib.pcdgpu_strerror.restype = ctypes.c_char_p
    lib.pcdgpu_strerror.argtypes = [ci]
    lib.pcdgpu_last_error.restype = ctypes.c_char_p
    lib.pcdgpu_last_error.argtypes = [vp]
    lib.pcdgpu_affine_bytes.restype = sz
    lib.pcdgpu_affine_bytes.argtypes = [ci]
    lib.pcdgpu_ctx_create.argtypes = [ci, ctypes.POINTER(vp)]
    lib.pcdgpu_ctx_destroy.argtypes = [vp]
    lib.pcdgpu_ctx_destroy.restype = None
    lib.pcdgpu_sync.argtypes = [vp]
    lib.pcdgpu_set_stream.argtypes = [vp, vp]
    lib.pcdgpu_set_msm_window.argtypes = [vp, ci]
    lib.pcdgpu_set_concurrency.argtypes = [vp, ci]
    lib.pcdgpu_set_proof_graphs.argtypes = [vp, ci]
    lib.pcdgpu_proof_graph_stats.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    lib.pcdgpu_ntt.argtypes = [vp, ci, vp, ctypes.c_uint32, ci, ci]
    lib.pcdgpu_ntt_dev.argtypes = [vp, ci, vp, ctypes.c_uint32, ci, ci]
    lib.pcdgpu_domain_size.restype = sz
    lib.pcdgpu_domain_size.argtypes = [ci, sz, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    lib.pcdgpu_ntt_general.argtypes = [vp, ci, vp, ci, ci, ci, ci]
    lib.pcdgpu_msm.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.pcdgpu_msm_dev.argtypes = [vp, ci, vp, vp, ci, sz, vp]
    lib.pcdgpu_bases_upload.argtypes = [vp, ci, vp, sz, ci, ctypes.POINTER(vp)]
    lib.pcdgpu_bases_free.argtypes = [vp]
    lib.pcdgpu_bases_free.restype = None
    lib.pcdgpu_msm_bases.argtypes = [vp, vp, sz, vp, sz, vp]
    lib.pcdgpu_msm_bases_dev.argtypes = [vp, vp, sz, vp, ci, sz, vp]
    lib.pcdgpu_xyzz_sum.argtypes = [vp, ci, vp, sz, vp]
    lib.pcdgpu_xyzz_download.argtypes = [vp, ci, vp, vp]
    lib.pcdgpu_fixed_base_mul.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.pcdgpu_fixed_base_mul_dev.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.pcdgpu_r1cs_upload.argtypes = [vp, ci, sz, sz, sz] + [vp] * 9 + [ctypes.POINTER(vp)]
    lib.pcdgpu_r1cs_free.argtypes = [vp]
    lib.pcdgpu_r1cs_free.restype = None
    lib.pcdgpu_r1cs_domain_size.argtypes = [vp]
    lib.pcdgpu_r1cs_domain_size.restype = sz
    lib.pcdgpu_witness_map.argtypes = [vp, vp, vp, vp]
    lib.pcdgpu_pk_upload.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10 + [ci, ctypes.POINTER(vp)]
    lib.pcdgpu_pk_free.argtypes = [vp]
    lib.pcdgpu_pk_free.restype = None
    lib.pcdgpu_groth16_prove.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.pcdgpu_groth16_prove_dev.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.pcdgpu_serialize_proof.argtypes = [vp, ci, vp, vp, ctypes.POINTER(sz)]
    lib.pcdgpu_profile_enable.argtypes = [vp, ci]
    lib.pcdgpu_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                        ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    lib.pcdgpu_profile_timeline.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                            ctypes.POINTER(ctypes.c_int), sz, ctypes.POINTER(sz)]
    lib.pcdgpu_bench_imad.argtypes = [vp, ci, ci, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    lib.pcdgpu_sap_domain_size.argtypes = [ci, sz, sz]
    lib.pcdgpu_sap_domain_size.restype = sz
    lib.pcdgpu_sap_witness_map.argtypes = [vp] * 7
    lib.pcdgpu_gm17_pk_upload.argtypes = [vp, ci, sz, sz, sz] + [vp] * 9 + [ci, ctypes.POINTER(vp)]
    lib.pcdgpu_gm17_pk_free.argtypes = [vp]
    lib.pcdgpu_gm17_pk_free.restype = None
    lib.pcdgpu_gm17_prove.argtypes = [vp] * 8
    lib.pcdgpu_gm17_prove_dev.argtypes = [vp] * 8
    lib.pcdgpu_set_msm_side_by_side.argtypes = [vp, ci]
    lib.pcdgpu_groth16_assemble_begin_dev.argtypes = [vp, ci, vp, vp, ci, vp, vp]
    lib.pcdgpu_groth16_assemble_finish_dev.argtypes = [vp, ci, ci, vp, vp]
    lib.pcdgpu_qap_vector_dev.argtypes = [vp, vp, ci, vp, vp]
    lib.pcdgpu_qap_combine_dev.argtypes = [vp, vp, vp, vp, vp]
    lib.pcdgpu_poly_divide_linear.argtypes = [vp, ci, vp, sz, vp, vp, vp]
    lib.pcdgpu_poly_mul.argtypes = [vp, ci, vp, sz, vp, sz, vp]
    lib.pcdgpu_kzg_commit.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp]
    lib.pcdgpu_kzg_open.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp, vp, vp, vp]
    lib.pcdgpu_comm_unique_id.argtypes = [vp]
    lib.pcdgpu_comm_init.argtypes = [vp, vp, ci, ci]
    lib.pcdgpu_comm_info.argtypes = [vp, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    lib.pcdgpu_comm_destroy.argtypes = [vp]
    lib.pcdgpu_comm_destroy.restype = None
    lib.pcdgpu_pk_upload_sharded.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10 + [ci, ctypes.POINTER(vp)]
    lib.pcdgpu_groth16_prove_sharded.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.pcdgpu_groth16_prove_sharded_dev.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.pcdgpu_msm_bases_sharded.argtypes = [vp, vp, vp, sz, vp]
    lib.pcdgpu_msm_bases_sharded_dev.argtypes = [vp, vp, vp, ci, sz, vp]
    lib.pcdgpu_dev_alloc.argtypes = [vp, sz, ctypes.POINTER(vp)]
    lib.pcdgpu_dev_free.argtypes = [vp, vp]
    lib.pcdgpu_dev_upload.argtypes = [vp, vp, vp, sz]
    lib.pcdgpu_dev_download.argtypes = [vp, vp, vp, sz]
    lib.pcdgpu_dev_copy.argtypes = [vp, vp, vp, sz]
    lib.pcdgpu_dev_zero.argtypes = [vp, vp, sz]
    lib.pcdgpu_vec_binary_dev.argtypes = [vp, ci, ci, vp, vp, vp, sz]
    lib.pcdgpu_vec_scalar_dev.argtypes = [vp, ci, ci, vp, vp, vp, sz]
    lib.pcdgpu_vec_axpy_dev.argtypes = [vp, ci, vp, vp, vp, sz]
    lib.pcdgpu_vec_inverse_dev.argtypes = [vp, ci, vp, sz]
    lib.pcdgpu_vec_powers_dev.argtypes = [vp, ci, vp, vp, vp, sz]
    lib.pcdgpu_vec_gather_dev.argtypes = [vp, ci, vp, vp, vp, sz]
    lib.pcdgpu_poly_eval_dev.argtypes = [vp, ci, vp, sz, vp, vp]
    lib.pcdgpu_poly_divide_vanishing_dev.argtypes = [vp, ci, vp, sz, sz, vp, vp]
    lib.pcdgpu_poly_divide_linear_dev.argtypes = [vp, ci, vp, sz, vp, vp, vp]
    lib.pcdgpu_ntt_general_dev.argtypes = [vp, ci, vp, ci, ci, ci, ci]
    lib.pcdgpu_csr_upload.argtypes = [vp, ci, sz, sz, vp, vp, vp, ctypes.POINTER(vp)]
    lib.pcdgpu_csr_free.argtypes = [vp]
    lib.pcdgpu_csr_free.restype = None
    lib.pcdgpu_csr_matvec_dev.argtypes = [vp, vp, vp, vp]
    lib.pcdgpu_kzg_commit_dev.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, vp]
    lib.pcdgpu_pairing.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.pcdgpu_groth16_pvk_create.argtypes = [vp, ci] + [vp] * 5 + [sz, ctypes.POINTER(vp)]
    lib.pcdgpu_groth16_pvk_free.argtypes = [vp]
    lib.pcdgpu_groth16_pvk_free.restype = None
    lib.pcdgpu_groth16_verify_batch.argtypes = [vp, vp, vp, vp, sz, vp]
    lib.pcdgpu_gm17_pvk_create.argtypes = [vp, ci] + [vp] * 6 + [sz, ctypes.POINTER(vp)]
    lib.pcdgpu_gm17_pvk_free.argtypes = [vp]
    lib.pcdgpu_gm17_pvk_free.restype = None
    lib.pcdgpu_gm17_verify_batch.argtypes = [vp, vp, vp, vp, sz, vp]
    lib.pcdgpu_deserialize_proofs.argtypes = [vp, ci, vp, sz, vp, vp]
    lib.pcdgpu_groth16_verify_batch_serialized.argtypes = [vp, vp, vp, vp, sz, vp]
    lib.pcdgpu_gm17_verify_batch_serialized.argtypes = [vp, vp, vp, vp, sz, vp]
    _lib = lib
    return lib


def domain_size(field: int, min_size: int):
    """GeneralEvaluationDomain::new(min_size) -> (n, pow7, pow2) or None"""
    a, b = ctypes.c_int(), ctypes.c_int()
    n = load().pcdgpu_domain_size(field, min_size, ctypes.byref(a), ctypes.byref(b))
    return (n, a.value, b.value) if n else None


def _u64(a, width=None):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    if width is not None:
        a = a.reshape(-1, width)
    return a


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


class Context:
    """One GPU + one stream (pcdgpu_ctx)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = ctypes.c_void_p()
        rc = self.lib.pcdgpu_ctx_create(device, ctypes.byref(h))
        if rc != 0:
            raise PcdGpuError(rc, self.lib.pcdgpu_strerror(rc).decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.pcdgpu_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            detail = self.lib.pcdgpu_last_error(self.h).decode() or self.lib.pcdgpu_strerror(rc).decode()
            raise PcdGpuError(rc, detail)

    def sync(self):
        self._check(self.lib.pcdgpu_sync(self.h))

    def set_stream(self, stream_ptr: int):
        self._check(self.lib.pcdgpu_set_stream(self.h, ctypes.c_void_p(stream_ptr)))

    def set_concurrency(self, on: bool):
        self._check(self.lib.pcdgpu_set_concurrency(self.h, int(on)))

    def set_proof_graphs(self, on: bool):
        """CUDA graphs of whole Groth16 proofs (include/pcdgpu.h: pcdgpu_set_proof_graphs); off by default (measured slower)"""
        self._check(self.lib.pcdgpu_set_proof_graphs(self.h, int(on)))

    def proof_graph_stats(self):
        """(graphs captured, proofs replayed from a graph) since the context exists"""
        a, b = ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self.lib.pcdgpu_proof_graph_stats(self.h, ctypes.byref(a), ctypes.byref(b)))
        return int(a.value), int(b.value)

    def set_msm_window(self, c: int):
        self._check(self.lib.pcdgpu_set_msm_window(self.h, c))

    # ---- NTT ----
    def ntt(self, field: int, data: np.ndarray, inverse: bool = False, coset: bool = False) -> np.ndarray:
        d = np.array(data, dtype=np.uint64, copy=True).reshape(-1, 5)
        n = d.shape[0]
        log_n = max(n, 1).bit_length() - 1
        if n == 0 or (1 << log_n) != n:
            raise ValueError("NTT length must be a power of two")
        self._check(self.lib.pcdgpu_ntt(self.h, field, _p(d), log_n, int(inverse), int(coset)))
        return d

    def ntt_general(self, field: int, data: np.ndarray, pow7: int, pow2: int, inverse: bool = False,
                    coset: bool = False) -> np.ndarray:
        """transform on the domain 7^pow7 * 2^pow2 (ark-poly GeneralEvaluationDomain)"""
        d = np.array(data, dtype=np.uint64, copy=True).reshape(-1, 5)
        if d.shape[0] != (7 ** pow7) << pow2:
            raise ValueError("data length does not match the domain")
        self._check(self.lib.pcdgpu_ntt_general(self.h, field, _p(d), pow7, pow2, int(inverse), int(coset)))
        return d

    def ntt_dev(self, field: int, d_ptr: int, log_n: int, inverse: bool = False, coset: bool = False):
        self._check(self.lib.pcdgpu_ntt_dev(self.h, field, ctypes.c_void_p(d_ptr), log_n, int(inverse), int(coset)))

    # ---- pairings ----
    def pairing(self, pairing: int, g1: np.ndarray, g2: np.ndarray) -> np.ndarray:
        """e(g1[i], g2[i]) for every row: (n, GT_LIMBS[pairing]) u64 limbs (ark-ec PairingEngine::pairing)"""
        g1 = _u64(g1, AFFINE_LIMBS[G1_OF[pairing]])
        g2 = _u64(g2, AFFINE_LIMBS[G2_OF[pairing]])
        if g1.shape[0] != g2.shape[0]:
            raise ValueError("g1 and g2 hold different numbers of points")
        out = np.zeros((g1.shape[0], GT_LIMBS[pairing]), dtype=np.uint64)
        self._check(self.lib.pcdgpu_pairing(self.h, pairing, _p(g1), _p(g2), g1.shape[0], _p(out)))
        return out

    # ---- MSM ----
    def msm(self, curve: int, bases: np.ndarray, scalars: np.ndarray) -> np.ndarray:
        bases = _u64(bases, AFFINE_LIMBS[curve])
        scalars = _u64(scalars, 5)
        n = min(bases.shape[0], scalars.shape[0])
        out = np.zeros(AFFINE_LIMBS[curve], dtype=np.uint64)
        self._check(self.lib.pcdgpu_msm(self.h, curve, _p(bases), _p(scalars), n, _p(out)))
        return out

    def msm_dev(self, curve: int, d_bases: int, d_scalars: int, n: int, d_out: int, scalars_mont: bool = False):
        self._check(self.lib.pcdgpu_msm_dev(self.h, curve, ctypes.c_void_p(d_bases), ctypes.c_void_p(d_scalars),
                                            int(scalars_mont), n, ctypes.c_void_p(d_out)))

    def xyzz_sum(self, curve: int, parts: np.ndarray) -> np.ndarray:
        parts = _u64(parts, XYZZ_LIMBS[curve])
        out = np.zeros(AFFINE_LIMBS[curve], dtype=np.uint64)
        self._check(self.lib.pcdgpu_xyzz_sum(self.h, curve, _p(parts), parts.shape[0], _p(out)))
        return out

    def xyzz_download(self, curve: int, d_ptr: int) -> np.ndarray:
        out = np.zeros(XYZZ_LIMBS[curve], dtype=np.uint64)
        self._check(self.lib.pcdgpu_xyzz_download(self.h, curve, ctypes.c_void_p(d_ptr), _p(out)))
        return out

    def fixed_base_mul(self, curve: int, base: np.ndarray, scalars: np.ndarray) -> np.ndarray:
        base = _u64(base)
        scalars = _u64(scalars, 5)
        out = np.zeros((scalars.shape[0], AFFINE_LIMBS[curve]), dtype=np.uint64)
        self._check(self.lib.pcdgpu_fixed_base_mul(self.h, curve, _p(base), _p(scalars), scalars.shape[0], _p(out)))
        return out

    def fixed_base_mul_dev(self, curve: int, base: np.ndarray, d_scalars: int, n: int, d_out: int):
        base = _u64(base)
        self._check(self.lib.pcdgpu_fixed_base_mul_dev(self.h, curve, _p(base), ctypes.c_void_p(d_scalars), n,
                                                       ctypes.c_void_p(d_out)))

    # ---- multi-GPU: the library's own collective (NCCL all-gather of partial sums, comm.cu) ----
    def comm_unique_id(self) -> bytes:
        """rank 0: the 128 bytes every rank passes to comm_init (ship them by any means)"""
        buf = ctypes.create_string_buffer(COMM_ID_BYTES)
        rc = self.lib.pcdgpu_comm_unique_id(buf)
        if rc != 0:
            raise PcdGpuError(rc, "libnccl.so.2 could not be loaded")
        return buf.raw

    def comm_init(self, uid: bytes, rank: int, world: int):
        self._check(self.lib.pcdgpu_comm_init(self.h, ctypes.c_char_p(uid) if uid else None, rank, world))

    def comm_init_torch(self, group=None):
        """comm_init with the id broadcast through an initialised torch.distributed group"""
        import torch
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return self.comm_init(None, 0, 1)
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        box = [self.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, group=group)
        self.comm_init(box[0], rank, world)

    def comm_info(self):
        r, w = ctypes.c_int(), ctypes.c_int()
        self._check(self.lib.pcdgpu_comm_info(self.h, ctypes.byref(r), ctypes.byref(w)))
        return r.value, w.value

    def bench_imad(self, mode: int = 0, iters: int = 2000):
        ops, ms = ctypes.c_double(), ctypes.c_double()
        self._check(self.lib.pcdgpu_bench_imad(self.h, mode, iters, ctypes.byref(ops), ctypes.byref(ms)))
        return ops.value, ms.value

    def serialize_proof(self, pairing: int, proof_affine: np.ndarray) -> bytes:
        proof_affine = _u64(proof_affine)
        out = np.zeros(192, dtype=np.uint8)
        n = ctypes.c_size_t()
        self._check(self.lib.pcdgpu_serialize_proof(self.h, pairing, _p(proof_affine), _p(out), ctypes.byref(n)))
        return out[:n.value].tobytes()

    def deserialize_proofs(self, pairing: int, rows: np.ndarray):
        """checked ark-serialize deserialization of n compressed proofs ((n, PROOF_BYTES[pairing]) uint8) ->
        ((n, A || B || C) affine limbs, zero rows for invalid proofs; (n,) bool verdicts)"""
        width = 2 * AFFINE_LIMBS[G1_OF[pairing]] + AFFINE_LIMBS[G2_OF[pairing]]
        out = np.zeros((rows.shape[0], width), dtype=np.uint64)
        ok = np.zeros(rows.shape[0], dtype=np.uint8)
        self._check(self.lib.pcdgpu_deserialize_proofs(self.h, pairing, _p(rows), rows.shape[0], _p(out), _p(ok)))
        return out, ok.astype(bool)


class Bases:
    """Device-resident MSM base vector (pcdgpu_bases)."""

    def __init__(self, ctx: Context, curve: int, points: np.ndarray, precompute: bool = False):
        self.ctx, self.curve = ctx, curve
        pts = _u64(points, AFFINE_LIMBS[curve])
        self.n = pts.shape[0]
        h = ctypes.c_void_p()
        ctx._check(ctx.lib.pcdgpu_bases_upload(ctx.h, curve, _p(pts), self.n, int(precompute), ctypes.byref(h)))
        self.h = h

    def msm(self, scalars: np.ndarray, offset: int = 0) -> np.ndarray:
        scalars = _u64(scalars, 5)
        out = np.zeros(AFFINE_LIMBS[self.curve], dtype=np.uint64)
        self.ctx._check(self.ctx.lib.pcdgpu_msm_bases(self.ctx.h, self.h, offset, _p(scalars), scalars.shape[0],
                                                      _p(out)))
        return out

    def msm_dev(self, d_scalars: int, n: int, d_out: int, offset: int = 0, scalars_mont: bool = False):
        self.ctx._check(self.ctx.lib.pcdgpu_msm_bases_dev(self.ctx.h, self.h, offset, ctypes.c_void_p(d_scalars),
                                                          int(scalars_mont), n, ctypes.c_void_p(d_out)))

    def msm_sharded(self, scalars: np.ndarray) -> np.ndarray:
        """collective: this Bases holds THIS rank's slice, `scalars` this rank's scalars; every rank gets the sum"""
        scalars = _u64(scalars, 5)
        out = np.zeros(AFFINE_LIMBS[self.curve], dtype=np.uint64)
        self.ctx._check(self.ctx.lib.pcdgpu_msm_bases_sharded(self.ctx.h, self.h, _p(scalars), scalars.shape[0], _p(out)))
        return out

    def msm_sharded_dev(self, d_scalars: int, n: int, d_out_affine: int, scalars_mont: bool = False):
        self.ctx._check(self.ctx.lib.pcdgpu_msm_bases_sharded_dev(self.ctx.h, self.h, ctypes.c_void_p(d_scalars),
                                                                  int(scalars_mont), n, ctypes.c_void_p(d_out_affine)))

    def close(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.lib.pcdgpu_bases_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
