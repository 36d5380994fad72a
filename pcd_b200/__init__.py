"""pcd_b200 -- B200 (sm_100a) prover backend for the Groth16 proving step of arkworks-rs/pcd.

Everything numeric runs in libpcdgpu.so (pcd_b200/csrc, C ABI in include/pcdgpu.h); this package is
the thin host mirror of the reference's SNARK interface used by the tests and the benchmark.
"""
from .lib import (Bases, Context, PcdGpuError, load, FIELD_R4, FIELD_Q4, MNT4_298, MNT6_298, MNT4_G1, MNT4_G2,  # noqa
                  MNT6_G1, MNT6_G2, G1_OF, G2_OF, SCALAR_FIELD_OF, AFFINE_LIMBS, XYZZ_LIMBS, TWO_ADICITY)
from .snark import (ConstraintMatrices, GM17, GM17ProverIndex, GM17ProvingKey, GM17VerifyingKey, Groth16,  # noqa
                    PreparedVerifyingKey, Proof, ProverIndex, ProvingKey, VerifyingKey)
from . import kzg  # noqa
