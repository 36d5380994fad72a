"""Checked deserialization of compressed proofs on the GPU (pcd_b200/csrc/deserialize.cu) and verification straight
from the bytes, against the oracle (oracle/deserialize_oracle.py) and proofs with known verdicts."""
import ctypes

import numpy as np
import pytest

import codec
import deserialize_helpers as dh
import deserialize_oracle as do
import synth
import verify_helpers as vh

pytestmark = pytest.mark.gpu
PIDS = (0, 1)
KINDS = dh.REJECTIONS + ["subgroup", "inf"]


@pytest.fixture(scope="module")
def ctx():
    import pcd_b200
    c = pcd_b200.Context(0)
    yield c
    c.close()


def _vk(ctx, inst, gm17):
    import pcd_b200
    if gm17:
        return pcd_b200.GM17(ctx, inst["pairing"]), pcd_b200.GM17VerifyingKey(**vh.gm17_vk(inst))
    return pcd_b200.Groth16(ctx, inst["pairing"]), pcd_b200.VerifyingKey(**vh.groth16_vk(inst))


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_prover_proofs_round_trip(ctx, pid, gm17):
    """a GPU-prover proof: serialize -> deserialize gives the identical limbs, and it verifies from its bytes; a
    corrupted encoding raises ValueError, as does a row of the wrong length"""
    import test_gpu_parity as tp
    p = codec.FIELD_P[pid]
    if gm17:
        inst = synth.make_gm17_instance(pid, 1000, seed=700 + 1000, bitlike=0.4, num_inputs=3)
        g, idx = tp._gm17_index(ctx, inst)
        proof = g.create_proof(idx, inst["z"], *(codec.int_to_limbs(pow(k, 99, p)) for k in (3, 5, 7)))
    else:
        inst = synth.make_instance(pid, 1000, seed=900 + 1000, bitlike=0.4, num_inputs=3)
        g, idx = tp._index(ctx, inst)
        proof = g.create_proof_with_reduction(idx, inst["z"], codec.int_to_limbs(pow(3, 200, p)),
                                              codec.int_to_limbs(pow(7, 190, p)))
    idx.close()
    blob = g.serialize(proof)
    assert blob == dh.proof_bytes(pid, proof.affine_limbs())
    back = g.deserialize(blob)
    assert np.array_equal(back.affine_limbs(), proof.affine_limbs())
    v, vk = _vk(ctx, inst, gm17)
    pvk = v.process_vk(vk)
    x = vh.public_inputs(inst)
    assert v.verify_batch_serialized(pvk, x.reshape(1, -1), [blob]).tolist() == [True]
    pvk.close()
    off, curve_id = dh.point_offsets(pid)[1]
    with pytest.raises(ValueError):
        g.deserialize(dh.tamper_point(blob, off, curve_id, "subgroup"))
    with pytest.raises(ValueError):
        g.deserialize(blob[:-1])
    with pytest.raises(ValueError):
        g.deserialize_batch(np.zeros((2, len(blob) + 1), dtype=np.uint8))


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_batch_of_serialized_proofs(ctx, pid, gm17):
    """4096 simulated valid proofs serialized by the oracle, a seeded 10 % corrupted in their bytes (every rejection
    kind at every point, B replaced by twist points outside the subgroup, the infinity flag over a valid x): the ok mask
    and the rows equal the oracle's decoding; verify_batch_serialized = ok & verify_batch(rows), all true untampered;
    batches of 1 and 0 too"""
    inst = (synth.make_gm17_instance if gm17 else synth.make_instance)(pid, 64, num_inputs=3)
    v, vk = _vk(ctx, inst, gm17)
    pvk = v.process_vk(vk)
    n = 4096
    proofs, xs = vh.simulated(inst, n, 4321 + pid, gm17)
    blobs = [dh.proof_bytes(pid, r) for r in proofs]
    rng = np.random.Generator(np.random.Philox(199 + pid))
    bad = np.nonzero(rng.random(n) < 0.10)[0]
    want_rows, want_ok = proofs.copy(), np.ones(n, dtype=bool)
    pairing = synth.PAIRINGS[pid]
    offsets = dh.point_offsets(pid)
    for j, i in enumerate(bad):
        kind = KINDS[j % len(KINDS)]
        off, curve_id = offsets[1] if kind == "subgroup" else offsets[(j // len(KINDS)) % 3]
        blobs[i] = dh.tamper_point(blobs[i], off, curve_id, kind, j // len(KINDS) % 3)
        try:
            want_rows[i] = dh.proof_row(pid, do.deserialize_proof(pairing, blobs[i]))
        except do.InvalidData:
            want_rows[i] = 0
            want_ok[i] = False
        assert want_ok[i] == (kind == "inf"), (i, kind)
    data = np.stack([np.frombuffer(b, dtype=np.uint8) for b in blobs])
    rows, ok = v.deserialize_batch(data)
    assert np.array_equal(ok, want_ok)
    assert np.array_equal(rows, want_rows)
    ver = v.verify_batch(pvk, xs, rows)
    got = v.verify_batch_serialized(pvk, xs, data)
    assert np.array_equal(got, ok & ver)
    assert not got[bad].any()  # the infinity flags break the proofs too
    clean = np.setdiff1d(np.arange(n), bad)
    assert v.verify_batch_serialized(pvk, xs[clean], data[clean]).all()
    assert v.verify_batch_serialized(pvk, xs[:1], data[:1]).tolist() == [got[0]]
    assert v.verify_batch_serialized(pvk, xs[:0], data[:0]).shape == (0,)
    r1, ok1 = v.deserialize_batch(data[bad[:1]])
    assert ok1.tolist() == [want_ok[bad[0]]] and np.array_equal(r1[0], want_rows[bad[0]])
    r0, ok0 = v.deserialize_batch(data[:0])
    assert r0.shape == (0, proofs.shape[1]) and ok0.shape == (0,)
    pvk.close()


@pytest.mark.parametrize("pid", PIDS)
def test_abi_argument_errors(ctx, pid):
    """null pointers with n > 0 and an unknown pairing are PCDGPU_E_ARG; n = 0 with null pointers is PCDGPU_OK"""
    lib, h = ctx.lib, ctx.h
    nb = dh.PROOF_BYTES[pid]
    data = np.zeros(nb, dtype=np.uint8)
    out = np.zeros(2 * codec.POINT_LIMBS[codec.G1_OF[pid]] + codec.POINT_LIMBS[codec.G2_OF[pid]], dtype=np.uint64)
    ok = np.zeros(1, dtype=np.uint8)
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)
    assert lib.pcdgpu_deserialize_proofs(h, 2, vp(data), 1, vp(out), vp(ok)) == -1
    assert lib.pcdgpu_deserialize_proofs(h, pid, None, 1, vp(out), vp(ok)) == -1
    assert lib.pcdgpu_deserialize_proofs(h, pid, vp(data), 1, None, vp(ok)) == -1
    assert lib.pcdgpu_deserialize_proofs(h, pid, vp(data), 1, vp(out), None) == -1
    assert lib.pcdgpu_deserialize_proofs(None, pid, vp(data), 1, vp(out), vp(ok)) == -1
    assert lib.pcdgpu_deserialize_proofs(h, pid, None, 0, None, None) == 0
    # all-zero bytes: x = 0 with no flags, a point only if x^3 + a x + b is a square -- and a verdict either way
    assert lib.pcdgpu_deserialize_proofs(h, pid, vp(data), 1, vp(out), vp(ok)) == 0
    inst = synth.make_instance(pid, 16, num_inputs=1)
    import pcd_b200
    g = pcd_b200.Groth16(ctx, pid)
    pvk = g.process_vk(pcd_b200.VerifyingKey(**vh.groth16_vk(inst)))
    for fn in (lib.pcdgpu_groth16_verify_batch_serialized, lib.pcdgpu_gm17_verify_batch_serialized):
        assert fn(h, None, vp(data), None, 1, vp(ok)) == -1
        assert fn(None, None, vp(data), None, 1, vp(ok)) == -1
    assert lib.pcdgpu_groth16_verify_batch_serialized(h, pvk.h, None, None, 1, vp(ok)) == -1
    assert lib.pcdgpu_groth16_verify_batch_serialized(h, pvk.h, vp(data), None, 1, None) == -1
    assert lib.pcdgpu_groth16_verify_batch_serialized(h, pvk.h, None, None, 0, None) == 0
    assert lib.pcdgpu_groth16_verify_batch_serialized(h, pvk.h, vp(data), None, 1, vp(ok)) == 0 and ok[0] == 0
    pvk.close()
