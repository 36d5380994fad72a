"""GPU pairings and batched Groth16 / GM17 verification (pcd_b200/csrc/pairing.cu) against the oracle
(oracle/pairing_oracle.py) and proofs with known verdicts."""
import numpy as np
import pytest

import codec
import pairing_oracle as po
import pcd_oracle as o
import synth
import verify_helpers as vh

pytestmark = pytest.mark.gpu
PIDS = (0, 1)


@pytest.fixture(scope="module")
def ctx():
    import pcd_b200
    c = pcd_b200.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("pid", PIDS)
def test_pairing_bytes_and_bilinearity(ctx, pid):
    P = po.PARAMS[pid]
    G1, G2 = P.pairing.g1, P.pairing.g2
    g, h = o.generator(G1), o.generator(G2)
    c1, c2 = codec.G1_OF[pid], codec.G2_OF[pid]
    rng = o.SplitMix64(61 + pid)
    a, b = rng.field(P.r), rng.field(P.r)
    pairs = [(G1.mul(g, rng.field(P.r)), G2.mul(h, rng.field(P.r))) for _ in range(6)]
    pairs += [(None, h), (g, None), (g, h), (G1.mul(g, a), G2.mul(h, b)), (G1.mul(g, a * b % P.r), h)]
    got = ctx.pairing(pid, np.stack([synth.point_limbs(c1, p) for p, _ in pairs]),
                      np.stack([synth.point_limbs(c2, q) for _, q in pairs]))
    for i, (p, q) in enumerate(pairs[:-3]):
        assert np.array_equal(got[i], po.gt_to_limbs(P, po.pairing(P, p, q))), i
    # e([a]G, [b]H) = e([ab]G, H) on the device, and it is not e(G, H)
    assert np.array_equal(got[-2], got[-1]) and not np.array_equal(got[-3], got[-1])


def _vk(ctx, inst, gm17):
    import pcd_b200
    if gm17:
        return pcd_b200.GM17(ctx, inst["pairing"]), pcd_b200.GM17VerifyingKey(**vh.gm17_vk(inst))
    return pcd_b200.Groth16(ctx, inst["pairing"]), pcd_b200.VerifyingKey(**vh.groth16_vk(inst))


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_honest_proofs_verify_and_tamperings_fail(ctx, pid, gm17):
    """a GPU-prover proof verifies (one call and in a batch with every tampering of it, each rejected)"""
    import pcd_b200
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
    v, vk = _vk(ctx, inst, gm17)
    x = vh.public_inputs(inst)
    assert v.verify(vk, x, proof)
    pvk = v.process_vk(vk)
    assert v.verify_with_processed_vk(pvk, x, proof)
    other, _ = vh.simulated(inst, 1, 3, gm17)
    rows, xs = [proof.affine_limbs()], [x]
    for kind in vh.TAMPERINGS:
        pr, xx = vh.tamper(pid, proof.affine_limbs(), x, kind, other=other[0])
        rows.append(pr)
        xs.append(xx)
    assert v.verify_batch(pvk, np.stack(xs), np.stack(rows)).tolist() == [True] + [False] * len(vh.TAMPERINGS)
    # ark: a public-input count the key does not have is an error, not a verdict
    with pytest.raises(pcd_b200.PcdGpuError) as e:
        v.verify_batch(pvk, np.stack(xs)[:, :1], np.stack(rows))
    assert e.value.code == -1
    pvk.close()


@pytest.mark.parametrize("pid", PIDS)
@pytest.mark.parametrize("gm17", [False, True], ids=["groth16", "gm17"])
def test_batch_of_simulated_proofs(ctx, pid, gm17):
    """4096 distinct valid proofs with distinct public inputs, a seeded 10 % corrupted: exactly the expected mask;
    batches of 1 and 0 too"""
    inst = (synth.make_gm17_instance if gm17 else synth.make_instance)(pid, 64, num_inputs=3)
    v, vk = _vk(ctx, inst, gm17)
    pvk = v.process_vk(vk)
    proofs, xs = vh.simulated(inst, 4096, 1234 + pid, gm17)
    rng = np.random.Generator(np.random.Philox(99 + pid))
    bad = rng.random(4096) < 0.10
    a1, _ = vh.widths(pid)
    for i in np.nonzero(bad)[0]:
        kind = vh.TAMPERINGS[i % len(vh.TAMPERINGS)]
        proofs[i], xs[i] = vh.tamper(pid, proofs[i], xs[i], kind, other=proofs[(i + 1) % 4096])
    ok = v.verify_batch(pvk, xs, proofs)
    assert np.array_equal(ok, ~bad)
    assert v.verify_batch(pvk, xs[:1], proofs[:1]).tolist() == [not bad[0]]
    assert v.verify_batch(pvk, xs[:0], proofs[:0]).shape == (0,)
    pvk.close()


@pytest.mark.parametrize("pid", PIDS)
def test_bad_keys_are_argument_errors(ctx, pid):
    import pcd_b200
    inst = synth.make_instance(pid, 16, num_inputs=2)
    g = pcd_b200.Groth16(ctx, pid)
    vk = vh.groth16_vk(inst)
    off = dict(vk)
    off["alpha_g1"] = vk["alpha_g1"].copy()
    off["alpha_g1"][5] ^= 1  # y changed: off the curve
    with pytest.raises(pcd_b200.PcdGpuError) as e:
        g.process_vk(pcd_b200.VerifyingKey(**off))
    assert e.value.code == -1
    empty = dict(vk)
    empty["gamma_abc_g1"] = vk["gamma_abc_g1"][:0]
    with pytest.raises(pcd_b200.PcdGpuError) as e:
        g.process_vk(pcd_b200.VerifyingKey(**empty))
    assert e.value.code == -1
