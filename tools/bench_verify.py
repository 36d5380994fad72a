#!/usr/bin/env python3
"""Throughput of batched proof verification on the GPU: one JSON line with proofs/s and ms per call for batches of
1, 64, 1024 and 16384 proofs, per pairing and proof system.  Proofs are simulated valid proofs with distinct public
inputs (2 public inputs); the host clock runs around the synchronous call, after one warm-up call of the same size,
and every timed call's verdicts must all be true.

--serialized adds, next to each verify_batch row (op "verify"), the same proofs as compressed bytes (152 / 190 B,
serialized by the oracle): deserialize_batch alone (op "deserialize", once per pairing) and verify_batch_serialized
(op "verify_serialized").

    python tools/bench_verify.py [--batches 1,64,1024,16384] [--reps 3] [--serialized] [--out bench_verify.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402

import deserialize_helpers as dh  # noqa: E402
import pcd_b200  # noqa: E402
import synth  # noqa: E402
import verify_helpers as vh  # noqa: E402


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(device=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers still stand; say what is missing
        return dict(device="unknown (%s)" % e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,64,1024,16384")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--serialized", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    batches = [int(b) for b in a.batches.split(",")]
    ctx = pcd_b200.Context(0)
    res = dict(info=device_info(), results=[])
    nmax = max(batches)
    for pid in (0, 1):
        for gm17 in (False, True):
            inst = (synth.make_gm17_instance if gm17 else synth.make_instance)(pid, 64, num_inputs=3)
            v = (pcd_b200.GM17 if gm17 else pcd_b200.Groth16)(ctx, pid)
            vk = pcd_b200.GM17VerifyingKey(**vh.gm17_vk(inst)) if gm17 else pcd_b200.VerifyingKey(**vh.groth16_vk(inst))
            pvk = v.process_vk(vk)
            base_p, base_x = vh.simulated(inst, min(nmax, 2048), 77 + pid, gm17)
            base_b = np.stack([np.frombuffer(dh.proof_bytes(pid, r), dtype=np.uint8) for r in base_p]) \
                if a.serialized else None
            ops = [("verify", lambda p, b, x: v.verify_batch(pvk, x, p))]
            if a.serialized:
                if not gm17:
                    ops.append(("deserialize", lambda p, b, x: v.deserialize_batch(b)[1]))
                ops.append(("verify_serialized", lambda p, b, x: v.verify_batch_serialized(pvk, x, b)))
            for n in batches:
                reps = -(-n // base_p.shape[0])
                proofs = np.ascontiguousarray(np.concatenate([base_p] * reps)[:n])
                xs = np.ascontiguousarray(np.concatenate([base_x] * reps)[:n])
                blobs = np.ascontiguousarray(np.concatenate([base_b] * reps)[:n]) if a.serialized else None
                for op, fn in ops:
                    assert fn(proofs, blobs, xs).all()  # warm-up, same shape
                    ts = []
                    for _ in range(a.reps):
                        t0 = time.perf_counter()
                        ok = fn(proofs, blobs, xs)
                        ts.append(time.perf_counter() - t0)
                        assert ok.all(), "a valid proof was rejected"
                    t = min(ts)
                    res["results"].append(dict(pairing="mnt4_298" if pid == 0 else "mnt6_298",
                                               scheme="gm17" if gm17 else "groth16", op=op, batch=n,
                                               ms_per_call=t * 1e3, ms_per_call_all=[x * 1e3 for x in ts],
                                               proofs_per_s=n / t))
                    print(json.dumps(res["results"][-1]), file=sys.stderr, flush=True)
            pvk.close()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
