#!/usr/bin/env python3
"""End-to-end statements/s of csg_prove_many batches, witness included: host builders then prove_many, against the batch witness
builders on the device then prove_many_device.

  python tools/many_witness_throughput.py [--reps 3] [--ks 16,64,256,1024] [--out profiles/r4_many_witness.json]

Cases (the reference's bench sizes, one statement per proof): a Rescue chain of 128 (1024 x 14, blowup 4), one signature (512 x 56),
one Merkle update (512 x 65), one transfer (1024 x 94), at each K with count * width <= 65535.  The inputs (seeds, the signature or
transfer batch of K) exist before the timed window; what is timed is building the K traces and proving them:
  (a) host: the Rescue chains with csg_build_trace_rescue on a thread pool of every host core (ctypes releases the GIL); the
      signature and transfer batches with their host builders, which run over every host core (OpenMP), then cut into K traces
      (Merkle update: with row 1 of columns 14 and 43 set in each, as MerkleProver::build_trace sets them); then prove_many.
  (b) device: build_many_* into a CUDA tensor, then prove_many_device.
Both paths must give the same proofs (checked on the warm-up batch).  Per point: statements/s, the builder's own wall time and the
proof's, means over --reps batches after one warm-up.  The card's name, power limit and the host core count are recorded."""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import certificate_stark_b200 as csg  # noqa: E402

CASES = [   # name, air, rows, blowup
    ("rescue chain 128", csg.AIR_RESCUE, 1024, 4),
    ("schnorr 1 signature", csg.AIR_SCHNORR, 512, 8),
    ("merkle-update 1 tx", csg.AIR_MERKLE_UPDATE, 512, 8),
    ("state-transition 1 tx", csg.AIR_TRANSACTION, 1024, 8),
]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # noqa: BLE001 - recorded, not fatal
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def inputs(air, K):
    if air == csg.AIR_RESCUE:
        return np.arange(7 * K, dtype=np.uint64).reshape(K, 7) + 1
    if air == csg.AIR_SCHNORR:
        return csg.SignatureBatch(seed=K, num_sig=K)
    return csg.TransactionBatch(seed=K, num_tx=K)


def host_build(air, K, R, x, pool):
    if air == csg.AIR_RESCUE:
        built = list(pool.map(lambda s: csg.build_rescue_trace(s, 128), x))
        return [t for t, _ in built], np.stack([p for _, p in built])
    if air == csg.AIR_SCHNORR:
        trace, pub = x.schnorr_trace()
        pubs = pub.reshape(K, 38)
    else:
        trace, pub = x.merkle_update_trace() if air == csg.AIR_MERKLE_UPDATE else x.transaction_trace()
        pubs = np.zeros((K, 14), dtype=np.uint64)
        for k in range(K):   # (root before transfer k, root after it): rows 0 and R-1 of the root columns (58..64) of its slice
            pubs[k, :7], pubs[k, 7:] = trace[58:65, k * R], trace[58:65, (k + 1) * R - 1]

    def cut(k):
        t = np.ascontiguousarray(trace[:, k * R:(k + 1) * R])
        if air == csg.AIR_MERKLE_UPDATE:
            t[14, 1] = t[43, 1] = 1
        return t
    return list(pool.map(cut, range(K))), pubs


def device_build(ctx, air, x):
    if air == csg.AIR_RESCUE:
        return ctx.build_many_rescue(x, 128)
    if air == csg.AIR_SCHNORR:
        return ctx.build_many_schnorr(x)
    return ctx.build_many_merkle_update(x) if air == csg.AIR_MERKLE_UPDATE else ctx.build_many_transaction(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3, help="timed batches per point")
    ap.add_argument("--ks", default="16,64,256,1024")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    ks = [int(x) for x in args.ks.split(",")]
    cores = os.cpu_count()
    result = {"card": card(), "host_cores": cores, "reps": args.reps, "cases": []}
    print(json.dumps(result["card"] | {"host_cores": cores}), flush=True)
    with csg.Context(0) as ctx, ThreadPoolExecutor(cores) as pool:
        for name, air, R, blowup in CASES:
            opt = csg.ProofOptions(blowup_factor=blowup)
            w = csg.TRACE_WIDTH[air]
            rec = {"case": name, "trace": f"{R} x {w}", "blowup": blowup, "points": {}}
            for K in ks:
                if K * w > 65535:
                    continue
                x = inputs(air, K)
                traces, pubs = host_build(air, K, R, x, pool)   # warm-up of both paths, and the check that they agree
                dev, dpubs = device_build(ctx, air, x)
                assert np.array_equal(pubs, dpubs)
                assert ctx.prove_many(air, traces, pubs, opt) == ctx.prove_many_device(air, dev, dpubs, opt)
                del dev
                point = {}
                for path in ("host", "device"):
                    build_s = prove_s = 0.0
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        if path == "host":
                            traces, pubs = host_build(air, K, R, x, pool)
                        else:
                            dev, pubs = device_build(ctx, air, x)
                        t1 = time.perf_counter()
                        if path == "host":
                            ctx.prove_many(air, traces, pubs, opt)
                        else:
                            ctx.prove_many_device(air, dev, pubs, opt)
                            del dev
                        t2 = time.perf_counter()
                        build_s += t1 - t0
                        prove_s += t2 - t1
                    point[path] = {"statements_per_s": round(K * args.reps / (build_s + prove_s), 1),
                                   "build_ms": round(build_s / args.reps * 1e3, 3), "prove_ms": round(prove_s / args.reps * 1e3, 3)}
                point["device_over_host"] = round(point["device"]["statements_per_s"] / point["host"]["statements_per_s"], 2)
                rec["points"][str(K)] = point
                torch.cuda.empty_cache()
                print(json.dumps({"case": name, "K": K} | point), flush=True)
            result["cases"].append(rec)
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
