#!/usr/bin/env python3
"""Wall time of trace validation (csg_validate_*), against the proof of the same trace.

  python tools/validate_time.py [--reps 5] [--out profiles/r5_validate_time.json]

Measured in one run, each point the mean of --reps calls after one warm-up call (every call ends in a device synchronise):
  * the 1024-transaction trace (2^20 x 94), built on the device: validate_resident; validate of the same trace from page-locked
    memory (a HostBuffer) and from pageable memory (a numpy array); prove_loaded of the resident trace (default options);
  * validate_many_device of Rescue-128 batches (1024 x 14 per trace) and one-signature Schnorr batches (512 x 56) at K = 64, 256
    and 1024, built on the device.
Every trace validated is a valid witness: the figures are the pass itself, not the host localisation of failures.  The card's
name and power limit are recorded with the numbers."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import certificate_stark_b200 as csg  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # noqa: BLE001 - recorded, not fatal
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def mean_ms(fn, reps):
    out = fn()   # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    return round((time.perf_counter() - t0) / reps * 1e3, 3), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    result = {"card": card(), "reps": args.reps}
    print(json.dumps(result["card"]), flush=True)
    n = 1 << 20
    with csg.Context(0) as ctx:
        pub = ctx.build_batch(1, 1024)
        ctx.set_air(csg.AIR_TRANSACTION, n, pub, csg.ProofOptions())
        ctx.build_transaction_trace_resident()
        tx = {"trace": f"{n} x 94", "transactions": 1024}
        tx["validate_resident_ms"], r = mean_ms(ctx.validate_resident, args.reps)
        assert r.ok
        pageable = ctx.download_trace(94, n)
        pinned = csg.HostBuffer(94, n)
        pinned.array[:] = pageable
        tx["validate_pinned_ms"], r = mean_ms(lambda: ctx.validate(csg.AIR_TRANSACTION, pinned.array, pub), args.reps)
        assert r.ok
        tx["validate_pageable_ms"], r = mean_ms(lambda: ctx.validate(csg.AIR_TRANSACTION, pageable, pub), args.reps)
        assert r.ok
        pinned.close()
        del pageable
        tx["prove_loaded_ms"], _ = mean_ms(ctx.prove_loaded, args.reps)
        tx["validate_resident_over_prove_loaded"] = round(tx["validate_resident_ms"] / tx["prove_loaded_ms"], 4)
        result["transaction_2^20"] = tx
        print(json.dumps(tx), flush=True)

        import torch
        batches = []
        for name, air, build in [("rescue chain 128 (1024 x 14)", csg.AIR_RESCUE, lambda K: ctx.build_many_rescue(np.arange(7 * K, dtype=np.uint64).reshape(K, 7) + 1, 128)),
                                 ("schnorr 1 signature (512 x 56)", csg.AIR_SCHNORR, lambda K: ctx.build_many_schnorr(csg.SignatureBatch(seed=K, num_sig=K)))]:
            for K in (64, 256, 1024):
                dev, pubs = build(K)
                ms, reports = mean_ms(lambda: ctx.validate_many_device(air, dev, pubs), args.reps)
                assert all(r.ok for r in reports)
                point = {"case": name, "K": K, "validate_many_device_ms": ms, "traces_per_s": round(K / ms * 1e3, 1)}
                batches.append(point)
                print(json.dumps(point), flush=True)
                del dev
                torch.cuda.empty_cache()
        result["batches"] = batches
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
