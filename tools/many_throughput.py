#!/usr/bin/env python3
"""Throughput of csg_prove_many against the single-proof path on the small proofs of tools/small_latency.py (the reference's own
bench sizes), where launches and Fiat-Shamir round trips, not arithmetic, set the time.

  python tools/many_throughput.py [--reps 5] [--ks 1,16,64,256,1024] [--threads 1,4,8] [--out profiles/r3_many_throughput.json]

Per case: proofs/s of one context proving batches of K (every batch holds the same trace K times: the work does not depend on the
values, and building K distinct witnesses on the host would dominate the run), K capped by count * width <= 65535, with the stage
times and launches of the batch; and in the same run the proofs/s of 1, 4 and 8 contexts proving one at a time (small_latency.py).
The card's name and power limit are recorded with the numbers."""
import argparse
import json
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import certificate_stark_b200 as csg  # noqa: E402
from small_latency import run as run_single  # noqa: E402

STAGES = ("h2d", "lde", "commit_trace", "constraints", "composition", "ood_deep", "fri", "queries")


def cases():
    seed = np.arange(42, 49, dtype=np.uint64)
    yield "range 64-bit", csg.AIR_RANGE, csg.build_range_trace(2**63 - 1), 8
    yield "rescue chain 128", csg.AIR_RESCUE, csg.build_rescue_trace(seed, 128), 4
    yield "merkle-update 1 tx", csg.AIR_MERKLE_UPDATE, csg.TransactionBatch(seed=2, num_tx=1).merkle_update_trace(), 8
    yield "schnorr 1 signature", csg.AIR_SCHNORR, csg.SignatureBatch(seed=3, num_sig=1).schnorr_trace(), 8
    yield "state-transition 1 tx", csg.AIR_TRANSACTION, csg.TransactionBatch(seed=1, num_tx=1).transaction_trace(), 8


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # noqa: BLE001 - recorded, not fatal
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5, help="timed batches per K")
    ap.add_argument("--single-reps", type=int, default=200, help="timed proofs per context of the single-proof figures")
    ap.add_argument("--ks", default="1,16,64,256,1024")
    ap.add_argument("--threads", default="1,4,8")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    ks, tlist = [int(x) for x in args.ks.split(",")], [int(x) for x in args.threads.split(",")]
    result = {"card": card(), "cases": []}
    print(json.dumps(result["card"]), flush=True)
    for name, air, (trace, pub), blowup in cases():
        opt = csg.ProofOptions(blowup_factor=blowup)
        rec = {"case": name, "trace": f"{trace.shape[1]} x {trace.shape[0]}", "many": {}}
        with csg.Context(0) as ctx:
            single = ctx.prove(air, trace, pub, opt)
            for K in ks:
                if K * trace.shape[0] > 65535:
                    continue
                traces, pubs = [trace] * K, np.stack([pub] * K)
                proofs = ctx.prove_many(air, traces, pubs, opt)   # warm-up: buffers, tables, modules
                assert all(p == single for p in proofs)
                t0 = time.perf_counter()
                for _ in range(args.reps):
                    ctx.prove_many(air, traces, pubs, opt)
                dt = time.perf_counter() - t0
                t = ctx.timings()
                rec["many"][str(K)] = {"proofs_per_s": round(K * args.reps / dt, 1), "ms_per_batch": round(dt / args.reps * 1e3, 3),
                                       "kernel_launches": int(t["kernel_launches"]), "host_total_ms": round(t["total"], 3),
                                       "stage_ms": {s: round(t[s], 3) for s in STAGES}}
        ctxs = [csg.Context(0) for _ in range(max(tlist))]
        for c in ctxs:
            c.set_air(air, trace.shape[1], pub, opt)
            c.load_trace(trace)
            assert c.prove_loaded() == single
            run_single(c, 5)
        for T in tlist:
            th = [threading.Thread(target=run_single, args=(ctxs[i], args.single_reps)) for i in range(T)]
            t0 = time.perf_counter()
            for x in th:
                x.start()
            for x in th:
                x.join()
            rec[f"single_proofs_per_s_{T}ctx"] = round(T * args.single_reps / (time.perf_counter() - t0), 1)
        for c in ctxs:
            c.close()
        result["cases"].append(rec)
        print(json.dumps(rec), flush=True)
    if args.out:
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
