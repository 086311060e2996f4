#!/usr/bin/env python3
"""bench.py -- proving throughput of the state-transition AIR (BASELINE.json: "prove ms & tx/s, state-transition AIR").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--num-tx T] [--impl reference] [--dump-outputs DIR]

A "step" is one complete proof (Prover::prove, /root/reference/src/lib.rs:140) of one synthetic batch of T transactions
(default 1024: trace 2^20 rows x 94 columns, blowup 8 -> 2^23 LDE rows; BASELINE.json configs[3]).  With N > 1 (launched
by torchrun, one rank per GPU) every rank proves its own batch: the path shards by independent proofs, there is no
data-path collective, scaling is weak -- that is `value`.  The same run then also proves ONE batch with all N GPUs together
(coset-sharded proof, NCCL exchanges; `sharded_proof` in the JSON line): the latency view of the same hardware.

  value     tx/s with the trace already resident in HBM when the timed region starts (device-event time, max over ranks)
  e2e       the same through csg_prove_trace() with the trace in page-locked HOST memory (csg_host_alloc): H2D copy and proof D2H
            inside the region; e2e_pageable: the same from ordinary pageable memory (what a Rust Vec<u64> is)
  roofline  the dominant kernel family by time (the 1024-point NTT passes: the whole LDE stage is launches of that one kernel):
            integer-issue fraction (warp instructions / s against 148 SMs x 4 schedulers x SM clock) with the HBM fraction beside it
  stage_roofline  every stage against both rooflines
  cpu_baseline  the CPU oracle (a port: the Rust reference cannot be built here) proving the SAME batch once, N=1 rank 0 only;
            its proof bytes are compared with the GPU's (`parity`)
--impl reference times that CPU port alone, with all host threads, on full-size batches.
--dump-outputs DIR writes the proof of the last timed step, one float32 value per byte, to DIR/proof.npy (DIR/proof_rank<r>.npy
with N > 1): the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True       # the tree may be read-only: no __pycache__ of the modules imported below

METRIC, UNIT = "state_transition_prove_throughput", "tx/s"
TRACE_WIDTH, ROWS_PER_TX, BLOWUP = 94, 1024, 8
CONSTRAINT_BYTES_PER_ROW = 8 * TRACE_WIDTH + 8      # every LDE row read once, one combined value written (SURVEY.md 8(d))
MODMUL_PER_ROW = 5922                               # SURVEY.md Appendix I: instrumented count of src/air.rs:383-610
# The constraint stage is four kernels (csrc/constraints.cu).  Algorithmic bytes per ce row of each: the columns it has to
# read once (8 B each) plus the partial sums it writes / reads (8 B each); DESIGN.md section 3.
CONS_KERNELS = {   # name: (description, algorithmic bytes per ce row, fraction of the ce rows visited, one kernel launch?)
    "cons_rescue": ("cons_low_kernel<TRANSACTION,0> (5 Rescue residuals per row, even ce cosets, split mode)", 5 * 14 * 8 + 5 * 6 * 8, 0.5, True),
    "cons_ecc_banks": ("phase: cons_ecc_low_kernel<TRANSACTION> (2 banks x 2 curve formulas, even ce cosets) + extension transforms + "
                       "cons_ecc_merge_kernel", 2 * 19 * 8 + 12 * 8 + 2 * 8, 1.0, False),
    # inside cons_ecc_banks: the largest single launch of a proof.  Per even-coset row: the 18 point columns of each bank and the
    # 12 key columns of the second one read once, 10 merged formula polynomials written
    "cons_ecc_low": ("cons_ecc_low_kernel<TRANSACTION> (doubling and mixed-addition formulas of both scalar-multiplication banks, "
                     "even ce cosets, split mode)", (2 * 18 + 12) * 8 + 10 * 8, 0.5, True),
    "cons_ecc_final": ("cons_item_kernel<TRANSACTION,2> (final point addition)", 36 * 8 + 4 * 8 + 8, 1.0, True),
    "cons_rest": ("phase: cons_low_kernel<TRANSACTION,3> (linear constraints, even cosets) + extension transforms + cons_final_kernel",
                  8 * TRACE_WIDTH + 8 * 8 + 8, 1.0, False),
}


# csrc/ files that hold no kernel of a single-GPU proof: the C++ host driver, the C-ABI wrappers and the collectives of sharded proofs.
# A change there moves launches around, not the instructions a launch executes (the launch counts per stage are measured live).
HOST_DRIVER_FILES = {"prover_ctx.cuh", "prover.cu", "abi_kernels.cu", "abi_witness.cu", "comm.cu", "comm.cuh"}


def csrc_sha16(read=None, include_host_driver=False):
    """fingerprint of the kernel sources: profiles/traffic.json (ncu counters of one proof) is only quoted when it was captured
    from exactly these sources.  read(name) -> bytes overrides the working tree (tools/restamp_traffic.py reads a commit)."""
    import hashlib
    h = hashlib.sha256()
    d = ROOT / "certificate_stark_b200" / "csrc"
    for f in sorted(list(d.glob("*.cu")) + list(d.glob("*.cuh")) + list(d.glob("*.h"))):
        if f.name in HOST_DRIVER_FILES and not include_host_driver:
            continue
        h.update(f.name.encode()); h.update(read(f.name) if read else f.read_bytes())
    return h.hexdigest()[:16]


# ncu counters of ONE proof of this workload (tools/make_traffic.py from the launch list of `bench.py --profile --steps 1`):
# per stage and for the dominant kernel, warp instructions executed and DRAM bytes.  Instruction counts are a property of the
# code and the workload, not of the run -- but only of the code they were taken from: stale captures are dropped, not restated.
TRAFFIC = {}
_t = ROOT / "profiles" / "traffic.json"
if _t.exists():
    try:
        TRAFFIC = json.loads(_t.read_text())
    except Exception:
        TRAFFIC = {}
TRAFFIC_FRESH = bool(TRAFFIC) and TRAFFIC.get("_captured_at", {}).get("kernel_sha16") == csrc_sha16()


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def stage_bytes(n):
    """algorithmic HBM bytes of each stage of one proof (SURVEY.md 8(d) per-unit figures x units; DESIGN.md section 3)"""
    rows, w, ce = n * BLOWUP, TRACE_WIDTH, BLOWUP
    fri = 0
    m = rows
    while m > 256:
        fri += 8 * m + 8 * m // 4 + 32 * m // 4 + 32 * (2 * (m // 4) - 1)   # layer in, folded layer out, row digests, tree
        m //= 4
    return {
        "lde": w * n * (16 + 8 + 8 * BLOWUP),                                    # K1 16 n + K2 8 n + 8 b n per column
        "commit_trace": rows * (8 * w + 32) + 32 * (2 * rows - 1),              # K3 8 w + 32 per row, K4 32 L + 32 (L - 1)
        "constraints": rows * CONSTRAINT_BYTES_PER_ROW,                          # K5: every LDE row read once, one merged value written
        "composition": 8 * rows * 2 + ce * n * (8 + 8 * BLOWUP) + rows * (8 * ce + 32) + 32 * (2 * rows - 1),   # K6 + LDE of ce columns + K3/K4
        "ood_deep": 8 * n * (w + ce) * 2 + 3 * n * (8 + 8 * BLOWUP) + rows * 32,  # K7 reads every coefficient; K8 combines them, extends 3 columns, 24 B in + 8 out per row
        "fri": fri,
    }


def stage_roofline(stage_ms, n, hbm_peak, int_peak_gwips=None, stage_insts=None):
    """Every stage against both rooflines.  HBM: the algorithmic bytes above / the stage's CUDA-event time against the measured
    copy bandwidth.  INT: warp instructions executed in the stage (ncu, profiles/traffic.json, only when captured from these
    sources) / the same time, against 148 SMs x 4 schedulers x the SM clock sampled during the run.  The arithmetic stages are
    integer-issue-bound (64-bit modular multiplication has no native instruction); the fractions say how far each is from either roof."""
    out = {}
    for k, nbytes in stage_bytes(n).items():
        ms = stage_ms.get(k) or 0.0
        gbs = nbytes / (ms / 1e3) / 1e9 if ms > 0 else None
        rec = {"algorithmic_bytes": int(nbytes), "ms": ms, "achieved": gbs, "unit": "GB/s", "peak": hbm_peak,
               "frac": gbs / hbm_peak if gbs and hbm_peak else None}
        wi = (stage_insts or {}).get(k, {}).get("warp_insts") if stage_insts else None
        if wi and ms > 0 and int_peak_gwips:
            gw = wi / (ms / 1e3) / 1e9
            rec["int"] = {"warp_insts": int(wi), "achieved": gw, "peak": int_peak_gwips, "unit": "Gwarp-inst/s", "frac": gw / int_peak_gwips}
            dram = (stage_insts or {}).get(k, {}).get("dram_bytes")
            if dram:
                rec["traffic"] = int(dram)
        out[k] = rec
    return out


class ClockSampler:
    """nvidia-smi clocks and throttle reasons sampled DURING the timed region"""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], threading.Event(), None

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def __enter__(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop_flag.set()
        self.thread.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mhz = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(s) > 2 + k and s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


def cpu_port_run(num_tx, steps, warmup, seed=1, want_proof=False):
    """the CPU oracle's prover (OpenMP, all host threads) on num_tx transactions; returns mean seconds per proof"""
    import certificate_stark_b200 as csg
    from oracle import pyoracle as O
    batch = csg.TransactionBatch(seed=seed, num_tx=num_tx)
    trace, pub = batch.transaction_trace()
    opt = O.options()
    for _ in range(warmup):
        O.prove(O.AIR_TRANSACTION, trace, pub, opt)
    t0 = time.perf_counter()
    for _ in range(steps):
        proof = O.prove(O.AIR_TRANSACTION, trace, pub, opt)
    sec = (time.perf_counter() - t0) / max(steps, 1)
    return (sec, proof) if want_proof else sec


def dump_proof(directory, name, proof):
    """--dump-outputs: proof bytes as float32 (exact for 0..255)"""
    np.save(Path(directory) / f"{name}.npy", np.frombuffer(proof, dtype=np.uint8).astype(np.float32))


def run_reference(args, rank, world):
    """--impl reference: the reference path's CPU implementation.  The reference is Rust over an un-vendored winterfell fork
    and no Rust toolchain exists in this image, so what runs is the C/OpenMP port of that path (oracle/) with all host threads,
    on FULL-SIZE batches of the configured workload.  One proof takes 20-100 s, so the number of steps actually run is capped by a
    time budget (`steps_run`; no warm-up beyond one small proof that loads the library and its tables)."""
    if rank != 0:
        return
    cpu_port_run(min(args.num_tx, 16), 1, 0)            # load the library, build the tables
    budget_s, times = float(os.environ.get("CSG_REFERENCE_BUDGET_S", "150")), []
    t_all = time.perf_counter()
    while len(times) < max(args.steps, 1) and (not times or time.perf_counter() - t_all + times[-1] <= budget_s):
        sec, proof = cpu_port_run(args.num_tx, 1, 0, seed=1000, want_proof=True)
        times.append(sec)
    if args.dump_outputs:
        dump_proof(args.dump_outputs, "proof", proof)
    sec = sum(times) / len(times)
    value = args.num_tx / sec
    cores = os.cpu_count() or 1
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "steps_run": len(times),
            "warmup": 0, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (f63 modular)",
            "data": "synthetic", "config": workload_config(args.num_tx, 1),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{len(times)} full proof(s) of a {args.num_tx}-transaction batch (trace {args.num_tx * ROWS_PER_TX} x 94, blowup 8), "
                                       f"{sec:.1f} s each, out of the {args.steps} steps asked for (time budget {budget_s:.0f} s); C/OpenMP port of the path, "
                                       "the Rust reference cannot be built here"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(num_tx, world):
    return {"workload": f"benches/state_transition.rs shape at {num_tx} transactions per proof: trace {num_tx * ROWS_PER_TX} x {TRACE_WIDTH}, blowup {BLOWUP}, "
                        f"42 queries, Blake3_256, FRI folding 4 (BASELINE.json configs[3]); one proof per GPU per step",
            "num_transactions": num_tx, "trace_rows": num_tx * ROWS_PER_TX, "lde_rows": num_tx * ROWS_PER_TX * BLOWUP, "proofs_per_step": world,
            "l2_policy": f"inputs larger than L2: {num_tx * ROWS_PER_TX * TRACE_WIDTH * 8 / 2**20:.0f} MiB trace, {num_tx * ROWS_PER_TX * BLOWUP * TRACE_WIDTH * 8 / 2**30:.2f} GiB LDE"
                         if num_tx >= 256 else "small batch: working set may fit L2",
            "parallelism": f"independent proofs x{world}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--num-tx", type=int, default=1024)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: 1 warm-up, no e2e leg, no CPU baseline (not a bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof of the last timed step to DIR/proof.npy (float32, one value per byte)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)      # a bad path fails before the timed work, not after it
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    # torchrun pins OMP_NUM_THREADS=1; the host-side witness builder and the CPU port are OpenMP code: give them the cores
    # (the reference arm runs on rank 0 alone and takes all of them)
    ncpu = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(ncpu if args.impl == "reference" else max(1, ncpu // max(world, 1)))
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's banner off stdout: rank 0 prints exactly one JSON line
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import certificate_stark_b200 as csg

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA path is the product, there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    num_tx = args.num_tx
    n = num_tx * ROWS_PER_TX
    opt = csg.ProofOptions()
    # synthetic batch (seeded per rank), witness built on the host straight into page-locked memory (csg_host_alloc)
    ctx = csg.Context(local_rank)
    pinned = csg.HostBuffer(TRACE_WIDTH, n)
    trace = pinned.array
    batch = csg.TransactionBatch(seed=1000 + rank, num_tx=num_tx)
    _, pub = batch.transaction_trace(out=trace)
    ctx.set_air(csg.AIR_TRANSACTION, n, pub, opt)

    def prove_resident():
        ctx.reload_resident_trace()
        return ctx.prove_loaded()

    def prove_e2e():
        return ctx.prove_trace_ptr(pinned.ptr)      # csg_prove_trace: host buffer in, proof bytes out

    ctx.load_trace_ptr(pinned.ptr)
    proof = None
    warmup = 1 if args.profile else max(args.warmup, 3)
    for _ in range(warmup):
        proof = prove_resident()

    # ---- timed region 1: trace resident in HBM
    stage_sum, launches, stage_launches = {}, 0, {}
    with ClockSampler(local_rank) as clocks:
        barrier()
        ctx.timer_start()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            p = prove_resident()
            t = ctx.timings()
            launches += int(t["kernel_launches"])
            for k, v in t.items():
                if k not in ("total", "kernel_launches", "stage_launches"):
                    stage_sum[k] = stage_sum.get(k, 0.0) + v
            stage_launches = t["stage_launches"]
            assert p == proof, "non-deterministic proof"
        dev_ms = ctx.timer_stop()     # CUDA events on the proving stream around the K steps
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
    clock_summary = clocks.summary()
    if args.dump_outputs:
        dump_proof(args.dump_outputs, "proof" if world == 1 else f"proof_rank{rank}", p)

    # ---- timed region 2: end to end through the C ABI with host buffers (a) page-locked, (b) pageable
    e2e_ms, e2e_h2d_ms, e2e_pg_ms, e2e_pipe_ms = 0.0, 0.0, 0.0, 0.0
    if not args.profile:
        assert prove_e2e() == proof, "the end-to-end path gives a different proof"
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            p = prove_e2e()
            e2e_h2d_ms += ctx.timings()["h2d"]     # first byte .. last byte of the copy, on the copy stream (it runs under the extension)
        e2e_ms = ctx.timer_stop()
        barrier()
        pageable = np.array(trace)                 # ordinary host memory: what a Rust Vec<u64> is
        assert ctx.prove_trace_ptr(pageable.ctypes.data) == proof
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            ctx.prove_trace_ptr(pageable.ctypes.data)
        e2e_pg_ms = ctx.timer_stop()
        barrier()
        del pageable
        # (c) a stream of batches (csg_prefetch_trace / csg_prove_prefetched): every step proves the trace copied under the
        # previous step and starts the copy of the next one -- K proofs and K copies of 788 MB inside the region
        ctx.prefetch_trace_ptr(pinned.ptr)
        assert ctx.prove_prefetched_ptr(pinned.ptr) == proof
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            ctx.prove_prefetched_ptr(pinned.ptr)
        e2e_pipe_ms = ctx.timer_stop()
        barrier()
        assert ctx.prove_prefetched_ptr() == proof      # the copy still waiting

    # ---- timed region 3: TransactionExample::prove() as a whole = build_trace + prove, with the witness built on the device
    wit_ms = 0.0
    if not args.profile:
        ctx.build_transaction_trace(batch)
        assert ctx.prove_loaded() == proof, "device-built witness gives a different proof"
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            ctx.build_transaction_trace(batch)
            p = ctx.prove_loaded()
        wit_ms = ctx.timer_stop()
        barrier()

    # ---- timed region 4 (N > 1): ONE proof sharded over the N GPUs by LDE coset (csg_dist_*, NCCL exchanges on the proving
    # stream): the batch of rank 0, proved by all ranks together; every rank must return rank 0's single-GPU proof bytes
    sh_ms, sh_e2e_ms, sh_comm_ms, sh_stage = 0.0, 0.0, 0.0, {}
    if world > 1 and not args.profile and BLOWUP % world == 0:
        import hashlib
        if rank != 0:
            _, pub0 = csg.TransactionBatch(seed=1000, num_tx=num_tx).transaction_trace(out=trace)
        else:
            pub0 = pub
        sctx = csg.Context(local_rank)
        ok = torch.ones(1, device="cuda")
        try:
            sctx.dist_init_torch()
        except csg.CsgError as e:          # e.g. libnccl not loadable: the throughput numbers above do not depend on this leg
            print(f"[bench] sharded-proof leg skipped on rank {rank}: {e}", file=sys.stderr)
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        run_sharded = bool(ok.item())
    else:
        run_sharded = False
    if run_sharded:
        import hashlib
        sctx.set_air(csg.AIR_TRANSACTION, n, pub0, opt)
        sctx.load_trace_ptr(pinned.ptr)
        for _ in range(3):
            sctx.reload_resident_trace()
            sp = sctx.prove_loaded()
        digests = [None] * world
        dist.all_gather_object(digests, hashlib.sha256(sp).hexdigest())
        if rank == 0:
            assert all(d == hashlib.sha256(proof).hexdigest() for d in digests), "sharded proof differs from the single-GPU proof"
        barrier()
        sctx.timer_start()
        for _ in range(args.steps):
            sctx.reload_resident_trace()
            sctx.prove_loaded()
            t = sctx.timings()
            sh_comm_ms += t["comm"]
            for k, v in t.items():
                if k not in ("total", "kernel_launches", "stage_launches"):
                    sh_stage[k] = sh_stage.get(k, 0.0) + v
        sh_ms = sctx.timer_stop()
        barrier()
        sctx.prove_trace_ptr(pinned.ptr)
        barrier()
        sctx.timer_start()
        for _ in range(args.steps):
            sctx.prove_trace_ptr(pinned.ptr)
        sh_e2e_ms = sctx.timer_stop()
        barrier()
        sctx.close()

    times = torch.tensor([dev_ms, wall_ms, e2e_ms, wit_ms, sh_ms, sh_e2e_ms, sh_comm_ms, e2e_pg_ms, e2e_pipe_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms, e2e_ms, wit_ms, sh_ms, sh_e2e_ms, sh_comm_ms, e2e_pg_ms, e2e_pipe_ms = [float(x) for x in times.cpu()]

    if rank == 0:
        steps = max(args.steps, 1)
        ms_per_step = dev_ms / steps
        value = world * num_tx / (ms_per_step / 1e3)
        hbm_peak, peak_src, sm_max = measured_peaks()
        cons_ms = stage_sum.get("constraints", 0.0) / steps
        rows = n * BLOWUP
        kernels = {k: {"kernel": CONS_KERNELS[k][0], "launch_ms": stage_sum.get(k, 0.0) / steps,
                       "algorithmic_bytes_per_launch": int(rows * CONS_KERNELS[k][2]) * CONS_KERNELS[k][1]} for k in CONS_KERNELS}
        for v in kernels.values():
            v["achieved_gbs"] = v["algorithmic_bytes_per_launch"] / (v["launch_ms"] / 1e3) / 1e9 if v["launch_ms"] > 0 else None
        # The dominant kernel FAMILY by time is the 1024-point NTT pass (`ntt1024_kernel`, ~40 % of a proof); the LDE stage is
        # nothing but launches of it (the representation change rides on the inverse transform), so its per-launch time is measured
        # live: stage CUDA-event time / launches in the stage.  It is integer-issue-bound, so the headline fraction is the INT one
        # (warp instructions from the ncu capture of these very sources / time, against 148 x 4 schedulers x the sampled SM clock);
        # the HBM fraction of the algorithmic bytes (DESIGN.md section 3) stands beside it.
        stage_ms = {k: v / steps for k, v in stage_sum.items()}
        lde_ms, lde_launches = stage_ms.get("lde", 0.0), int(stage_launches.get("lde", 0)) or 1
        launch_ms = lde_ms / lde_launches
        alg_bytes = stage_bytes(n)["lde"] / lde_launches
        hbm_achieved = alg_bytes / (launch_ms / 1e3) / 1e9 if launch_ms > 0 else None
        clk_mhz = clock_summary.get("sm_mhz") or sm_max
        int_peak = 148 * 4 * clk_mhz * 1e6 / 1e9          # Gwarp-inst/s: one warp instruction per scheduler per clock
        fresh = TRAFFIC if TRAFFIC_FRESH else {}
        lde_cap = fresh.get("stages", {}).get("lde", {})
        roof = {"kernel": f"ntt1024_kernel (1024-point sub-transform passes of every size-2^20 NTT; the LDE stage = {lde_launches} launches of it per proof)",
                "launch_ms": launch_ms, "launches_per_step": lde_launches, "algorithmic_bytes_per_launch": int(alg_bytes),
                "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": (hbm_achieved / hbm_peak) if hbm_achieved else None, "peak_source": peak_src},
                "traffic": None}
        if lde_cap.get("warp_insts") and launch_ms > 0:
            wi = lde_cap["warp_insts"] / lde_launches
            gw = wi / (launch_ms / 1e3) / 1e9
            roof.update({"bound": "int", "achieved": gw, "peak": int_peak, "unit": "Gwarp-inst/s", "frac": gw / int_peak,
                         "warp_insts_per_launch": int(wi), "thread_insts_per_element": lde_cap["warp_insts"] * 32 / (TRACE_WIDTH * n * (1 + BLOWUP)) / 2,
                         "peak_source": f"148 SMs x 4 schedulers x {clk_mhz:.0f} MHz (SM clock sampled during the timed region)",
                         "pipes": lde_cap.get("pipes"), "traffic": int(lde_cap["dram_bytes"] / lde_launches) if lde_cap.get("dram_bytes") else None,
                         "captured_at": TRAFFIC.get("_captured_at")})
        else:   # no ncu capture of these sources: only the HBM view can be stated
            roof.update({"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": (hbm_achieved / hbm_peak) if hbm_achieved else None,
                         "note": "integer-issue-bound kernel; profiles/traffic.json was not captured from these sources, so no instruction counts are quoted"})
        roof["constraint_stage"] = {"ms": cons_ms, "kernels": kernels,
                                    "reference_modmul_per_s": rows * MODMUL_PER_ROW / (cons_ms / 1e3) if cons_ms > 0 else None}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (f63 modular)",
            "data": "synthetic", "config": workload_config(num_tx, world),
            "proofs_per_s": world / (ms_per_step / 1e3), "wall_ms_per_step": wall_ms / steps, "proof_bytes": len(proof),
            "stage_ms": stage_ms, "stage_launches": stage_launches,
            "e2e": {"value": (world * num_tx / (e2e_ms / steps / 1e3)) if e2e_ms else None, "unit": UNIT, "ms_per_step": e2e_ms / steps,
                    "h2d_ms_per_step": e2e_h2d_ms / steps, "h2d_bytes_per_step": int(TRACE_WIDTH * n * 8), "d2h_bytes_per_step": int(len(proof)),
                    "host_memory": "page-locked (csg_host_alloc); the copy runs on its own stream under the trace extension"},
            "e2e_pageable": {"value": (world * num_tx / (e2e_pg_ms / steps / 1e3)) if e2e_pg_ms else None, "unit": UNIT, "ms_per_step": e2e_pg_ms / steps,
                             "host_memory": "pageable (numpy array): staged through the library's pinned ring by the host threads"},
            "e2e_pipelined": {"value": (world * num_tx / (e2e_pipe_ms / steps / 1e3)) if e2e_pipe_ms else None, "unit": UNIT, "ms_per_step": e2e_pipe_ms / steps,
                              "note": "a stream of batches through csg_prefetch_trace / csg_prove_prefetched: the 788 MB copy of the NEXT batch runs on its own "
                                      "stream under the proof of the current one (page-locked memory, two trace buffers in HBM); K proofs and K copies in the region. "
                                      "`e2e` above is the strict form: copy and proof of the SAME batch inside every step"},
            "build_trace_and_prove": {"value": (world * num_tx / (wit_ms / steps / 1e3)) if wit_ms else None, "unit": UNIT, "ms_per_step": wit_ms / steps,
                                      "note": "TransactionExample::prove() as a whole: witness generated on the device (csg_build_trace_transaction_device), "
                                              "2.2 KB per transaction H2D, then the proof; the host builder needs ~0.4 s for the same batch.  With "
                                              "csg_tx_batch_build_device the batch metadata (account tree, paths, signatures) is built by kernels too: +23 ms "
                                              "instead of 1.3 s on the host (tools/batch_time.py, profiles/r2_batch_time.json)"},
            "gpu_launches": launches,
            "clocks": clock_summary,
            "roofline": roof,
        }
        try:
            line["stage_roofline"] = stage_roofline(stage_ms, n, hbm_peak, int_peak, fresh.get("stages"))
        except Exception as e:   # a reporting extra: never lets the bench line go missing
            line["stage_roofline"] = {"error": repr(e)}
        if sh_ms:
            line["sharded_proof"] = {
                "note": f"ONE proof of the same {num_tx}-transaction batch split over the {world} GPUs by LDE coset (each GPU owns {BLOWUP // world} of the "
                        f"{BLOWUP} cosets and the Merkle subtree of 1/{world} of the leaves; NCCL all-gathers of coefficients, composition slices, out-of-domain values, "
                        "DEEP evaluations and subtree roots, one all-to-all of leaf digests per commitment, sums of opened rows and path nodes); proof bytes "
                        "identical to the single-GPU proof on every rank; times are device events, max over ranks",
                "ms_per_proof": sh_ms / steps, "tx_per_s": num_tx / (sh_ms / steps / 1e3), "speedup_vs_one_gpu": ms_per_step / (sh_ms / steps),
                "comm_ms_per_proof": sh_comm_ms / steps, "stage_ms_rank0": {k: v / steps for k, v in sh_stage.items()},
                "e2e_ms_per_proof": sh_e2e_ms / steps, "e2e_tx_per_s": num_tx / (sh_e2e_ms / steps / 1e3),
                "e2e_h2d_bytes_per_rank": int(-(-TRACE_WIDTH // world) * n * 8)}
        if world == 1 and not args.no_cpu_baseline and not args.profile:
            # the CPU port proves the SAME batch once (20-100 s on the box's cores): the baseline at the metric's own config, and
            # the byte-for-byte check of the timed GPU proof against the oracle, outside every timed region
            import hashlib
            sec, cpu_proof = cpu_port_run(num_tx, 1, 0, seed=1000 + rank, want_proof=True)
            line["cpu_baseline"] = {"value": num_tx / sec, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                    "sample": f"one proof of the same {num_tx}-transaction batch (trace {num_tx * ROWS_PER_TX} x 94, blowup 8): {sec:.2f} s; "
                                              "C/OpenMP port of the path (oracle/), the Rust reference cannot be built here"}
            line["parity"] = {"gpu_proof_sha256": hashlib.sha256(proof).hexdigest(), "oracle_proof_sha256": hashlib.sha256(cpu_proof).hexdigest(),
                              "identical": proof == cpu_proof, "oracle": "oracle/ (C restatement; parity unpinned against the Rust reference)"}
            assert proof == cpu_proof, "the timed GPU proof differs from the CPU oracle's proof of the same batch"
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException as exc:   # noqa: BLE001
        if isinstance(exc, SystemExit) and exc.code in (0, None):
            raise
        # A rank that fails must END, at once: its peers are blocked inside collectives that it will never join, and the normal
        # interpreter shutdown of a process whose CUDA context has faulted can itself block in the NCCL / CUDA teardown -- the
        # launcher then never sees the failure and the whole job sits there until someone's time limit kills it.
        import traceback
        traceback.print_exc()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(exc.code if isinstance(exc, SystemExit) and isinstance(exc.code, int) else 1)
