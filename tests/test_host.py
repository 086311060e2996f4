"""CPU tests of the product's host side: the C-ABI library loads and exports what include/csg.h declares, the host-compiled
halves (AIR descriptors, fused per-row constraint evaluation, batch-opening shapes, transcript hashes) agree with the oracle,
and nothing pretends to work without the CUDA device."""
import ctypes as C
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol(csg):
    header = (ROOT / "include" / "csg.h").read_text()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    names = sorted(set(re.findall(r"\b(csg_[a-z0-9_]+)\s*\(", header)))
    assert len(names) >= 35
    L = C.CDLL(str(csg.LIB_PATH))
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, f"declared in csg.h but not exported: {missing}"


def test_ctypes_mirrors_match_the_header_layout(csg, tmp_path):
    # the structs that cross the C ABI by value or by pointer: size and the offset of the last field, as gcc lays out include/csg.h
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "csg.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(csg_options), sizeof(csg_shard_plan), sizeof(csg_timings), '
                   'offsetof(csg_timings, kernel_launches), offsetof(csg_timings, cons_ecc_low), offsetof(csg_timings, stage_launches)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)])
    opt, plan, tim, off_launches, off_last, off_stage = map(int, subprocess.check_output([str(exe)]).split())
    assert C.sizeof(csg.ProofOptions) == opt
    assert C.sizeof(csg.ShardPlan) == plan
    assert C.sizeof(csg.Timings) == tim
    assert csg.Timings.kernel_launches.offset == off_launches and csg.Timings.cons_ecc_low.offset == off_last
    assert csg.Timings.stage_launches.offset == off_stage


NO_DEVICE = r"""
import sys
sys.path.insert(0, sys.argv[1])
import certificate_stark_b200 as csg
for make in (lambda: csg.Context(0), lambda: csg.get_example(2)):
    try:
        make()
    except csg.CsgError as e:
        print(e)
    else:
        raise SystemExit("created without a CUDA device")
assert b"no context" in csg.lib().csg_last_error(None)
"""


def test_no_cpu_fallback(csg):
    # with no CUDA device visible (hidden from a child process, so that this also runs on a machine with a GPU) every entry
    # point raises instead of computing on the CPU
    out = subprocess.run([sys.executable, "-c", NO_DEVICE, str(ROOT)], capture_output=True, text=True,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, (out.stdout + out.stderr)[-2000:]
    assert "no CPU fallback" in out.stdout.splitlines()[0]


def test_host_harness_against_oracle(oracle, tmp_path):
    # compiles airs.cuh / air_desc.cpp / transcript.hpp for the host and checks them against the oracle (see host_harness.cpp)
    exe = tmp_path / "host_harness"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fopenmp", str(ROOT / "tests" / "host_harness.cpp"), "-x", "c++",
                           str(ROOT / "certificate_stark_b200" / "csrc" / "host" / "air_desc.cpp"), f"-L{ROOT / 'oracle'}", "-l:liboracle.so",
                           f"-Wl,-rpath,{ROOT / 'oracle'}", "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and "all checks passed" in out.stdout, out.stdout[-2000:]


def test_witness_builders_reject_bad_shapes(csg):
    with pytest.raises(csg.CsgError):
        csg.build_rescue_trace(np.arange(7, dtype=np.uint64), 3)
    with pytest.raises(csg.CsgError):
        csg.TransactionBatch(seed=1, num_tx=3).transaction_trace()
    with pytest.raises(csg.CsgError):
        csg.TransactionBatch(seed=1, num_tx=0)
    with pytest.raises(csg.CsgError):
        csg.TransactionExample(csg.ProofOptions(), 3)          # src/lib.rs:100-103


def test_witness_is_deterministic_in_the_seed(csg):
    a, pa = csg.TransactionBatch(seed=11, num_tx=2).transaction_trace()
    b, pb = csg.TransactionBatch(seed=11, num_tx=2).transaction_trace()
    c, _ = csg.TransactionBatch(seed=12, num_tx=2).transaction_trace()
    assert np.array_equal(a, b) and np.array_equal(pa, pb) and not np.array_equal(a, c)
    assert a.shape == (94, 2048) and int(a.max()) < csg.P


def test_range_trace_layout(csg):
    # src/range/prover.rs:74-84: column 0 = bits from the most significant one, column 1 = running value
    trace, pub = csg.build_range_trace(0b1011)
    assert int(pub[0]) == 0b1011 and int(trace[1, 63]) == 0b1011 and [int(v) for v in trace[0, 60:64]] == [1, 0, 1, 1]
    assert int(trace[1, 0]) == 0


def test_proof_options_mirror(csg):
    o = csg.ProofOptions()
    assert (o.num_queries, o.blowup_factor, o.grinding_factor, o.hash_fn, o.field_extension, o.fri_folding_factor, o.fri_max_remainder_size) == \
        (42, 8, 0, csg.HASH_BLAKE3_256, 1, 4, 256)      # get_example, src/lib.rs:78-86


def test_product_verifier_accepts_valid_and_rejects_invalid_proofs(csg, oracle):
    # csg_verify = winterfell::verify (src/lib.rs:144-150): host-only, so it is tested here against proofs from the CPU oracle,
    # with the reference's own test pattern: accept, reject wrong public inputs (src/tests.rs:32-37), reject tampering
    z = np.zeros(14, dtype=np.uint64)
    batch = csg.TransactionBatch(seed=2, num_tx=2)
    cases = [(csg.AIR_RESCUE, csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 16), 4, 2),
             (csg.AIR_RANGE, csg.build_range_trace(2**63 - 1), 8, 3),
             (csg.AIR_MERKLE_INIT, csg.build_merkle_init_trace(z, z, 1), 4, 2),
             (csg.AIR_MERKLE_UPDATE, batch.merkle_update_trace(), 8, 2),
             (csg.AIR_TRANSACTION, batch.transaction_trace(), 8, 2),
             (csg.AIR_SCHNORR, csg.SignatureBatch(seed=2, num_sig=2).schnorr_trace(), 8, 2)]
    for air, (trace, pub), blowup, hash_fn in cases:
        proof = oracle.prove(air, trace, pub, oracle.options(blowup=blowup, hash_fn=hash_fn))
        assert csg.verify(air, pub, proof) == 0
        assert oracle.verify(air, pub, proof) == 0
        wrong = pub.copy()
        wrong[-1] = (int(wrong[-1]) + 1) % csg.P
        assert csg.verify(air, wrong, proof) == 17                      # inconsistent out-of-domain evaluations
        for where in (len(proof) // 3, len(proof) // 2, len(proof) - 20):
            bad = bytearray(proof)
            bad[where] ^= 0x40
            assert csg.verify(air, pub, bytes(bad)) != 0, f"air {air}: flipped bit at {where} accepted"
        assert csg.verify(air, pub, proof[:-1]) == 16 and csg.verify(air, pub, proof + b"\0") == 16
        assert csg.verify((air + 1) % 6, pub, proof) != 0


def test_verifier_rejects_weak_or_malformed_contexts(csg, oracle):
    # ADVICE round 1: the context bytes of a proof are attacker-controlled.  (a) log2 fields out of range must not be shifted
    # (a blowup byte of 35 used to behave like 3); (b) a non-empty trace-meta blob is bound to nothing; (c) options that end the
    # FRI domain below 8 elements used to index before the start of a heap buffer; (d) an acceptance check needs a floor.
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 16)
    proof = oracle.prove(csg.AIR_RESCUE, trace, pub, oracle.options(blowup=4))
    assert csg.verify(csg.AIR_RESCUE, pub, proof) == 0
    # context layout: width, log n, meta length (2), modulus length, modulus (8), queries, log blowup, grinding, hash, extension, log folding, log remainder
    assert proof[0] == 14 and proof[2:4] == b"\0\0" and proof[4] == 8 and proof[14] == 2
    for off, val in [(14, 34), (14, 0), (14, 6), (18, 3), (18, 34), (19, 1), (19, 11), (19, 40), (15, 32), (1, 41)]:
        bad = bytearray(proof)
        bad[off] = val
        assert csg.verify(csg.AIR_RESCUE, pub, bytes(bad)) == 16, f"context byte {off} = {val} not rejected as malformed"
    meta = proof[:2] + b"\x01\x00\xaa" + proof[4:]
    assert csg.verify(csg.AIR_RESCUE, pub, meta) == 16
    # blowup 2 and remainder 4 on a 4^k domain end at 2 elements: the prover refuses these options, so must the verifier
    rt, rp = csg.build_range_trace(77)
    rproof = bytearray(oracle.prove(csg.AIR_RANGE, rt, rp, oracle.options(blowup=8)))
    rproof[14], rproof[19] = 1, 2          # 64 * 2 = 128 -> 32 -> 8 -> 2
    assert csg.verify(csg.AIR_RANGE, rp, bytes(rproof)) == 16
    # the floor: 42 queries expected, a proof with 8 (or grinding below, another hash, a smaller blowup) is refused before any work
    weak = oracle.prove(csg.AIR_RESCUE, trace, pub, oracle.options(blowup=4, num_queries=8))
    assert csg.verify(csg.AIR_RESCUE, pub, weak) == 0
    assert csg.verify(csg.AIR_RESCUE, pub, weak, csg.ProofOptions(blowup_factor=4)) == 22
    assert csg.verify(csg.AIR_RESCUE, pub, proof, csg.ProofOptions(blowup_factor=4)) == 0
    assert csg.verify(csg.AIR_RESCUE, pub, proof, csg.ProofOptions(blowup_factor=8)) == 22
    assert csg.verify(csg.AIR_RESCUE, pub, proof, csg.ProofOptions(blowup_factor=4, grinding_factor=8)) == 22
    assert csg.verify(csg.AIR_RESCUE, pub, proof, csg.ProofOptions(blowup_factor=4, hash_fn=csg.HASH_SHA3_256)) == 22
    assert csg.verify(csg.AIR_RESCUE, pub, proof, csg.ProofOptions(blowup_factor=2, num_queries=10, fri_max_remainder_size=1024)) == 0


@pytest.mark.parametrize("seed,num_tx,depth", [(1, 1, 15), (7, 8, 15), (5, 4, 3), (9, 16, 7), (3, 64, 15)])
def test_device_batch_plan_executed_on_the_host_gives_the_host_builders_records(csg, seed, num_tx, depth):
    # the plan of the device-side batch builder (csrc/host/batch_plan.hpp: node versions of the account tree, the children each
    # merges, the versions every path reads) executed with host hashes must reproduce the sequential builder bit for bit;
    # depth 3 (the reference's cfg(test) tree) makes slots collide: repeated accounts, senders that were receivers before
    L = csg.lib()
    L.csg_debug_tx_batch_plan_records.restype = C.c_int
    L.csg_debug_tx_batch_plan_records.argtypes = [C.c_uint64, C.c_size_t, C.c_uint, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    got, pub = np.zeros((num_tx, 278), dtype=np.uint64), np.zeros(14, dtype=np.uint64)
    assert L.csg_debug_tx_batch_plan_records(seed, num_tx, depth, got.ctypes.data_as(C.POINTER(C.c_uint64)), pub.ctypes.data_as(C.POINTER(C.c_uint64))) == 0
    want = csg.TransactionBatch(seed=seed, num_tx=num_tx, tree_depth=depth)
    assert np.array_equal(pub, want.public_inputs())
    bad = np.argwhere(got != want.packed_records())
    assert bad.size == 0, f"first differing (transfer, word): {bad[0]}"
    assert L.csg_debug_tx_batch_plan_records(seed, 0, depth, got.ctypes.data_as(C.POINTER(C.c_uint64)), pub.ctypes.data_as(C.POINTER(C.c_uint64))) != 0


def test_bench_stage_roofline_arithmetic():
    # bench.py's HBM view of the LDE and commitment stages: SURVEY.md 8(d) bytes / stage time, on the round-1 stage times
    import bench
    n = 1 << 20
    r = bench.stage_roofline({"lde": 18.94, "commit_trace": 4.38}, n, 6544.0)
    assert r["lde"]["algorithmic_bytes"] == 94 * n * 88 and r["commit_trace"]["algorithmic_bytes"] == (8 * n) * 784 + 32 * (16 * n - 1)
    assert abs(r["lde"]["achieved"] - 94 * n * 88 / 18.94e-3 / 1e9) < 1e-6 and 0.06 < r["lde"]["frac"] < 0.08
    assert 0.2 < r["commit_trace"]["frac"] < 0.3
    assert bench.stage_roofline({}, n, 6544.0)["lde"]["achieved"] is None   # a missing stage does not raise


def test_committed_counters_belong_to_the_committed_kernels():
    # profiles/traffic.json (ncu counters of one proof) is what bench.py's INT roofline quotes; it carries a fingerprint of the kernel
    # sources it was captured from and bench.py drops it when the kernels have changed since.  In a committed tree the two must agree:
    # a kernel change without a new counter pass would silently turn the bench line's roofline back into the HBM-only form.
    import bench
    cap = bench.TRAFFIC.get("_captured_at", {})
    assert cap.get("kernel_sha16") == bench.csrc_sha16(), "kernel sources changed since the ncu counter pass: re-run tools/gpu_calls/run_s3a.sh (tools/make_traffic.py)"
    assert bench.TRAFFIC_FRESH
    # host-driver files are outside the fingerprint, kernels are inside
    assert "prover_ctx.cuh" in bench.HOST_DRIVER_FILES and "ntt.cu" not in bench.HOST_DRIVER_FILES and "airs.cuh" not in bench.HOST_DRIVER_FILES
    assert bench.csrc_sha16(include_host_driver=True) != bench.csrc_sha16()


def test_verifier_survives_mutated_proofs(csg, oracle, tmp_path):
    # A proof is attacker-controlled input.  tests/fuzz_verifier.cpp mutates valid proofs (bit flips, blown-up length fields,
    # truncation, insertions, deletions, spliced and zeroed runs; half of the single-byte mutations aim at the context bytes) and
    # calls the product's verifier, compiled here with AddressSanitizer and UBSan: every mutation must be rejected -- no crash, no
    # sanitizer report, no acceptance.  (A longer campaign -- 20 000 mutations x 4 seeds x 5 proofs, plus 3 000 each of the
    # transaction, Schnorr and Merkle-update proofs -- ran clean at the end of round 2.)
    exe = tmp_path / "fuzz_verifier"
    host = ROOT / "certificate_stark_b200" / "csrc" / "host"
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fopenmp", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                           str(ROOT / "tests" / "fuzz_verifier.cpp"), "-x", "c++", str(host / "verifier.cpp"), str(host / "air_desc.cpp"), "-o", str(exe)])
    cases = [(csg.AIR_RESCUE, csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 16), dict(blowup=4), 600),
             (csg.AIR_RANGE, csg.build_range_trace(77), dict(blowup=8, field_extension=2), 600),
             (csg.AIR_RESCUE, csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 16), dict(blowup=4, field_extension=3, hash_fn=3), 250),
             (csg.AIR_SCHNORR, csg.SignatureBatch(seed=2, num_sig=1).schnorr_trace(), dict(blowup=8), 100)]
    for k, (air, (trace, pub), opts, iters) in enumerate(cases):
        proof = oracle.prove(air, trace, pub, oracle.options(**opts))
        (tmp_path / f"{k}.proof").write_bytes(proof)
        pub.astype(np.uint64).tofile(tmp_path / f"{k}.pub")
        out = subprocess.run([str(exe), str(air), str(tmp_path / f"{k}.pub"), str(tmp_path / f"{k}.proof"), str(iters), str(1000 + k)],
                             capture_output=True, text=True, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
        assert out.returncode == 0 and "accepted 0" in out.stdout, (out.stdout + out.stderr)[-3000:]


def test_host_builders_are_sanitizer_clean(tmp_path):
    # the host witness / batch builders write into caller buffers sized by the header's comments (94 x 1024*num_tx, 65 x 512*num_tx,
    # 56 x 512*num_sig, 38*num_sig, ...): tests/host_sanitize.cpp gives them exact-size heap buffers under ASan + UBSan + LSan
    exe = tmp_path / "host_sanitize"
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fopenmp", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                           str(ROOT / "tests" / "host_sanitize.cpp"), "-x", "c++", str(ROOT / "certificate_stark_b200" / "csrc" / "host" / "witness.cpp"), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=1"))
    assert out.returncode == 0 and "0 failures" in out.stdout, (out.stdout + out.stderr)[-3000:]
