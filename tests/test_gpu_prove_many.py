"""csg_prove_many (-m gpu): K independent proofs of one AIR through one launch sequence.  Every proof of a batch must be the byte
string csg_prove returns for the same trace and public inputs (and, where marked, the CPU oracle's), and every proof of a valid
witness must verify."""
import ctypes as C
import hashlib
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
P = 0x4180000000000001


# ---------------------------------------------------------------------------------------------- witnesses: K distinct ones per AIR
def witnesses(csg, air_id, count, seed=0):
    rng = np.random.default_rng(seed + 1000 * air_id + count)
    out = []
    for k in range(count):
        s = seed + k + 1
        if air_id == csg.AIR_RANGE:
            out.append(csg.build_range_trace(int(rng.integers(0, 2**63))))
        elif air_id == csg.AIR_RESCUE:
            out.append(csg.build_rescue_trace(np.arange(s, s + 7, dtype=np.uint64), 128))
        elif air_id == csg.AIR_MERKLE_INIT:
            z = np.zeros(14, dtype=np.uint64)
            out.append(csg.build_merkle_init_trace(z, z, s))
        elif air_id == csg.AIR_MERKLE_UPDATE:
            out.append(csg.TransactionBatch(seed=s, num_tx=1).merkle_update_trace())
        elif air_id == csg.AIR_SCHNORR:
            out.append(csg.SignatureBatch(seed=s, num_sig=1).schnorr_trace())
        else:
            out.append(csg.TransactionBatch(seed=s, num_tx=1).transaction_trace())
    return [t for t, _ in out], np.stack([p for _, p in out])


def oracle_options(oracle, opt):
    return oracle.options(num_queries=opt.num_queries, blowup=opt.blowup_factor, grinding=opt.grinding_factor, hash_fn=opt.hash_fn,
                          max_remainder=opt.fri_max_remainder_size)


def check_batch(ctx, csg, air_id, traces, pubs, opt, oracle=None, oracle_at=None, repr=0):
    proofs = ctx.prove_many(air_id, traces, pubs, opt, repr=repr)
    assert len(proofs) == len(traces)
    for k, proof in enumerate(proofs):
        assert proof == ctx.prove(air_id, traces[k], pubs[k], opt, repr=repr), f"proof {k} differs from the single-proof path"
    for k in (range(len(traces)) if oracle_at is None else oracle_at):
        if oracle is not None:
            t = traces[k] if repr == 0 else oracle.from_mont_fast(traces[k])
            assert proofs[k] == oracle.prove(air_id, t, pubs[k], oracle_options(oracle, opt)), f"proof {k} differs from the oracle's"
    return proofs


AIRS = ["TRANSACTION", "MERKLE_UPDATE", "MERKLE_INIT", "SCHNORR", "RANGE", "RESCUE"]


@pytest.mark.parametrize("count", [1, 3, 16])
@pytest.mark.parametrize("air", AIRS)
def test_each_air_matches_single_path_and_oracle(ctx, oracle, csg, air, count):
    air_id = getattr(csg, "AIR_" + air)
    traces, pubs = witnesses(csg, air_id, count)
    opt = csg.ProofOptions(blowup_factor=4 if air_id == csg.AIR_RESCUE else 8)
    proofs = check_batch(ctx, csg, air_id, traces, pubs, opt, oracle)
    for k, proof in enumerate(proofs):
        assert csg.verify(air_id, pubs[k], proof) == 0


@pytest.mark.parametrize("air,kw", [
    ("RANGE", dict(hash_fn=3)), ("RESCUE", dict(hash_fn=3, blowup_factor=4)),
    ("RANGE", dict(blowup_factor=4)), ("RANGE", dict(blowup_factor=16)), ("RESCUE", dict(blowup_factor=16)),
    ("TRANSACTION", dict(blowup_factor=16)), ("SCHNORR", dict(blowup_factor=16)),
    ("RANGE", dict(num_queries=1)), ("RANGE", dict(num_queries=255)), ("RESCUE", dict(num_queries=255, blowup_factor=4)),
    ("RANGE", dict(grinding_factor=8)), ("RESCUE", dict(grinding_factor=8, blowup_factor=4)),
    ("RANGE", dict(fri_max_remainder_size=64)), ("RESCUE", dict(fri_max_remainder_size=16, blowup_factor=4)),
    ("MERKLE_UPDATE", dict(hash_fn=3, num_queries=1)),
])
def test_options_match_single_path(ctx, oracle, csg, air, kw):
    air_id = getattr(csg, "AIR_" + air)
    traces, pubs = witnesses(csg, air_id, 4, seed=7)
    opt = csg.ProofOptions(**kw)
    proofs = check_batch(ctx, csg, air_id, traces, pubs, opt, oracle, oracle_at=[0])
    for k, proof in enumerate(proofs):
        assert csg.verify(air_id, pubs[k], proof) == 0


def test_montgomery_repr(ctx, oracle, csg):
    traces, pubs = witnesses(csg, csg.AIR_RESCUE, 3)
    mont = [oracle.to_mont_fast(t) for t in traces]
    check_batch(ctx, csg, csg.AIR_RESCUE, mont, pubs, csg.ProofOptions(blowup_factor=4), oracle, oracle_at=[1], repr=csg.REPR_MONTGOMERY)


@pytest.mark.parametrize("air,count,blowup", [("RANGE", 1024, 8), ("RESCUE", 256, 4)])
def test_large_batches(ctx, oracle, csg, air, count, blowup):
    air_id = getattr(csg, "AIR_" + air)
    traces, pubs = witnesses(csg, air_id, count, seed=11)
    check_batch(ctx, csg, air_id, traces, pubs, csg.ProofOptions(blowup_factor=blowup), oracle, oracle_at=[0, count // 2, count - 1])


def test_longest_trace_accepted_and_longer_refused(ctx, csg):
    traces, pubs = zip(*[csg.build_rescue_trace(np.arange(s, s + 7, dtype=np.uint64), 8192) for s in (3, 4)])   # 2^16 rows
    opt = csg.ProofOptions(blowup_factor=4)
    proofs = check_batch(ctx, csg, csg.AIR_RESCUE, list(traces), np.stack(pubs), opt)
    assert csg.verify(csg.AIR_RESCUE, pubs[1], proofs[1]) == 0
    t, p = csg.build_rescue_trace(np.arange(1, 8, dtype=np.uint64), 16384)   # 2^17 rows
    with pytest.raises(csg.CsgError, match="^unsupported"):
        ctx.prove_many(csg.AIR_RESCUE, [t, t], np.stack([p, p]), opt)


def test_equal_and_permuted_inputs(ctx, csg):
    traces, pubs = witnesses(csg, csg.AIR_RESCUE, 5, seed=3)
    opt = csg.ProofOptions(blowup_factor=4)
    base = ctx.prove_many(csg.AIR_RESCUE, traces, pubs, opt)
    twice = ctx.prove_many(csg.AIR_RESCUE, [traces[2], traces[2]], np.stack([pubs[2], pubs[2]]), opt)
    assert twice[0] == twice[1] == base[2]
    perm = [4, 2, 0, 3, 1]
    permuted = ctx.prove_many(csg.AIR_RESCUE, [traces[i] for i in perm], pubs[perm], opt)
    assert permuted == [base[i] for i in perm]


def test_corrupted_trace_affects_only_its_proof(ctx, csg):
    traces, pubs = witnesses(csg, csg.AIR_RESCUE, 4, seed=5)
    opt = csg.ProofOptions(blowup_factor=4)
    good = ctx.prove_many(csg.AIR_RESCUE, traces, pubs, opt)
    bad = [t.copy() for t in traces]
    bad[2][5, 17] = (int(bad[2][5, 17]) + 1) % P
    proofs = ctx.prove_many(csg.AIR_RESCUE, bad, pubs, opt)
    assert proofs[2] == ctx.prove(csg.AIR_RESCUE, bad[2], pubs[2], opt)
    assert proofs[2] != good[2] and csg.verify(csg.AIR_RESCUE, pubs[2], proofs[2]) != 0
    for k in (0, 1, 3):
        assert proofs[k] == good[k] and csg.verify(csg.AIR_RESCUE, pubs[k], proofs[k]) == 0


def test_launches_do_not_grow_with_the_batch(ctx, csg):
    traces, pubs = witnesses(csg, csg.AIR_RANGE, 256, seed=9)
    opt = csg.ProofOptions()
    ctx.prove_many(csg.AIR_RANGE, traces[:1], pubs[:1], opt)
    one = ctx.timings()["kernel_launches"]
    ctx.prove_many(csg.AIR_RANGE, traces, pubs, opt)
    t = ctx.timings()
    assert t["kernel_launches"] == one > 0
    assert sum(t["stage_launches"].values()) == one


def test_bytes_do_not_depend_on_the_thread_count(ctx, csg):
    traces, pubs = witnesses(csg, csg.AIR_RESCUE, 16, seed=13)
    want = [hashlib.sha256(p).hexdigest() for p in ctx.prove_many(csg.AIR_RESCUE, traces, pubs, csg.ProofOptions(blowup_factor=4))]
    code = ("import sys, hashlib, numpy as np; sys.path.insert(0, sys.argv[1]); import certificate_stark_b200 as csg\n"
            "tr = [csg.build_rescue_trace(np.arange(s, s + 7, dtype=np.uint64), 128) for s in range(14, 30)]\n"
            "with csg.Context(0) as c:\n"
            "    ps = c.prove_many(csg.AIR_RESCUE, [t for t, _ in tr], np.stack([p for _, p in tr]), csg.ProofOptions(blowup_factor=4))\n"
            "print(' '.join(hashlib.sha256(p).hexdigest() for p in ps))\n")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-c", code, str(ROOT)], env=env, capture_output=True, text=True, check=True).stdout.split()
    assert out == want


def test_single_proof_state_is_left_alone(ctx, csg):
    opt = csg.ProofOptions(blowup_factor=4)
    (t1, t2), pubs = witnesses(csg, csg.AIR_RESCUE, 2, seed=17)
    with csg.Context(0) as ref:   # what the prefetched trace proves to without a batch in between
        ref.set_air(csg.AIR_RESCUE, t2.shape[1], pubs[0], opt)
        ref.load_trace(t2)
        want_prefetched = ref.prove_loaded()
    ctx.set_air(csg.AIR_RESCUE, t1.shape[1], pubs[0], opt)
    ctx.load_trace(t1)
    want_loaded = ctx.prove_loaded()
    t2 = np.ascontiguousarray(t2)
    ctx.prefetch_trace_ptr(t2.ctypes.data)
    rt, rp = witnesses(csg, csg.AIR_RANGE, 8, seed=19)
    ctx.prove_many(csg.AIR_RANGE, rt, rp, csg.ProofOptions())   # (ctx.prove would replace the AIR: compared elsewhere)
    assert ctx.prove_loaded() == want_loaded
    assert ctx.prove_prefetched_ptr() == want_prefetched


def test_rejections_leave_the_context_usable(ctx, csg):
    traces, pubs = witnesses(csg, csg.AIR_RANGE, 2, seed=21)
    opt = csg.ProofOptions()
    lib = csg.lib()

    def rejected(kind, *args, **kw):
        with pytest.raises(csg.CsgError, match="^" + kind):
            ctx.prove_many(*args, **kw)

    rejected("unsupported", csg.AIR_RANGE, traces, pubs, csg.ProofOptions(field_extension=2))
    rejected("unsupported", csg.AIR_RANGE, traces, pubs, csg.ProofOptions(field_extension=3))
    rejected("invalid argument", csg.AIR_RANGE, traces, pubs, opt, repr=7)
    rejected("invalid argument", csg.AIR_RANGE, traces, np.zeros((2, 2), dtype=np.uint64), opt)   # npub
    rejected("invalid argument", csg.AIR_RANGE, traces * 513, np.concatenate([pubs] * 513), opt)  # 1026 proofs
    tx = np.zeros((94, 1024), dtype=np.uint64)
    rejected("invalid argument", csg.AIR_TRANSACTION, [tx] * 698, np.zeros((698, 14), dtype=np.uint64), opt)   # 65612 columns
    big = np.zeros((94, 1 << 16), dtype=np.uint64)   # one buffer, 697 times: 275 GB of LDE alone
    with pytest.raises(csg.CsgError, match="device memory"):
        ctx.prove_many(csg.AIR_TRANSACTION, [big] * 697, np.zeros((697, 14), dtype=np.uint64), opt)
    # the C ABI directly: count 0 and null pointers
    outs, lens = (C.POINTER(C.c_uint8) * 2)(), (C.c_size_t * 2)()
    ptrs = (C.POINTER(C.c_uint64) * 2)(*[t.ctypes.data_as(C.POINTER(C.c_uint64)) for t in traces])
    pp = pubs.ctypes.data_as(C.POINTER(C.c_uint64))
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 0, ptrs, 0, 64, pp, 1, C.byref(opt), outs, lens) == 1
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 2, None, 0, 64, pp, 1, C.byref(opt), outs, lens) == 1
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 2, ptrs, 0, 64, None, 1, C.byref(opt), outs, lens) == 1
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 2, ptrs, 0, 64, pp, 1, None, outs, lens) == 1
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 2, ptrs, 0, 64, pp, 1, C.byref(opt), None, lens) == 1
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 2, ptrs, 0, 64, pp, 1, C.byref(opt), outs, None) == 1
    # too many proofs: the caller's output arrays are cleared all the same
    many_outs = (C.POINTER(C.c_uint8) * 1025)(*[C.cast(C.c_void_p(8), C.POINTER(C.c_uint8))] * 1025)
    many_lens = (C.c_size_t * 1025)(*[5] * 1025)
    many_ptrs = (C.POINTER(C.c_uint64) * 1025)(*[ptrs[0]] * 1025)
    many_pubs = np.zeros(1025, dtype=np.uint64)
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 1025, many_ptrs, 0, 64, many_pubs.ctypes.data_as(C.POINTER(C.c_uint64)), 1, C.byref(opt),
                              many_outs, many_lens) == 1
    assert not any(many_outs[i] for i in range(1025)) and not any(many_lens)
    ptrs[1] = C.POINTER(C.c_uint64)()
    assert lib.csg_prove_many(ctx._h, csg.AIR_RANGE, 2, ptrs, 0, 64, pp, 1, C.byref(opt), outs, lens) == 1
    assert not outs[0] and not outs[1]
    # a context attached to a group
    with csg.LocalGroup(2) as g:
        with pytest.raises(csg.CsgError, match="^unsupported"):
            g.ctxs[0].prove_many(csg.AIR_RANGE, traces, pubs, opt)
        assert g.prove(csg.AIR_RANGE, traces[0], pubs[0], opt) == [ctx.prove(csg.AIR_RANGE, traces[0], pubs[0], opt)] * 2
    check_batch(ctx, csg, csg.AIR_RANGE, traces, pubs, opt)


def test_oversized_batch_allocates_nothing(csg):
    torch = pytest.importorskip("torch")
    opt = csg.ProofOptions()
    big = np.zeros((94, 1 << 16), dtype=np.uint64)   # one buffer, 697 times: 275 GB of LDE alone, 34 GB of trace staging
    with csg.Context(0) as fresh:
        free0 = torch.cuda.mem_get_info(0)[0]
        with pytest.raises(csg.CsgError, match="device memory"):
            fresh.prove_many(csg.AIR_TRANSACTION, [big] * 697, np.zeros((697, 14), dtype=np.uint64), opt)
        assert abs(torch.cuda.mem_get_info(0)[0] - free0) < 2 << 30   # the GPU may be shared: 2 GB of slack, far below one buffer
        traces, pubs = witnesses(csg, csg.AIR_RANGE, 2, seed=23)
        assert fresh.prove_many(csg.AIR_RANGE, traces, pubs, opt) == [fresh.prove(csg.AIR_RANGE, t, p, opt) for t, p in zip(traces, pubs)]
