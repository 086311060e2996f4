"""csg_validate_* (-m gpu): winterfell's debug-build trace.validate on the GPU.  Valid witnesses of every AIR validate clean in both
representations; a corrupted cell is reported exactly as oracle.check_trace and oracle/pyair.py's assertions see it; the verdict
agrees with csg_verify on the proof of the same trace; the 2^20-row transaction trace validates at size from the device builder and
from the host; batches from the device builders validate clean and a corrupted trace in a batch is reported alone; the calls leave
the single-proof state alone and refuse malformed arguments."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_prove_many import AIRS, witnesses

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
P = 0x4180000000000001


@pytest.fixture(scope="module")
def pyair():
    from oracle import pyair as A
    return A


def up(traces):
    """host traces -> one contiguous int64 CUDA tensor (K, w, n)"""
    return torch.from_numpy(np.stack(traces).view(np.int64)).to("cuda:0")


def air_of(csg, air):
    return getattr(csg, "AIR_" + air)


def failing_cells(pyair, air_id, trace, pub):
    """(column, step) of every asserted cell whose word differs from its value, ascending by step then column (pyair's assertions)"""
    n = trace.shape[1]
    bad = []
    for kind, col, first, stride, values in pyair.AIRS[air_id](n, [int(v) for v in pub]).assertions():
        steps = [first] if stride == 0 else list(range(first, n, stride))
        for j, s in enumerate(steps):
            v = values[j] if kind == "sequence" else values[0]
            if int(trace[col, s]) % P != v % P:
                bad.append((col, s))
    return sorted(bad, key=lambda cs: (cs[1], cs[0]))


def expected(oracle, pyair, air_id, trace, pub):
    pairs = sorted(oracle.check_trace(air_id, trace % np.uint64(P), pub, pyair.AIRS[air_id].num_constraints))
    return pairs, failing_cells(pyair, air_id, trace, pub)


def check_report(r, pairs, cells, cap=256):
    assert r.transition == [tuple(p) for p in pairs[:cap]]
    assert r.failed_steps == len({s for s, _ in pairs})
    assert r.boundary == cells[:cap]
    assert r.failed_cells == len(cells)
    assert r.ok == (not pairs and not cells)


# ---------------------------------------------------------------------------------------------- valid traces
@pytest.mark.parametrize("repr", [0, 1])
@pytest.mark.parametrize("air", AIRS)
def test_witnesses_validate_clean(ctx, oracle, csg, air, repr):
    air_id = air_of(csg, air)
    traces, pubs = witnesses(csg, air_id, 2)
    for t, p in zip(traces, pubs):
        words = oracle.to_mont_fast(t) if repr == csg.REPR_MONTGOMERY else t
        r = ctx.validate(air_id, words, p, repr=repr)
        assert r.ok and r.failed_steps == 0 and r.failed_cells == 0 and r.transition == [] and r.boundary == [], r
        # a word >= p counts as its residue
        lifted = words.copy()
        lifted[:, ::2] += np.uint64(P)
        lifted[:, 1::4] += np.uint64(2 * P)
        assert ctx.validate(air_id, lifted, p, repr=repr).ok


# ---------------------------------------------------------------------------------------------- single-cell corruptions
@pytest.mark.parametrize("air", AIRS)
def test_single_cell_corruptions(ctx, oracle, csg, pyair, air):
    air_id = air_of(csg, air)
    (trace,), (pub,) = witnesses(csg, air_id, 1)
    n, w = trace.shape[1], trace.shape[0]
    kind, acol, afirst, _, _ = pyair.AIRS[air_id](n, [int(v) for v in pub]).assertions()[-1]
    rng = np.random.default_rng(air_id)
    cases = [(int(rng.integers(0, w)), 0), (int(rng.integers(0, w)), n // 2 + 3), (int(rng.integers(0, w)), n - 1), (acol, afirst)]
    for col, row in cases:
        bad = trace.copy()
        bad[col, row] = (int(bad[col, row]) + 1 + int(rng.integers(0, 1000))) % P
        pairs, cells = expected(oracle, pyair, air_id, bad, pub)
        assert pairs or cells or (col, row) != (acol, afirst)
        for repr in (0, 1):
            r = ctx.validate(air_id, bad if repr == 0 else oracle.to_mont_fast(bad), pub, repr=repr)
            check_report(r, pairs, cells)


def test_agrees_with_the_verifier(ctx, oracle, csg):
    """random single-cell corruptions of small traces: validate's verdict is csg_verify's verdict on csg_prove's proof"""
    rng = np.random.default_rng(7)
    seen = set()
    for air_id in (csg.AIR_RANGE, csg.AIR_RESCUE, csg.AIR_MERKLE_INIT):
        (trace,), (pub,) = witnesses(csg, air_id, 1)
        opt = csg.ProofOptions(blowup_factor=4 if air_id == csg.AIR_RESCUE else 8)
        for _ in range(5):
            bad = trace.copy()
            col, row = int(rng.integers(0, bad.shape[0])), int(rng.integers(0, bad.shape[1]))
            bad[col, row] = int(rng.integers(0, P))
            ok = ctx.validate(air_id, bad, pub).ok
            proof = ctx.prove(air_id, bad, pub, opt)
            assert ok == (csg.verify(air_id, pub, proof) == 0), (air_id, col, row)
            seen.add(ok)
    assert False in seen


# ---------------------------------------------------------------------------------------------- at size: 1024 transactions, 2^20 x 94
def pairs_at(oracle, air, trace, steps, nc):
    out = []
    for s in steps:
        r = air.eval_row(s, oracle.to_mont_fast(trace[:, s] % np.uint64(P)), oracle.to_mont_fast(trace[:, s + 1] % np.uint64(P)), nc)
        out += [(s, int(i)) for i in np.nonzero(r)[0]]
    return out


def test_transaction_trace_at_size(csg, oracle, pyair):
    n, nc = 1 << 20, csg.NUM_CONSTRAINTS[csg.AIR_TRANSACTION]
    with csg.Context(0) as ctx:
        pub = ctx.build_batch(11, 1024)
        ctx.set_air(csg.AIR_TRANSACTION, n, pub, csg.ProofOptions())
        ctx.build_transaction_trace_resident()
        r = ctx.validate_resident()
        assert r.ok, r
        trace = ctx.download_trace(94, n)
        assert ctx.validate(csg.AIR_TRANSACTION, trace, pub).ok
        air = oracle.Air(csg.AIR_TRANSACTION, n, pub)
        row = 700_001
        trace[50, row] = (int(trace[50, row]) + 5) % P
        r = ctx.validate(csg.AIR_TRANSACTION, trace, pub)
        want = pairs_at(oracle, air, trace, (row - 1, row), nc)
        assert want and r.transition == want and r.failed_steps == len({s for s, _ in want}) and r.failed_cells == 0
        # random words: every step fails; the first CSG_REPORT_CAP pairs, ascending
        del trace
        rnd = np.random.default_rng(5).integers(0, 2**64, size=(94, n), dtype=np.uint64)
        r = ctx.validate(csg.AIR_TRANSACTION, rnd, pub)
        assert r.failed_steps == n - 1 and r.num_transition == csg.REPORT_CAP
        assert r.transition == sorted(r.transition)
        want = []
        s = 0
        while len(want) < csg.REPORT_CAP:
            want += pairs_at(oracle, air, rnd, (s,), nc)
            s += 1
        assert r.transition == want[:csg.REPORT_CAP]
        cells = failing_cells(pyair, csg.AIR_TRANSACTION, rnd, pub)
        assert r.failed_cells == len(cells) and r.boundary == cells


# ---------------------------------------------------------------------------------------------- batches
def test_device_built_batches_validate_clean(ctx, csg):
    seeds = np.arange(16 * 7, dtype=np.uint64).reshape(16, 7) * np.uint64(977)
    builds = [(csg.AIR_RESCUE, ctx.build_many_rescue(seeds, 64)),
              (csg.AIR_SCHNORR, ctx.build_many_schnorr(csg.SignatureBatch(seed=5, num_sig=8))),
              (csg.AIR_MERKLE_UPDATE, ctx.build_many_merkle_update(csg.TransactionBatch(seed=5, num_tx=8))),
              (csg.AIR_TRANSACTION, ctx.build_many_transaction(csg.TransactionBatch(seed=6, num_tx=4)))]
    for air_id, (dev, pubs) in builds:
        reports = ctx.validate_many_device(air_id, dev, pubs)
        assert len(reports) == dev.shape[0] and all(r.ok for r in reports), (air_id, [r for r in reports if not r.ok][:2])


@pytest.mark.parametrize("air", ["MERKLE_UPDATE", "SCHNORR", "RESCUE", "RANGE"])
def test_batch_with_one_corrupted_trace(ctx, oracle, csg, air):
    air_id = air_of(csg, air)
    traces, pubs = witnesses(csg, air_id, 5)
    traces = [t.copy() for t in traces]
    n = traces[2].shape[1]
    traces[2][1, n // 3] = (int(traces[2][1, n // 3]) + 1) % P
    traces[2][0, 0] = (int(traces[2][0, 0]) + 1) % P
    for repr in (0, 1):
        words = [oracle.to_mont_fast(t) for t in traces] if repr else traces
        dev = up(words)
        before = dev.clone()
        reports = ctx.validate_many_device(air_id, dev, pubs, repr=repr)
        assert torch.equal(dev, before), "the library wrote to the caller's buffer"
        assert [r.ok for r in reports] == [True, True, False, True, True]
        for k, r in enumerate(reports):
            alone = ctx.validate(air_id, words[k], pubs[k], repr=repr)
            assert (r.failed_steps, r.failed_cells, r.transition, r.boundary) == (alone.failed_steps, alone.failed_cells, alone.transition, alone.boundary)


# ---------------------------------------------------------------------------------------------- state and rejections
def test_leaves_the_single_proof_state_alone(csg):
    (trace,), (pub,) = witnesses(csg, csg.AIR_RESCUE, 1)
    (other,), (opub,) = witnesses(csg, csg.AIR_SCHNORR, 1)
    opt = csg.ProofOptions(blowup_factor=4)
    with csg.Context(0) as ref:
        ref.set_air(csg.AIR_RESCUE, trace.shape[1], pub, opt)
        ref.load_trace(trace)
        want = ref.prove_loaded()
    buf = csg.HostBuffer(*trace.shape)
    buf.array[:] = trace
    with csg.Context(0) as ctx:
        ctx.set_air(csg.AIR_RESCUE, trace.shape[1], pub, opt)
        assert ctx.validate(csg.AIR_SCHNORR, other, opub).ok
        ctx.load_trace(trace)
        assert ctx.validate_many_device(csg.AIR_SCHNORR, up([other]), opub[None])[0].ok
        assert ctx.validate_resident().ok
        assert ctx.prove_loaded() == want
        ctx.prefetch_trace_ptr(buf.ptr)
        assert not ctx.validate(csg.AIR_SCHNORR, other ^ np.uint64(1), opub).ok
        assert ctx.prove_prefetched_ptr() == want
        assert ctx.prove_loaded() == want
    buf.close()


def test_rejections(csg):
    L = csg.lib()
    (trace,), (pub,) = witnesses(csg, csg.AIR_RESCUE, 1)
    n = trace.shape[1]
    r = csg.TraceReport()
    p64, null = csg._p64, C.POINTER(C.c_uint64)()
    with csg.Context(0) as ctx:
        h = ctx._h
        assert L.csg_validate_resident_trace(h, C.byref(r)) == 3                                    # no resident trace
        assert L.csg_validate_trace(h, 9, p64(trace), 0, n, p64(pub), 14, C.byref(r)) == 1           # bad AIR id
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, p64(trace), 0, n, p64(pub), 13, C.byref(r)) == 1
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, p64(trace), 2, n, p64(pub), 14, C.byref(r)) == 1
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, null, 0, n, p64(pub), 14, C.byref(r)) == 1
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, p64(trace), 0, n, null, 14, C.byref(r)) == 1
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, p64(trace), 0, n, p64(pub), 14, None) == 1
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, p64(trace), 0, n - 8, p64(pub), 14, C.byref(r)) == 1
        assert L.csg_validate_trace(h, csg.AIR_RESCUE, p64(trace), 0, 1 << 23, p64(pub), 14, C.byref(r)) == 1
        dev = up([trace, trace])
        pubs = np.stack([pub, pub])
        many = (csg.TraceReport * 1100)()
        def vm(air_id=csg.AIR_RESCUE, count=2, ptr=dev.data_ptr(), repr=0, rows=n, pp=p64(pubs), npub=14, out=many):
            return L.csg_validate_many_device(h, air_id, count, ptr, repr, rows, pp, npub, out)
        assert vm() == 0 and many[0].ok and many[1].ok
        assert vm(count=0) == 1 and vm(count=1025) == 1 and vm(repr=5) == 1 and vm(npub=7) == 1 and vm(air_id=-1) == 1
        assert vm(ptr=None) == 1 and vm(pp=null) == 1 and vm(out=None) == 1
        assert vm(ptr=trace.ctypes.data) == 1                                                         # host memory
        assert vm(rows=1 << 17) == 4                                                                  # above 2^16 rows
        assert vm(air_id=csg.AIR_TRANSACTION, count=700, rows=1024, pp=p64(np.zeros((700, 14), np.uint64))) == 1   # count * width
        assert ctx.validate(csg.AIR_RESCUE, trace, pub).ok                                             # still usable
    with csg.LocalGroup(2) as g:
        for c in g.ctxs:
            assert L.csg_validate_trace(c._h, csg.AIR_RESCUE, p64(trace), 0, n, p64(pub), 14, C.byref(r)) == 4
            assert L.csg_validate_many_device(c._h, csg.AIR_RESCUE, 2, dev.data_ptr(), 0, n, p64(pubs), 14, many) == 4
