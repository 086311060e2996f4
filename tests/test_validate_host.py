"""Trace validation, the parts that need no GPU: the new entry points are exported, csg_trace_report has the layout gcc gives it and
the ctypes mirror assumes, and csg_debug_transition_at -- the host evaluation that localises the failing (step, constraint) pairs of
csg_validate_* -- gives every constraint slot as oracle/airs.c and the independent oracle/pyair.py do, on witness rows (all zero) and
on random frames."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
AIRS = ["TRANSACTION", "MERKLE_UPDATE", "MERKLE_INIT", "SCHNORR", "RANGE", "RESCUE"]
NEW = ("csg_validate_trace", "csg_validate_resident_trace", "csg_validate_many_device", "csg_debug_transition_at")


@pytest.mark.parametrize("name", NEW)
def test_exported(csg, name):
    assert hasattr(C.CDLL(str(csg.LIB_PATH)), name)
    assert callable(getattr(csg.lib(), name))


def test_report_layout_matches_gcc(csg, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "csg.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %d\\n", sizeof(csg_trace_report), offsetof(csg_trace_report, failed_steps),\n'
                   '         offsetof(csg_trace_report, failed_cells), offsetof(csg_trace_report, num_transition),\n'
                   '         offsetof(csg_trace_report, num_boundary), offsetof(csg_trace_report, transition),\n'
                   '         offsetof(csg_trace_report, boundary), CSG_REPORT_CAP);\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", f"-I{ROOT / 'include'}", str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    R = csg.TraceReport
    assert got == [C.sizeof(R), R.failed_steps.offset, R.failed_cells.offset, R.num_transition.offset, R.num_boundary.offset,
                   R._transition.offset, R._boundary.offset, csg.REPORT_CAP]


def witness(csg, air_id):
    """one small witness of each AIR from the library's host builders: (trace (w, n), pub)"""
    if air_id == csg.AIR_RANGE:
        return csg.build_range_trace(0x1234_5678_9ABC)
    if air_id == csg.AIR_RESCUE:
        return csg.build_rescue_trace(np.arange(3, 10, dtype=np.uint64), 16)
    if air_id == csg.AIR_MERKLE_INIT:
        return csg.build_merkle_init_trace(np.arange(1, 15, dtype=np.uint64), np.arange(20, 34, dtype=np.uint64), 5)
    if air_id == csg.AIR_MERKLE_UPDATE:
        return csg.TransactionBatch(seed=3, num_tx=1).merkle_update_trace()
    if air_id == csg.AIR_SCHNORR:
        return csg.SignatureBatch(seed=3, num_sig=1).schnorr_trace()
    return csg.TransactionBatch(seed=3, num_tx=1).transaction_trace()


def reference_values(oracle, pyair, air_id, n, pub, step, cur, nxt):
    """(oracle/airs.c, oracle/pyair.py) result[] of evaluate_transition at `step`, canonical"""
    nc = pyair.AIRS[air_id].num_constraints
    a = oracle.Air(air_id, n, pub).eval_row(step, oracle.to_mont(cur), oracle.to_mont(nxt), nc)
    p = pyair.AIRS[air_id](n, [int(v) for v in pub]).evaluate([int(v) for v in cur], [int(v) for v in nxt],
                                                               pyair.periodic_row(pyair.AIRS[air_id](n, [int(v) for v in pub]), step))
    return oracle.from_mont(a), np.array(p, dtype=np.uint64)


@pytest.fixture(scope="module")
def pyair():
    from oracle import pyair as A
    return A


@pytest.mark.parametrize("air", AIRS)
def test_debug_transition_at_matches_the_oracles(csg, oracle, pyair, air):
    air_id = getattr(csg, "AIR_" + air)
    trace, pub = witness(csg, air_id)
    n = trace.shape[1]
    rng = np.random.default_rng(air_id)
    steps = sorted({0, 1, 7, n // 2 - 1, n - 2} | {int(s) for s in rng.integers(0, n - 1, 3)})
    for s in steps:   # witness rows: every slot vanishes
        got = csg.debug_transition_at(air_id, n, pub, s, trace[:, s], trace[:, s + 1])
        assert got.shape == (csg.NUM_CONSTRAINTS[air_id],) and not got.any(), f"step {s}: {np.nonzero(got)[0]}"
    for s in steps:   # random frames: slot by slot
        cur, nxt = (rng.integers(0, csg.P, size=trace.shape[0], dtype=np.uint64) for _ in range(2))
        got = csg.debug_transition_at(air_id, n, pub, s, cur, nxt)
        want_c, want_py = reference_values(oracle, pyair, air_id, n, pub, s, cur, nxt)
        assert np.array_equal(got, want_c), f"step {s}: slots {np.nonzero(got != want_c)[0]} differ from oracle/airs.c"
        assert np.array_equal(got, want_py), f"step {s}: slots {np.nonzero(got != want_py)[0]} differ from oracle/pyair.py"
        assert got.any()


def test_debug_transition_at_one_corrupted_cell(csg, oracle, pyair):
    """a witness with one changed word: the same non-zero slots as the oracles at the two steps that read it"""
    trace, pub = witness(csg, csg.AIR_RESCUE)
    n, r = trace.shape[1], 37
    trace[4, r] ^= 1
    for s in (r - 1, r):
        got = csg.debug_transition_at(csg.AIR_RESCUE, n, pub, s, trace[:, s], trace[:, s + 1])
        want_c, want_py = reference_values(oracle, pyair, csg.AIR_RESCUE, n, pub, s, trace[:, s], trace[:, s + 1])
        assert got.any() and np.array_equal(got, want_c) and np.array_equal(got, want_py)


def test_debug_transition_at_rejects(csg):
    trace, pub = witness(csg, csg.AIR_RANGE)
    with pytest.raises(csg.CsgError):
        csg.debug_transition_at(csg.AIR_RANGE, 64, pub, 64, trace[:, 0], trace[:, 1])        # step outside the trace
    with pytest.raises(csg.CsgError):
        csg.debug_transition_at(csg.AIR_RANGE, 48, pub, 0, trace[:, 0], trace[:, 1])         # not a power of two
    with pytest.raises(csg.CsgError):
        csg.debug_transition_at(csg.AIR_RANGE, 64, np.zeros(2, np.uint64), 0, trace[:, 0], trace[:, 1])   # npub
    with pytest.raises(KeyError):
        csg.debug_transition_at(9, 64, pub, 0, trace[:, 0], trace[:, 1])
    p = C.POINTER(C.c_uint64)()
    assert csg.lib().csg_debug_transition_at(9, 64, csg._p64(pub), 1, 0, p, p, p) != 0
