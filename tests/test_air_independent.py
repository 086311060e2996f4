"""The AIR side against a SECOND, independent restatement (oracle/pyair.py: plain Python big integers, its own parse of the
reference's constants, its own witness builders) -- removes the single-author common mode between oracle/airs.c and the
product's airs.cuh / air_desc.cpp / witness.cpp on src/air.rs:114-173,383-610, src/schnorr/air.rs:394-531,
src/merkle/update/air.rs:215-369 (VERDICT round 1).  CPU only; the GPU legs are in tests/test_gpu_parity.py.

tests/golden/air_vectors.txt holds, for all six AIRs: degrees, periodic-column fingerprints, assertions, and full result[]
vectors of evaluate_transition on witness rows (all zero) and random frames (dense).  tests/host_harness.cpp checks oracle/airs.c
slot by slot and the product's fused evaluation through random linear combinations of the golden slots."""
import json
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden" / "air_vectors.txt"


@pytest.fixture(scope="module")
def pyair():
    from oracle import pyair as A
    return A


@pytest.fixture(scope="module")
def harness(tmp_path_factory, oracle):
    exe = tmp_path_factory.mktemp("hh") / "host_harness"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fopenmp", str(ROOT / "tests" / "host_harness.cpp"), "-x", "c++",
                           str(ROOT / "certificate_stark_b200" / "csrc" / "host" / "air_desc.cpp"), f"-L{ROOT / 'oracle'}", "-l:liboracle.so",
                           f"-Wl,-rpath,{ROOT / 'oracle'}", "-o", str(exe)])
    return exe


def test_oracle_and_product_match_the_independent_golden_vectors(harness):
    out = subprocess.run([str(harness), str(GOLDEN)], capture_output=True, text=True)
    assert out.returncode == 0 and "7 AIR sections, 97 frames, all checks passed" in out.stdout, out.stdout[-3000:]


def test_the_golden_check_notices_a_wrong_slot(harness, tmp_path):
    # flip one hex digit of one result slot of a dense (random) transaction frame: both sides must be reported
    lines = GOLDEN.read_text().splitlines()
    idx = next(i for i, l in enumerate(lines) if l.startswith("ROW -1")) + 4
    assert lines[idx].startswith("RES ")
    words = lines[idx].split()
    words[60] = format(int(words[60], 16) ^ 1, "x")
    lines[idx] = " ".join(words)
    bad = tmp_path / "bad.txt"
    bad.write_text("\n".join(lines) + "\n")
    out = subprocess.run([str(harness), str(bad)], capture_output=True, text=True)
    assert out.returncode != 0 and "oracle/airs.c result[59] differs" in out.stdout and "product airs.cuh merged value differs" in out.stdout


def header_tables(text):
    """name -> values of the uint64 tables of a header written by tools/gen_constants.py (`NAME[n] = {...};` or `#define NAME_VALUES`)"""
    blocks = re.findall(r"(?:uint64_t (\w+)\[\d+\] = \{|#define (\w+)_VALUES)(.*?)(?:\};|\n(?!\s+0x))", text, re.S)
    return {a or b: [int(v, 16) for v in re.findall(r"0x([0-9a-f]{16})ULL", body)] for a, b, body in blocks}


def test_pyair_constants_are_its_own_parse_of_the_reference(pyair):
    # pyair's stored parse of the reference (tests/golden/make_air_vectors.py) is what it runs on, and it agrees with the tables
    # tools/gen_constants.py parsed separately from the same sources for the C oracle (canonical) and the product (Montgomery)
    names = ("MDS", "INV_MDS", "ARK", "GENERATOR", "B3")
    stored = json.loads((ROOT / "tests" / "golden" / "air_constants.json").read_text())
    assert [pyair._K[k] for k in names] == [stored[k] for k in names]
    P = pyair.P
    oracle_h = header_tables((ROOT / "oracle" / "ref_constants.h").read_text())
    product_h = header_tables((ROOT / "certificate_stark_b200" / "csrc" / "ref_constants.h").read_text())
    for k in names:
        assert oracle_h["REF_" + k] == stored[k], k
        assert product_h["CSG_" + k] == [v * 2**64 % P for v in stored[k]], k
    # MDS * INV_MDS = I, generator on the curve
    assert all(sum(pyair.MDS[i][k] * pyair.INV_MDS[k][j] for k in range(14)) % P == (1 if i == j else 0) for i in range(14) for j in range(14))
    gx, gy = pyair.GENERATOR[0:6], pyair.GENERATOR[6:12]
    b = [v * pow(3, -1, P) % P for v in pyair.B3]
    assert pyair.f6mul(gy, gy) == pyair.f6add(pyair.f6add(pyair.f6mul(pyair.f6mul(gx, gx), gx), gx), b)      # y^2 = x^3 + x + B3/3


def test_pyair_rescue_known_answers(pyair):
    # SURVEY.md Appendix D (tests/golden/rescue_kat.json comes from the survey session's restatement: a third derivation)
    kat = json.loads((ROOT / "tests" / "golden" / "rescue_kat.json").read_text())
    hx = lambda v: ["%016x" % x for x in v]      # noqa: E731
    assert hx(pyair.apply_permutation([0] * 14)[:7]) == kat["permutation_of_zero"]
    assert hx(pyair.merge(list(range(1, 8)), list(range(8, 15)))) == kat["merge_1to7_8to14"]
    assert hx(pyair.digest(list(range(1, 7)))) == kat["digest_1to6"]
    v, r = list(range(42, 49)), [0] * 7              # compute_hash_chain, benches/rescue.rs:104-121
    for i in range(1, 129):
        r = pyair.merge(v, r)
        v = r
        if i in (1, 128):
            assert hx(r) == kat[f"hash_chain_seed42_n{i}"]


def test_pyair_field_tower(pyair):
    import random
    rnd = random.Random(5)
    for _ in range(20):
        a = [rnd.randrange(pyair.P) for _ in range(6)]
        assert pyair.f6mul(a, pyair.f6inv(a)) == [1, 0, 0, 0, 0, 0]
    # group law sanity on the independent formulas: 2G + 3G = 5G, mixed addition = full addition with Z = 1, doubling = adding to itself
    G = pyair.GENERATOR
    aff = lambda k: pyair.to_affine(pyair.scalar_mul(k, G))      # noqa: E731
    p2, p3 = pyair.scalar_mul(2, G), aff(3)
    assert pyair.to_affine(pyair.compute_add_mixed(p2, p3)) == aff(5)
    assert pyair.to_affine(pyair.compute_add(p2, p3 + [1, 0, 0, 0, 0, 0])) == aff(5)
    assert pyair.to_affine(pyair.compute_double(p2)) == aff(4) == pyair.to_affine(pyair.compute_add(p2, p2))


def as_columns(rows):
    return np.ascontiguousarray(np.array(rows, dtype=np.uint64).T)


def test_independent_witnesses_are_accepted_by_the_c_oracle_and_the_product_verifier(pyair, oracle, csg):
    # pyair's OWN witnesses (own metadata generator, own signing, own sparse Rescue tree) through the C oracle's prover and both
    # verifiers: the trace layouts of src/trace.rs / */trace.rs as read by two independent restatements must be the same tables
    batch = pyair.TransactionBatch(seed=3, num_tx=1)
    rows, pub = batch.transaction_trace(), np.array(batch.pub_inputs(), dtype=np.uint64)
    assert not pyair.violations(pyair.TransactionAir(len(rows), batch.pub_inputs()), rows)
    trace = as_columns(rows)
    assert oracle.check_trace(oracle.AIR_TRANSACTION, trace, pub, 115) == []
    proof = oracle.prove(oracle.AIR_TRANSACTION, trace, pub, oracle.options())
    assert oracle.verify(oracle.AIR_TRANSACTION, pub, proof) == 0 and csg.verify(csg.AIR_TRANSACTION, pub, proof, csg.ProofOptions()) == 0
    wrong = pub.copy()
    wrong[7] ^= np.uint64(1)
    assert csg.verify(csg.AIR_TRANSACTION, wrong, proof) != 0
    # Merkle update (with the bit tweak of MerkleProver::build_trace), Schnorr (2 signatures), range, Rescue chain
    mrows = batch.merkle_update_trace()
    cases = [(oracle.AIR_MERKLE_UPDATE, mrows, batch.pub_inputs(), 8), (oracle.AIR_SCHNORR, *pyair.schnorr_batch(seed=9, num_sig=2), 8),
             (oracle.AIR_RANGE, *pyair.range_trace(2**62 + 12345), 8), (oracle.AIR_RESCUE, *pyair.rescue_trace(list(range(42, 49)), 16), 4)]
    for air, r, p, blowup in cases:
        t, p = as_columns(r), np.array(p, dtype=np.uint64)
        proof = oracle.prove(air, t, p, oracle.options(blowup=blowup))
        assert oracle.verify(air, p, proof) == 0 and csg.verify(air, p, proof) == 0, f"air {air}"


def test_product_witness_builders_satisfy_the_independent_air(pyair, csg):
    # the other direction: the traces of the product's witness.cpp, judged by pyair's evaluate_transition with pyair's periodic columns
    batch = csg.TransactionBatch(seed=5, num_tx=1)
    trace, pub = batch.transaction_trace()
    rows = [[int(v) for v in r] for r in trace.T]
    air = pyair.TransactionAir(len(rows), [int(v) for v in pub])
    assert pyair.violations(air, rows) == []
    assert all(rows[st][col] == vals[0] for _, col, st, _, vals in air.assertions())
    strace, spub = csg.SignatureBatch(seed=5, num_sig=2).schnorr_trace()
    srows = [[int(v) for v in r] for r in strace.T]
    sair = pyair.SchnorrAir(len(srows), [int(v) for v in spub])
    assert pyair.violations(sair, srows) == []
    for kind, col, first, stride, vals in sair.assertions():
        for k in range(len(srows) // stride):
            assert srows[first + k * stride][col] == vals[k % len(vals)], (kind, col, first)
    mtrace, mpub = batch.merkle_update_trace()
    mrows = [[int(v) for v in r] for r in mtrace.T]
    assert pyair.violations(pyair.MerkleUpdateAir(len(mrows), [int(v) for v in mpub]), mrows) == []
