"""GPU parity (-m gpu) at shapes the other suites do not prove: blowup factors above the constraint-evaluation blowup of the
AIRs with the low-degree split, and the largest traces csg_set_air accepts.

Blowup 16 / 32 over ce blowup 8: the ce cosets are every 2nd / 4th LDE coset, so the split's even/odd coset mix, its coset
interpolation and extension read strided cosets; a sharded proof runs the split without the exchange (only ce == blowup
keeps it), and the first FRI layer folds from logm - logW = 4 / 5.  2^22 rows: both four-step NTT passes are 2^11 points,
and a 4096-transaction proof holds 94 x 2^25 > 2^31 LDE elements in one context.  Every proof is compared byte for byte
with the CPU oracle's (oracle/stark.c), except the 4096-transaction one, whose oracle proof would need tens of GB of host
memory: that one is checked by both verifiers, by a two-rank group whose ranks each hold fewer than 2^31 elements, and by
the device-built witness.
"""
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
P = 0x4180000000000001


def first_difference(got, want):
    return next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), min(len(got), len(want)))


@pytest.fixture(scope="module")
def oracle_proof(csg, oracle):
    """(air, num, blowup, ext) -> (trace, pub, oracle proof bytes), each computed once for the module"""
    cache = {}
    builders = {"tx": lambda k: csg.TransactionBatch(seed=17, num_tx=k).transaction_trace(),
                "sig": lambda k: csg.SignatureBatch(seed=19, num_sig=k).schnorr_trace()}
    airs = {"tx": oracle.AIR_TRANSACTION, "sig": oracle.AIR_SCHNORR}

    def get(kind, num, blowup, ext):
        key = (kind, num, blowup, ext)
        if key not in cache:
            trace, pub = builders[kind](num)
            opt = oracle.options(blowup=blowup, field_extension=ext)
            want = oracle.prove(airs[kind], trace, pub, opt) if ext == 1 else oracle.prove_generic(airs[kind], trace, pub, opt)
            cache[key] = (trace, pub, want)
        return cache[key]
    return get


def check_proof(csg, oracle, air, pub, got, want, ext, changed_input):
    """bytes equal to the oracle's; both verifiers accept; both reject a changed public input"""
    assert got == want, f"proof bytes differ (len {len(got)} vs {len(want)}), first difference at byte {first_difference(got, want)}"
    overify = oracle.verify if ext == 1 else oracle.verify_generic
    assert csg.verify(air, pub, got) == 0 and overify(air, pub, got) == 0
    wrong = pub.copy()
    wrong[changed_input] = (int(wrong[changed_input]) + 1) % P
    assert csg.verify(air, wrong, got) != 0 and overify(air, wrong, got) != 0


# ---------------------------------------------------------------------------------------------- blowup above ce blowup
@pytest.mark.parametrize("ext", [1, 2, 3])
@pytest.mark.parametrize("blowup", [16, 32])
def test_transaction_wide_blowup_identical_to_oracle(ctx, csg, oracle, oracle_proof, blowup, ext):
    # 16 transactions = 2^14 rows: the low-degree split runs at the default threshold
    trace, pub, want = oracle_proof("tx", 16, blowup, ext)
    got = ctx.prove(csg.AIR_TRANSACTION, trace, pub, csg.ProofOptions(blowup_factor=blowup, field_extension=ext))
    check_proof(csg, oracle, csg.AIR_TRANSACTION, pub, got, want, ext, 8)


@pytest.mark.parametrize("ext", [1, 2, 3])
@pytest.mark.parametrize("blowup", [16, 32])
def test_forced_split_and_direct_evaluation_at_wide_blowup(ctx, csg, oracle, oracle_proof, monkeypatch, blowup, ext):
    # 2 transactions: the direct evaluation by default, the split with CSG_SPLIT_MIN_ROWS=0; both must be the oracle's bytes
    trace, pub, want = oracle_proof("tx", 2, blowup, ext)
    opt = csg.ProofOptions(blowup_factor=blowup, field_extension=ext)
    direct = ctx.prove(csg.AIR_TRANSACTION, trace, pub, opt)
    launches_direct = ctx.timings()["kernel_launches"]
    check_proof(csg, oracle, csg.AIR_TRANSACTION, pub, direct, want, ext, 8)
    monkeypatch.setenv("CSG_SPLIT_MIN_ROWS", "0")
    with csg.Context(0) as forced:
        split = forced.prove(csg.AIR_TRANSACTION, trace, pub, opt)
        assert forced.timings()["kernel_launches"] > launches_direct     # the split really ran
    assert split == want, f"first difference at byte {first_difference(split, want)}"


@pytest.mark.parametrize("ext", [1, 3])
def test_schnorr_wide_blowup_identical_to_oracle(ctx, csg, oracle, oracle_proof, ext):
    # 32 signatures = 2^14 rows: split by default
    trace, pub, want = oracle_proof("sig", 32, 16, ext)
    got = ctx.prove(csg.AIR_SCHNORR, trace, pub, csg.ProofOptions(blowup_factor=16, field_extension=ext))
    check_proof(csg, oracle, csg.AIR_SCHNORR, pub, got, want, ext, 0)


@pytest.mark.parametrize("world,blowup,ext", [(2, 16, 1), (4, 16, 1), (8, 16, 1), (2, 16, 3), (4, 16, 3), (8, 16, 3), (8, 32, 1)])
def test_transaction_wide_blowup_sharded(csg, oracle_proof, world, blowup, ext):
    # ce blowup 8 < blowup: every rank splits on its own ce cosets, without the exchange of interpolants.  World 8 owns 2
    # (blowup 16) or 4 (blowup 32) LDE cosets and one ce coset per rank.
    trace, pub, want = oracle_proof("tx", 16, blowup, ext)
    with csg.LocalGroup(world) as grp:
        proofs = grp.prove(csg.AIR_TRANSACTION, trace, pub, csg.ProofOptions(blowup_factor=blowup, field_extension=ext))
    bad = [r for r, p in enumerate(proofs) if p != want]
    assert not bad, f"ranks {bad} differ from the oracle, first difference at byte {first_difference(proofs[bad[0]], want)}"


# ---------------------------------------------------------------------------------------------- the 2^22-row limit
def test_rescue_at_the_trace_length_limit_identical_to_oracle(ctx, csg, oracle):
    # 2^19 hashes = 2^22 rows x 14 columns, blowup 4: the only NTT size whose two four-step passes are both 2^11 points
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 1 << 19)
    assert trace.shape == (14, 1 << 22)
    got = ctx.prove(csg.AIR_RESCUE, trace, pub, csg.ProofOptions(blowup_factor=4))
    t0 = time.perf_counter()
    want = oracle.prove(oracle.AIR_RESCUE, trace, pub, oracle.options(blowup=4))
    print(f"oracle proof of 2^22 x 14 Rescue rows at blowup 4: {time.perf_counter() - t0:.1f} s")
    check_proof(csg, oracle, csg.AIR_RESCUE, pub, got, want, 1, 7)
    with pytest.raises(csg.CsgError, match="2\\^22"):
        ctx.set_air(csg.AIR_RESCUE, 1 << 23, pub, csg.ProofOptions(blowup_factor=4))


def test_transaction_proof_above_2_pow_31_lde_elements(csg, oracle):
    # 4096 transactions: 94 x 2^22 trace, 94 x 2^25 = 3.15e9 LDE elements in one context (about 25 GB of LDE).  Each context
    # is closed before the next one starts.
    num_tx, seed = 4096, 23
    trace, pub = csg.TransactionBatch(seed=seed, num_tx=num_tx).transaction_trace()
    opt = csg.ProofOptions()
    with csg.Context(0) as c:
        proof = c.prove(csg.AIR_TRANSACTION, trace, pub, opt)
    assert csg.verify(csg.AIR_TRANSACTION, pub, proof, opt) == 0 and oracle.verify(oracle.AIR_TRANSACTION, pub, proof) == 0
    wrong = pub.copy()
    wrong[8] = (int(wrong[8]) + 1) % P
    assert csg.verify(csg.AIR_TRANSACTION, wrong, proof) != 0 and oracle.verify(oracle.AIR_TRANSACTION, wrong, proof) != 0
    # two ranks hold 1.58e9 LDE elements each, below 2^31: a 32-bit index in the single context would show as a difference
    with csg.LocalGroup(2) as grp:
        assert grp.prove(csg.AIR_TRANSACTION, trace, pub, opt) == [proof, proof]
    del trace
    ex = csg.TransactionExample(opt, num_tx, seed=seed, batch_on_device=True)   # metadata and witness built on the device
    try:
        assert ex.prove() == proof
        assert np.array_equal(ex.pub_inputs, pub)
    finally:
        ex.ctx.close()
