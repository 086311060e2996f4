"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI of include/csg.h, against the CPU oracle on the same
seeded inputs.  Integer arithmetic throughout: every comparison is bit-exact."""
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
P = 0x4180000000000001


def rand_field(rng, shape):
    return (rng.integers(0, 2**63, size=shape, dtype=np.uint64) % np.uint64(P)).astype(np.uint64)


# ---------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("logn,width,blowup", [(1, 3, 2), (3, 5, 4), (6, 2, 8), (10, 14, 4), (11, 3, 8), (12, 7, 8), (13, 2, 2), (16, 3, 8), (20, 1, 2),
                                               (19, 2, 4), (20, 3, 8), (21, 1, 2)])   # 2^19..2^21: the warp-per-lane 1024-point passes
def test_lde_matches_oracle(ctx, oracle, logn, width, blowup):
    rng = np.random.default_rng(logn * 100 + width)
    n = 1 << logn
    cols = rand_field(rng, (width, n))
    got = ctx.lde(cols, blowup)
    for c in range(width):
        want = oracle.from_mont_fast(oracle.lde_column(oracle.to_mont_fast(cols[c]), blowup))
        assert np.array_equal(got[c], want), f"column {c}"


def test_lde_of_low_degree_column_is_the_polynomial(ctx):
    # size-independent property at a large size: LDE of evaluations of x -> x^3 + 5 over the trace domain equals that
    # polynomial on the coset 3*<w>
    logn, blowup = 18, 8
    n = 1 << logn
    g = pow(pow(3, 131, P), 1 << (55 - logn), P)
    x = np.empty(n, dtype=object)
    acc = 1
    for i in range(n):
        x[i] = acc
        acc = acc * g % P
    col = np.array([(int(v) ** 3 + 5) % P for v in x], dtype=np.uint64).reshape(1, n)
    got = ctx.lde(col, blowup)[0]
    gl = pow(pow(3, 131, P), 1 << (55 - logn - 3), P)
    for j in [0, 1, 7, 8, 9, 12345, n * blowup - 1]:
        xj = 3 * pow(gl, j, P) % P
        assert int(got[j]) == (xj ** 3 + 5) % P


@pytest.mark.parametrize("hash_fn", [2, 3])
@pytest.mark.parametrize("width,rows", [(1, 4), (4, 300), (8, 64), (14, 1000), (17, 33), (56, 128), (94, 513), (128, 16)])
def test_row_hashes_match_oracle_and_hashlib(ctx, oracle, hash_fn, width, rows):
    rng = np.random.default_rng(width * 7 + rows)
    cols = rand_field(rng, (width, rows))
    got = ctx.hash_rows(cols, hash_fn)
    for r in [0, 1, rows // 2, rows - 1]:
        data = cols[:, r].astype("<u8").tobytes()
        want = oracle.blake3(data) if hash_fn == 2 else hashlib.sha3_256(data).digest()
        assert got[r].tobytes() == want
    mont = oracle.to_mont_fast(cols)
    for r in range(0, rows, max(1, rows // 16)):
        assert got[r].tobytes() == oracle.hash_elements(np.ascontiguousarray(mont[:, r]), hash_fn)


@pytest.mark.parametrize("hash_fn", [2, 3])
@pytest.mark.parametrize("logl", [1, 2, 9, 10, 11, 15])
def test_merkle_tree_matches_oracle(ctx, oracle, hash_fn, logl):
    rng = np.random.default_rng(logl)
    leaves = rng.integers(0, 256, size=(1 << logl, 32), dtype=np.uint8)
    got = ctx.merkle(leaves, hash_fn)
    want = oracle.merkle_nodes(leaves, hash_fn)
    assert np.array_equal(got[1:], want[1:])


@pytest.mark.parametrize("logm", [3, 6, 10, 16, 21])
def test_fri_fold_matches_oracle(ctx, oracle, logm):
    rng = np.random.default_rng(logm)
    evals = rand_field(rng, 1 << logm)
    alpha = int(rand_field(rng, 1)[0])
    got = ctx.fri_fold4(evals, alpha)
    want = oracle.from_mont_fast(oracle.fri_fold4(oracle.to_mont_fast(evals), int(oracle.to_mont_fast(np.array([alpha], dtype=np.uint64))[0])))
    assert np.array_equal(got, want)


def test_fri_fold_of_a_cubic_is_constant(ctx):
    # folding by 4 maps a polynomial of degree < 4 to a constant: sum_d c_d alpha^d
    m, alpha, c = 1 << 12, 987654321, [11, 22, 33, 44]
    gl = pow(pow(3, 131, P), 1 << (55 - 12), P)
    ev = np.array([sum(cd * pow(3 * pow(gl, j, P) % P, d, P) for d, cd in enumerate(c)) % P for j in range(m)], dtype=np.uint64)
    out = ctx.fri_fold4(ev, alpha)
    want = sum(cd * pow(alpha, d, P) for d, cd in enumerate(c)) % P
    assert np.all(out == np.uint64(want))


# ---------------------------------------------------------------------------------------------- whole proofs
def prove_both(ctx, oracle, csg, air_id, trace, pub, blowup=8, hash_fn=2):
    want = oracle.prove(air_id, trace, pub, oracle.options(blowup=blowup, hash_fn=hash_fn))
    got = ctx.prove(air_id, trace, pub, csg.ProofOptions(blowup_factor=blowup, hash_fn=hash_fn))
    return got, want


def assert_same_proof(got, want):
    if got != want:
        first = next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), min(len(got), len(want)))
        raise AssertionError(f"proof bytes differ: len {len(got)} vs {len(want)}, first difference at byte {first}")


@pytest.mark.parametrize("chain", [2, 8, 128, 1024])
@pytest.mark.parametrize("hash_fn", [2, 3])
def test_rescue_proof_identical_to_oracle(ctx, oracle, csg, chain, hash_fn):
    # config 2: benches/rescue.rs, seed [42..48], blowup 4
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), chain)
    got, want = prove_both(ctx, oracle, csg, csg.AIR_RESCUE, trace, pub, blowup=4, hash_fn=hash_fn)
    assert_same_proof(got, want)
    assert oracle.verify(oracle.AIR_RESCUE, pub, got) == 0


@pytest.mark.parametrize("blowup", [4, 8, 16])
def test_range_proof_identical_to_oracle(ctx, oracle, csg, blowup):
    for number in [0, 1, 123456789012345, 2**63 - 1]:
        trace, pub = csg.build_range_trace(number)
        got, want = prove_both(ctx, oracle, csg, csg.AIR_RANGE, trace, pub, blowup=blowup)
        assert_same_proof(got, want)
        assert oracle.verify(oracle.AIR_RANGE, pub, got) == 0


def test_merkle_init_proof_identical_to_oracle(ctx, oracle, csg):
    z = np.zeros(14, dtype=np.uint64)
    trace, pub = csg.build_merkle_init_trace(z, z, 1)   # PreMerkleExample::new (src/merkle/init/mod.rs:66-79)
    for blowup in (4, 8):
        got, want = prove_both(ctx, oracle, csg, csg.AIR_MERKLE_INIT, trace, pub, blowup=blowup)
        assert_same_proof(got, want)
        assert oracle.verify(oracle.AIR_MERKLE_INIT, pub, got) == 0


@pytest.mark.parametrize("num_tx", [1, 2, 16, 128])     # 128: the largest batch of benches/merkle.rs
def test_merkle_update_proof_identical_to_oracle(ctx, oracle, csg, num_tx):
    batch = csg.TransactionBatch(seed=3, num_tx=num_tx)
    trace, pub = batch.merkle_update_trace()
    got, want = prove_both(ctx, oracle, csg, csg.AIR_MERKLE_UPDATE, trace, pub, blowup=8)
    assert_same_proof(got, want)
    assert oracle.verify(oracle.AIR_MERKLE_UPDATE, pub, got) == 0


@pytest.mark.parametrize("num_sig", [1, 2, 8, 32, 128])   # from 32 signatures (2^14 rows) on the low-degree split runs; 128: benches/schnorr.rs
def test_schnorr_proof_identical_to_oracle(ctx, oracle, csg, num_sig):
    batch = csg.SignatureBatch(seed=5, num_sig=num_sig)
    trace, pub = batch.schnorr_trace()
    got, want = prove_both(ctx, oracle, csg, csg.AIR_SCHNORR, trace, pub, blowup=8)
    assert_same_proof(got, want)
    assert oracle.verify(oracle.AIR_SCHNORR, pub, got) == 0


@pytest.mark.parametrize("num_tx,hash_fn", [(1, 2), (4, 2), (2, 3), (16, 2), (128, 3)])
def test_transaction_proof_identical_to_oracle(ctx, oracle, csg, num_tx, hash_fn):
    # config 1: the state-transition example at its smallest batches, default options (src/lib.rs:78-86)
    batch = csg.TransactionBatch(seed=1, num_tx=num_tx)
    trace, pub = batch.transaction_trace()
    got, want = prove_both(ctx, oracle, csg, csg.AIR_TRANSACTION, trace, pub, blowup=8, hash_fn=hash_fn)
    assert_same_proof(got, want)
    assert oracle.verify(oracle.AIR_TRANSACTION, pub, got) == 0
    wrong = pub.copy()
    wrong[8] = (int(wrong[8]) + 1) % P
    assert oracle.verify(oracle.AIR_TRANSACTION, wrong, got) != 0      # src/tests.rs:32-37


@pytest.mark.parametrize("ext", [1, 2, 3])
def test_low_degree_split_and_direct_evaluation_give_the_same_proof(ctx, csg, monkeypatch, ext):
    # small traces evaluate every constraint on every coset (fewer launches); from 2^14 rows on the low-degree constraints are
    # evaluated on half of the cosets and extended.  CSG_SPLIT_MIN_ROWS=0 forces the second path on the small traces here.
    cases = [(csg.AIR_TRANSACTION, csg.TransactionBatch(seed=1, num_tx=2).transaction_trace()),
             (csg.AIR_SCHNORR, csg.SignatureBatch(seed=5, num_sig=2).schnorr_trace())]
    opt = csg.ProofOptions(field_extension=ext)
    direct = [ctx.prove(air, trace, pub, opt) for air, (trace, pub) in cases]
    launches_direct = ctx.timings()["kernel_launches"]
    monkeypatch.setenv("CSG_SPLIT_MIN_ROWS", "0")
    with csg.Context(0) as forced:
        split = [forced.prove(air, trace, pub, opt) for air, (trace, pub) in cases]
        assert forced.timings()["kernel_launches"] > launches_direct     # the split really ran
    assert split == direct


def test_reproving_a_resident_trace_gives_the_same_bytes(ctx, csg):
    batch = csg.TransactionBatch(seed=9, num_tx=2)
    trace, pub = batch.transaction_trace()
    opt = csg.ProofOptions()
    first = ctx.prove(csg.AIR_TRANSACTION, trace, pub, opt)
    ctx.reload_resident_trace()
    assert ctx.prove_loaded() == first
    t = ctx.timings()
    assert t["kernel_launches"] > 0 and t["total"] > 0


def test_stage_timings_are_read_on_demand(ctx, csg):
    # csg_get_timings: the stage times are event pairs collected when asked for, and describe the LAST proof only
    trace, pub = csg.TransactionBatch(seed=9, num_tx=4).transaction_trace()
    ctx.prove(csg.AIR_TRANSACTION, trace, pub, csg.ProofOptions())
    stages = ("lde", "commit_trace", "constraints", "composition", "ood_deep", "fri", "queries")
    t1 = ctx.timings()
    assert all(t1[k] > 0 for k in stages)
    assert sum(t1[k] for k in stages) <= t1["total"] * 1.02
    assert ctx.timings() == t1                                   # reading twice changes nothing
    for _ in range(3):                                           # proofs nobody asks about leave nothing behind
        ctx.reload_resident_trace()
        ctx.prove_loaded()
    t2 = ctx.timings()
    assert sum(t2[k] for k in stages) <= t2["total"] * 1.02
    assert t2["fri"] < 2 * t1["fri"] + 0.05
    # (the first proof took its trace from host memory: chunked extension, more launches than the resident one)
    assert 0 < sum(t2["stage_launches"].values()) <= t2["kernel_launches"] <= t1["kernel_launches"]


def test_batch_after_batch_of_one_shape(ctx, oracle, csg):
    # csg_set_air with the shape of the last call keeps the device tables and only takes the new public inputs -- unless the
    # periodic columns carry public inputs (Schnorr: keys and messages), then the tables follow
    for air, make in ((csg.AIR_TRANSACTION, lambda s: csg.TransactionBatch(seed=s, num_tx=2).transaction_trace()),
                      (csg.AIR_SCHNORR, lambda s: csg.SignatureBatch(seed=s, num_sig=2).schnorr_trace()),
                      (csg.AIR_MERKLE_UPDATE, lambda s: csg.TransactionBatch(seed=s, num_tx=2).merkle_update_trace())):
        pubs = []
        for seed in (31, 32, 31):
            trace, pub = make(seed)
            got, want = prove_both(ctx, oracle, csg, air, trace, pub)
            assert_same_proof(got, want)
            pubs.append(pub.tobytes())
        assert pubs[0] != pubs[1]


def test_prefetched_traces_prove_like_prove(ctx, csg):
    # csg_prefetch_trace / csg_prove_prefetched: a stream of traces, the copy of the next one under the proof of the current one
    opt = csg.ProofOptions()
    batches = [csg.TransactionBatch(seed=20 + i, num_tx=2).transaction_trace() for i in range(3)]
    pub = batches[0][1]
    want = [ctx.prove(csg.AIR_TRANSACTION, t, p, opt) for t, p in batches]
    bufs = [csg.HostBuffer(94, 2048) for _ in batches]
    for b, (t, _) in zip(bufs, batches):
        b.array[:] = t
    got = []
    for i, (t, p) in enumerate(batches):       # public inputs differ per batch: set_air per proof, one trace in flight
        ctx.set_air(csg.AIR_TRANSACTION, 2048, p, opt)
        ctx.prefetch_trace_ptr(bufs[i].ptr)
        got.append(ctx.prove_prefetched_ptr())
    assert got == want
    # same AIR and public inputs, three traces back to back: trace k+1 is copied while trace k is proved
    t0, p0 = batches[0]
    ctx.set_air(csg.AIR_TRANSACTION, 2048, p0, opt)
    ctx.prefetch_trace_ptr(bufs[0].ptr)
    first = ctx.prove_prefetched_ptr(bufs[0].ptr)
    second = ctx.prove_prefetched_ptr(bufs[0].ptr)
    third = ctx.prove_prefetched_ptr()
    assert first == second == third == want[0]
    assert ctx.timings()["h2d"] > 0
    with pytest.raises(csg.CsgError):
        ctx.prove_prefetched_ptr()              # nothing waiting
    ctx.prefetch_trace_ptr(bufs[1].ptr)
    with pytest.raises(csg.CsgError):
        ctx.prefetch_trace_ptr(bufs[2].ptr)     # one trace can wait at a time
    ctx.reload_resident_trace()                 # the last proved trace is still the resident one
    assert ctx.prove_loaded() == want[0]
    ctx.set_air(csg.AIR_TRANSACTION, 2048, batches[1][1], opt)   # same shape, new public inputs: the waiting trace stays
    assert ctx.prove_prefetched_ptr() == want[1]
    ctx.prefetch_trace_ptr(bufs[2].ptr)
    ctx.set_air(csg.AIR_TRANSACTION, 4096, csg.TransactionBatch(seed=20, num_tx=4).transaction_trace()[1], opt)   # another shape drops it
    with pytest.raises(csg.CsgError):
        ctx.prove_prefetched_ptr()
    for b in bufs:
        b.close()


def test_example_facade(csg, oracle):
    ex = csg.get_example(2, seed=4)
    proof = ex.prove()                                   # witness built on the device
    assert oracle.verify(oracle.AIR_TRANSACTION, ex.pub_inputs, proof) == 0
    assert ex.prove(witness_on_device=False) == proof    # witness built on the host: same trace, same proof
    assert ex.verify(proof) and not ex.verify_with_wrong_inputs(proof)     # src/tests.rs:12-37 with the product's own verifier


def test_errors_are_reported_not_swallowed(ctx, csg):
    trace, pub = csg.build_range_trace(5)
    with pytest.raises(csg.CsgError):
        ctx.prove(csg.AIR_RANGE, trace, pub, csg.ProofOptions(fri_folding_factor=8))
    with pytest.raises(csg.CsgError):
        ctx.prove(csg.AIR_RANGE, trace, pub[:0], csg.ProofOptions())
    with pytest.raises(csg.CsgError):   # blowup below the AIR's constraint-evaluation blowup
        batch = csg.TransactionBatch(seed=1, num_tx=1)
        t, p = batch.transaction_trace()
        ctx.prove(csg.AIR_TRANSACTION, t, p, csg.ProofOptions(blowup_factor=4))


def test_rejected_set_air_is_rejected_again(csg, oracle):
    # csg_set_air with the AIR, length and options of the last successful call keeps the device tables (the fast path of
    # test_batch_after_batch_of_one_shape).  A call that fails on a check after the context's members took the new shape must
    # not make the same arguments look like the last good shape: repeated, it has to fail again, with the same message, and
    # the prove and prefetch calls must refuse to run on what it left.  The repeated set_air comes first: a context that took
    # the fast path here would hold the tables of the old shape.
    L = csg.lib()
    rescue = lambda chain: csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), chain)     # noqa: E731
    r_trace, r_pub = rescue(32)                                                                   # 256 rows
    tx_trace, tx_pub = csg.TransactionBatch(seed=1, num_tx=1).transaction_trace()
    cases = [("constraint evaluation blowup", csg.AIR_TRANSACTION, tx_trace.shape[1], tx_pub, csg.ProofOptions(blowup_factor=4), tx_trace),
             ("above 2^22", csg.AIR_RESCUE, 1 << 23, r_pub, csg.ProofOptions(), None),
             ("FRI remainder", csg.AIR_RESCUE, r_trace.shape[1], r_pub, csg.ProofOptions(blowup_factor=32, fri_max_remainder_size=4), r_trace)]

    def rejected_twice(c, air, n, pub, opt):
        msgs = []
        for _ in range(2):
            with pytest.raises(csg.CsgError) as e:
                c.set_air(air, n, pub, opt)
            msgs.append((str(e.value), L.csg_last_error(c._h)))
        assert msgs[0] == msgs[1]
        return msgs[0][0]

    with csg.Context(0) as c:
        good = csg.ProofOptions(blowup_factor=4)
        for reason, air, n, pub, opt, trace in cases:
            c.set_air(csg.AIR_RESCUE, r_trace.shape[1], r_pub, good)          # a good shape first: the fast path is armed
            assert reason in rejected_twice(c, air, n, pub, opt)
            with pytest.raises(csg.CsgError):
                c.prove_loaded()
            with pytest.raises(csg.CsgError):
                c.reload_resident_trace()
            if trace is not None:
                for _ in range(2):
                    with pytest.raises(csg.CsgError):
                        c.prove(air, trace, pub, opt)
        # a prefetched trace does not survive a rejected set_air
        hb = csg.HostBuffer(14, r_trace.shape[1])
        try:
            hb.array[:] = r_trace
            c.set_air(csg.AIR_RESCUE, r_trace.shape[1], r_pub, good)
            c.prefetch_trace_ptr(hb.ptr)
            with pytest.raises(csg.CsgError):
                c.set_air(csg.AIR_RESCUE, r_trace.shape[1], r_pub, csg.ProofOptions(blowup_factor=32, fri_max_remainder_size=4))
            with pytest.raises(csg.CsgError):
                c.prove_prefetched_ptr()
            with pytest.raises(csg.CsgError):
                c.set_air(csg.AIR_RESCUE, r_trace.shape[1], r_pub, csg.ProofOptions(blowup_factor=32, fri_max_remainder_size=4))
            # and the context proves correctly afterwards, for the last good shape and for the others
            c.set_air(csg.AIR_RESCUE, r_trace.shape[1], r_pub, good)
            c.prefetch_trace_ptr(hb.ptr)
            want = oracle.prove(oracle.AIR_RESCUE, r_trace, r_pub, oracle.options(blowup=4))
            assert c.prove_prefetched_ptr() == want
        finally:
            hb.close()
        assert c.prove(csg.AIR_RESCUE, r_trace, r_pub, good) == want
        assert c.prove(csg.AIR_TRANSACTION, tx_trace, tx_pub, csg.ProofOptions()) == oracle.prove(oracle.AIR_TRANSACTION, tx_trace, tx_pub, oracle.options())
    # the shard plan: 8 ranks cannot share the 4 LDE cosets of blowup 4.  One rank's set_air runs no collective.
    with csg.LocalGroup(8) as grp:
        r0 = grp.ctxs[0]
        r0.set_air(csg.AIR_RESCUE, r_trace.shape[1], r_pub, csg.ProofOptions())
        assert "divide the blowup" in rejected_twice(r0, csg.AIR_RESCUE, r_trace.shape[1], r_pub, good)
        with pytest.raises(csg.CsgError):
            r0.prove_loaded()
        proofs = grp.prove(csg.AIR_RESCUE, r_trace, r_pub, csg.ProofOptions())
    assert proofs == [oracle.prove(oracle.AIR_RESCUE, r_trace, r_pub, oracle.options())] * 8


def test_device_field_arithmetic_selftest(ctx, csg):
    # the fused modular multiplication and the column-form accumulators (field.cuh) against mul_wide + the textbook reduction +
    # modular additions, on random operands and carry-path patterns; the same checker runs on the host in tests/host_harness.cpp
    import ctypes as C
    L = csg.lib()
    L.csg_debug_field_selftest.restype, L.csg_debug_field_selftest.argtypes = C.c_longlong, [C.c_void_p]
    assert L.csg_debug_field_selftest(ctx._h) == 0


def test_device_montgomery_reduction_selftest(ctx, csg):
    # the 32-bit word-serial reduction used by every kernel against the textbook 64-bit one, on random and edge operands
    import ctypes as C
    L = csg.lib()
    L.csg_debug_redc_selftest.restype, L.csg_debug_redc_selftest.argtypes = C.c_longlong, [C.c_void_p]
    assert L.csg_debug_redc_selftest(ctx._h) == 0


@pytest.mark.parametrize("num_tx", [1, 4, 32])
def test_device_witness_matches_host_builder(csg, oracle, num_tx):
    # SURVEY.md 8(f).1: TransactionProver::build_trace on the GPU, bit for bit the table the host builder produces
    batch = csg.TransactionBatch(seed=21 + num_tx, num_tx=num_tx)
    want, pub = batch.transaction_trace()
    assert np.array_equal(pub, batch.public_inputs())
    with csg.Context(0) as c:
        c.set_air(csg.AIR_TRANSACTION, 1024 * num_tx, pub, csg.ProofOptions())
        c.build_transaction_trace(batch)
        got = c.download_trace(94, 1024 * num_tx)
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"first differing (column, row): {bad[0]}"
        proof = c.prove_loaded()
    assert proof == oracle.prove(oracle.AIR_TRANSACTION, want, pub, oracle.options())


@pytest.mark.parametrize("num_queries,grinding,max_remainder,blowup", [(8, 0, 256, 4), (100, 0, 64, 8), (42, 8, 1024, 16), (1, 4, 16, 4), (27, 0, 16, 16)])
def test_proof_options_are_honoured(ctx, oracle, csg, num_queries, grinding, max_remainder, blowup):
    # ProofOptions::new(num_queries, blowup, grinding, hash, extension, folding, max_remainder) (src/lib.rs:78-86): every field
    # that changes the proof must change it the same way on both sides
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 32)
    want = oracle.prove(oracle.AIR_RESCUE, trace, pub, oracle.options(num_queries=num_queries, blowup=blowup, grinding=grinding, max_remainder=max_remainder))
    got = ctx.prove(csg.AIR_RESCUE, trace, pub, csg.ProofOptions(num_queries=num_queries, blowup_factor=blowup, grinding_factor=grinding,
                                                                   fri_max_remainder_size=max_remainder))
    assert_same_proof(got, want)
    assert csg.verify(csg.AIR_RESCUE, pub, got) == 0 and oracle.verify(oracle.AIR_RESCUE, pub, got) == 0


def test_degenerate_shapes_fail_cleanly(ctx, csg):
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 1)      # 8 rows: 32 LDE points < 42 queries
    with pytest.raises(csg.CsgError, match="query positions"):
        ctx.prove(csg.AIR_RESCUE, trace, pub, csg.ProofOptions(blowup_factor=4))
    with pytest.raises(csg.CsgError):
        ctx.prove(csg.AIR_RESCUE, trace[:, :6], pub, csg.ProofOptions(blowup_factor=4))  # not a power of two
    with pytest.raises(csg.CsgError):
        ctx.prove(csg.AIR_RANGE, *csg.build_range_trace(1), csg.ProofOptions(field_extension=4))   # FieldExtension is None / Quadratic / Cubic
    with pytest.raises(csg.CsgError, match="remainder"):
        ctx.prove(csg.AIR_RESCUE, *csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 32), csg.ProofOptions(blowup_factor=32, fri_max_remainder_size=4))
    # the context stays usable after errors
    t, p = csg.build_range_trace(123)
    assert csg.verify(csg.AIR_RANGE, p, ctx.prove(csg.AIR_RANGE, t, p, csg.ProofOptions())) == 0


def test_independent_python_witnesses_prove_identically(ctx, oracle, csg):
    # witnesses from oracle/pyair.py (second, independent restatement: own metadata, tree, signing and trace layout; tests/
    # test_air_independent.py) through the GPU prover: the bytes must be the C oracle's, and both verifiers accept
    from oracle import pyair
    cols = lambda rows: np.ascontiguousarray(np.array(rows, dtype=np.uint64).T)      # noqa: E731
    batch = pyair.TransactionBatch(seed=13, num_tx=2)
    cases = [(csg.AIR_TRANSACTION, batch.transaction_trace(), batch.pub_inputs(), 8),
             (csg.AIR_MERKLE_UPDATE, batch.merkle_update_trace(), batch.pub_inputs(), 8),
             (csg.AIR_SCHNORR, *pyair.schnorr_batch(seed=14, num_sig=2), 8),
             (csg.AIR_SCHNORR, *pyair.schnorr_batch(seed=15, num_sig=1), 8),
             (csg.AIR_RANGE, *pyair.range_trace(987654321987), 8),
             (csg.AIR_RESCUE, *pyair.rescue_trace(list(range(42, 49)), 32), 4)]
    for air, rows, pub, blowup in cases:
        trace, pub = cols(rows), np.array(pub, dtype=np.uint64)
        got, want = prove_both(ctx, oracle, csg, air, trace, pub, blowup=blowup)
        assert_same_proof(got, want)
        assert csg.verify(air, pub, got) == 0 and oracle.verify(air, pub, got) == 0
