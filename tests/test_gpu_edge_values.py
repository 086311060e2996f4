"""Values at the edges of their ranges (-m gpu).  The rest of the suite feeds uniform random canonical words; here:

A. trace words anywhere in [0, 2^64): a word counts as its residue (csg.h, DESIGN 1), so a trace whose words are random
   representatives v + k*p must prove, commit and validate exactly as its reduced form, on every input path and at every size
   whose inverse NTT reads the caller's words through another kernel route (the `clamp_in` subtraction of 2p in
   ntt_pass_kernel and in ntt1024_kernel's `scaled`);
B. structured columns (zero, constant, spike, monomial, alternating 0 / p-1) through ctx.lde, ctx.fri_fold4 and ctx.hash_rows,
   against exact closed forms in Python integers -- no oracle;
C. every stage buffer a level-2 call produces holds canonical words (csg_debug_count_unreduced): the proof bytes cannot show
   this, since hashing and serialisation map a stored p to 0;
D. the A/B tuning routes (CSG_NTT_GENERIC, CSG_NTT_SHAPE_A/B, CSG_NO_SPLIT, CSG_NO_ECC_SPLIT, CSG_H2D_CHUNKS,
   CSG_COEF_BLOCKWISE) give the default bytes.  Knobs read once per process run in a child process."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import blake3
import numpy as np
import pytest

from test_gpu_prove_many import AIRS, witnesses

pytestmark = pytest.mark.gpu
P = 0x4180000000000001
R = (1 << 64) % P                      # 2^64 mod p: the word 2^64 - 1 is the largest representative of R - 1
MONT_MINUS_ONE = P - pow(R, -1, P)     # the canonical value whose Montgomery form is p - 1
TOP = np.uint64(2**64 - 1)
HERE = Path(__file__).resolve().parent
KNOBS = ("CSG_NTT_GENERIC", "CSG_NTT_SHAPE_A", "CSG_NTT_SHAPE_B", "CSG_NO_SPLIT", "CSG_NO_ECC_SPLIT", "CSG_H2D_CHUNKS",
         "CSG_COEF_BLOCKWISE", "CSG_SPLIT_MIN_ROWS")


def root_of_unity(logn):
    return pow(pow(3, 131, P), 1 << (55 - logn), P)


# ---------------------------------------------------------------------------------------------- words anywhere in [0, 2^64)
def lift(words, rng, forced=8):
    """each word v < p -> v + k*p, k uniform in 0 .. floor((2^64 - 1 - v) / p) (about half the words end up >= 2p); every cell
    of residue R - 1 and `forced` random cells take their largest representative (2^64 - 1 for residue R - 1)"""
    v = np.ascontiguousarray(words, dtype=np.uint64)
    kmax = (TOP - v) // np.uint64(P)
    k = (rng.random(v.shape) * (kmax + np.uint64(1))).astype(np.uint64)
    flat_k, flat_max = k.reshape(-1), kmax.reshape(-1)
    pick = rng.integers(0, v.size, size=forced)
    flat_k[pick] = flat_max[pick]
    top = v == np.uint64(R - 1)
    k[top] = kmax[top]
    return v + k * np.uint64(P)


def random_trace(rng, width, n):
    """canonical words with cells of residue R - 1 planted at both corners and one random cell"""
    t = rng.integers(0, P, size=(width, n), dtype=np.uint64)
    t[0, 0] = t[width - 1, n - 1] = t[int(rng.integers(width)), int(rng.integers(n))] = R - 1
    return t


def lifted_case(logn, width=14, seed=0):
    rng = np.random.default_rng(seed * 1000 + logn)
    trace = random_trace(rng, width, 1 << logn)
    pub = rng.integers(0, P, size=14, dtype=np.uint64)
    return trace, lift(trace, rng), pub


def digest(proofs):
    return [hashlib.sha256(p).hexdigest() for p in proofs]


def up(traces):
    """host traces -> one contiguous int64 CUDA tensor (K, w, n): words >= 2^63 travel as negative int64"""
    import torch
    return torch.from_numpy(np.stack(traces).view(np.int64)).to("cuda:0")


def down_sha(t):
    import torch
    torch.cuda.synchronize()
    return hashlib.sha256(t.cpu().view(torch.int64).numpy().tobytes()).hexdigest()


@pytest.fixture(scope="module")
def tx1024(csg):
    """the 1024-transaction trace (2^20 x 94): column chunking and the pageable staging ring of stage 1"""
    return csg.TransactionBatch(seed=1000, num_tx=1024).transaction_trace()


# ---------------------------------------------------------------------------------------------- C: the stage-buffer check
def unreduced(csg, c, which):
    L = csg.lib()
    L.csg_debug_count_unreduced.restype, L.csg_debug_count_unreduced.argtypes = C.c_longlong, [C.c_void_p, C.c_int]
    return L.csg_debug_count_unreduced(c._h, which)


def stage_calls(c, csg, air_id, trace, pub, opt, repr=0, seed=0):
    """csg_set_air, csg_load_trace and the level-2 calls up to the composition commitment with arbitrary canonical coefficients;
    after each call the buffers it produced hold no word >= p.  Returns the trace and composition roots."""
    L, h = csg.lib(), c._h
    rng = np.random.default_rng(seed)
    ext = opt.field_extension
    c.set_air(air_id, trace.shape[1], pub, opt)
    c.load_trace(trace, repr)
    troot, croot = np.zeros(32, dtype=np.uint8), np.zeros(32, dtype=np.uint8)
    c._check(L.csg_extend_and_commit_trace(h, csg._p8(troot)))
    assert [unreduced(csg, c, k) for k in (0, 1, 2)] == [0, 0, 0], "trace coefficients / trace LDE / periodic tables"
    t_coeffs = rng.integers(0, P, size=2 * 128 * ext, dtype=np.uint64)      # at least 2 * constraints * ext words
    b_coeffs = rng.integers(0, P, size=2 * 64 * ext, dtype=np.uint64)       # at least 2 * assertions * ext words
    c._check(L.csg_eval_constraints(h, csg._p64(t_coeffs), csg._p64(b_coeffs)))
    assert unreduced(csg, c, 3) == 0, "merged constraint column"
    c._check(L.csg_commit_composition(h, csg._p8(croot)))
    assert [unreduced(csg, c, k) for k in (4, 5)] == [0, 0], "composition columns / composition LDE"
    return troot.tobytes(), croot.tobytes()


def test_count_unreduced_refuses_an_unknown_buffer(ctx, csg):
    # csg_debug_count_unreduced used to read the composition LDE for any `which` above 4
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 8)
    stage_calls(ctx, csg, csg.AIR_RESCUE, trace, pub, csg.ProofOptions(blowup_factor=4))
    assert [unreduced(csg, ctx, k) for k in (-1, 6, 1 << 20)] == [-1, -1, -1]


# ---------------------------------------------------------------------------------------------- A: one size per raw-pass route
# n = 2^6, 2^11: the single ntt_pass_kernel pass (ntt.cu:108); 2^12 .. 2^18: pass A of the split in ntt_pass_kernel; 2^19, 2^20:
# pass A in ntt1024_kernel<STAGE_IN=true> (the clamp in `scaled`, ntt.cu:212); 2^21, 2^22: pass A in ntt_pass_kernel, logS = 11
NTT_SIZES = [6, 11, 12, 16, 18, 19, 20, 21, 22]


@pytest.mark.parametrize("logn", NTT_SIZES)
def test_raw_words_prove_as_their_residues_at_every_ntt_size(ctx, oracle, csg, logn):
    # csg_prove, pageable, in both representations: the proof of the lifted words is the proof of the reduced ones; the level-2
    # trace and composition roots agree too, and every stage buffer is canonical -- for the lifted trace, an all-zero trace
    # and a constant p - 1 trace
    trace, lifted, pub = lifted_case(logn)
    assert (lifted == TOP).any() and 0.4 < (lifted >= np.uint64(2 * P)).mean() < 0.6
    opt = csg.ProofOptions(blowup_factor=4)
    for repr in (csg.REPR_CANONICAL, csg.REPR_MONTGOMERY):
        want = ctx.prove(csg.AIR_RESCUE, trace, pub, opt, repr=repr)
        assert ctx.prove(csg.AIR_RESCUE, lifted, pub, opt, repr=repr) == want, f"repr {repr}"
        if logn <= 12:   # a Montgomery word m is the Montgomery form of m mod p
            canon = trace if repr == csg.REPR_CANONICAL else oracle.from_mont_fast(trace)
            assert want == oracle.prove(oracle.AIR_RESCUE, canon, pub, oracle.options(blowup=4))
    assert stage_calls(ctx, csg, csg.AIR_RESCUE, lifted, pub, opt) == stage_calls(ctx, csg, csg.AIR_RESCUE, trace, pub, opt)
    n = 1 << logn
    for const in (0, P - 1):
        stage_calls(ctx, csg, csg.AIR_RESCUE, np.full((14, n), const, dtype=np.uint64), pub, opt)


@pytest.mark.parametrize("logn", [6, 11, 12, 16])
def test_lifted_rescue_witness_proves_and_verifies(ctx, oracle, csg, logn):
    # a valid witness, lifted: same proof as the witness, and csg_verify accepts it
    trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), (1 << logn) // 8)
    lifted = lift(trace, np.random.default_rng(logn))
    opt = csg.ProofOptions(blowup_factor=4)
    want = ctx.prove(csg.AIR_RESCUE, trace, pub, opt)
    got = ctx.prove(csg.AIR_RESCUE, lifted, pub, opt)
    assert got == want
    assert csg.verify(csg.AIR_RESCUE, pub, got) == 0
    if logn <= 12:
        assert want == oracle.prove(oracle.AIR_RESCUE, trace, pub, oracle.options(blowup=4))


@pytest.mark.parametrize("num_tx", [2, 1024])
def test_raw_words_on_every_host_input_path(ctx, oracle, csg, tx1024, num_tx):
    # a lifted transaction witness (94 columns: the ramped column chunks of stage 1) through csg_prove (pageable: the staging
    # ring; both representations), csg_prove_columns, a csg_host_alloc buffer (csg_prove_trace), csg_load_trace +
    # csg_prove_loaded and csg_prefetch_trace + csg_prove_prefetched: always the proof of the reduced words, and it verifies
    trace, pub = tx1024 if num_tx == 1024 else csg.TransactionBatch(seed=77, num_tx=num_tx).transaction_trace()
    rng = np.random.default_rng(num_tx)
    n = trace.shape[1]
    opt = csg.ProofOptions()
    lifted = lift(trace, rng)
    want = ctx.prove(csg.AIR_TRANSACTION, trace, pub, opt)
    if num_tx == 2:
        assert want == oracle.prove(oracle.AIR_TRANSACTION, trace, pub, oracle.options())
    assert ctx.prove(csg.AIR_TRANSACTION, lifted, pub, opt) == want
    assert csg.verify(csg.AIR_TRANSACTION, pub, want) == 0
    mont = lift(oracle.to_mont_fast(trace), rng)
    assert ctx.prove(csg.AIR_TRANSACTION, mont, pub, opt, repr=csg.REPR_MONTGOMERY) == want
    assert ctx.prove_columns(csg.AIR_TRANSACTION, [np.array(lifted[c]) for c in range(94)], pub, opt) == want
    del mont
    hb = csg.HostBuffer(94, n)
    try:
        hb.array[:] = lifted
        ctx.set_air(csg.AIR_TRANSACTION, n, pub, opt)
        assert ctx.prove_trace_ptr(hb.ptr) == want
        ctx.load_trace_ptr(hb.ptr)
        assert ctx.prove_loaded() == want
        ctx.prefetch_trace_ptr(hb.ptr)
        assert ctx.prove_prefetched_ptr() == want
    finally:
        hb.close()


@pytest.mark.parametrize("logn", [6, 11, 12, 16])
def test_raw_words_in_proof_batches(ctx, csg, logn):
    # csg_prove_many (both representations) and csg_prove_many_device from an int64 tensor, whose words >= 2^63 are negative:
    # the proofs of the reduced traces, and the caller's buffer is left as it was
    cases = [lifted_case(logn, seed=s) for s in range(3)]
    traces, lifted, pubs = [c[0] for c in cases], [c[1] for c in cases], np.stack([c[2] for c in cases])
    opt = csg.ProofOptions(blowup_factor=4)
    for repr in (csg.REPR_CANONICAL, csg.REPR_MONTGOMERY):
        want = [ctx.prove(csg.AIR_RESCUE, t, p, opt, repr=repr) for t, p in zip(traces, pubs)]
        assert ctx.prove_many(csg.AIR_RESCUE, lifted, pubs, opt, repr=repr) == want, f"repr {repr}"
        dev = up(lifted)
        assert (dev < 0).any()
        before = down_sha(dev)
        assert ctx.prove_many_device(csg.AIR_RESCUE, dev, pubs, opt, repr=repr) == want, f"repr {repr}"
        assert down_sha(dev) == before, "the library wrote to the caller's buffer"


@pytest.mark.parametrize("world", [2, 4])
def test_raw_words_in_sharded_proofs(ctx, csg, world):
    # LocalGroup: every rank interpolates its own column block straight from the caller's words
    for logn in (12, 19):
        trace, lifted, pub = lifted_case(logn, seed=world)
        opt = csg.ProofOptions(blowup_factor=4)
        want = ctx.prove(csg.AIR_RESCUE, trace, pub, opt)
        with csg.LocalGroup(world) as grp:
            assert grp.prove(csg.AIR_RESCUE, lifted, pub, opt) == [want] * world, f"2^{logn}"


def same_report(a, b):
    return (a.failed_steps, a.failed_cells, a.transition, a.boundary) == (b.failed_steps, b.failed_cells, b.transition, b.boundary)


@pytest.mark.parametrize("air", AIRS)
def test_raw_words_validate_as_their_residues(ctx, oracle, csg, air):
    # csg_validate_trace / csg_validate_many_device (the validator's own conversion, validate/kernels.cu:25): a lifted witness
    # validates clean in both representations; a lifted corrupted trace gets exactly the report of its reduced form
    air_id = getattr(csg, "AIR_" + air)
    traces, pubs = witnesses(csg, air_id, 2)
    rng = np.random.default_rng(air_id)
    for t, p in zip(traces, pubs):
        assert ctx.validate(air_id, lift(t, rng), p).ok
        assert ctx.validate(air_id, lift(oracle.to_mont_fast(t), rng), p, repr=csg.REPR_MONTGOMERY).ok
    from oracle import pyair
    bad = [t.copy() for t in traces]
    for b, t, p in zip(bad, traces, pubs):
        for _ in range(3):
            col, row = int(rng.integers(b.shape[0])), int(rng.integers(b.shape[1]))
            b[col, row] = int(rng.integers(0, P))
        _, acol, afirst, _, _ = pyair.AIRS[air_id](b.shape[1], [int(v) for v in p]).assertions()[-1]
        b[acol, afirst] = (int(t[acol, afirst]) + R) % P    # an asserted cell: the trace fails whatever else it does
    bad[0][0, 0] = R - 1
    lifted_bad = [lift(b, rng) for b in bad]
    for b, lb, p in zip(bad, lifted_bad, pubs):
        want = ctx.validate(air_id, b, p)
        assert not want.ok
        assert same_report(ctx.validate(air_id, lb, p), want)
    many = ctx.validate_many_device(air_id, up([lift(t, rng) for t in traces]), pubs)
    assert all(r.ok for r in many)
    many = ctx.validate_many_device(air_id, up(lifted_bad), pubs)
    assert all(same_report(r, ctx.validate(air_id, b, p)) for r, b, p in zip(many, bad, pubs))


# ---------------------------------------------------------------------------------------------- B: closed forms
def lde_columns(n, rng):
    """(name, column of evaluations on <w_n>, f(x) of its interpolant) -- the inputs whose butterflies meet the >= boundaries"""
    w = root_of_unity(n.bit_length() - 1)
    pw = np.empty(n, dtype=np.uint64)
    acc = 1
    for i in range(n):
        pw[i] = acc
        acc = acc * w % P
    r = int(rng.integers(n))
    wr = int(pw[r])
    spike = np.zeros(n, dtype=np.uint64)
    spike[r] = P - 1
    ninv, half = pow(n, -1, P), pow(2, -1, P)
    alt = np.zeros(n, dtype=np.uint64)
    alt[1::2] = P - 1
    return [("zero", np.zeros(n, dtype=np.uint64), lambda x: 0),
            ("p-1", np.full(n, P - 1, dtype=np.uint64), lambda x: P - 1),
            ("mont(p-1)", np.full(n, MONT_MINUS_ONE, dtype=np.uint64), lambda x: MONT_MINUS_ONE),
            # (p-1) e_r interpolates to -(w^r / n) (x^n - 1) / (x - w^r)
            ("spike", spike, lambda x: (P - 1) * wr * ninv * (pow(x, n, P) - 1) * pow(x - wr, -1, P) % P),
            ("x", pw, lambda x: x),
            ("x^(n-1)", np.ascontiguousarray(pw[(n - np.arange(n)) % n]), lambda x: pow(x, n - 1, P)),
            # 0, p-1, 0, p-1, ... = (x^(n/2) - 1) / 2
            ("0/p-1", alt, lambda x: (pow(x, n // 2, P) - 1) * half % P)]


@pytest.mark.parametrize("blowup", [2, 8, 32])
@pytest.mark.parametrize("logn", [1, 2, 11, 12, 18, 19, 20, 21, 22])
def test_lde_of_edge_columns_is_the_closed_form(ctx, logn, blowup):
    # ctx.lde (intt_columns + coset_ntt_columns) on columns with known interpolants; output j is the interpolant at 3 * w_{nb}^j.
    # Every point up to 2^14 outputs; above, 4096 sampled points and the first and last row of every coset.
    n, rng = 1 << logn, np.random.default_rng(logn * 64 + blowup)
    nb = n * blowup
    cols = lde_columns(n, rng)
    if nb <= 1 << 14:
        js = list(range(nb))
    else:
        js = sorted(set(rng.integers(0, nb, size=4096).tolist()) | set(range(blowup)) | set(range(nb - blowup, nb)))
    gl = root_of_unity(logn + blowup.bit_length() - 1)
    xs = [3 * pow(gl, j, P) % P for j in js]
    per_call = max(1, (1 << 27) // nb)        # at most 2^27 output words per call
    for c0 in range(0, len(cols), per_call):
        group = cols[c0:c0 + per_call]
        got = ctx.lde(np.stack([c for _, c, _ in group]), blowup)
        for (name, _, f), row in zip(group, got):
            sel = row[js]
            want = [f(x) for x in xs]
            bad = [j for j, g, v in zip(js, sel.tolist(), want) if g != v]
            assert not bad, f"{name}: {len(bad)} wrong points, first at {bad[0]}"


def fold_layers(m, rng):
    """(name, evaluations on 3 * <w_m>, {degree: coefficient}) -- zero, constant and sparse layers of degree < m with coefficients p - 1"""
    w = root_of_unity(m.bit_length() - 1)
    pw = np.empty(m, dtype=object)
    acc = 1
    for i in range(m):
        pw[i] = acc
        acc = acc * w % P
    j = np.arange(m, dtype=np.int64)

    def evaluate(poly):
        acc = np.zeros(m, dtype=object)
        for d, c in poly.items():
            acc = acc + (c * pow(3, d, P) % P) * pw[(d * j) % m]
        return np.array([int(v) % P for v in acc], dtype=np.uint64)
    c = int(rng.integers(1, P))
    sparse = {d: P - 1 for d in {0, 1, 2, 3, m - 1, m - 4, int(rng.integers(m))}}
    top = {d: P - 1 for d in {m - 1, m - 2, m // 2 + 1}}
    return pw, [("zero", np.zeros(m, dtype=np.uint64), {}), ("constant", np.full(m, c, dtype=np.uint64), {0: c}),
                ("sparse", evaluate(sparse), sparse), ("top", evaluate(top), top)]


@pytest.mark.parametrize("logm", [3, 10, 16, 21])
def test_fri_fold_of_edge_layers_is_the_closed_form(ctx, logm):
    # folding sum_d c_d x^d by 4 with alpha gives sum_d c_d alpha^(d mod 4) y^(d div 4) at y_i = (3 w_m^i)^4 (every output point)
    m, rng = 1 << logm, np.random.default_rng(logm)
    pw, layers = fold_layers(m, rng)
    i = np.arange(m // 4, dtype=np.int64)
    for alpha in (int(rng.integers(1, P)), P - 1):
        for name, ev, poly in layers:
            got = ctx.fri_fold4(ev, alpha)
            want = np.zeros(m // 4, dtype=object)
            for d, c in poly.items():
                e = d // 4        # y_i^e = 81^e w_m^(4 i e)
                want = want + (c * pow(alpha, d % 4, P) * pow(81, e, P) % P) * pw[(4 * e * i) % m]
            want = np.array([int(v) % P for v in want], dtype=np.uint64)
            bad = np.flatnonzero(got != want)
            assert bad.size == 0, f"{name}, alpha {alpha}: {bad.size} wrong points, first at {bad[0]}"


@pytest.mark.parametrize("hash_fn", [2, 3])
@pytest.mark.parametrize("width", [16, 34, 51, 64, 127])
def test_row_hashes_of_edge_rows(ctx, hash_fn, width):
    # rows of 0, p - 1 and mont(p - 1) words at multiples of the SHA3 rate (17 words) and the Blake3 block (8 words) and one word
    # short of the Blake3 chunk (128 words), against hashlib / blake3 of the canonical little-endian words
    vals = [0, P - 1, MONT_MINUS_ONE]
    cols = np.array([vals] * width, dtype=np.uint64)
    got = ctx.hash_rows(cols, hash_fn)
    for r, v in enumerate(vals):
        data = np.full(width, v, dtype="<u8").tobytes()
        want = blake3.blake3(data).digest() if hash_fn == 2 else hashlib.sha3_256(data).digest()
        assert got[r].tobytes() == want, f"row of {v:#x}"


# ---------------------------------------------------------------------------------------------- C: witnesses of every AIR
@pytest.fixture(scope="module")
def split_ctx(csg):
    """a context that takes the low-degree split at every size (CSG_SPLIT_MIN_ROWS=0 is read when a context is created)"""
    old = os.environ.get("CSG_SPLIT_MIN_ROWS")
    os.environ["CSG_SPLIT_MIN_ROWS"] = "0"
    try:
        c = csg.Context(0)
    finally:
        if old is None:
            del os.environ["CSG_SPLIT_MIN_ROWS"]
        else:
            os.environ["CSG_SPLIT_MIN_ROWS"] = old
    yield c
    c.close()


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("ext", [1, 2, 3])
@pytest.mark.parametrize("air", AIRS)
def test_stage_buffers_of_witnesses_stay_canonical(ctx, split_ctx, csg, air, ext, split):
    # csg_extend_and_commit_trace, csg_eval_constraints (direct, or the low-degree split) and csg_commit_composition leave no
    # word >= p in the buffers they produce
    air_id = getattr(csg, "AIR_" + air)
    (trace,), pubs = witnesses(csg, air_id, 1)
    opt = csg.ProofOptions(blowup_factor=4 if air_id == csg.AIR_RESCUE else 8, field_extension=ext)
    stage_calls(split_ctx if split else ctx, csg, air_id, trace, pubs[0], opt, seed=ext)


# ---------------------------------------------------------------------------------------------- D: the A/B routes
def workload(csg, ctx, name):
    """sha256 of each proof of a fixed workload; run in this process with the default routes, and in a child with a knob set"""
    if name == "ntt":      # pass A in ntt1024_kernel<STAGE_IN> at 2^19 / 2^20, pass B in ntt1024_kernel<!STAGE_IN> at 2^20 / 2^21
        proofs = [ctx.prove(csg.AIR_RESCUE, lifted, pub, csg.ProofOptions(blowup_factor=4)) for _, lifted, pub in map(lifted_case, (19, 20, 21))]
        trace, pub = csg.TransactionBatch(seed=1000, num_tx=1024).transaction_trace()
        return digest(proofs + [ctx.prove(csg.AIR_TRANSACTION, trace, pub, csg.ProofOptions())])
    if name == "split":    # 2^14 rows: the first size that takes the low-degree split by default
        cases = [(csg.AIR_TRANSACTION, csg.TransactionBatch(seed=1, num_tx=16).transaction_trace()),
                 (csg.AIR_SCHNORR, csg.SignatureBatch(seed=5, num_sig=32).schnorr_trace())]
        return digest([ctx.prove(air, t, p, csg.ProofOptions(field_extension=ext)) for air, (t, p) in cases for ext in (1, 3)])
    if name == "h2d":      # pinned and pageable 2^20 x 94 traces, copied in the chunks of the schedule
        trace, pub = csg.TransactionBatch(seed=1000, num_tx=1024).transaction_trace()
        hb = csg.HostBuffer(94, trace.shape[1])
        try:
            hb.array[:] = trace
            ctx.set_air(csg.AIR_TRANSACTION, trace.shape[1], pub, csg.ProofOptions())
            pinned = ctx.prove_trace_ptr(hb.ptr)
        finally:
            hb.close()
        return digest([pinned, ctx.prove(csg.AIR_TRANSACTION, trace, pub, csg.ProofOptions())])
    if name == "sharded":  # the coefficient exchange of a sharded proof
        trace, pub = csg.TransactionBatch(seed=1, num_tx=16).transaction_trace()
        _, lifted, rpub = lifted_case(12)
        out = []
        for world in (2, 4):
            with csg.LocalGroup(world) as grp:
                out += grp.prove(csg.AIR_TRANSACTION, trace, pub, csg.ProofOptions())
                out += grp.prove(csg.AIR_RESCUE, lifted, rpub, csg.ProofOptions(blowup_factor=4))
        return digest(out)
    raise ValueError(name)


def child_main(name):
    import certificate_stark_b200 as csg
    with csg.Context(0) as c:
        print(json.dumps(workload(csg, c, name)))


_DEFAULT = {}


@pytest.mark.parametrize("name,env", [("ntt", {"CSG_NTT_GENERIC": "1"}),
                                      ("ntt", {"CSG_NTT_SHAPE_A": "4", "CSG_NTT_SHAPE_B": "5"}),
                                      ("ntt", {"CSG_NTT_SHAPE_A": "5", "CSG_NTT_SHAPE_B": "4"}),
                                      ("split", {"CSG_NO_ECC_SPLIT": "1"}),
                                      ("h2d", {"CSG_H2D_CHUNKS": "5,2,7"}),
                                      ("sharded", {"CSG_COEF_BLOCKWISE": "1"})],
                         ids=["generic", "shapeA4-B5", "shapeA5-B4", "no-ecc-split", "h2d-chunks", "coef-blockwise"])
def test_ab_route_gives_the_default_bytes(ctx, csg, name, env):
    # knobs read once per process (static const in ntt.cu, constraints_kernels.cuh, prover_ctx.cuh): a child process per knob
    if name not in _DEFAULT:
        _DEFAULT[name] = workload(csg, ctx, name)
    child_env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    child_env.update(env)
    code = f"import sys; sys.path[:0] = [{str(HERE.parent)!r}, {str(HERE)!r}]; import test_gpu_edge_values as t; t.child_main({name!r})"
    out = subprocess.run([sys.executable, "-c", code], env=child_env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    got = json.loads([line for line in out.stdout.splitlines() if line.startswith("[")][-1])
    assert got == _DEFAULT[name]


def test_no_split_gives_the_default_bytes(ctx, csg, monkeypatch):
    # CSG_NO_SPLIT is read when a context is created (prover_ctx.cuh:224): every constraint on every coset at 2^14 rows
    want = workload(csg, ctx, "split")
    monkeypatch.setenv("CSG_NO_SPLIT", "1")
    with csg.Context(0) as c:
        assert workload(csg, c, "split") == want
