"""csg_prove_many_device and the batch witness builders (-m gpu): a batch whose traces are already in device memory must give the
proofs csg_prove_many gives for the same traces, without writing the buffer; the builders must write, trace for trace, what the
host builders write, and the public inputs each proof verifies with."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from test_gpu_prove_many import AIRS, oracle_options, witnesses

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
P = 0x4180000000000001


def up(traces):
    """host traces -> one contiguous int64 CUDA tensor (K, w, n)"""
    return torch.from_numpy(np.stack(traces).view(np.int64)).to("cuda:0")


def down(t):
    return t.cpu().view(torch.int64).numpy().view(np.uint64)


def sha(t):
    torch.cuda.synchronize()
    return hashlib.sha256(down(t).tobytes()).hexdigest()


def opt_for(csg, air_id):
    return csg.ProofOptions(blowup_factor=4 if air_id == csg.AIR_RESCUE else 8)


# ---------------------------------------------------------------------------------------------- prove_many_device
@pytest.mark.parametrize("repr", [0, 1])
@pytest.mark.parametrize("count", [1, 3, 16])
@pytest.mark.parametrize("air", AIRS)
def test_matches_prove_many(ctx, oracle, csg, air, count, repr):
    air_id = getattr(csg, "AIR_" + air)
    traces, pubs = witnesses(csg, air_id, count)
    if repr == csg.REPR_MONTGOMERY:
        traces = [oracle.to_mont_fast(t) for t in traces]
    opt = opt_for(csg, air_id)
    dev = up(traces)
    before = sha(dev)
    got = ctx.prove_many_device(air_id, dev, pubs, opt, repr=repr)
    assert got == ctx.prove_many(air_id, traces, pubs, opt, repr=repr)
    assert sha(dev) == before, "the library wrote to the caller's buffer"


def test_longest_trace(ctx, csg):
    traces, pubs = zip(*[csg.build_rescue_trace(np.arange(s, s + 7, dtype=np.uint64), 8192) for s in (3, 4)])   # 2^16 rows
    opt = csg.ProofOptions(blowup_factor=4)
    dev = up(traces)
    before = sha(dev)
    got = ctx.prove_many_device(csg.AIR_RESCUE, dev, np.stack(pubs), opt)
    assert got == ctx.prove_many(csg.AIR_RESCUE, list(traces), np.stack(pubs), opt)
    assert sha(dev) == before


# ---------------------------------------------------------------------------------------------- Rescue builder
def rescue_seeds(count, seed):
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 2**64, size=(count, 7), dtype=np.uint64)
    s[0, :3] = [P, P + 5, 2**64 - 1]   # seeds at and above p are reduced
    return s


@pytest.mark.parametrize("chain,count", [(1, 1), (1, 5), (128, 1), (128, 5), (128, 256), (8192, 1), (8192, 5)])
def test_rescue_builder_matches_host(ctx, oracle, csg, chain, count):
    seeds = rescue_seeds(count, chain + count)
    dev, pubs = ctx.build_many_rescue(seeds, chain)
    assert dev.shape == (count, 14, 8 * chain) and dev.dtype == torch.uint64
    got = down(dev)
    host = [csg.build_rescue_trace(s, chain) for s in seeds]
    for k, (t, p) in enumerate(host):
        assert np.array_equal(got[k], t), f"trace {k} differs from csg_build_trace_rescue"
        assert np.array_equal(pubs[k], p), f"public inputs {k} differ"
    if chain == 1:
        return
    opt = csg.ProofOptions(blowup_factor=4)
    proofs = ctx.prove_many_device(csg.AIR_RESCUE, dev, pubs, opt)
    assert proofs == ctx.prove_many(csg.AIR_RESCUE, [t for t, _ in host], pubs, opt)
    if chain == 128 and count == 5:
        for k in (0, 2, 4):
            assert proofs[k] == oracle.prove(csg.AIR_RESCUE, host[k][0], pubs[k], oracle_options(oracle, opt))


# ---------------------------------------------------------------------------------------------- signature / transfer builders
ITEMS = {   # air: (batch, device builder, host builder, rows)
    "SCHNORR": (lambda csg, s, k: csg.SignatureBatch(seed=s, num_sig=k), "build_many_schnorr", "schnorr_trace", 512),
    "MERKLE_UPDATE": (lambda csg, s, k: csg.TransactionBatch(seed=s, num_tx=k), "build_many_merkle_update", "merkle_update_trace", 512),
    "TRANSACTION": (lambda csg, s, k: csg.TransactionBatch(seed=s, num_tx=k), "build_many_transaction", "transaction_trace", 1024),
}


def tamper(pub, i):
    bad = pub.copy()
    bad[i] = (int(bad[i]) + 1) % P
    return bad


@pytest.mark.parametrize("count", [1, 4])
@pytest.mark.parametrize("air", list(ITEMS))
def test_item_builders(ctx, oracle, csg, air, count):
    air_id = getattr(csg, "AIR_" + air)
    make, dev_build, host_build, R = ITEMS[air]
    batch = make(csg, 31 + count, count)
    dev, pubs = getattr(ctx, dev_build)(batch)
    host, host_pub = getattr(batch, host_build)()
    got = down(dev)
    assert got.shape == (count, csg.TRACE_WIDTH[air_id], R)
    for k in range(count):
        want = host[:, k * R:(k + 1) * R].copy()
        if air == "MERKLE_UPDATE":
            want[14, 1] = want[43, 1] = 1   # set in every proof, as MerkleProver::build_trace sets them in a single one
        assert np.array_equal(got[k], want), f"trace {k} is not columns [{k * R}, {(k + 1) * R}) of the host trace"
    if count == 1:
        assert np.array_equal(got[0], host) and np.array_equal(pubs[0], host_pub)
    if air == "SCHNORR":
        assert np.array_equal(pubs.reshape(-1), host_pub)
    else:   # a chain of roots from the batch's initial root to its final one
        assert np.array_equal(pubs[0, :7], host_pub[:7]) and np.array_equal(pubs[-1, 7:], host_pub[7:])
        for k in range(count - 1):
            assert np.array_equal(pubs[k, 7:], pubs[k + 1, :7])
    opt = csg.ProofOptions()
    proofs = ctx.prove_many_device(air_id, dev, pubs, opt)
    assert proofs == ctx.prove_many(air_id, list(got), pubs, opt)
    changed = 0 if air == "SCHNORR" else 7   # a message word; the root after the transfer
    for k, proof in enumerate(proofs):
        assert csg.verify(air_id, pubs[k], proof) == 0 and oracle.verify(air_id, pubs[k], proof) == 0
        assert csg.verify(air_id, tamper(pubs[k], changed), proof) != 0
        assert oracle.verify(air_id, tamper(pubs[k], changed), proof) != 0
        assert csg.verify(air_id, tamper(pubs[k], 3), proof) != 0   # the root before / a message word
    if count == 4:
        assert proofs[1] == oracle.prove(air_id, got[1], pubs[1], oracle_options(oracle, opt))


# ---------------------------------------------------------------------------------------------- launches
@pytest.mark.parametrize("air", ["RESCUE", "SCHNORR", "MERKLE_UPDATE", "TRANSACTION"])
def test_launches_do_not_grow_with_the_batch(ctx, csg, air):
    air_id = getattr(csg, "AIR_" + air)
    counts = []
    for count in (1, 16):
        if air == "RESCUE":
            dev, pubs = ctx.build_many_rescue(rescue_seeds(count, 3), 128)
        else:
            make, dev_build, _, _ = ITEMS[air]
            dev, pubs = getattr(ctx, dev_build)(make(csg, 5, count))
        build = ctx.timings()["kernel_launches"]
        ctx.prove_many_device(air_id, dev, pubs, opt_for(csg, air_id))
        counts.append((build, ctx.timings()["kernel_launches"]))
    assert counts[0] == counts[1] and counts[0][0] > 0


# ---------------------------------------------------------------------------------------------- rejections
def test_rejections_leave_the_context_usable(ctx, csg):
    lib = csg.lib()
    traces, pubs = witnesses(csg, csg.AIR_RANGE, 2, seed=21)
    opt = csg.ProofOptions()
    dev = up(traces)
    u64p = C.POINTER(C.c_uint64)
    pp = pubs.ctypes.data_as(u64p)
    outs, lens = (C.POINTER(C.c_uint8) * 1025)(), (C.c_size_t * 1025)()

    def abi(ptr, count=2, o=opt, air=csg.AIR_RANGE, n=64, npub=1, p=pp):
        return lib.csg_prove_many_device(ctx._h, air, count, ptr, 0, n, p, npub, C.byref(o), outs, lens)

    host = np.stack(traces)
    pinned = torch.from_numpy(host.view(np.int64)).pin_memory()
    assert abi(host.ctypes.data) == 1, "a numpy buffer"
    assert abi(pinned.data_ptr()) == 1, "a pinned host buffer"
    assert abi(None) == 1
    assert abi(dev.data_ptr(), count=0) == 1
    assert abi(dev.data_ptr(), count=1025, p=np.zeros(1025, dtype=np.uint64).ctypes.data_as(u64p)) == 1
    assert abi(dev.data_ptr(), o=csg.ProofOptions(field_extension=2)) == 4
    assert abi(dev.data_ptr(), o=csg.ProofOptions(field_extension=3)) == 4
    assert not any(outs[i] for i in range(1025))
    wide = torch.zeros((698, 94, 1024), dtype=torch.int64, device="cuda:0")   # 65612 columns
    with pytest.raises(csg.CsgError, match="^invalid argument.*65535"):
        ctx.prove_many_device(csg.AIR_TRANSACTION, wide, np.zeros((698, 14), dtype=np.uint64), opt)
    del wide
    for bad in (host, pinned, dev.float()):
        with pytest.raises(csg.CsgError):
            ctx.prove_many_device(csg.AIR_RANGE, bad, pubs, opt)
    with csg.LocalGroup(2) as g:
        with pytest.raises(csg.CsgError, match="^unsupported"):
            g.ctxs[0].prove_many_device(csg.AIR_RANGE, dev, pubs, opt)
    if torch.cuda.device_count() > 1:
        with pytest.raises(csg.CsgError, match="^invalid argument.*device memory"):
            ctx.prove_many_device(csg.AIR_RANGE, dev.to("cuda:1"), pubs, opt)

    # the builders
    seeds = rescue_seeds(2, 1)
    out = torch.empty((2, 14, 8 * 128), dtype=torch.uint64, device="cuda:0")
    pub_out = np.zeros((2, 14), dtype=np.uint64)
    sp, pb = seeds.ctypes.data_as(u64p), pub_out.ctypes.data_as(u64p)
    rescue = lib.csg_build_traces_many_rescue
    assert rescue(ctx._h, sp, 2, 128, out.data_ptr(), pb) == 0
    for chain in (0, 3, 96, 16384):
        assert rescue(ctx._h, sp, 2, chain, out.data_ptr(), pb) == 1
    assert rescue(ctx._h, None, 2, 128, out.data_ptr(), pb) == 1
    assert rescue(ctx._h, sp, 2, 128, None, pb) == 1
    assert rescue(ctx._h, sp, 2, 128, out.data_ptr(), None) == 1
    assert rescue(ctx._h, sp, 0, 128, out.data_ptr(), pb) == 1
    assert rescue(ctx._h, sp, 1025, 128, out.data_ptr(), pb) == 1
    assert rescue(ctx._h, sp, 2, 128, host.ctypes.data, pb) == 1
    assert rescue(ctx._h, sp, 2, 128, pinned.data_ptr(), pb) == 1
    with pytest.raises(csg.CsgError, match="^invalid argument"):
        ctx.build_many_rescue(seeds, 6)
    sigs, tx = csg.SignatureBatch(seed=1, num_sig=2), csg.TransactionBatch(seed=1, num_tx=2)
    for fn in (lib.csg_build_traces_many_schnorr, lib.csg_build_traces_many_merkle_update, lib.csg_build_traces_many_transaction):
        assert fn(ctx._h, None, out.data_ptr(), pb) == 1
    assert lib.csg_build_traces_many_schnorr(ctx._h, sigs._h, host.ctypes.data, pb) == 1
    assert lib.csg_build_traces_many_transaction(ctx._h, tx._h, pinned.data_ptr(), pb) == 1
    with pytest.raises(csg.CsgError, match="^invalid argument.*depth 15"):
        ctx.build_many_transaction(csg.TransactionBatch(seed=1, num_tx=2, tree_depth=7))
    with pytest.raises(csg.CsgError, match="^invalid argument.*1..1024"):
        ctx.build_many_schnorr(csg.SignatureBatch(seed=1, num_sig=1025))

    assert ctx.prove_many_device(csg.AIR_RANGE, dev, pubs, opt) == ctx.prove_many(csg.AIR_RANGE, traces, pubs, opt)


# ---------------------------------------------------------------------------------------------- isolation
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
    dev, rp = ctx.build_many_rescue(rescue_seeds(3, 19), 16)
    ctx.prove_many_device(csg.AIR_RESCUE, dev, rp, opt)
    for build in ("build_many_schnorr", "build_many_merkle_update", "build_many_transaction"):
        batch = csg.SignatureBatch(seed=3, num_sig=2) if build == "build_many_schnorr" else csg.TransactionBatch(seed=3, num_tx=2)
        getattr(ctx, build)(batch)
    assert ctx.prove_loaded() == want_loaded
    assert ctx.prove_prefetched_ptr() == want_prefetched
