"""Level-2 C ABI (include/csg.h): the per-stage calls a patched winterfell `generate_proof` would make, driven here by a
transcript that lives OUTSIDE the library (a Python RandomCoin + proof writer).  The proof assembled this way must be the
very bytes csg_prove() returns, and the product verifier must accept it."""
import ctypes as C
import struct

import blake3
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
P = 0x4180000000000001


class Coin:   # winterfell RandomCoin over Blake3_256, as the library's built-in transcript implements it
    def __init__(self, seed_bytes):
        self.seed, self.counter = blake3.blake3(seed_bytes).digest(), 0

    def reseed(self, digest):
        self.seed, self.counter = blake3.blake3(self.seed + bytes(digest)).digest(), 0

    def reseed_int(self, v):
        self.seed, self.counter = blake3.blake3(self.seed + struct.pack("<Q", v)).digest(), 0

    def next_u64(self):
        self.counter += 1
        return struct.unpack("<Q", blake3.blake3(self.seed + struct.pack("<Q", self.counter)).digest()[:8])[0]

    def draw(self):
        while True:
            v = self.next_u64()
            if v < P:
                return v

    def draw_x(self, d):
        """an element of the degree-d extension: the first 8*d bytes of one output, all d words canonical (coin.draw::<E>())"""
        while True:
            self.counter += 1
            out = blake3.blake3(self.seed + struct.pack("<Q", self.counter)).digest()
            words = struct.unpack(f"<{d}Q", out[:8 * d])
            if all(v < P for v in words):
                return list(words)

    def draw_integers(self, count, domain):
        out = []
        while len(out) < count:
            v = self.next_u64() & (domain - 1)
            if v not in out:
                out.append(v)
        return out


def hash_elements(vals):
    return blake3.blake3(b"".join(struct.pack("<Q", int(v)) for v in vals)).digest()


@pytest.mark.parametrize("ext", [1, 2, 3])
@pytest.mark.parametrize("kind", ["rescue", "transaction"])
def test_stage_calls_with_external_transcript_reproduce_csg_prove(ctx, csg, kind, ext):
    if kind == "rescue":
        trace, pub = csg.build_rescue_trace(np.arange(42, 49, dtype=np.uint64), 64)
        stage_calls_reproduce_csg_prove(ctx, csg, csg.AIR_RESCUE, trace, pub, 4, ext, ncons=14, nassert=14, ce=4)
    else:
        trace, pub = csg.TransactionBatch(seed=6, num_tx=1).transaction_trace()
        stage_calls_reproduce_csg_prove(ctx, csg, csg.AIR_TRANSACTION, trace, pub, 8, ext, ncons=115, nassert=4, ce=8)


@pytest.mark.parametrize("num_tx,ext", [(16, 1), (16, 3), (2048, 1)])
def test_transaction_stage_calls_at_size_reproduce_csg_prove(ctx, csg, num_tx, ext):
    # 16 transactions (2^14 rows): csg_eval_constraints takes the low-degree split, with E-valued coefficients at ext 3;
    # 2048 transactions (2^21 rows): the 1024-point NTT passes.  test_gpu_headline.py pins csg_prove at this shape to the oracle.
    trace, pub = csg.TransactionBatch(seed=6, num_tx=num_tx).transaction_trace()
    stage_calls_reproduce_csg_prove(ctx, csg, csg.AIR_TRANSACTION, trace, pub, 8, ext, ncons=115, nassert=4, ce=8)


def stage_calls_reproduce_csg_prove(ctx, csg, air, trace, pub, blowup, ext, ncons, nassert, ce):
    L = csg.lib()
    opt = csg.ProofOptions(blowup_factor=blowup, field_extension=ext)
    want = ctx.prove(air, trace, pub, opt)
    flat = lambda elems: [w_ for e in elems for w_ in e]      # an element of E crosses the ABI as its `ext` words in order

    w, n = trace.shape
    lde_n, nq = n * blowup, opt.num_queries
    logn = n.bit_length() - 1
    context = struct.pack("<BBHBQ7B", w, logn, 0, 8, P, nq, blowup.bit_length() - 1, 0, 2, ext, 2, 8)
    coin = Coin(b"".join(struct.pack("<Q", int(v)) for v in pub) + context)
    h, p64, p8 = ctx._h, csg._p64, csg._p8
    u64 = lambda xs: np.array(xs, dtype=np.uint64)

    ctx.set_air(air, n, pub, opt)
    ctx.load_trace(trace)
    root = np.zeros(32, dtype=np.uint8)
    ctx._check(L.csg_extend_and_commit_trace(h, p8(root)))
    trace_root = root.tobytes()
    coin.reseed(trace_root)
    t_coeffs = u64(flat(coin.draw_x(ext) for _ in range(2 * ncons)))
    b_coeffs = u64(flat(coin.draw_x(ext) for _ in range(2 * nassert)))
    ctx._check(L.csg_eval_constraints(h, p64(t_coeffs), p64(b_coeffs)))
    ctx._check(L.csg_commit_composition(h, p8(root)))
    comp_root = root.tobytes()
    coin.reseed(comp_root)
    z = coin.draw_x(ext)
    cur, nxt, comp = np.zeros(w * ext, dtype=np.uint64), np.zeros(w * ext, dtype=np.uint64), np.zeros(ce * ext, dtype=np.uint64)
    if ext == 1:
        ctx._check(L.csg_ood(h, z[0], p64(cur), p64(nxt), p64(comp)))
    else:
        assert L.csg_ood(h, z[0], p64(cur), p64(nxt), p64(comp)) != 0       # the by-value form is for the base field
        ctx._check(L.csg_ood_ext(h, p64(u64(z)), p64(cur), p64(nxt), p64(comp)))
    for frame in (cur, nxt, comp):
        coin.reseed(hash_elements(frame))
    ab = []
    for _ in range(w):
        ab += coin.draw_x(ext) + coin.draw_x(ext)
        coin.draw_x(ext)
    deltas = u64(flat(coin.draw_x(ext) for _ in range(ce)))
    lam_mu = u64(coin.draw_x(ext) + coin.draw_x(ext))
    ctx._check(L.csg_deep(h, p64(u64(ab)), p64(deltas), p64(lam_mu)))
    nlayers, d = 1, lde_n
    while d > opt.fri_max_remainder_size:
        d //= 4
        nlayers += 1
    fri_roots = []
    for layer in range(nlayers):
        ctx._check(L.csg_fri_commit_layer(h, p8(root)))
        fri_roots.append(root.tobytes())
        coin.reseed(fri_roots[-1])
        alpha = coin.draw_x(ext)
        if layer + 1 < nlayers:
            if ext == 1:
                ctx._check(L.csg_fri_fold(h, alpha[0]))
            else:
                ctx._check(L.csg_fri_fold_ext(h, p64(u64(alpha))))
    nonce = 1
    coin.reseed_int(nonce)
    pos = coin.draw_integers(nq, lde_n)

    def opening(fn, positions, width, *extra):
        positions = u64(positions)
        rows, paths, plen = np.zeros(len(positions) * width, dtype=np.uint64), np.zeros(1 << 20, dtype=np.uint8), C.c_size_t()
        ctx._check(fn(h, *extra, p64(positions), len(positions), p64(rows), p8(paths), paths.size, C.byref(plen)))
        return rows.astype("<u8").tobytes(), paths[:plen.value].tobytes()

    out = bytearray(context)
    out += struct.pack("<H", (2 + nlayers) * 32) + trace_root + comp_root + b"".join(fri_roots)
    for fn, width in ((L.csg_open_trace, w), (L.csg_open_composition, ce * ext)):
        rows, paths = opening(fn, pos, width)
        out += struct.pack("<I", len(rows)) + rows + struct.pack("<I", len(paths)) + paths
    out += struct.pack("<H", w * ext * 8) + cur.astype("<u8").tobytes() + nxt.astype("<u8").tobytes()
    out += struct.pack("<H", ce * ext * 8) + comp.astype("<u8").tobytes()
    out += struct.pack("<B", nlayers - 1)
    fp, domain = pos, lde_n
    for layer in range(nlayers - 1):
        folded = []
        for p in fp:
            if p % (domain // 4) not in folded:
                folded.append(p % (domain // 4))
        fp = folded
        rows, paths = opening(L.csg_open_fri_layer, fp, 4 * ext, layer)
        out += struct.pack("<I", len(rows)) + rows + struct.pack("<I", len(paths)) + paths
        domain //= 4
    rem, rlen = np.zeros(opt.fri_max_remainder_size * ext, dtype=np.uint64), C.c_size_t()
    ctx._check(L.csg_fri_remainder(h, p64(rem), rem.size, C.byref(rlen)))
    out += struct.pack("<H", rlen.value * 8) + rem[:rlen.value].astype("<u8").tobytes() + b"\x01" + struct.pack("<Q", nonce)
    assert bytes(out) == want
    assert csg.verify(air, pub, bytes(out)) == 0


def test_stage_calls_out_of_order_are_refused(csg):
    with csg.Context(0) as c:
        L, root = csg.lib(), np.zeros(32, dtype=np.uint8)
        assert L.csg_extend_and_commit_trace(c._h, csg._p8(root)) == 3          # CSG_ERR_STATE: no AIR, no trace
        trace, pub = csg.build_range_trace(9)
        c.set_air(csg.AIR_RANGE, 64, pub, csg.ProofOptions())
        assert L.csg_commit_composition(c._h, csg._p8(root)) == 3
        assert b"first" in L.csg_last_error(c._h)
