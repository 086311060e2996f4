"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Second, independent restatement of the AIR side of the reference, in plain Python
big-integer arithmetic on CANONICAL field elements (no Montgomery form, no shared code or generated tables with oracle/*.c
or with the product).

What it restates, each from the reference file it cites (paths relative to /root/reference):
  * Rescue-XLIX round / permutation / digest / merge        src/utils/rescue.rs:96-130, 143-152, 237-263, 327-375
  * enforce_round                                           src/utils/rescue.rs:269-300
  * Fp2 / Fp6 arithmetic, complete projective group law     src/utils/ecc.rs:186-404 (formulas), 407-548 (tower)
  * enforce_point_doubling / _addition_mixed / _reduce_x    src/utils/ecc.rs:73-172
  * the six `impl Air`: evaluate_transition, degrees, periodic columns, assertions
        TransactionAir   src/air.rs:76-189, 194-380, 383-610          MerkleAir     src/merkle/update/air.rs:36-401
        PreMerkleAir     src/merkle/init/air.rs:40-211                 SchnorrAir    src/schnorr/air.rs:41-585
        RangeProofAir    src/range/air.rs:36-105                       RescueAir     benches/rescue.rs:136-268
  * witnesses (build_trace of each prover)                  src/prover.rs:37-98, src/trace.rs:28-142, src/merkle/update/trace.rs,
        src/schnorr/trace.rs, src/range/prover.rs:36-84, benches/rescue.rs:279-321, SURVEY.md Appendix G
  * the batch metadata of TransactionMetadata::build_random src/lib.rs:235-464 (own PRNG; keys by the SURVEY.md 8(d) recipe)

Constants (MDS, INV_MDS, ARK, GENERATOR, B3) come from this module's OWN parse of src/utils/rescue.rs:385-996 and
src/utils/ecc.rs:23-45 (`parse_reference_constants`), not from tools/gen_constants.py.  tests/golden/make_air_vectors.py
stores the parse in tests/golden/air_constants.json, and the module reads it from there: it runs without the reference
sources.  Only tests/ and tests/golden/make_air_vectors.py import this file.
"""
import json
import re
from pathlib import Path

P = 0x4180000000000001            # src/range/tests.rs:59
R_MONT = (1 << 64) % P            # BaseElement::from_raw_unchecked values are Montgomery words (R = 2^64)
INV_ALPHA = 3146514939656186539   # src/utils/rescue.rs:383
HERE = Path(__file__).resolve().parent
CONSTANTS_JSON = HERE.parent / "tests" / "golden" / "air_constants.json"

STATE, RATE, ROUNDS, CYCLE = 14, 7, 7, 8     # src/utils/rescue.rs:25-37
COORD, AFFINE, PROJ = 6, 12, 18              # src/utils/ecc.rs:16-20


# ---------------------------------------------------------------------------------------------- constants
def _numbers(block):
    return [int(m, 0) for m in re.findall(r"BaseElement::(?:new|from_raw_unchecked)\((0x[0-9a-fA-F]+|\d+)\)", block)]


def _const_block(text, name):
    m = re.search(r"const %s\b[^=]*=\s*\[" % name, text)
    depth, i = 1, m.end()
    while depth:
        depth += {"[": 1, "]": -1}.get(text[i], 0)
        i += 1
    return text[m.end():i - 1]


def parse_reference_constants(root):
    """the constant tables of a checkout of the reference at `root`"""
    rescue = (root / "src/utils/rescue.rs").read_text()
    ecc = (root / "src/utils/ecc.rs").read_text()
    mds, inv_mds = _numbers(_const_block(rescue, "MDS")), _numbers(_const_block(rescue, "INV_MDS"))
    ark_block = _const_block(rescue, "ARK")
    ark = _numbers(ark_block)
    assert len(mds) == 196 and len(inv_mds) == 196 and len(ark) == 7 * 28 and "[BaseElement::ZERO; STATE_WIDTH * 2]" in ark_block
    ark += [0] * 28                                               # the eighth row: src/utils/rescue.rs:995
    gen_raw, b3 = _numbers(_const_block(ecc, "GENERATOR")), _numbers(_const_block(ecc, "B3"))
    assert len(gen_raw) == 12 and len(b3) == 6
    rinv = pow(R_MONT, -1, P)
    return {"MDS": mds, "INV_MDS": inv_mds, "ARK": ark, "GENERATOR": [g * rinv % P for g in gen_raw], "B3": b3}


_K = json.loads(CONSTANTS_JSON.read_text())
MDS = [_K["MDS"][i * 14:(i + 1) * 14] for i in range(14)]
INV_MDS = [_K["INV_MDS"][i * 14:(i + 1) * 14] for i in range(14)]
ARK = [_K["ARK"][i * 28:(i + 1) * 28] for i in range(8)]
GENERATOR, B3 = _K["GENERATOR"], _K["B3"]


class View:
    """a slice of a list that writes through: &mut result[a..b] of the reference"""

    def __init__(self, base, off=0):
        self.base, self.off = base, off

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self.base[self.off + k] for k in range(i.start or 0, i.stop)]
        return self.base[self.off + i]

    def __setitem__(self, i, v):
        self.base[self.off + i] = v

    def sub(self, a):
        return View(self.base, self.off + a)


def agg(result, index, flag, value):      # src/utils/mod.rs:58-62
    result[index] = (result[index] + flag * value) % P


def are_equal(a, b):
    return (a - b) % P


def is_binary(a):
    return (a * a - a) % P


def not_(a):
    return (1 - a) % P


# ---------------------------------------------------------------------------------------------- Rescue
def apply_round(state, step):             # src/utils/rescue.rs:246-263
    ark = ARK[step % CYCLE]
    s = [pow(x, 3, P) for x in state]
    s = [(sum(MDS[i][j] * s[j] for j in range(14)) + ark[i]) % P for i in range(14)]
    s = [pow(x, INV_ALPHA, P) for x in s]
    return [(sum(MDS[i][j] * s[j] for j in range(14)) + ark[14 + i]) % P for i in range(14)]


def apply_permutation(state):
    for i in range(ROUNDS):
        state = apply_round(state, i)
    return state


def merge(a, b):                          # src/utils/rescue.rs:143-152
    return apply_permutation(list(a) + list(b))[:7]


def digest(data):                         # src/utils/rescue.rs:108-130 (no padding)
    state, i = [0] * 14, 0
    for e in data:
        state[i] = (state[i] + e) % P
        i += 1
        if i % RATE == 0:
            state, i = apply_permutation(state), 0
    if i > 0:
        state = apply_permutation(state)
    return state[:7]


def enforce_round(result, current, nxt, ark, flag):   # src/utils/rescue.rs:269-300
    s1 = [pow(current[i], 3, P) for i in range(14)]
    s1 = [(sum(MDS[i][j] * s1[j] for j in range(14)) + ark[i]) % P for i in range(14)]
    s2 = [(nxt[i] - ark[14 + i]) % P for i in range(14)]
    s2 = [sum(INV_MDS[i][j] * s2[j] for j in range(14)) % P for i in range(14)]
    s2 = [pow(x, 3, P) for x in s2]
    for i in range(14):
        agg(result, i, flag, are_equal(s2[i], s1[i]))


# ---------------------------------------------------------------------------------------------- Fp6 = Fp[u]/(u^2-2u-2)[v]/(v^3+v+1)
# src/utils/ecc.rs:424-439 gives (a0 + a1 u)(b0 + b1 u) = a0 b0 + 2 a1 b1 + (a0 b1 + a1 b0 + 2 a1 b1) u, i.e. u^2 = 2u + 2; :506-548 gives
# v^3 = -v - 1.  Products here are schoolbook polynomial products reduced by those relations, not the reference's Karatsuba steps.
def f2mul(a, b):
    t = a[1] * b[1]
    return [(a[0] * b[0] + 2 * t) % P, (a[0] * b[1] + a[1] * b[0] + 2 * t) % P]


def f2add(a, b):
    return [(a[0] + b[0]) % P, (a[1] + b[1]) % P]


def f2sub(a, b):
    return [(a[0] - b[0]) % P, (a[1] - b[1]) % P]


def f6mul(a, b):
    A, B = [a[0:2], a[2:4], a[4:6]], [b[0:2], b[2:4], b[4:6]]
    c = [[0, 0] for _ in range(5)]
    for i in range(3):
        for j in range(3):
            c[i + j] = f2add(c[i + j], f2mul(A[i], B[j]))
    # v^4 = -v^2 - v, v^3 = -v - 1
    c[2] = f2sub(c[2], c[4]); c[1] = f2sub(c[1], c[4])
    c[1] = f2sub(c[1], c[3]); c[0] = f2sub(c[0], c[3])
    return c[0] + c[1] + c[2]


def f6add(a, b):
    return [(x + y) % P for x, y in zip(a, b)]


def f6sub(a, b):
    return [(x - y) % P for x, y in zip(a, b)]


def f6dbl(a):
    return [2 * x % P for x in a]


def f2inv(a):                             # src/utils/ecc.rs:442-446: norm a0^2 + 2 a0 a1 - 2 a1^2
    t = pow((a[0] * a[0] + 2 * a[0] * a[1] - 2 * a[1] * a[1]) % P, P - 2, P)
    return [(a[0] + 2 * a[1]) * t % P, (-a[1]) * t % P]


def f6inv(a):
    """inverse by solving a * x = 1 as a 6 x 6 linear system over Fp (independent of invert_fp6's closed form, ecc.rs:551-591)"""
    cols = []
    for k in range(6):
        e = [0] * 6
        e[k] = 1
        cols.append(f6mul(a, e))
    M = [[cols[c][r] for c in range(6)] + [1 if r == 0 else 0] for r in range(6)]
    for c in range(6):
        piv = next(r for r in range(c, 6) if M[r][c])
        M[c], M[piv] = M[piv], M[c]
        inv = pow(M[c][c], P - 2, P)
        M[c] = [x * inv % P for x in M[c]]
        for r in range(6):
            if r != c and M[r][c]:
                f = M[r][c]
                M[r] = [(x - f * y) % P for x, y in zip(M[r], M[c])]
    return [M[r][6] for r in range(6)]


def compute_double(s):                    # src/utils/ecc.rs:186-240 (RCB15 algorithm 3, a = 1)
    X, Y, Z = s[0:6], s[6:12], s[12:18]
    t0, t1, t2 = f6mul(X, X), f6mul(Y, Y), f6mul(Z, Z)
    t3 = f6dbl(f6mul(X, Y))
    z3 = f6dbl(f6mul(X, Z))
    y3 = f6add(z3, f6mul(B3, t2))
    x3 = f6sub(t1, y3)
    y3 = f6add(t1, y3)
    y3 = f6mul(x3, y3)
    x3 = f6mul(t3, x3)
    z3 = f6mul(B3, z3)
    t3 = f6add(f6sub(t0, t2), z3)
    t0 = f6add(f6add(f6dbl(t0), t0), t2)
    t0 = f6mul(t0, t3)
    y3 = f6add(y3, t0)
    t2 = f6dbl(f6mul(Y, Z))
    x3 = f6sub(x3, f6mul(t2, t3))
    z3 = f6dbl(f6dbl(f6mul(t2, t1)))
    return x3 + y3 + z3


def compute_add(s, q):                    # src/utils/ecc.rs:242-318 (RCB15 algorithm 1, a = 1)
    X1, Y1, Z1, X2, Y2, Z2 = s[0:6], s[6:12], s[12:18], q[0:6], q[6:12], q[12:18]
    t0, t1, t2 = f6mul(X1, X2), f6mul(Y1, Y2), f6mul(Z1, Z2)
    t3 = f6sub(f6mul(f6add(X1, Y1), f6add(X2, Y2)), f6add(t0, t1))
    t4 = f6sub(f6mul(f6add(X1, Z1), f6add(X2, Z2)), f6add(t0, t2))
    t5 = f6sub(f6mul(f6add(Y1, Z1), f6add(Y2, Z2)), f6add(t1, t2))
    z3 = f6add(f6mul(B3, t2), t4)
    x3 = f6sub(t1, z3)
    z3 = f6add(t1, z3)
    y3 = f6mul(x3, z3)
    t1 = f6add(f6add(f6dbl(t0), t0), t2)
    t4 = f6add(f6mul(B3, t4), f6sub(t0, t2))
    y3 = f6add(y3, f6mul(t1, t4))
    x3 = f6sub(f6mul(t3, x3), f6mul(t5, t4))
    z3 = f6add(f6mul(t5, z3), f6mul(t3, t1))
    return x3 + y3 + z3


def compute_add_mixed(s, q):              # src/utils/ecc.rs:320-388 (RCB15 algorithm 2, a = 1, Z2 = 1)
    X1, Y1, Z1, X2, Y2 = s[0:6], s[6:12], s[12:18], q[0:6], q[6:12]
    t0, t1 = f6mul(X1, X2), f6mul(Y1, Y2)
    t3 = f6sub(f6mul(f6add(X2, Y2), f6add(X1, Y1)), f6add(t0, t1))
    t4 = f6add(f6mul(X2, Z1), X1)
    t5 = f6add(f6mul(Y2, Z1), Y1)
    z3 = f6add(f6mul(Z1, B3), t4)
    x3 = f6sub(t1, z3)
    z3 = f6add(t1, z3)
    y3 = f6mul(x3, z3)
    t1 = f6add(f6add(f6dbl(t0), t0), Z1)
    t4 = f6add(f6mul(t4, B3), f6sub(t0, Z1))
    y3 = f6add(y3, f6mul(t1, t4))
    x3 = f6sub(f6mul(t3, x3), f6mul(t5, t4))
    z3 = f6add(f6mul(t5, z3), f6mul(t3, t1))
    return x3 + y3 + z3


def enforce_point_doubling(result, current, nxt, flag):            # src/utils/ecc.rs:73-99
    s1 = compute_double(current[0:18])
    for i in range(18):
        agg(result, i, flag, are_equal(nxt[i], s1[i]))
    agg(result, 18, flag, is_binary(current[18]))


def enforce_point_addition_mixed(result, current, nxt, point, flag):   # src/utils/ecc.rs:102-139
    s1 = compute_add_mixed(current[0:18], point)
    bit = current[18]
    for i in range(18):
        agg(result, i, flag, are_equal(nxt[i], (bit * s1[i] + not_(bit) * current[i]) % P))
    agg(result, 18, flag, are_equal(current[18], nxt[18]))


def enforce_point_addition_reduce_x(result, current, nxt, point, flag):   # src/utils/ecc.rs:146-172
    s1 = compute_add(current[0:18], point)
    x_z = f6mul(nxt[0:6], s1[12:18])
    for i in range(6):
        agg(result, i, flag, are_equal(x_z[i], s1[i]))
    for i in range(6, 18):
        agg(result, i, flag, are_equal(nxt[i], s1[i]))


def enforce_double_and_add_step(result, current, nxt, value_pos, bit_pos, flag, constrained=False):   # src/utils/field.rs:31-70
    agg(result, value_pos, flag, are_equal(nxt[value_pos], (2 * current[value_pos] + nxt[bit_pos]) % P))
    if not constrained:
        agg(result, bit_pos, flag, is_binary(nxt[bit_pos]))


# ---------------------------------------------------------------------------------------------- layout (src/constants.rs, src/merkle/constants.rs)
MERKLE_DEPTH = 15
HASH_LEN = CYCLE * MERKLE_DEPTH + ROUNDS                       # TRANSACTION_HASH_LENGTH = 127
S_INIT, S_BIT, S_UPD, R_INIT, R_BIT, R_UPD, ROOT_POS = 0, 14, 15, 29, 43, 44, 58
MERKLE_WIDTH = ROOT_POS + RATE                                 # 65
VALUE_RES = MERKLE_WIDTH                                       # 65
BALANCE_RES = MERKLE_WIDTH + AFFINE * 2 + 1                    # 90
NONCE_RES, INT_ROOT_RES = BALANCE_RES + 1, BALANCE_RES + 2     # 91, 92
PREV_MATCH_RES = INT_ROOT_RES + RATE                           # 99
S_KEY_POS, R_KEY_POS = MERKLE_WIDTH, MERKLE_WIDTH + AFFINE     # 65, 77
DELTA_POS, SIGMA_POS, NONCE_POS = MERKLE_WIDTH + 24, MERKLE_WIDTH + 25, MERKLE_WIDTH + 26   # 89, 90, 91
TX_WIDTH = NONCE_POS + 3                                       # 94
S_KEY_RES = PREV_MATCH_RES + 2                                 # 101  (strides of 2 while the loops run 12 wide: overlaps are the reference's)
R_KEY_RES, DELTA_RES = S_KEY_RES + 2, S_KEY_RES + 4            # 103, 105
SIGMA_RES, NONCE_COPY_RES, DELTA_RANGE_RES, SIGMA_RANGE_RES = DELTA_RES + 1, DELTA_RES + 2, DELTA_RES + 3, DELTA_RES + 4   # 106..109
SCHNORR_WIDTH = 2 * PROJ + 2 + 4 + STATE                        # 56
DELTA_BIT, DELTA_ACC, SIGMA_BIT, SIGMA_ACC = SCHNORR_WIDTH, SCHNORR_WIDTH + 1, NONCE_POS + 1, NONCE_POS + 2
TX_CYCLE, MERKLE_CYCLE, SIG_CYCLE, SCALAR_MUL_LEN, NUM_HASH_ITER, RANGE_LOG = 1024, 512, 512, 510, 5, 64
# periodic column indices of the transaction AIR (src/constants.rs:85-115)
(SETUP_M, MERKLE_M, HASH_INPUT_M, FINISH_M, HASH_M, SCHNORR_M, SCALAR_MULT_M, DOUBLING_M) = range(8)
DIGEST_M, SCHNORR_HASH_M, INTERNAL_INPUT_M = 8, 12, 13
RANGE_STEP_M, RANGE_FINISH_M, VALUE_COPY_M, ARK_INDEX = 17, 18, 19, 20


def round_constant_columns():             # rescue::get_round_constants, src/utils/rescue.rs:305-321
    return [[ARK[i][j] for i in range(8)] for j in range(28)]


def single(column, step, value):          # Assertion::single(column, step, value)
    return ("single", column, step, 0, [value])


class Degree:
    def __init__(self, base, cycles=()):
        self.base, self.cycles = base, list(cycles)

    def evaluation_degree(self, n):       # TransitionConstraintDegree::get_evaluation_degree [winterfell]
        return self.base * (n - 1) + sum((n // c) * (c - 1) for c in self.cycles)

    def key(self):
        return (self.base, tuple(self.cycles))


# ---------------------------------------------------------------------------------------------- the six AIRs
def merkle_update_degrees(cycle):         # src/merkle/update/air.rs:371-401
    h = [Degree(3, [cycle])] * 14
    auth = h + [Degree(2, [cycle])] + h
    return auth + auth + [Degree(1, [cycle])] * (PREV_MATCH_RES + RATE - ROOT_POS)


def schnorr_degrees(num_sig, cycle):      # src/schnorr/air.rs:533-585
    bit_degree = 3 if num_sig == 1 else 5
    d = [Degree(5, [cycle, cycle])] * COORD + [Degree(4, [cycle, cycle])] * AFFINE + [Degree(2, [cycle])]
    d += [Degree(bit_degree, [cycle, cycle])] * PROJ + [Degree(2, [cycle])]
    return d + [Degree(1, [cycle, cycle])] * 4 + [Degree(3, [cycle])] * STATE


def merkle_update_periodic():             # src/merkle/update/air.rs:182-212
    setup = [1] + [0] * (MERKLE_CYCLE - 1)
    hashing = [1] * HASH_LEN + [0] * (MERKLE_CYCLE - HASH_LEN)
    hash_input = [0] * 7 + [1]
    finish = [0] * MERKLE_CYCLE
    finish[HASH_LEN - 1] = 1
    hash_mask = [hashing[i] * (1 if i % 8 < 7 else 0) for i in range(MERKLE_CYCLE)]
    return [setup, hashing, hash_input, finish, hash_mask] + round_constant_columns()


def schnorr_periodic():                   # src/schnorr/air.rs:282-343 (the eight masks shared with the transaction AIR, then ARK)
    hash_flag = ([1] * 7 + [0]) * NUM_HASH_ITER
    hash_flag += [0] * (SIG_CYCLE - len(hash_flag))
    scalar_mult = [1] * SCALAR_MUL_LEN + [0] * (SIG_CYCLE - SCALAR_MUL_LEN)
    doubling = [1, 0] * (SCALAR_MUL_LEN // 2) + [0] * (SIG_CYCLE - SCALAR_MUL_LEN)
    digest_flags = [[0] * SIG_CYCLE for _ in range(4)]
    for k, (a, b) in enumerate([(0, 126), (126, 254), (254, 382), (382, 510)]):
        for i in range(a, b):
            digest_flags[k][i] = 1
    global_mask = [1] * (SCALAR_MUL_LEN + 1) + [0] * (SIG_CYCLE - SCALAR_MUL_LEN - 1)
    return [global_mask, scalar_mult, doubling] + digest_flags + [hash_flag] + round_constant_columns()


def merkle_init_constraints(result, current, nxt, ark, flag):      # src/merkle/init/air.rs:159-202
    for res, pos in [(S_INIT, S_INIT), (S_UPD - 1, S_UPD), (R_INIT - 1, R_INIT), (R_UPD - 2, R_UPD)]:
        enforce_round(result.sub(res), current.sub(pos), nxt.sub(pos), ark, flag)


def merkle_update_auth(result, current, nxt, ark, hash_flag_tx, hash_input_flag, hash_flag):   # src/merkle/update/air.rs:291-369
    copy_flag = hash_flag_tx * not_(hash_flag + hash_input_flag) % P
    init_flag = hash_flag_tx * hash_input_flag % P
    bit = nxt[STATE]
    agg(result, STATE, hash_flag_tx, is_binary(bit))
    nbit = not_(bit)
    for res, reg in [(0, 0), (STATE + 1, STATE + 1)]:
        enforce_round(result.sub(res), current.sub(reg), nxt.sub(reg), ark, hash_flag)
        for i in range(RATE):
            agg(result, res + i, copy_flag, are_equal(current[reg + i], nxt[reg + i]))
            agg(result, res + i, init_flag, nbit * are_equal(current[reg + i], nxt[reg + i]) % P)
            agg(result, res + RATE + i, init_flag, bit * are_equal(current[reg + i], nxt[reg + RATE + i]) % P)
    for i in range(RATE):
        agg(result, i, init_flag, bit * are_equal(nxt[STATE + 1 + i], nxt[i]) % P)
    for i in range(RATE, STATE):
        agg(result, i, init_flag, nbit * are_equal(nxt[STATE + 1 + i], nxt[i]) % P)


def merkle_update_constraints(result, current, nxt, ark, hash_flag_tx, hash_input_flag, hash_flag, finish_flag):   # :215-289
    merkle_update_auth(result.sub(S_INIT), current.sub(S_INIT), nxt.sub(S_INIT), ark, hash_flag_tx, hash_input_flag, hash_flag)
    merkle_update_auth(result.sub(R_INIT), current.sub(R_INIT), nxt.sub(R_INIT), ark, hash_flag_tx, hash_input_flag, hash_flag)
    for i in range(RATE):
        agg(result, ROOT_POS + i, not_(finish_flag), are_equal(nxt[ROOT_POS + i], current[ROOT_POS + i]))
        agg(result, ROOT_POS + i, finish_flag, are_equal(nxt[ROOT_POS + i], nxt[R_UPD + i]))
    for i in range(RATE):
        agg(result, INT_ROOT_RES + i, finish_flag, are_equal(current[S_UPD + i], current[R_INIT + i]))
    for i in range(RATE):
        agg(result, PREV_MATCH_RES + i, finish_flag, are_equal(nxt[S_INIT + i], current[ROOT_POS + i]))


def setup_value_constraints(result, current, flag):   # shared head of src/air.rs:405-454 and src/merkle/update/air.rs:77-128
    for i in range(AFFINE):
        agg(result, VALUE_RES + i, flag, are_equal(current[S_INIT + i], current[S_UPD + i]))
        agg(result, VALUE_RES + AFFINE + i, flag, are_equal(current[R_INIT + i], current[R_UPD + i]))
    agg(result, VALUE_RES + 2 * AFFINE, flag, are_equal(current[R_INIT + AFFINE + 1], current[R_UPD + AFFINE + 1]))
    agg(result, BALANCE_RES, flag, are_equal((current[S_INIT + AFFINE] - current[S_UPD + AFFINE]) % P, (current[R_UPD + AFFINE] - current[R_INIT + AFFINE]) % P))
    agg(result, NONCE_RES, flag, are_equal(current[S_UPD + AFFINE + 1], (current[S_INIT + AFFINE + 1] + 1) % P))


def schnorr_hash_copy(result, current, nxt, flag, inputs):         # src/schnorr/air.rs:309-330
    for i in range(RATE):
        agg(result, i, flag, are_equal(current[i], nxt[i]))
    for i in range(RATE):
        agg(result, RATE + i, flag, (nxt[RATE + i] - inputs[i]) % P)


def schnorr_constraints(result, current, nxt, ark, doubling, addition, digest_flags, pkey, final_add, hash_flag, copy_hash, inputs):   # :394-531
    H = 2 * PROJ                                                     # 36
    enforce_point_doubling(result, current, nxt, doubling)
    enforce_point_addition_mixed(result, current, nxt, GENERATOR, addition)
    enforce_point_doubling(result.sub(PROJ + 1), current.sub(PROJ + 1), nxt.sub(PROJ + 1), doubling)
    enforce_point_addition_mixed(result.sub(PROJ + 1), current.sub(PROJ + 1), nxt.sub(PROJ + 1), pkey, addition)
    for i in range(4):
        enforce_double_and_add_step(result.sub(H + 1), current.sub(H + 1), nxt.sub(H + 1), 4 - i, 0, digest_flags[i] * doubling % P, constrained=True)
    for i in range(4):
        agg(result, H + 2 + i, addition, are_equal(current[H + 2 + i], nxt[H + 2 + i]))
    for i in range(4):
        agg(result, H + 5 - i, not_(digest_flags[i]) * doubling % P, are_equal(current[H + 5 - i], nxt[H + 5 - i]))
    enforce_round(result.sub(H + 6), current.sub(H + 6), nxt.sub(H + 6), ark, hash_flag)
    schnorr_hash_copy(result.sub(H + 6), current.sub(H + 6), nxt.sub(H + 6), copy_hash, inputs)
    enforce_point_addition_reduce_x(result, current, nxt, current[PROJ + 1:2 * PROJ + 1], final_add)
    for i in range(4):
        agg(result, H + 2 + i, final_add, are_equal(current[H + 2 + i], current[H + 6 + i]))


class TransactionAir:
    air_id, width, num_constraints, name = 0, TX_WIDTH, 115, "transaction"

    def __init__(self, trace_len, pub):
        self.n, self.pub = trace_len, list(pub)      # initial_root[7] final_root[7]

    def degrees(self):                    # src/air.rs:76-108
        d = merkle_update_degrees(TX_CYCLE)
        d[R_BIT] = Degree(3, [TX_CYCLE])
        d[INT_ROOT_RES] = Degree(2, [TX_CYCLE])
        sd = schnorr_degrees(2, TX_CYCLE)
        for i in range(PROJ):
            d[i] = sd[i]
            d[i + PROJ + 1] = sd[i + PROJ + 1]
        return d + [Degree(1, [TX_CYCLE])] * (SIGMA_RANGE_RES - S_KEY_RES + 1)

    def periodic_columns(self):           # src/air.rs:194-380, as the stitch / fill / pad sequence the reference runs
        cols = [[] for _ in range(ARK_INDEX + 28)]
        for j, c in enumerate(round_constant_columns()):
            cols[ARK_INDEX + j] += c
        pad = lambda idx, length, v: [cols[i].extend([v] * (length - len(cols[i]))) for i in idx]   # noqa: E731
        pad([SETUP_M], 1, 1)
        pad([VALUE_COPY_M], 1, 0)
        pad([MERKLE_M, FINISH_M, HASH_M], 0, 0)
        mcols = merkle_update_periodic()
        cols[HASH_INPUT_M] += mcols[2]
        for a, o in [(1, MERKLE_M), (3, FINISH_M), (4, HASH_M)]:
            for i in range(len(cols[o]), HASH_LEN):
                cols[o].append(mcols[a][i % len(mcols[a])])
        pad([SETUP_M, MERKLE_M, FINISH_M, HASH_M, SCHNORR_M, SCALAR_MULT_M, DOUBLING_M, SCHNORR_HASH_M, RANGE_STEP_M, RANGE_FINISH_M], MERKLE_CYCLE, 0)
        pad(range(DIGEST_M, SCHNORR_HASH_M), MERKLE_CYCLE, 0)
        pad([VALUE_COPY_M], MERKLE_CYCLE, 1)
        scols = schnorr_periodic()
        for a, o in enumerate([SCHNORR_M, SCALAR_MULT_M, DOUBLING_M, DIGEST_M, DIGEST_M + 1, DIGEST_M + 2, DIGEST_M + 3, SCHNORR_HASH_M]):
            cols[o] += scols[a]
        pad(range(INTERNAL_INPUT_M, RANGE_STEP_M), MERKLE_CYCLE, 0)
        for k in range(RANGE_STEP_M - INTERNAL_INPUT_M):
            mask = [0] * SIG_CYCLE
            mask[(k + 1) * CYCLE - 1] = 1
            cols[INTERNAL_INPUT_M + k] += mask
        cols[RANGE_STEP_M] += [1] * RANGE_LOG
        cols[RANGE_FINISH_M] += [0] * (RANGE_LOG - 1) + [1]
        length = MERKLE_CYCLE + max(3 * CYCLE - 1, RANGE_LOG)
        pad([VALUE_COPY_M], length, 1)
        pad([SETUP_M, MERKLE_M, FINISH_M, HASH_M, SCHNORR_M, SCALAR_MULT_M, DOUBLING_M, SCHNORR_HASH_M, RANGE_STEP_M, RANGE_FINISH_M, VALUE_COPY_M], TX_CYCLE, 0)
        pad(range(DIGEST_M, DIGEST_M + 4), TX_CYCLE, 0)
        pad(range(INTERNAL_INPUT_M, INTERNAL_INPUT_M + 3), TX_CYCLE, 0)
        return cols

    def assertions(self):                 # src/air.rs:175-184: (kind, column, first_step, stride, values); kind = the Assertion constructor called
        last = self.n - 1
        return [single(ROOT_POS, 0, self.pub[0]), single(ROOT_POS + 1, 0, self.pub[1]), single(ROOT_POS, last, self.pub[7]), single(ROOT_POS + 1, last, self.pub[8])]

    def evaluate(self, current, nxt, pv):  # src/air.rs:114-173 + 383-610
        result = [0] * self.num_constraints
        res, cur, nx = View(result), View(list(current)), View(list(nxt))
        setup, hashing, hash_input, finish, hash_flag = pv[SETUP_M], pv[MERKLE_M], pv[HASH_INPUT_M], pv[FINISH_M], pv[HASH_M]
        schnorr_mask, scalar_mult, doubling = pv[SCHNORR_M], pv[SCALAR_MULT_M], pv[DOUBLING_M]
        digest_flags, schnorr_hash = pv[DIGEST_M:SCHNORR_HASH_M], pv[SCHNORR_HASH_M]
        input_flags = pv[INTERNAL_INPUT_M:RANGE_STEP_M]
        range_flag, range_finish, copy_values = pv[RANGE_STEP_M], pv[RANGE_FINISH_M], pv[VALUE_COPY_M]
        ark = pv[ARK_INDEX:]
        copy_hash = not_(schnorr_hash) * schnorr_mask % P
        final_add = not_(scalar_mult) * schnorr_mask % P
        addition = not_(doubling) * scalar_mult % P

        merkle_init_constraints(res, cur, nx, ark, setup)
        setup_value_constraints(res, cur, setup)
        for r, origin, copy in [(S_KEY_RES, S_INIT, S_KEY_POS), (R_KEY_RES, R_INIT, R_KEY_POS)]:
            for o in range(AFFINE):
                agg(res, r + o, setup, are_equal(nx[copy + o], cur[origin + o]))
        agg(res, DELTA_RES, setup, are_equal(nx[DELTA_POS], (cur[S_INIT + AFFINE] - cur[S_UPD + AFFINE]) % P))
        for r, origin, copy in [(SIGMA_RES, S_UPD + AFFINE, SIGMA_POS), (NONCE_COPY_RES, S_INIT + AFFINE + 1, NONCE_POS)]:
            agg(res, r, setup, are_equal(nx[copy], cur[origin]))
        for r, copy in [(S_KEY_RES, S_KEY_POS), (R_KEY_RES, R_KEY_POS)]:
            for o in range(AFFINE):
                agg(res, r + o, copy_values, are_equal(nx[copy + o], cur[copy + o]))
        for r, copy in [(DELTA_RES, DELTA_POS), (SIGMA_RES, SIGMA_POS), (NONCE_COPY_RES, NONCE_POS)]:
            agg(res, r, copy_values, are_equal(nx[copy], cur[copy]))
        merkle_update_constraints(res, cur, nx, ark, hashing, hash_input, hash_flag, finish)
        inputs = [0] * RATE
        for k in range(NUM_HASH_ITER - 1):
            for i in range(RATE):
                m = k * RATE + i
                cell = nx[S_KEY_POS + m] if m < AFFINE else nx[R_KEY_POS + m - AFFINE] if m < 2 * AFFINE else \
                    nx[DELTA_POS] if m == 2 * AFFINE else nx[NONCE_POS] if m == 2 * AFFINE + 1 else 0
                inputs[i] = (inputs[i] + input_flags[k] * cell) % P
        # result[0..56], current[0..56], next[0..56]; the public key is next[65..77]
        schnorr_constraints(res, cur, nx, ark, doubling, addition, digest_flags, nx[S_KEY_POS:S_KEY_POS + AFFINE], final_add, schnorr_hash, copy_hash, inputs)
        enforce_double_and_add_step(res, cur, nx, DELTA_ACC, DELTA_BIT, range_flag)
        enforce_double_and_add_step(res, cur, nx, SIGMA_ACC, SIGMA_BIT, range_flag)
        agg(res, DELTA_RANGE_RES, range_finish, are_equal(nx[DELTA_ACC], nx[DELTA_POS]))
        agg(res, SIGMA_RANGE_RES, range_finish, are_equal(nx[DELTA_ACC], nx[DELTA_POS]))   # sic: delta again (src/air.rs:605-609)
        return result


class MerkleUpdateAir:
    air_id, width, num_constraints, name = 1, MERKLE_WIDTH, 106, "merkle_update"

    def __init__(self, trace_len, pub):
        self.n, self.pub = trace_len, list(pub)

    def degrees(self):
        return merkle_update_degrees(MERKLE_CYCLE)

    def periodic_columns(self):
        return merkle_update_periodic()

    def assertions(self):                 # src/merkle/update/air.rs:158-177
        last = self.n - 1
        return [single(ROOT_POS + i, 0, self.pub[i]) for i in range(7)] + [single(ROOT_POS + i, last, self.pub[7 + i]) for i in range(7)]

    def evaluate(self, current, nxt, pv):  # src/merkle/update/air.rs:57-156
        result = [0] * self.num_constraints
        res, cur, nx = View(result), View(list(current)), View(list(nxt))
        setup_value_constraints(res, cur, pv[0])
        merkle_update_constraints(res, cur, nx, pv[5:], pv[1], pv[2], pv[4], pv[3])
        return result


class MerkleInitAir:
    air_id, width, num_constraints, name = 2, 58, 56, "merkle_init"

    def __init__(self, trace_len, pub):
        self.n, self.pub = trace_len, list(pub)      # s_inputs[14] r_inputs[14] delta

    def degrees(self):
        return [Degree(3)] * 56

    def periodic_columns(self):
        return round_constant_columns()

    def assertions(self):                 # src/merkle/init/air.rs:77-141
        s, r, delta = self.pub[0:14], self.pub[14:28], self.pub[28]
        a = [single(S_INIT + i, 0, s[i]) for i in range(14)] + [single(S_UPD + i, 0, s[i]) for i in range(12)]
        a += [single(S_UPD + 12, 0, (s[12] - delta) % P), single(S_UPD + 13, 0, (s[13] + 1) % P)]
        a += [single(R_INIT + i, 0, r[i]) for i in range(14)] + [single(R_UPD + i, 0, r[i]) for i in range(12)]
        return a + [single(R_UPD + 12, 0, (r[12] + delta) % P), single(R_UPD + 13, 0, r[13])]

    def evaluate(self, current, nxt, pv):
        result = [0] * self.num_constraints
        merkle_init_constraints(View(result), View(list(current)), View(list(nxt)), pv, 1)
        return result


class SchnorrAir:
    air_id, width, num_constraints, name = 3, SCHNORR_WIDTH, 56, "schnorr"

    def __init__(self, trace_len, pub):
        self.n, self.pub = trace_len, list(pub)      # per signature: message[28] Rx[6] s[4 LE words]
        self.nsig = trace_len // SIG_CYCLE
        self.messages = [self.pub[38 * k:38 * k + 28] for k in range(self.nsig)]
        self.rx = [self.pub[38 * k + 28:38 * k + 34] for k in range(self.nsig)]

    def degrees(self):
        return schnorr_degrees(self.nsig, SIG_CYCLE)

    def periodic_columns(self):           # src/schnorr/air.rs:229-299
        base = schnorr_periodic()
        cols = [[] for _ in range(COORD + PROJ + 3)]          # 27
        for a, o in [(0, 0), (1, 1), (2, 2), (3, 3), (4, 4), (5, 5), (6, 6), (7, 7 + AFFINE)]:
            cols[o] += base[a]
        n = SIG_CYCLE * self.nsig
        inputs, keys = [[0] * n for _ in range(RATE)], [[0] * n for _ in range(AFFINE)]
        for m in range(self.nsig):
            for i in range(SIG_CYCLE):
                if i < NUM_HASH_ITER - 1:
                    for j in range(RATE):
                        inputs[j][i * CYCLE + ROUNDS + m * SIG_CYCLE] = self.messages[m][j + i * RATE]
                for j in range(AFFINE):
                    keys[j][i + m * SIG_CYCLE] = self.messages[m][j]
        for j in range(AFFINE):
            cols[7 + j] += keys[j]
        for j in range(RATE):
            cols[8 + AFFINE + j] += inputs[j]
        return cols + round_constant_columns()

    def assertions(self):                 # src/schnorr/air.rs:111-227
        per = lambda c, v: ("periodic", c, 0, SIG_CYCLE, [v])             # noqa: E731  Assertion::periodic(column, first_step, stride, value)
        seq = lambda c, first: ("sequence", c, first, SIG_CYCLE, [self.rx[m][c if first else c - 2 * PROJ - 6] for m in range(self.nsig)])   # noqa: E731
        a = [per(i, 1 if i == COORD else 0) for i in range(PROJ)] + [per(PROJ, 0)]
        a += [per(i + PROJ + 1, 1 if i == COORD else 0) for i in range(PROJ)]
        a += [per(i + 2 * PROJ + 1, 0) for i in range(5)]
        a += [seq(2 * PROJ + 6 + k, 0) for k in range(6)]
        a += [per(i + 2 * PROJ + COORD + 6, 0) for i in range(RATE)]
        return a + [seq(k, SCALAR_MUL_LEN + 1) for k in range(6)]

    def evaluate(self, current, nxt, pv):  # src/schnorr/air.rs:59-109
        result = [0] * self.num_constraints
        global_mask, scalar_mult, doubling = pv[0], pv[1], pv[2]
        hash_flag = pv[AFFINE + 7]
        schnorr_constraints(View(result), View(list(current)), View(list(nxt)), pv[AFFINE + 15:], doubling, not_(doubling) * scalar_mult % P, pv[3:7],
                            pv[7:AFFINE + 7], not_(scalar_mult) * global_mask % P, hash_flag, not_(hash_flag) * global_mask % P, pv[AFFINE + 8:AFFINE + 15])
        return result


class RangeAir:
    air_id, width, num_constraints, name = 4, 2, 2, "range"

    def __init__(self, trace_len, pub):
        self.n, self.pub = trace_len, list(pub)

    def degrees(self):
        return [Degree(2), Degree(1)]

    def periodic_columns(self):
        return []

    def assertions(self):                 # src/range/air.rs:82-87
        return [single(1, 0, 0), single(1, self.n - 1, self.pub[0])]

    def evaluate(self, current, nxt, pv):
        result = [0, 0]
        enforce_double_and_add_step(result, current, nxt, 1, 0, 1)
        return result


class RescueAir:
    air_id, width, num_constraints, name = 5, 14, 14, "rescue"

    def __init__(self, trace_len, pub):
        self.n, self.pub = trace_len, list(pub)      # seed[7] result[7]

    def degrees(self):
        return [Degree(3, [CYCLE])] * 14

    def periodic_columns(self):           # benches/rescue.rs:262-267
        return [[1] * 7 + [0]] + round_constant_columns()

    def assertions(self):
        last = self.n - 1
        return [single(i, 0, self.pub[i]) for i in range(7)] + [single(i, last, self.pub[7 + i]) for i in range(7)]

    def evaluate(self, current, nxt, pv):  # benches/rescue.rs:210-268
        result = [0] * 14
        hash_flag = pv[0]
        enforce_round(result, current, nxt, pv[1:], hash_flag)
        copy = not_(hash_flag)
        for i in range(RATE):
            agg(result, i, copy, are_equal(current[i], nxt[i]))
        for i in range(RATE):
            agg(result, RATE + i, copy, nxt[RATE + i] % P)
        return result


AIRS = [TransactionAir, MerkleUpdateAir, MerkleInitAir, SchnorrAir, RangeAir, RescueAir]


def ce_blowup(air):                       # AirContext::new [winterfell]: max over constraints of next_power_of_two(base + #cycles), at least 2
    m = 2
    for d in air.degrees():
        v = d.base + len(d.cycles)
        m = max(m, 1 << (v - 1).bit_length())
    return m


def periodic_row(air, step):
    return [c[step % len(c)] for c in air.periodic_columns()]


# ---------------------------------------------------------------------------------------------- witnesses
class Rng:
    """SplitMix64 (own stream; the reference draws from OsRng)"""

    def __init__(self, seed):
        self.s = seed & (2**64 - 1)

    def u64(self):
        self.s = (self.s + 0x9E3779B97F4A7C15) & (2**64 - 1)
        z = self.s
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2**64 - 1)
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2**64 - 1)
        return z ^ (z >> 31)

    def field(self):
        return self.u64() % P


IDENTITY = [0] * 6 + [1] + [0] * 11          # (0 : 1 : 0)


def scalar_mul(k, point_affine):
    """k * point by MSB-first double-and-add with the complete formulas (k a plain integer: no group order is needed)"""
    acc = list(IDENTITY)
    for b in bin(k)[2:] if k else "":
        acc = compute_double(acc)
        if b == "1":
            acc = compute_add_mixed(acc, point_affine)
    return acc


def to_affine(pt):
    zi = f6inv(pt[12:18])
    return f6mul(pt[0:6], zi) + f6mul(pt[6:12], zi)


def hash_message(rx, message):            # src/schnorr/mod.rs:247-288
    h = digest(rx)
    for k in range(4):
        h = merge(h, message[7 * k:7 * k + 7])
    return h


def sign(rng, message, sk):
    """SURVEY.md 8(d): r in [2^254 + 2^251, 2^255), s = r - sk * h as a plain non-negative integer below 2^255"""
    while True:
        r = (1 << 254) + (1 << 251) + ((rng.u64() | (rng.u64() << 64) | (rng.u64() << 128) | (rng.u64() << 192)) % ((1 << 254) - (1 << 251)))
        rx = to_affine(scalar_mul(r, GENERATOR))[0:6]
        h = hash_message(rx, message)
        h_int = sum(h[i] << (64 * i) for i in range(4)) & ((1 << 255) - 1)
        s = r - sk * h_int
        if 0 <= s < (1 << 255):
            return rx, s


def schnorr_rows(message, rx, s_int):
    """rows 0..511 of one signature fragment (56 columns): init_sig_verification_state + update (src/schnorr/trace.rs:18-122)"""
    h = hash_message(rx, message)
    h_int = sum(h[i] << (64 * i) for i in range(4))
    pkey = message[0:12]
    st = [0] * SCHNORR_WIDTH
    st[COORD] = 1
    st[PROJ + COORD + 1] = 1
    st[2 * PROJ + 6:2 * PROJ + 12] = rx
    rows = [list(st)]
    for step in range(SIG_CYCLE - 1):
        st = list(st)
        H = 2 * PROJ + 6
        if step < CYCLE * NUM_HASH_ITER:
            if step % CYCLE < ROUNDS:
                st[H:H + 14] = apply_round(st[H:H + 14], step)
            elif step < (NUM_HASH_ITER - 1) * CYCLE:
                st[H + 7:H + 14] = message[7 * (step // CYCLE):7 * (step // CYCLE) + 7]
            else:
                st[H + 7:H + 14] = [0] * 7
        if step < SCALAR_MUL_LEN:
            real = step // 2
            chunk = 0 if real < 63 else (real - 63) // 64 + 1
            st[PROJ] = (s_int >> (254 - real)) & 1
            st[2 * PROJ + 1] = (h_int >> (254 - real)) & 1
            if step % 2 == 0:
                st[0:PROJ] = compute_double(st[0:PROJ])
                st[PROJ + 1:2 * PROJ + 1] = compute_double(st[PROJ + 1:2 * PROJ + 1])
                pos = 2 * PROJ + 1 + 4 - chunk
                st[pos] = (2 * st[pos] + st[2 * PROJ + 1]) % P
            else:
                if st[PROJ] == 1:
                    st[0:PROJ] = compute_add_mixed(st[0:PROJ], GENERATOR)
                if st[2 * PROJ + 1] == 1:
                    st[PROJ + 1:2 * PROJ + 1] = compute_add_mixed(st[PROJ + 1:2 * PROJ + 1], pkey)
        elif step == SCALAR_MUL_LEN:
            st[PROJ] = 1
            st[0:PROJ] = compute_add(st[0:PROJ], st[PROJ + 1:2 * PROJ + 1])
            st[0:COORD] = f6mul(st[0:COORD], f6inv(st[2 * COORD:PROJ]))
        rows.append(list(st))
    return rows


class SparseTree:
    """MerkleTree::<Rescue63>::build_empty(depth) + update_leaf + prove (src/lib.rs:261-422): leaves default to the zero digest"""

    def __init__(self, depth):
        self.depth, self.nodes = depth, {}
        self.empty = [[0] * 7]
        for _ in range(depth):
            self.empty.append(merge(self.empty[-1], self.empty[-1]))

    def node(self, level, index):         # level 0 = leaves
        return self.nodes.get((level, index), self.empty[level])

    def update_leaf(self, index, leaf):
        self.nodes[(0, index)] = list(leaf)
        for level in range(1, self.depth + 1):
            index >>= 1
            self.nodes[(level, index)] = merge(self.node(level - 1, 2 * index), self.node(level - 1, 2 * index + 1))

    def root(self):
        return self.node(self.depth, 0)

    def prove(self, index):               # [leaf, sibling at level 0, sibling at level 1, ...]
        path = [self.node(0, index)]
        for level in range(self.depth):
            path.append(self.node(level, (index >> level) ^ 1))
        return path


def leaf_of(value):
    return merge(value[0:7], value[7:14])


class TransactionBatch:
    """TransactionMetadata::build_random (src/lib.rs:235-464) with a seeded generator"""

    def __init__(self, seed, num_tx, depth=MERKLE_DEPTH):
        rng = Rng(seed)
        size = 1 << depth
        self.depth, self.num_tx = depth, num_tx
        tree, values, keys = SparseTree(depth), {}, {}

        def new_account(index):
            sk = 1 + rng.u64() % 3
            pk = to_affine(scalar_mul(sk, GENERATOR))
            values[index] = pk + [rng.u64() % P, rng.u64() % P]
            keys[index] = sk
            tree.update_leaf(index, leaf_of(values[index]))
        self.s_indices = []
        for _ in range(num_tx):
            i = rng.u64() % size
            self.s_indices.append(i)
            new_account(i)
        self.r_indices = []
        for t in range(num_tx):
            r = rng.u64() % size
            while r == self.s_indices[t]:
                r = rng.u64() % size
            self.r_indices.append(r)
            if r not in keys:
                new_account(r)
        self.initial_roots, self.s_old, self.r_old, self.s_paths, self.r_paths, self.deltas, self.sks = [], [], [], [], [], [], []
        for t in range(num_tx):
            s, r = self.s_indices[t], self.r_indices[t]
            delta = rng.u64() % max(1, min(values[s][12], 2**64 - 1 - values[r][12]))
            self.initial_roots.append(tree.root())
            self.sks.append(keys[s]); self.s_old.append(list(values[s])); self.r_old.append(list(values[r])); self.deltas.append(delta)
            self.s_paths.append(tree.prove(s))
            values[s][12] = (values[s][12] - delta) % P
            values[s][13] = (values[s][13] + 1) % P
            values[r][12] = (values[r][12] + delta) % P
            tree.update_leaf(s, leaf_of(values[s]))
            tree.update_leaf(r, leaf_of(values[r]))
            self.r_paths.append(tree.prove(r))
        self.final_root = tree.root()
        self.messages = [self.s_old[t][0:12] + self.r_old[t][0:12] + [self.deltas[t], self.s_old[t][13], 0, 0] for t in range(num_tx)]   # build_tx_message
        self.signatures = [sign(rng, self.messages[t], self.sks[t]) for t in range(num_tx)]

    def pub_inputs(self):
        return list(self.initial_roots[0]) + list(self.final_root)

    def merkle_rows(self, t, count):
        """rows 0..count-1 of transaction t's Merkle phase (65 columns): init_merkle_update_state + update (src/merkle/update/trace.rs)"""
        s, r, delta = self.s_old[t], self.r_old[t], self.deltas[t]
        st = [0] * MERKLE_WIDTH
        st[S_INIT:S_INIT + 14] = s
        st[S_UPD:S_UPD + 14] = s[0:12] + [(s[12] - delta) % P, (s[13] + 1) % P]
        st[R_INIT:R_INIT + 14] = r
        st[R_UPD:R_UPD + 14] = r[0:12] + [(r[12] + delta) % P, r[13]]
        st[ROOT_POS:ROOT_POS + 7] = self.initial_roots[t]
        rows = [list(st)]
        for step in range(count - 1):
            st = list(st)
            if step < HASH_LEN:
                for base, index, branch in [(S_INIT, self.s_indices[t], self.s_paths[t]), (R_INIT, self.r_indices[t], self.r_paths[t])]:
                    level, pos = step // CYCLE, step % CYCLE
                    if pos < ROUNDS:
                        st[base:base + 14] = apply_round(st[base:base + 14], step)
                        st[base + 15:base + 29] = apply_round(st[base + 15:base + 29], step)
                    else:
                        node, bit = branch[level + 1], (index >> level) & 1
                        if bit == 0:
                            st[base + 7:base + 14] = node
                            st[base + 15 + 7:base + 15 + 14] = node
                        else:
                            st[base + 7:base + 14] = st[base:base + 7]
                            st[base + 15 + 7:base + 15 + 14] = st[base + 15:base + 15 + 7]
                            st[base:base + 7] = node
                            st[base + 15:base + 15 + 7] = node
                        st[base + 14] = bit
            if step == HASH_LEN - 1:
                st[ROOT_POS:ROOT_POS + 7] = st[R_UPD:R_UPD + 7]
            rows.append(list(st))
        return rows

    def transaction_trace(self):
        """TransactionProver::build_trace (src/prover.rs:37-98): rows as lists of 94 canonical values"""
        out = []
        for t in range(self.num_tx):
            s, delta = self.s_old[t], self.deltas[t]
            sigma = (s[12] - delta) % P
            tail = self.s_old[t][0:12] + self.r_old[t][0:12] + [delta, sigma, s[13], 0, 0]       # columns 65..93
            rows = [m + tail for m in self.merkle_rows(t, MERKLE_CYCLE)]
            rx, s_int = self.signatures[t]
            sch = schnorr_rows(self.messages[t], rx, s_int)
            dacc = sacc = 0
            for k, srow in enumerate(sch):          # row 512 + k; k = 0 is the state written by step 511
                dbit = sbit = 0
                if 1 <= k <= RANGE_LOG:             # written by schnorr_step = k - 1 < 64
                    dbit, sbit = (delta >> (RANGE_LOG - k)) & 1, (sigma >> (RANGE_LOG - k)) & 1
                    dacc, sacc = (2 * dacc + dbit) % P, (2 * sacc + sbit) % P
                elif k > RANGE_LOG:                 # registers keep their last values
                    dbit, sbit = delta & 1, sigma & 1
                prev = rows[-1]
                rows.append(srow + [dbit, dacc] + prev[ROOT_POS:NONCE_POS + 1] + [sbit, sacc])
            out += rows
        return out

    def merkle_update_trace(self):
        """MerkleProver::build_trace (src/merkle/update/prover.rs:37-80), including the bit tweak at step 1 (:72-77)"""
        out = []
        for t in range(self.num_tx):
            out += self.merkle_rows(t, MERKLE_CYCLE)
        out[1][S_BIT] = 1
        out[1][R_BIT] = 1
        return out


def schnorr_batch(seed, num_sig):
    """SchnorrExample::new (src/schnorr/mod.rs:79-141): messages = public key + 16 random elements; returns (rows, pub)"""
    rng = Rng(seed)
    rows, pub = [], []
    for _ in range(num_sig):
        sk = 1 + rng.u64() % 3
        message = to_affine(scalar_mul(sk, GENERATOR)) + [rng.field() for _ in range(16)]
        rx, s = sign(rng, message, sk)
        rows += schnorr_rows(message, rx, s)
        pub += message + rx + [(s >> (64 * i)) & (2**64 - 1) for i in range(4)]
    return rows, pub


def range_trace(number):                  # src/range/prover.rs:36-84 (range_log - 1 = 63 passed to the update)
    rows, acc = [[0, 0]], 0
    for step in range(63):
        bit = (number >> (62 - step)) & 1
        acc = (2 * acc + bit) % P
        rows.append([bit, acc])
    return rows, [rows[-1][1]]


def rescue_trace(seed, chain):            # benches/rescue.rs:279-321
    st = list(seed) + [0] * 7
    rows = [list(st)]
    for step in range(8 * chain - 1):
        st = apply_round(st, step) if step % 8 < 7 else st[0:7] + [0] * 7
        rows.append(list(st))
    return rows, list(seed) + rows[-1][0:7]


def merkle_init_trace(s_inputs, r_inputs, delta):   # src/merkle/init/trace.rs:18-72, src/merkle/init/prover.rs:35-53
    st = [0] * 58
    # the reference never writes the sender's INITIAL coins and nonce: it stores them in the updated slots first and then
    # overwrites those (src/merkle/init/trace.rs:26-35; SURVEY.md Appendix E).  Harmless for its own all-zero example only.
    st[S_INIT:S_INIT + 12] = s_inputs[0:12]
    st[S_UPD:S_UPD + 14] = s_inputs[0:12] + [(s_inputs[12] - delta) % P, (s_inputs[13] + 1) % P]
    st[R_INIT:R_INIT + 14] = r_inputs
    st[R_UPD:R_UPD + 14] = r_inputs[0:12] + [(r_inputs[12] + delta) % P, r_inputs[13]]
    rows = [list(st)]
    for step in range(15):                # a round on EVERY step: the eighth uses the all-zero constants
        st = list(st)
        for base in (S_INIT, S_UPD, R_INIT, R_UPD):
            st[base:base + 14] = apply_round(st[base:base + 14], step)
        rows.append(list(st))
    return rows, rows[0][S_INIT:S_INIT + 14] + rows[0][R_INIT:R_INIT + 14] + [delta]


def violations(air, rows, wrap=True):
    """(step, constraint) pairs that do not vanish on consecutive rows (the last row wraps to the first only for the
    transition the engine never checks, so it is skipped)"""
    bad = []
    cols = air.periodic_columns()
    for step in range(len(rows) - 1):
        pv = [c[step % len(c)] for c in cols]
        res = air.evaluate(rows[step], rows[step + 1], pv)
        bad += [(step, i) for i, v in enumerate(res) if v]
    return bad
