"""The shared-memory, lazily reduced Fp12 tower of the verification kernels (csrc/lazy.cuh: lz_f12mul_g, lz_f12sqr, lz_mul_line,
lz_cyc_sqr, lz_f12inv, lz_frob, lz_final_exp_stage, lz_mul_nline, lz_miller_norm_seg) on the device, through the parity hook
zkv_fp12_op_batch op 16 + k (k_lz_fp12_op), against the CPU oracle bit for bit (12 x BE-32, tower order) and against the round-1 tower
(op k, k_fp12_op) on the same operands.  Operands at the edges of lazy reduction (oracle_lib.fp12_operand_classes) sit in one batch
with random ones; batch sizes around the 128-thread block, a full wave plus a partial block, lane isolation and stale shared memory
cover what can go wrong in the launch rather than in the arithmetic."""
import functools
import random

import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

P = O.P
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
ONE, ZERO = O.FP12_ONE, bytes(384)
SIZES = (1, 127, 128, 129, 300)
ROUND1 = {16: 0, 17: 1, 18: 2, 19: 3, 20: 4, 21: 5, 22: 6, 23: 7, 24: 8, 26: 9}     # the round-1 hook op of the same operation
UNARY = (17, 19, 20, 21, 22, 23, 24)
CLASSES = O.fp12_operand_classes(0x1A2)


@pytest.fixture(scope="module")
def Z():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import stylus_zkvm_verifiers_b200 as Z
    return Z


def run(Z, op, A, B=None):
    n = len(A)
    out = Z.fp12_op_batch(op, b"".join(A), None if B is None else b"".join(B), n)
    assert len(out) == 384 * n
    return [out[384 * i:384 * i + 384] for i in range(n)]


def line_dense(b):
    """l0 + l3 w + l4 v w as a dense Fp12 (l0, l3, l4 = b's first three Fp2): what ops 2 / 18 multiply by"""
    return b[0:64] + bytes(128) + b[64:192] + bytes(64)


def nline_dense(b):
    """1 + c3 w + c4 v w (c3, c4 = b's first two Fp2): what op 25 multiplies by"""
    return w32(1) + bytes(160) + b[0:128] + bytes(64)


def neg_g1(p):
    return p[:32] + w32((P - int.from_bytes(p[32:64], "big")) % P)


def neg_g2(q):
    return q[:64] + b"".join(w32((P - int.from_bytes(q[k:k + 32], "big")) % P) for k in (64, 96))


@functools.lru_cache(maxsize=None)
def frobs(a):
    """(a^p, a^(p^2), a^(p^3)) by square-and-multiply over the oracle's product"""
    f1 = O.fp12_frob(a, 1); f2 = O.fp12_frob(f1, 1)
    return f1, f2, O.fp12_frob(f2, 1)


@functools.lru_cache(maxsize=None)
def expected(op, a, b):
    """the oracle's value of op on (a, b), or None where the check is not a value (20: inverse by product; 21-23: see check)"""
    if op == 16: return O.fp12_mul(a, b)
    if op == 17: return O.fp12_mul(a, a)
    if op == 18: return O.fp12_mul(a, line_dense(b))
    if op == 19: return O.fp12_cyc_sqr(a)
    if op == 24: return O.final_exp(a)
    if op == 25: return O.fp12_mul(a, nline_dense(b))
    if op == 26: return O.ec_pairing(b[:192], debug=True)[1]
    return None


def check(op, A, B, out, pow_frob=None):
    """every output of an op-`op` batch against the oracle; for the Frobenius ops, a^(p^k) on the operands listed in pow_frob"""
    for i, a in enumerate(A):
        b = None if B is None else B[i]
        if op == 20:
            assert (out[i] == ZERO) if a == ZERO else (O.fp12_mul(a, out[i]) == ONE), (op, i, a.hex())
        elif op in (21, 22, 23):
            if pow_frob is not None and a in pow_frob:
                assert out[i] == frobs(a)[op - 21], (op, i, a.hex())
        else:
            assert out[i] == expected(op, a, b), (op, i, a.hex(), b.hex() if b else None)


# ------------------------------------------------------------------------------------------------ operands
def rand12(rnd):
    return b"".join(w32(rnd.getrandbits(256) % P) for _ in range(12))


def edge_batch(n, seed):
    """n operand pairs: every operand class of oracle_lib (at random lanes) next to random pairs when n allows, else a sample of them"""
    rnd = random.Random(seed)
    items = [(a, b) for _, a, b in CLASSES]
    if n < len(items):
        return [list(t) for t in zip(*rnd.sample(items, n))]
    pairs = [(rand12(rnd), rand12(rnd)) for _ in range(n)]
    for pos, it in zip(rnd.sample(range(n), len(items)), items):
        pairs[pos] = it
    return [list(t) for t in zip(*pairs)]


@functools.lru_cache(maxsize=None)
def cyclotomic_pool():
    return [g for _, g in O.fp12_cyclotomic_operands(0x1A2, nfrob=2)]


@functools.lru_cache(maxsize=None)
def pair_pool():
    """(P, Q) for op 26: P = [k]G1 and -P, Q = [k]G2 for k in {1, 2, 5, r - 1, r - 2, random}, Q = -G2"""
    from stylus_zkvm_verifiers_b200.synth import G1_GEN, G2_GEN
    rnd = random.Random(0x26)
    ks = [1, 2, 5, R - 1, R - 2, rnd.randrange(3, R - 2)]
    ps = [O.g1_mul(G1_GEN, k) for k in ks]
    ps += [neg_g1(p) for p in ps]
    qs = [O.g2_mul(G2_GEN, k) for k in ks] + [neg_g2(G2_GEN)]
    return [p + q for p in ps for q in qs]


def inputs(op, n, seed):
    """(A, B) of n operands for op"""
    rnd = random.Random(seed)
    if op == 19:
        pool = cyclotomic_pool()
        A = pool[:n] + [rnd.choice(pool) for _ in range(n - len(pool))]
        rnd.shuffle(A)
        return A, None
    if op == 26:
        pool = pair_pool()
        B = pool[:n] + [rnd.choice(pool) for _ in range(n - len(pool))]
        rnd.shuffle(B)
        return [ZERO] * n, [pq + bytes(192) for pq in B]
    A, B = edge_batch(n, seed)
    return A, (None if op in UNARY else B)


LAZY_OPS = (16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26)


# ------------------------------------------------------------------------------------------------ tests
def test_argument_checks(Z):
    for op in (15, 27, -1, 10):
        with pytest.raises(Z.ZkvError) as e:
            Z.fp12_op_batch(op, ZERO, ZERO, 1)
        assert e.value.code == -1, op
    for op in (16, 18, 25, 26):
        with pytest.raises(Z.ZkvError) as e:
            Z.fp12_op_batch(op, ZERO, None, 1)
        assert e.value.code == -1, op
    for op in LAZY_OPS:
        assert Z.fp12_op_batch(op, b"", b"", 0) == b""


@pytest.mark.parametrize("op", (16, 17, 18, 20, 21, 22, 23, 24, 25))
def test_lazy_op_matches_oracle_and_round1(Z, op):
    """Every size around the block of 128 threads; the operand classes with random operands in the larger batches."""
    for n in SIZES:
        A, B = inputs(op, n, 1000 * (21 if op in (21, 22, 23) else op) + n)       # one batch for the three Frobenius ops: a^(p^k) once
        out = run(Z, op, A, B)
        pow_frob = set(A[:4]) if n < 300 else set(A[:24]) | {a for _, a, _ in CLASSES[::4]}
        check(op, A, B, out, pow_frob)
        if op in ROUND1:
            assert out == run(Z, ROUND1[op], A, B), (op, n)
    if op == 20:
        assert run(Z, 20, [ZERO]) == run(Z, 4, [ZERO]) == [ZERO]                   # inv(0) = 0, as the safegcd inversion gives


def test_cyclotomic_square_on_cyclotomic_elements(Z):
    """op 19 (lz_cyc_sqr) is only defined on the cyclotomic subgroup: final-exponentiation outputs, their conjugates and Frobenius images, one."""
    for n in SIZES:
        A, _ = inputs(19, n, 1900 + n)
        out = run(Z, 19, A)
        check(19, A, None, out)
        assert all(out[i] == O.fp12_mul(a, a) for i, a in enumerate(A))
        assert out == run(Z, 3, A)


def test_verification_miller_loop_single_pair(Z):
    """op 26 (lz_miller_norm_seg in three segments, fixed pairs off) against the oracle's Miller value and the round-1 loop (op 9); twist
    points outside G2 have no oracle value (the precompile reverts) and must still give op 9's value."""
    for n in SIZES:
        A, B = inputs(26, n, 2600 + n)
        out = run(Z, 26, A, B)
        check(26, A, B, out)
        assert out == run(Z, 9, A, B), n
    from stylus_zkvm_verifiers_b200.synth import G1_GEN, SplitMix64, random_twist_point
    rng = SplitMix64(0x2626)
    ps = [G1_GEN, O.g1_mul(G1_GEN, 7), neg_g1(O.g1_mul(G1_GEN, 11))]
    B = [ps[i % 3] + random_twist_point(rng) + bytes(192) for i in range(6)]
    assert all(O.ec_pairing(b[:192]) is None for b in B)
    assert run(Z, 26, [ZERO] * 6, B) == run(Z, 9, [ZERO] * 6, B)


def test_full_wave_and_a_partial_block(Z):
    """ops 16 and 17 on one full wave of the kernel (SMs x 2 blocks x 128 threads) plus 129 operands, every output against the oracle."""
    n = Z.wave_proofs(0, 0) + 129
    for op in (16, 17):
        A, B = edge_batch(n, 0xA0 + op)
        B = None if op == 17 else B
        out = run(Z, op, A, B)
        bad = [i for i in range(n) if out[i] != expected(op, A[i], A[i] if op == 17 else B[i])]
        assert not bad, (op, bad[:10])
    expected.cache_clear()


@pytest.mark.parametrize("op", LAZY_OPS)
def test_lane_isolation(Z, op):
    """Slots are word-interleaved across the block: a routine that touches a neighbour's slot is wrong only on the device.  A batch rotated
    by 37 lanes gives outputs rotated the same way, and one operand repeated with a different one at lane 0, 31, 32 or 127 gives the
    repeated operand's value everywhere else."""
    n = 300
    A, B = inputs(op, n, 3700 + op)
    out = run(Z, op, A, B)
    rot = lambda xs: None if xs is None else xs[37:] + xs[:37]
    assert run(Z, op, rot(A), rot(B)) == rot(out), op
    x, y = 0, 1
    while (A[x], B[x] if B else None) == (A[y], B[y] if B else None):
        y += 1
    m = 160
    for lane in (0, 31, 32, 127):
        A2 = [A[x]] * m; A2[lane] = A[y]
        B2 = None if B is None else [B[x]] * m
        if B2 is not None:
            B2[lane] = B[y]
        got = run(Z, op, A2, B2)
        assert got[lane] == out[y] and all(got[i] == out[x] for i in range(m) if i != lane), (op, lane)


@pytest.mark.parametrize("op", LAZY_OPS)
def test_stale_shared_memory(Z, op):
    """The slots are not cleared between launches: op X on a batch right after another op on unrelated data gives the bytes of its first run."""
    A, B = inputs(op, 300, 4100 + op)
    first = run(Z, op, A, B)
    for other in (24, 26, 16 if op != 16 else 17):
        if other == op:
            continue
        C, D = inputs(other, 300, 4200 + other)
        if other != 26:
            C = [b"".join(w32(P - 1) for _ in range(12))] * 150 + C[150:]
        run(Z, other, C, D)
        assert run(Z, op, A, B) == first, (op, other)
