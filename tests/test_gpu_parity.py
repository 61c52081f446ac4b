"""Parity tests proper: the sm_100a path, called through the C ABI (ctypes mirror in the package), against
the CPU oracle on the same seeded inputs, the reference's golden fixtures, and size-independent properties."""
import numpy as np
import pytest

import oracle_lib as O
from conftest import oracle_vk

pytestmark = pytest.mark.gpu

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
G1 = w32(1) + w32(2)


@pytest.fixture(scope="module")
def Z():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import stylus_zkvm_verifiers_b200 as Z
    return Z


@pytest.fixture(scope="module")
def gpu(Z):
    return Z.GpuBackend(0)


def test_fp_mul(Z):
    from stylus_zkvm_verifiers_b200.synth import SplitMix64
    rng = SplitMix64(1)
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, (1 << 256) % P, 1 << 253]
    pairs = [(x, y) for x in edge for y in edge] + [(rng.u256() % P, rng.u256() % P) for _ in range(20000)]
    a = b"".join(w32(x) for x, _ in pairs); b = b"".join(w32(y) for _, y in pairs)
    out = Z.fp_mul_batch(a, b, len(pairs)).tobytes()
    for i, (x, y) in enumerate(pairs):
        assert out[32 * i:32 * i + 32] == w32(x * y % P), (hex(x), hex(y))


def test_fp12_tower_ops(Z):
    """Every Fp12 routine the pairing kernels are built from, against the oracle's tower (bit-exact, 12 x BE-32)."""
    from stylus_zkvm_verifiers_b200.synth import SplitMix64
    rng = SplitMix64(12)
    n = 200                                           # more than one block: the routines rendezvous block-wide
    rnd12 = lambda: b"".join(w32(rng.u256() % P) for _ in range(12))
    one = w32(1) + bytes(352)
    A = [rnd12() for _ in range(n)]; B = [rnd12() for _ in range(n)]
    A[0] = one; B[1] = one; A[2] = b"".join(w32(P - 1) for _ in range(12)); B[2] = A[2]; A[3] = bytes(384)
    a, b = b"".join(A), b"".join(B)
    mul = Z.fp12_op_batch(0, a, b, n)
    sqr = Z.fp12_op_batch(1, a, None, n)
    inv = Z.fp12_op_batch(4, a, None, n)
    for i in range(n):
        assert mul[384 * i:384 * i + 384] == O.fp12_mul(A[i], B[i]), ("mul", i)
        assert sqr[384 * i:384 * i + 384] == O.fp12_mul(A[i], A[i]), ("sqr", i)
        if i != 3:
            assert O.fp12_mul(A[i], inv[384 * i:384 * i + 384]) == one, ("inv", i)
    # sparse line product: a * (l0 + l3 w + l4 v w) == a * dense(l0,0,0 | l3,l4,0)
    L = [B[i][:192] for i in range(n)]
    dense = [L[i][0:64] + bytes(128) + L[i][64:192] + bytes(64) for i in range(n)]
    line = Z.fp12_op_batch(2, a, b"".join(L[i] + bytes(192) for i in range(n)), n)
    for i in range(n):
        assert line[384 * i:384 * i + 384] == O.fp12_mul(A[i], dense[i]), ("line", i)
    # Frobenius: x^(p^k) for k = 1, 2, 3 must be multiplicative and frob1 o frob1 = frob2, frob1 o frob2 = frob3
    f1 = Z.fp12_op_batch(5, a, None, n); f2 = Z.fp12_op_batch(6, a, None, n); f3 = Z.fp12_op_batch(7, a, None, n)
    assert Z.fp12_op_batch(5, f1, None, n) == f2 and Z.fp12_op_batch(5, f2, None, n) == f3
    fm = Z.fp12_op_batch(5, mul, None, n); fb = Z.fp12_op_batch(5, b, None, n)
    assert Z.fp12_op_batch(0, f1, fb, n) == fm
    # final exponentiation and cyclotomic squaring (on elements of the cyclotomic subgroup = final-exponentiation outputs)
    m = 64
    fe = Z.fp12_op_batch(8, a[:384 * m], None, m)
    cs = Z.fp12_op_batch(3, fe, None, m)
    for i in range(4, m):
        g = O.final_exp(A[i])
        assert fe[384 * i:384 * i + 384] == g, ("final_exp", i)
        assert cs[384 * i:384 * i + 384] == O.fp12_cyc_sqr(g) == O.fp12_mul(g, g), ("cyc_sqr", i)


def test_single_pair_miller_loop_hook(Z, gpu):
    """Miller loop of one (P, Q) pair with a variable Q, bit-exact against the oracle (the variable-pair code path on its own: doubling
    and addition steps on the fly plus the two Frobenius lines; this is the path a compiler stack-slot bug once broke, DESIGN.md 5)."""
    ks = [(5, 9), (77, 31), (12345, 999), (R - 1, 2), (3, R - 2)]
    ps = gpu.g1_mul([k for k, _ in ks]); qs = gpu.g2_mul([k for _, k in ks])
    n = len(ks)
    got = Z.fp12_op_batch(9, bytes(384 * n), b"".join(p + q + bytes(192) for p, q in zip(ps, qs)), n)
    for i, (p, q) in enumerate(zip(ps, qs)):
        assert got[384 * i:384 * i + 384] == O.ec_pairing(p + q, debug=True)[1], i


def test_ec_add_mul_services(Z):
    from stylus_zkvm_verifiers_b200.synth import SplitMix64
    rng = SplitMix64(2)
    pts = [G1, bytes(64), O.g1_mul(G1, 5), O.g1_mul(G1, R - 5), w32(1) + w32(3), w32(P) + w32(2), w32(1) + w32(P + 2)] + [O.g1_mul(G1, rng.fr()) for _ in range(8)]
    adds = [a + b for a in pts for b in pts]
    out, rev = Z.ec_add_batch(b"".join(adds), len(adds)); out = out.tobytes()
    for i, d in enumerate(adds):
        want = O.ec_add(d)
        assert (rev[i] == 1) == (want is None)
        assert out[64 * i:64 * i + 64] == (want or bytes(64))
    scal = [0, 1, 2, R - 1, R, R + 1, (1 << 256) - 1] + [rng.u256() for _ in range(6)]
    muls = [p + w32(s) for p in pts for s in scal]
    out, rev = Z.ec_mul_batch(b"".join(muls), len(muls)); out = out.tobytes()
    for i, d in enumerate(muls):
        want = O.ec_mul(d)
        assert (rev[i] == 1) == (want is None)
        assert out[64 * i:64 * i + 64] == (want or bytes(64))


def test_g2_mul_and_subgroup_check(Z):
    from stylus_zkvm_verifiers_b200.synth import G2_GEN, SplitMix64, random_twist_point
    rng = SplitMix64(3)
    ks = [1, 2, R - 1, R, rng.fr(), rng.fr(), rng.u256()]
    out, rev = Z.g2_mul_batch(G2_GEN, b"".join(w32(k) for k in ks), len(ks), broadcast=True); out = out.tobytes()
    assert not rev.any()
    sub = []
    for i, k in enumerate(ks):
        assert out[128 * i:128 * i + 128] == O.g2_mul(G2_GEN, k)
        sub.append(out[128 * i:128 * i + 128])
    wrong = [random_twist_point(rng) for _ in range(12)]
    mixed = [O.g2_add(wq, O.g2_mul(G2_GEN, rng.fr())) for wq in wrong[:4]]
    bad = bytearray(G2_GEN); bad[77] ^= 8
    pts = sub + wrong + mixed + [bytes(128), bytes(bad), w32(P) + G2_GEN[32:]]
    got = Z.g2_check_batch(b"".join(pts), len(pts))
    want = [1] * len(sub) + [0] * (len(wrong) + len(mixed)) + [1, 2, 2]
    assert list(got) == want
    # multiples of a wrong-subgroup point through the hook agree with the oracle as well
    out, rev = Z.g2_mul_batch(b"".join(wrong[:4]), b"".join(w32(k) for k in ks[:4]), 4); out = out.tobytes()
    for i in range(4):
        assert out[128 * i:128 * i + 128] == O.g2_mul(wrong[i], ks[i])


def test_pairing4_fp12_bit_exact(Z, gpu):
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 2, 5)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    n = 96
    g1s, g2s, expect = S.make_pairing4_batch(gpu, vk, n, 0xB2000005, pool=16)
    # edge instances: infinity members, invalid points
    g1s[0] = bytes(64) + g1s[0][64:]; g2s[1] = bytes(128); g1s[2] = g1s[2][:64] + bytes(64) + g1s[2][128:]
    g1s[3] = w32(1) + w32(3) + g1s[3][64:]; g2s[4] = S.random_twist_point(S.SplitMix64(9)); g1s[5] = g1s[5][:192] + w32(P) + w32(0)
    ok, gt, ml = Z.pairing4_batch(kv, b"".join(g1s), b"".join(g2s), n, want_gt=True, want_miller=True)
    blob = b"".join(g1s[i][0:64] + g2s[i] + g1s[i][64:128] + vk.beta + g1s[i][128:192] + vk.gamma + g1s[i][192:256] + vk.delta for i in range(n))
    ook, ogt, oml = O.pairing4_batch(blob, n, want_gt=True, want_miller=True)
    assert list(ok) == list(ook)
    assert list(ok[3:6]) == [2, 2, 2]
    for i in range(n):
        if ook[i] != 2:
            assert ml[384 * i:384 * i + 384].tobytes() == oml[384 * i:384 * i + 384].tobytes(), i
            assert gt[384 * i:384 * i + 384].tobytes() == ogt[384 * i:384 * i + 384].tobytes(), i
    assert list(ok[6:]) == expect[6:]


def test_vk_x_matches_precompile_chain(Z, gpu):
    from stylus_zkvm_verifiers_b200 import synth as S
    rng = S.SplitMix64(21)
    vk = S.make_vk(gpu, 0, 6, 21)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    sigs = [[rng.fr() for _ in range(5)] for _ in range(20)] + [[0] * 5, [R - 1] * 5, [1, 0, 0, 0, 0], [0, 0, (1 << 128) - 1, 1 << 127, 7]]
    # a signal vector whose vk_x is the point at infinity: s0 = -(ic0 + ...)/ic1
    t = vk.trap["ic"]
    s = [0, 3, 5, 7, 11]; s[0] = (-(t[0] + sum(a * b for a, b in zip(s[1:], t[2:])))) * pow(t[1], -1, R) % R
    sigs.append(s)
    out = Z.vk_x_batch(kv, b"".join(w32(v) for sg in sigs for v in sg), 5, len(sigs)).tobytes()
    for i, sg in enumerate(sigs):
        acc = vk.ic[0]
        for j in range(5):
            acc = O.ec_add(acc + O.ec_mul(vk.ic[j + 1] + w32(sg[j])))
        assert out[64 * i:64 * i + 64] == acc, i
    assert out[-64:] == bytes(64)


def test_reference_fixtures_through_the_mirror(Z, fx):
    E = Z.errors
    v = Z.RiscZeroVerifier()
    seal, im, jd = fx["seal"], fx["image_id"], fx["journal_digest"]
    assert not v.is_initialized() and v.get_selector() == bytes(4)
    with pytest.raises(E.InvalidInitialization):
        v.verify(seal, im, jd)
    v.initialize(fx["control_root"], fx["bn254_control_id"])
    with pytest.raises(E.AlreadyInitialized):
        v.initialize(fx["control_root"], fx["bn254_control_id"])
    assert v.is_initialized() and v.get_selector().hex() == "9f39696c"
    assert v.get_verifier_key_digest().hex() == "21c5fdd9b4d576b17581f50b755482ba7a2134a3b5186e8e454acfa1f69511ab"
    assert v.get_bn254_control_id() == fx["bn254_control_id"]
    c0, c1 = v.get_control_root()
    assert int.from_bytes(c0, "big") == 0x4c2d7bb17348241967b0276818329053 and int.from_bytes(c1, "big") == 0x7645843b52b258e94f99b1cf022d2e12
    assert v.verify(seal, im, jd) is True
    assert v.verify_integrity(seal, O.claim_digest(im, jd)) is True
    flip = lambda b, i: b[:i] + bytes([b[i] ^ 1]) + b[i + 1:]
    with pytest.raises(E.VerificationFailed):
        v.verify(seal, flip(im, 3), jd)
    with pytest.raises(E.VerificationFailed):
        v.verify(flip(seal, 100), im, jd)
    with pytest.raises(E.SelectorMismatch) as ei:
        v.verify(flip(seal, 1), im, jd)
    assert ei.value.received == flip(seal, 1)[:4] and ei.value.expected == seal[:4]
    for bad in (b"", seal[:3], seal[:200], seal + b"\0"):
        with pytest.raises(E.InvalidProofData):
            v.verify(bad, im, jd)
    s = Z.Sp1Verifier()
    assert s.version() == "v5.0.0" and s.verifier_hash()[:4].hex() == "a4594c59"
    assert s.verify_proof(fx["sp1_vkey"], fx["sp1_public_values"], fx["sp1_proof"]) is None
    with pytest.raises(E.VerificationFailed):
        s.verify_proof(fx["sp1_vkey"], flip(fx["sp1_public_values"], 95), fx["sp1_proof"])
    with pytest.raises(E.VerificationFailed):
        s.verify_proof(w32(R), fx["sp1_public_values"], fx["sp1_proof"])
    with pytest.raises(E.WrongVerifierSelector):
        s.verify_proof(fx["sp1_vkey"], fx["sp1_public_values"], flip(fx["sp1_proof"], 0))
    with pytest.raises(E.InvalidProofData):
        s.verify_proof(fx["sp1_vkey"], fx["sp1_public_values"], fx["sp1_proof"][:259])
    # empty and ragged public values
    for pv in (b"", b"\x01", bytes(55), bytes(56), bytes(64), bytes(119), bytes(120), bytes(1000)):
        st = s.verify_batch([fx["sp1_vkey"]], [pv], [fx["sp1_proof"]])
        assert st[0] == O.sp1_verify(O.sp1_vk(), fx["sp1_selector"], fx["sp1_vkey"], pv, fx["sp1_proof"])


def test_negate_quirk_and_bn254_id_range(Z, fx):
    v = Z.RiscZeroVerifier(); v.initialize(fx["control_root"], fx["bn254_control_id"])
    ro = O.Risc0Oracle(); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    seal, im, jd = fx["seal"], fx["image_id"], fx["journal_digest"]
    variants = [seal[:4] + bytes(64) + seal[68:], seal[:4] + w32(0) + w32(P) + seal[68:], seal[:36] + w32(0) + seal[68:],
                seal[:36] + w32(P) + seal[68:], seal[:4] + w32(P) + seal[36:], seal[:68] + bytes(128) + seal[196:], seal[:196] + bytes(64)]
    st = v.verify_batch(variants, [im] * len(variants), [jd] * len(variants))
    assert list(st) == [ro.verify(s, im, jd) for s in variants]
    big = Z.RiscZeroVerifier(); big.initialize(fx["control_root"], w32(R))           # bn254_control_id >= R: every proof fails (groth16.rs:32-34)
    ob = O.Risc0Oracle(); ob.initialize(fx["control_root"], w32(R))
    s2 = ob.selector() + seal[4:]
    assert big.get_selector() == ob.selector()
    assert big.verify_batch([s2], [im], [jd])[0] == ob.verify(s2, im, jd) == O.ST_VERIFICATION_FAILED


@pytest.mark.parametrize("seed", [0xB2000001, 0xB2000004])
def test_risc0_shape_mixed_batch_vs_oracle(Z, gpu, fx, seed):
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB2000001)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    ro = O.Risc0Oracle(oracle_vk(vk)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    assert v.get_selector() == ro.selector() and v.get_verifier_key_digest() == ro.vk_digest()
    n = 768
    batch = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, seed, pool=64)
    assert (v.verify_batch(batch.seals, batch.image_ids, batch.journals) == 0).all()
    claims = [O.claim_digest(batch.image_ids[i], batch.journals[i]) for i in range(n)]
    assert (v.verify_integrity_batch(batch.seals, claims) == 0).all()
    rng = S.SplitMix64(seed ^ 0x55)
    S.mutate_risc0(batch, gpu, rng, S.Pools(gpu, rng, 16))
    got = v.verify_batch(batch.seals, batch.image_ids, batch.journals)
    want = ro.verify_batch(batch.seals, batch.image_ids, batch.journals)
    bad = [(i, batch.classes[i], int(got[i]), int(want[i])) for i in range(n) if got[i] != want[i]]
    assert not bad, bad[:10]
    for i in range(n):
        if batch.expect[i] is not None:
            assert got[i] == batch.expect[i]
    assert len(set(got)) >= 4          # OK, INVALID_PROOF_DATA, SELECTOR_MISMATCH, VERIFICATION_FAILED all occur


def test_normalised_and_unscaled_lines_agree(Z, gpu, fx):
    """The verification path scales the gamma / delta lines by subfield elements (10 instead of 13 Fp2 products per line): every status
    byte must equal both the oracle's and the one obtained with the unscaled lines of the pairing service."""
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB2000009)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    n = 300
    batch = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 0xB2000009, pool=32)
    S.mutate_risc0(batch, gpu, S.SplitMix64(0xB200000A))
    ro = O.Risc0Oracle(oracle_vk(vk)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    want = ro.verify_batch(batch.seals, batch.image_ids, batch.journals)
    assert v.tune("normalised_lines") == 1 and v.tune("layout") == 1          # the defaults; tuning is per key, not process-wide
    a = v.verify_batch(batch.seals, batch.image_ids, batch.journals)          # shared-memory kernels, normalised lines
    v.tune("layout", 0)
    a0 = v.verify_batch(batch.seals, batch.image_ids, batch.journals)         # round-1 kernels, normalised lines
    v.tune("normalised_lines", 0)
    b = v.verify_batch(batch.seals, batch.image_ids, batch.journals)          # round-1 kernels, unscaled lines (the pairing service's loop)
    v.tune("layout", 1)
    b1 = v.verify_batch(batch.seals, batch.image_ids, batch.journals)         # unscaled lines + shared-memory final exponentiation
    assert a.tolist() == want.tolist() and b.tolist() == want.tolist() and a0.tolist() == want.tolist() and b1.tolist() == want.tolist()
    other = Z.RiscZeroVerifier(Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic))
    assert other.tune("normalised_lines") == 1                                # another key handle keeps its own settings
    assert 0 < int((want == 0).sum()) < n


def test_sp1_shape_mixed_batch_vs_oracle(Z, gpu):
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 1, 3, 0xB2000003)
    kv = Z.VerificationKey(1, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.Sp1Verifier(kv)
    ovk = oracle_vk(vk)
    n = 768
    batch = S.make_sp1_batch(gpu, vk, n, 0xB2000003, pool=64)
    for i in range(0, n, 7):                                  # ragged public values
        batch.public_values[i] = batch.public_values[i][: i % 96]
    if True:
        # re-solve the proofs whose public values changed
        rng0 = S.SplitMix64(99); pools = S.Pools(gpu, rng0, 16)
        idx = list(range(0, n, 7))
        sigs = [S.sp1_signals(batch.vkeys[i], batch.public_values[i]) for i in idx]
        prs = S.make_proofs(gpu, vk, sigs, rng0, pools)
        for i, p in zip(idx, prs):
            batch.proofs[i] = S.SP1_SELECTOR + p
    assert (v.verify_batch(batch.vkeys, batch.public_values, batch.proofs) == 0).all()
    rng = S.SplitMix64(0xB2000004)
    S.mutate_sp1(batch, gpu, rng)
    got = v.verify_batch(batch.vkeys, batch.public_values, batch.proofs)
    want = O.sp1_verify_batch(ovk, S.SP1_SELECTOR, batch.vkeys, batch.public_values, batch.proofs)
    bad = [(i, batch.classes[i], int(got[i]), int(want[i])) for i in range(n) if got[i] != want[i]]
    assert not bad, bad[:10]


def test_generic_groth16_and_invalid_keys(Z, gpu):
    from stylus_zkvm_verifiers_b200 import synth as S
    rng = S.SplitMix64(31)
    vk = S.make_vk(gpu, 0, 4, 31)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    n = 40
    sigs = [[rng.fr() for _ in range(3)] for _ in range(n)]
    sigs[5][1] = R; sigs[6][2] = (1 << 256) - 1                 # signal >= R
    prs = S.make_proofs(gpu, vk, [[s % R for s in sg] for sg in sigs], rng, S.Pools(gpu, rng, 8))
    sb = b"".join(w32(v) for sg in sigs for v in sg)
    got = Z.Groth16Verifier.verify_batch(kv, b"".join(prs), sb, 3, n)
    want = O.groth16_verify_batch(oracle_vk(vk), b"".join(prs), sb, n)
    assert list(got) == list(want) and got[5] == got[6] == 4 and got[0] == 0
    # wrong number of signals: groth16.rs:32
    assert (Z.Groth16Verifier.verify_batch(kv, b"".join(prs), sb, 2, n) == 4).all()
    a = [int.from_bytes(prs[0][0:32], "big"), int.from_bytes(prs[0][32:64], "big")]
    b = [[int.from_bytes(prs[0][64:96], "big"), int.from_bytes(prs[0][96:128], "big")], [int.from_bytes(prs[0][128:160], "big"), int.from_bytes(prs[0][160:192], "big")]]
    c = [int.from_bytes(prs[0][192:224], "big"), int.from_bytes(prs[0][224:256], "big")]
    assert Z.Groth16Verifier.verify_proof_with_key(kv, a, b, c, sigs[0]) is True
    assert Z.Groth16Verifier.verify_proof_with_key(kv, a, b, c, sigs[1]) is False
    # a key with an invalid point makes every precompile call revert -> false (groth16.rs:38,106)
    for mod in ("ic", "gamma", "alpha"):
        ic, gamma, alpha = list(vk.ic), vk.gamma, vk.alpha
        if mod == "ic":
            ic[2] = w32(1) + w32(3)
        elif mod == "gamma":
            gamma = S.random_twist_point(S.SplitMix64(4))
        else:
            alpha = w32(P) + w32(1)
        kb = Z.VerificationKey(0, alpha, vk.beta, gamma, vk.delta, ic)
        ob = O.Vk(0, alpha, vk.beta, gamma, vk.delta, ic)
        g = Z.Groth16Verifier.verify_batch(kb, b"".join(prs[:4]), sb[:4 * 96], 3, 4)
        assert list(g) == list(O.groth16_verify_batch(ob, b"".join(prs[:4]), sb[:4 * 96], 4)) == [4] * 4


def test_device_resident_entry_points_match_host_path(Z, gpu, fx):
    import torch
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 41)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    n = 300
    batch = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 41, pool=32)
    rng = S.SplitMix64(42)
    S.mutate_risc0(batch, gpu, rng)
    keep = [i for i in range(n) if len(batch.seals[i]) == 260]     # the device entry point takes fixed 260-byte records
    seals = [batch.seals[i] for i in keep]; ims = [batch.image_ids[i] for i in keep]; jds = [batch.journals[i] for i in keep]
    host = v.verify_batch(seals, ims, jds)
    t = lambda blobs: torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()
    d_s, d_i, d_j = t(seals), t(ims), t(jds)
    d_st = torch.full((len(keep),), 255, dtype=torch.uint8, device="cuda")
    v.verify_batch_device(0, d_s.data_ptr(), d_i.data_ptr(), d_j.data_ptr(), len(keep), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert d_st.cpu().numpy().tolist() == host.tolist()
    assert 3 in host.tolist()


def test_full_size_properties(Z, gpu, fx):
    """BASELINE config-2 size (2^16): all trapdoor proofs accept; the same batch with every journal bit-flipped rejects;
    replicating the reference's real seal accepts everywhere."""
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB2000001)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    n = 1 << 16
    batch = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 0xB2000001, pool=4096)
    st = v.verify_batch(batch.seals, batch.image_ids, batch.journals)
    assert int((st == 0).sum()) == n
    flipped = [bytes([j[0] ^ 0x80]) + j[1:] for j in batch.journals]
    st = v.verify_batch(batch.seals, batch.image_ids, flipped)
    assert int((st == 4).sum()) == n
    real = Z.RiscZeroVerifier(); real.initialize(fx["control_root"], fx["bn254_control_id"])
    m = 4096
    st = real.verify_batch([fx["seal"]] * m, [fx["image_id"]] * m, [fx["journal_digest"]] * m)
    assert int((st == 0).sum()) == m


@pytest.mark.gpu
def test_scale_sp1_mixed_and_pairing(Z, gpu, fx):
    """BASELINE configs 3-5 at a size that exercises several waves and the stream-overlap chunks (2^16 SP1-shape proofs, a 2^16 mixed
    RISC Zero-shape batch, 2^15 pairing instances).  Full batches are checked through what the generator knows by construction (valid
    proofs accept, every mutated class rejects); a 2048-element prefix is compared 1:1 with the oracle, Fp12 values included."""
    from stylus_zkvm_verifiers_b200 import synth as S
    sub = 2048
    # config 3: SP1 shape, all valid
    vk = S.make_vk(gpu, 1, 3, 0xB2000003)
    kv = Z.VerificationKey(1, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.Sp1Verifier(kv)
    n = 1 << 16
    b = S.make_sp1_batch(gpu, vk, n, 0xB2000003, pool=2048)
    st = v.verify_batch(b.vkeys, b.public_values, b.proofs)
    assert int((st == 0).sum()) == n
    # config 4 (SP1 flavour): mixed classes; expect[] is what the mutation guarantees, the oracle decides the prefix
    S.mutate_sp1(b, gpu, S.SplitMix64(0xB2000004))
    st = v.verify_batch(b.vkeys, b.public_values, b.proofs)
    for i in range(n):
        if b.expect[i] is not None:
            assert st[i] == b.expect[i], (i, b.classes[i], int(st[i]))
    want = O.sp1_verify_batch(oracle_vk(vk), S.SP1_SELECTOR, b.vkeys[:sub], b.public_values[:sub], b.proofs[:sub])
    assert st[:sub].tolist() == want.tolist()
    assert {"valid", "tampered", "off_curve", "wrong_subgroup", "infinity", "malformed"} <= set(b.classes)
    # config 4 (RISC Zero flavour)
    vk0 = S.make_vk(gpu, 0, 6, 0xB2000001)
    kv0 = Z.VerificationKey(0, vk0.alpha, vk0.beta, vk0.gamma, vk0.delta, vk0.ic)
    r = Z.RiscZeroVerifier(kv0); r.initialize(fx["control_root"], fx["bn254_control_id"])
    b0 = S.make_risc0_batch(gpu, vk0, r.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 0xB2000004, pool=2048)
    S.mutate_risc0(b0, gpu, S.SplitMix64(0xB2000004))
    st0 = r.verify_batch(b0.seals, b0.image_ids, b0.journals)
    for i in range(n):
        if b0.expect[i] is not None:
            assert st0[i] == b0.expect[i], (i, b0.classes[i], int(st0[i]))
    ro = O.Risc0Oracle(oracle_vk(vk0)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    assert st0[:sub].tolist() == ro.verify_batch(b0.seals[:sub], b0.image_ids[:sub], b0.journals[:sub]).tolist()
    # config 5: pairing service, ok bits for all, Fp12 values on the prefix
    m = 1 << 15
    g1s, g2s, expect = S.make_pairing4_batch(gpu, vk0, m, 0xB2000005, pool=1024)
    ok, gt, ml = Z.pairing4_batch(kv0, b"".join(g1s), b"".join(g2s), m, want_gt=True, want_miller=True)
    assert ok.tolist() == expect
    blob = b"".join(g1s[i][0:64] + g2s[i] + g1s[i][64:128] + vk0.beta + g1s[i][128:192] + vk0.gamma + g1s[i][192:256] + vk0.delta for i in range(sub))
    ook, ogt, oml = O.pairing4_batch(blob, sub, want_gt=True, want_miller=True)
    assert ok[:sub].tolist() == list(ook) and bytes(gt[:384 * sub]) == bytes(ogt) and bytes(ml[:384 * sub]) == bytes(oml)


def test_segmented_miller_loop_matches(Z, gpu, fx):
    """The verification Miller loop run as 2, 4 and 7 segment kernels (state carried in HBM) gives the same status bytes as the single
    kernel and as the oracle, on a mixed batch large enough to be cut into stream chunks."""
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB200000B)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    n = 9000
    batch = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 0xB200000B, pool=64)
    S.mutate_risc0(batch, gpu, S.SplitMix64(0xB200000C))
    ro = O.Risc0Oracle(oracle_vk(vk)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    sub = 600
    want = ro.verify_batch(batch.seals[:sub], batch.image_ids[:sub], batch.journals[:sub])
    for layout in (1, 0):                                  # shared-memory kernels (default), round-1 kernels
        v.tune("layout", layout)
        v.tune("miller_segments", 1)
        base = v.verify_batch(batch.seals, batch.image_ids, batch.journals)
        assert base[:sub].tolist() == want.tolist(), layout
        for segs in (2, 4, 7):
            v.tune("miller_segments", segs)
            assert v.verify_batch(batch.seals, batch.image_ids, batch.journals).tolist() == base.tolist(), (layout, segs)
        for fe in (0, 1):                                  # one-kernel / staged final exponentiation
            v.tune("final_exp_stages", fe)
            assert v.verify_batch(batch.seals, batch.image_ids, batch.journals).tolist() == base.tolist(), (layout, "fe", fe)


@pytest.mark.gpu
def test_launch_counter_and_wave_size(Z, gpu, fx):
    """zkv_launch_count counts every kernel of the verification chains (bench.py's gpu_launches); zkv_wave_proofs is SMs x resident blocks
    x 128 threads: two blocks per SM for the shared-memory Miller / final-exponentiation kernels, three / two for the round-1 kernels."""
    import torch
    from stylus_zkvm_verifiers_b200 import synth as S
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert Z.wave_proofs(0, 0) == sms * 2 * 128 and Z.wave_proofs(0, 1) == sms * 2 * 128
    assert Z.wave_proofs(0, 2) == sms * 3 * 128 and Z.wave_proofs(0, 3) == sms * 2 * 128
    vk = S.make_vk(gpu, 0, 6, 0xB200000D)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    small = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], 64, 0xB200000D, pool=8)
    c0 = Z.launch_count()
    assert set(v.verify_batch(small.seals, small.image_ids, small.journals).tolist()) == {0}
    assert Z.launch_count() - c0 == 6                      # one serial chain: decode, signals, vk_x, G2 check, Miller loop, final exponentiation
    n = 8192 + 300
    big = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 0xB200000E, pool=8)
    assert v.tune("overlap") == 0                          # default: automatic: one chain below half a wave (SMs x 128 proofs), four chunks above
    c0 = Z.launch_count()
    assert set(v.verify_batch(big.seals, big.image_ids, big.journals).tolist()) == {0}
    assert Z.launch_count() - c0 == 6
    v.tune("overlap", 4)
    chunks, segs, fe = v.tune("overlap"), v.tune("miller_segments"), v.tune("final_exp_stages")
    c0 = Z.launch_count()
    assert set(v.verify_batch(big.seals, big.image_ids, big.journals).tolist()) == {0}
    per_chain = 4 + segs + (4 if fe else 1)
    assert chunks == 4 and Z.launch_count() - c0 == chunks * per_chain
    v.tune("overlap", 0)
    m = sms * 128 + 1                                      # just over half a wave -> four chunks
    mid = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], m, 0xB200000F, pool=8)
    c0 = Z.launch_count()
    assert set(v.verify_batch(mid.seals, mid.image_ids, mid.journals).tolist()) == {0}
    assert Z.launch_count() - c0 == 4 * per_chain


def test_concurrent_calls_on_shared_and_separate_handles(Z, gpu, fx):
    """SURVEY 8b, threading row: handles are immutable after create and the library serialises the calls of one device, so host threads
    that call one handle (or two handles of different keys) at the same time must each get the oracle's status bytes."""
    import threading
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB2000011)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    ro = O.Risc0Oracle(oracle_vk(vk)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    svk = S.make_vk(gpu, 1, 3, 0xB2000012)
    sv = Z.Sp1Verifier(Z.VerificationKey(1, svk.alpha, svk.beta, svk.gamma, svk.delta, svk.ic))
    jobs = []
    for t in range(3):
        b = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], 200 + 37 * t, 0xB2000013 + t, pool=16)
        S.mutate_risc0(b, gpu, S.SplitMix64(0xB2000020 + t))
        want = ro.verify_batch(b.seals, b.image_ids, b.journals)
        jobs.append((lambda b=b: v.verify_batch(b.seals, b.image_ids, b.journals), want))
    sb = S.make_sp1_batch(gpu, svk, 256, 0xB2000016, pool=16)
    S.mutate_sp1(sb, gpu, S.SplitMix64(0xB2000017))
    jobs.append((lambda: sv.verify_batch(sb.vkeys, sb.public_values, sb.proofs),
                 O.sp1_verify_batch(oracle_vk(svk), S.SP1_SELECTOR, sb.vkeys, sb.public_values, sb.proofs)))
    got, errs = [None] * len(jobs), []

    def run(i):
        try:
            for _ in range(3):
                got[i] = jobs[i][0]()
                assert got[i].tolist() == jobs[i][1].tolist(), "thread %d: status bytes differ from the oracle's" % i
        except Exception as e:                                 # surfaced in the main thread below
            errs.append(e)

    th = [threading.Thread(target=run, args=(i,)) for i in range(len(jobs))]
    [t.start() for t in th]; [t.join() for t in th]
    assert not errs, errs
    assert all(0 < int((w == 0).sum()) < len(w) for _, w in jobs)


def test_general_ec_pairing_service_vs_oracle(Z, gpu):
    """zkv_ec_pairing_batch / zkv_ec_pairing: precompile 0x08 with every G2 point variable (the seam groth16.rs:109-128 calls), k = 0..6
    pairs, against the oracle's zkvo_ec_pairing: return word, failure (revert) and the Miller-loop value bit for bit; products that are
    one by bilinearity, members at infinity, points off the curve / twist, coordinates >= p, G2 points outside the subgroup, bad lengths."""
    from stylus_zkvm_verifiers_b200 import synth as S
    rng = S.SplitMix64(0xB2000041)
    G1, G2 = S.G1_GEN, S.G2_GEN
    neg = lambda p: p[:32] + O.w32((P - int.from_bytes(p[32:], "big")) % P)
    wrong = S.random_twist_point(rng)

    def pairs(k, kind):
        """k pairs; kind: 'one' product is 1 by construction, 'rand' random, plus mutations"""
        ps = []
        if kind == "one" and k >= 2:
            tot = 0
            for j in range(k - 1):
                a, b = rng.fr(), rng.fr(); tot = (tot + a * b) % R
                ps.append(O.g1_mul(G1, a) + O.g2_mul(G2, b))
            ps.append(neg(O.g1_mul(G1, tot)) + G2)
        else:
            ps = [O.g1_mul(G1, rng.fr()) + O.g2_mul(G2, rng.fr()) for _ in range(k)]
        return ps
    for k in range(0, 7):
        n = 24
        inst = []
        for i in range(n):
            ps = pairs(k, "one" if i % 2 == 0 else "rand")
            if k:
                j = rng.below(k)
                m = i % 12
                if m == 3: ps[j] = bytes(64) + ps[j][64:]                       # G1 at infinity: the pair contributes 1
                elif m == 5: ps[j] = ps[j][:64] + bytes(128)                    # G2 at infinity
                elif m == 7: ps[j] = O.w32(1) + O.w32(3) + ps[j][64:]           # G1 off the curve -> the call fails
                elif m == 9: ps[j] = ps[j][:64] + wrong                         # G2 on the twist, outside the subgroup -> fails
                elif m == 10: ps[j] = ps[j][:64] + O.w32(P) + ps[j][96:]        # coordinate >= p -> fails
                elif m == 11: b = bytearray(ps[j]); b[191] ^= 1; ps[j] = bytes(b)   # G2 off the twist -> fails
            inst.append(b"".join(ps))
        words, rev, ml = Z.ec_pairing_batch(b"".join(inst), k, n, want_miller=True)
        for i in range(n):
            ret = O.ec_pairing(inst[i], debug=True) if k else (O.ec_pairing(b""), None, None)
            want = ret[0] if isinstance(ret, tuple) else ret
            if want is None:
                assert rev[i] == 1 and not words[32 * i:32 * i + 32].any(), (k, i)
            else:
                assert rev[i] == 0 and bytes(words[32 * i:32 * i + 32]) == want, (k, i)
                if k:
                    assert bytes(ml[384 * i:384 * i + 384]) == ret[1], (k, i, "Miller value")
        if k >= 2:
            assert any(bytes(words[32 * i:32 * i + 32])[31] == 1 for i in range(n)) and any(rev)
    one = O.w32(1)
    assert Z.ec_pairing(b"") == one and Z.ec_pairing(G1 + bytes(128)) == one and Z.ec_pairing(G1 + G2) == O.w32(0)
    assert Z.ec_pairing((G1 + G2)[:-1]) is None and Z.ec_pairing(G1 + G2 + neg(G1) + G2) == one


def test_one_handle_across_all_devices_matches_one_device(Z, gpu, fx):
    """North star: 'partitioned across the GPUs ... results gathered on the host'.  ONE handle created over devices [0..N-1] splits a mixed
    batch call into contiguous ranges (for_each_device in csrc/zkv.cu), one host thread per device, and gathers the status bytes; they must
    equal the single-device handle's bytes everywhere and the oracle's on a prefix and on the range boundaries.  Skipped on a 1-GPU box."""
    import torch
    nd = Z.device_count() if hasattr(Z, "device_count") else torch.cuda.device_count()
    if nd < 2:
        pytest.skip("needs at least two CUDA devices")
    from stylus_zkvm_verifiers_b200 import synth as S
    devs = list(range(nd))
    n = 1 << 17
    for shape in ("risc0", "sp1"):
        if shape == "risc0":
            vk = S.make_vk(gpu, 0, 6, 0xB2000001)
            mk = lambda d: Z.RiscZeroVerifier(Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, devices=d), devices=d)
            one, many = mk([0]), mk(devs)
            for v in (one, many):
                v.initialize(fx["control_root"], fx["bn254_control_id"])
            b = S.make_risc0_batch(gpu, vk, one.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, 0xB2000021, pool=512)
            S.mutate_risc0(b, gpu, S.SplitMix64(0xB2000022))
            run = lambda v: v.verify_batch(b.seals, b.image_ids, b.journals)
            ro = O.Risc0Oracle(oracle_vk(vk)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
            oracle = lambda idx: ro.verify_batch([b.seals[i] for i in idx], [b.image_ids[i] for i in idx], [b.journals[i] for i in idx])
        else:
            vk = S.make_vk(gpu, 1, 3, 0xB2000003)
            mk = lambda d: Z.Sp1Verifier(Z.VerificationKey(1, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, devices=d), devices=d)
            one, many = mk([0]), mk(devs)
            b = S.make_sp1_batch(gpu, vk, n, 0xB2000023, pool=512)
            S.mutate_sp1(b, gpu, S.SplitMix64(0xB2000024))
            run = lambda v: v.verify_batch(b.vkeys, b.public_values, b.proofs)
            ovk = oracle_vk(vk)
            oracle = lambda idx: O.sp1_verify_batch(ovk, S.SP1_SELECTOR, [b.vkeys[i] for i in idx], [b.public_values[i] for i in idx], [b.proofs[i] for i in idx])
        a, m = np.asarray(run(one)), np.asarray(run(many))
        assert a.shape == m.shape == (n,) and (a == m).all(), (shape, int((a != m).sum()))
        idx = list(range(512))
        for d in range(1, nd):                      # both sides of every device-range boundary
            cut = n * d // nd
            idx += list(range(cut - 32, cut + 32))
        want = np.asarray(oracle(idx))
        assert (m[idx] == want).all(), shape
        assert 0 < int((m == 0).sum()) < n and len(set(m.tolist())) >= 3


def test_campaign_batches_match_committed_oracle_digests(Z, gpu, consts):
    """Two batches of the round-2 exactness campaign (2^16 mixed proofs each, one per proof shape) rebuilt from their seeds and verified
    through the C ABI: the status bytes must hash to what the CPU oracle produced for the same batch (profiles/r2_campaign_oracle_digests.json,
    written by tools/campaign_oracle.py from 10 092 544 oracle-verified proofs); the input fingerprints must agree as well."""
    import hashlib, json, os, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "tools"))
    import campaign_common as CC
    dg = {b["k"]: b for b in json.load(open(os.path.join(root, "profiles", "r2_campaign_oracle_digests.json")))["batches"]}
    h = bytes.fromhex; r = consts["risc0_fixture"]
    vk0, vk1 = CC.keys(gpu)
    v0 = Z.RiscZeroVerifier(Z.VerificationKey(0, vk0.alpha, vk0.beta, vk0.gamma, vk0.delta, vk0.ic)); v0.initialize(h(r["control_root"]), h(r["bn254_control_id"]))
    v1 = Z.Sp1Verifier(Z.VerificationKey(1, vk1.alpha, vk1.beta, vk1.gamma, vk1.delta, vk1.ic))
    for k in (0, 1):
        shape, b, fpr = CC.batch(gpu, k, vk0, vk1, v0.get_selector(), consts, CC.BATCH)
        st = v0.verify_batch(b.seals, b.image_ids, b.journals) if shape == "risc0" else v1.verify_batch(b.vkeys, b.public_values, b.proofs)
        st = np.asarray(st, dtype=np.uint8)
        assert fpr == dg[k]["fingerprint"] and shape == dg[k]["shape"]
        assert int((st == 0).sum()) == dg[k]["accepted"]
        assert hashlib.sha256(st.tobytes()).hexdigest() == dg[k]["status_sha256"], k


def test_large_batch_schedules_agree(Z, gpu, fx):
    """Large batches through every schedule the library has (csrc/zkv.cu chunk_count, run_verify, host_pipeline): a mixed 6.4-wave batch
    through (a) the host-buffer call (automatic: four chunks, fronts first), (b) the device-resident call, (c) the same with page-locked
    inputs uploaded in place, (d) a forced 7-chunk host call (more pieces than side streams) and (e) a forced single chain must give the same
    status bytes, equal to the generator's expectation everywhere and to the oracle on a sample; a 2.5-wave batch as well."""
    import torch
    from stylus_zkvm_verifiers_b200 import synth as S
    wave = Z.wave_proofs(0, 0)
    vk = S.make_vk(gpu, 0, 6, 0xB2000001)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    ro = O.Risc0Oracle(oracle_vk(vk)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    for n, seed in ((6 * wave + (2 * wave) // 5 + 37, 0xB2000041), (2 * wave + wave // 2 + 5, 0xB2000043)):
        b = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, seed, pool=512)
        S.mutate_risc0(b, gpu, S.SplitMix64(seed + 1))
        for i in range(n):                               # the device entry point takes fixed 260-byte records: keep malformed lengths out
            if len(b.seals[i]) != 260:
                b.seals[i] = (b.seals[i] + bytes(260))[:260]; b.expect[i] = None
        assert v.tune("overlap") == 0
        host = np.asarray(v.verify_batch(b.seals, b.image_ids, b.journals))
        t = lambda blobs: torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()
        d_s, d_i, d_j = t(b.seals), t(b.image_ids), t(b.journals)
        d_st = torch.full((n,), 255, dtype=torch.uint8, device="cuda")
        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            v.verify_batch_device(0, d_s.data_ptr(), d_i.data_ptr(), d_j.data_ptr(), n, d_st.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        dev = d_st.cpu().numpy()
        # the same call with every input array in page-locked memory: uploaded in place, no staging pass (include/zkv.h zkv_host_alloc)
        pin = [Z.pinned_copy(np.frombuffer(b"".join(x), dtype=np.uint8)) for x in (b.seals, b.image_ids, b.journals)]
        poff = Z.pinned_copy(np.arange(n + 1, dtype=np.uint64) * 260)
        pinned = np.asarray(v.verify_batch_packed(pin[0], poff, pin[1], pin[2], n))
        assert (host == pinned).all()
        v.tune("overlap", 7); forced4 = np.asarray(v.verify_batch(b.seals, b.image_ids, b.journals))
        v.tune("overlap", 1); serial = np.asarray(v.verify_batch(b.seals, b.image_ids, b.journals))
        v.tune("overlap", 0)
        assert (host == dev).all() and (host == forced4).all() and (host == serial).all(), n
        bad = [i for i in range(n) if b.expect[i] is not None and host[i] != b.expect[i]]
        assert not bad, bad[:10]
        idx = list(range(64)) + list(range(n - 64, n)) + [wave * k + d for k in range(1, n // wave + 1) for d in (-1, 0, 1) if wave * k + d < n]
        want = ro.verify_batch([b.seals[i] for i in idx], [b.image_ids[i] for i in idx], [b.journals[i] for i in idx])
        assert host[idx].tolist() == np.asarray(want).tolist()
        assert 0 < int((host == 0).sum()) < n and len(set(host.tolist())) >= 3


def test_async_device_calls_share_the_workspace_safely(Z, gpu, fx):
    """ADVICE round 1: the *_device entry points return before their kernels finish and share one workspace per key and device.  A device call
    on stream X followed immediately by a host batch call on the same key, and two device calls on two different streams back to back, must
    each produce their own correct status bytes (the library orders later users of the workspace behind a busy event); a NULL stream means the
    legacy default stream, so work queued there before the call is ordered before it."""
    import torch
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB2000051)
    kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    v = Z.RiscZeroVerifier(kv); v.initialize(fx["control_root"], fx["bn254_control_id"])
    t = lambda blobs: torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()

    def mk(n, seed):
        b = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, seed, pool=64)
        S.mutate_risc0(b, gpu, S.SplitMix64(seed + 7))
        keep = [i for i in range(n) if len(b.seals[i]) == 260]
        return [b.seals[i] for i in keep], [b.image_ids[i] for i in keep], [b.journals[i] for i in keep]
    A, B = mk(9000, 0xB2000052), mk(7000, 0xB2000053)          # > 8192 proofs: A is cut into chunks on side streams
    wantA = np.asarray(v.verify_batch(*A)); wantB = np.asarray(v.verify_batch(*B))
    assert 0 < int((wantA == 0).sum()) < len(wantA) and wantA[:len(wantB)].tolist() != wantB.tolist()
    dA, dB = [t(x) for x in A], [t(x) for x in B]
    for rep in range(3):
        sx, sy = torch.cuda.Stream(), torch.cuda.Stream()
        stA = torch.full((len(wantA),), 255, dtype=torch.uint8, device="cuda"); stB = torch.full((len(wantB),), 255, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        # device call on stream X, then at once a host call on the same key
        v.verify_batch_device(0, dA[0].data_ptr(), dA[1].data_ptr(), dA[2].data_ptr(), len(wantA), stA.data_ptr(), sx.cuda_stream)
        hostB = np.asarray(v.verify_batch(*B))
        sx.synchronize()
        assert hostB.tolist() == wantB.tolist() and stA.cpu().numpy().tolist() == wantA.tolist(), rep
        # two device calls on two streams back to back
        stA.fill_(255); stB.fill_(255); torch.cuda.synchronize()
        v.verify_batch_device(0, dA[0].data_ptr(), dA[1].data_ptr(), dA[2].data_ptr(), len(wantA), stA.data_ptr(), sx.cuda_stream)
        v.verify_batch_device(0, dB[0].data_ptr(), dB[1].data_ptr(), dB[2].data_ptr(), len(wantB), stB.data_ptr(), sy.cuda_stream)
        torch.cuda.synchronize()
        assert stA.cpu().numpy().tolist() == wantA.tolist() and stB.cpu().numpy().tolist() == wantB.tolist(), rep
    # NULL stream = legacy default stream: the fill queued on it before the call must not overwrite the results
    stB = torch.empty((len(wantB),), dtype=torch.uint8, device="cuda")
    with torch.cuda.stream(torch.cuda.default_stream()):
        stB.fill_(255)
        v.verify_batch_device(0, dB[0].data_ptr(), dB[1].data_ptr(), dB[2].data_ptr(), len(wantB), stB.data_ptr(), None)
    torch.cuda.synchronize()
    assert stB.cpu().numpy().tolist() == wantB.tolist()


def test_workspace_growth_under_an_async_device_call(Z, gpu, fx):
    """A device call that has to grow the workspace frees buffers an earlier, still running device call on another stream uses, so it must
    wait for that call first.  On a fresh key handle (empty workspace): a small device call on stream X, at once a chunked one on stream Y
    that grows every workspace buffer, then a still larger pairing-service device call on the same key.  Each must give the host path's
    bytes, taken on a second handle of the same key so that its workspace does not pre-grow the first one's."""
    import torch
    from stylus_zkvm_verifiers_b200 import synth as S
    from stylus_zkvm_verifiers_b200 import _native as N
    vk = S.make_vk(gpu, 0, 6, 0xB2000071)
    kref, kv = [Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic) for _ in range(2)]
    ref, v = Z.RiscZeroVerifier(kref), Z.RiscZeroVerifier(kv)
    for h in (ref, v):
        h.initialize(fx["control_root"], fx["bn254_control_id"])
    t = lambda blobs: torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()

    def mk(n, seed):
        b = S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, seed, pool=64)
        S.mutate_risc0(b, gpu, S.SplitMix64(seed + 7))
        keep = [i for i in range(n) if len(b.seals[i]) == 260]
        return [b.seals[i] for i in keep], [b.image_ids[i] for i in keep], [b.journals[i] for i in keep]
    A, B = mk(300, 0xB2000072), mk(9500, 0xB2000073)
    wantA, wantB = np.asarray(ref.verify_batch(*A)), np.asarray(ref.verify_batch(*B))
    assert len(wantB) > 8192 and 0 < int((wantB == 0).sum()) < len(wantB)
    npair = len(wantB) + 2000
    g1s, g2s, _ = S.make_pairing4_batch(gpu, vk, npair, 0xB2000074, pool=16)
    wantP = Z.pairing4_batch(kref, b"".join(g1s), b"".join(g2s), npair)[0]
    assert 0 < int((wantP == 1).sum()) < npair
    dA, dB, dg1, dg2 = [t(x) for x in A], [t(x) for x in B], t(g1s), t(g2s)
    sx, sy = torch.cuda.Stream(), torch.cuda.Stream()
    stA = torch.full((len(wantA),), 255, dtype=torch.uint8, device="cuda"); stB = torch.full((len(wantB),), 255, dtype=torch.uint8, device="cuda")
    okP = torch.full((npair,), 255, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    v.verify_batch_device(0, dA[0].data_ptr(), dA[1].data_ptr(), dA[2].data_ptr(), len(wantA), stA.data_ptr(), sx.cuda_stream)
    v.verify_batch_device(0, dB[0].data_ptr(), dB[1].data_ptr(), dB[2].data_ptr(), len(wantB), stB.data_ptr(), sy.cuda_stream)
    N.check(N.lib().zkv_pairing4_batch_device(kv._h, 0, dg1.data_ptr(), dg2.data_ptr(), npair, okP.data_ptr(), None, sx.cuda_stream))
    torch.cuda.synchronize()
    assert stA.cpu().numpy().tolist() == wantA.tolist()
    assert stB.cpu().numpy().tolist() == wantB.tolist()
    assert okP.cpu().numpy().tolist() == wantP.tolist()


def test_staging_copy_covers_every_byte(Z, gpu, fx):
    """Regression (round 2): large blocks are gathered into the pinned staging buffer by several copy threads; slicing by floor(n / parts)
    once left the last n mod parts bytes of a chunk's seal blob uncopied whenever floor(n / parts) was a multiple of 64 - five valid proofs in
    the 10^7-proof campaign came back rejected, caught by the committed oracle digests.  Here chunk 0's blob is 16384 x 260 + 1 bytes (one seal
    a byte too long), i.e. exactly that case, and the staging buffer is dirtied by a different batch first."""
    from stylus_zkvm_verifiers_b200 import synth as S
    vk = S.make_vk(gpu, 0, 6, 0xB2000001)
    v = Z.RiscZeroVerifier(Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)); v.initialize(fx["control_root"], fx["bn254_control_id"])
    n = 1 << 16
    mk = lambda seed: S.make_risc0_batch(gpu, vk, v.get_selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], n, seed, pool=256)
    dirty, b = mk(0xB2000061), mk(0xB2000062)
    assert (np.asarray(v.verify_batch(dirty.seals, dirty.image_ids, dirty.journals)) == 0).all()
    for odd in (5, 16384 + 9, 3 * 16384 + 1):              # one over-long seal in chunks 0, 1 and 3: their blobs have odd lengths
        b.seals[odd] = b.seals[odd] + b"\\x00"
    st = np.asarray(v.verify_batch(b.seals, b.image_ids, b.journals))
    want = np.zeros(n, dtype=np.uint8); want[[5, 16384 + 9, 3 * 16384 + 1]] = 2          # InvalidProofData for the three, every other proof valid
    assert (st == want).all(), np.nonzero(st != want)[0][:10]
