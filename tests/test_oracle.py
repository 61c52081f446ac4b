"""Pins the CPU oracle (oracle/) against every golden datum the reference holds for this path
(SURVEY.md section 4 / 8c): the two embedded fixtures, the known-answer table derived from them, the
independent Python referee, and algebraic self-checks of the precompile restatement."""
import hashlib

import pytest

import oracle_lib as O

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
G1 = w32(1) + w32(2)


def test_sha256_matches_hashlib():
    for n in (0, 1, 55, 56, 63, 64, 65, 98, 119, 120, 128, 170, 183, 184, 194, 447, 448, 1000, 4096, 65536, 1 << 20):
        m = bytes((i * 7 + n) & 0xFF for i in range(n))
        assert O.sha256(m) == hashlib.sha256(m).digest()


def test_known_answers_risc0(fx):
    # SURVEY.md section 4 table
    assert O.sha256(b"risc0.ReceiptClaim").hex() == "cb1fefcd1f2d9a64975cbbbf6e161e2914434b0cbb9960b84df5d717e86b48af"
    assert O.sha256(b"risc0.Output").hex() == "77eafeb366a78b47747de0d7bb176284085ff5564887009a5be63da32d3559d4"
    r = O.Risc0Oracle()
    assert r.verify(fx["seal"], fx["image_id"], fx["journal_digest"]) == O.ST_INVALID_INITIALIZATION
    assert r.initialize(fx["control_root"], fx["bn254_control_id"]) == 0
    assert r.initialize(fx["control_root"], fx["bn254_control_id"]) == -1            # AlreadyInitialized
    assert r.vk_digest().hex() == "21c5fdd9b4d576b17581f50b755482ba7a2134a3b5186e8e454acfa1f69511ab"
    assert r.selector().hex() == "9f39696c" == fx["seal"][:4].hex()                   # pinned by the reference's own fixture
    claim = O.claim_digest(fx["image_id"], fx["journal_digest"])
    assert claim.hex() == "da64ae8d4ca166ae88e79a55dbaebe6479cb3f383bf963fc2c9bb48dd10169b6"
    sig = r.signals(claim)
    want = [0x4c2d7bb17348241967b0276818329053, 0x7645843b52b258e94f99b1cf022d2e12, 0x64beaedb559ae788ae66a14c8dae64da,
            0xb66901d18db49b2cfc63f93b383fcb79, int.from_bytes(fx["bn254_control_id"], "big")]
    assert [int.from_bytes(sig[32 * i:32 * i + 32], "big") for i in range(5)] == want
    # vk_x through the ecMul / ecAdd restatement
    vk = O.risc0_vk()
    acc = vk.ic[0]
    for i in range(5):
        acc = O.ec_add(acc + O.ec_mul(vk.ic[i + 1] + sig[32 * i:32 * i + 32]))
    assert acc.hex() == ("16c84fab9b8b745138532ae504d77ff206fbff38bd074311b12ad877f1dfd58a"
                         "1b12af2913caa5a3301bf6fcb1422a83f5c331d2aea78340e338a386801db136")


def test_fixture_risc0_accepts_and_tampers_reject(fx):
    r = O.Risc0Oracle(); r.initialize(fx["control_root"], fx["bn254_control_id"])
    seal, im, jd = fx["seal"], fx["image_id"], fx["journal_digest"]
    assert r.verify(seal, im, jd) == O.ST_OK
    assert r.verify_integrity(seal, O.claim_digest(im, jd)) == O.ST_OK
    flip = lambda b, i: b[:i] + bytes([b[i] ^ 1]) + b[i + 1:]
    assert r.verify(seal, flip(im, 5), jd) == O.ST_VERIFICATION_FAILED
    assert r.verify(seal, im, flip(jd, 31)) == O.ST_VERIFICATION_FAILED
    assert r.verify(flip(seal, 0), im, jd) == O.ST_SELECTOR_MISMATCH
    assert r.verify(seal[:3], im, jd) == O.ST_INVALID_PROOF_DATA
    assert r.verify(seal[:259], im, jd) == O.ST_INVALID_PROOF_DATA
    assert r.verify(seal + b"\0", im, jd) == O.ST_INVALID_PROOF_DATA
    assert r.verify(b"\0\0\0\0" + seal[4:], im, jd) == O.ST_SELECTOR_MISMATCH
    for i in (4, 40, 70, 140, 200, 259):
        assert r.verify(flip(seal, i), im, jd) == O.ST_VERIFICATION_FAILED


def test_fixture_sp1_accepts_and_tampers_reject(fx):
    vk, sel = O.sp1_vk(), fx["sp1_selector"]
    vkey, pv, pr = fx["sp1_vkey"], fx["sp1_public_values"], fx["sp1_proof"]
    assert sel.hex() == "a4594c59"
    assert O.sp1_hash_public_values(pv).hex() == "0f1cb7decf31e49c7934c3740bec5df3ead27bc947af739782930df6e37e9d90"
    assert O.sp1_verify(vk, sel, vkey, pv, pr) == O.ST_OK
    flip = lambda b, i: b[:i] + bytes([b[i] ^ 1]) + b[i + 1:]
    assert O.sp1_verify(vk, sel, flip(vkey, 9), pv, pr) == O.ST_VERIFICATION_FAILED
    assert O.sp1_verify(vk, sel, vkey, flip(pv, 40), pr) == O.ST_VERIFICATION_FAILED
    assert O.sp1_verify(vk, sel, vkey, pv + b"\0", pr) == O.ST_VERIFICATION_FAILED
    assert O.sp1_verify(vk, sel, vkey, pv, flip(pr, 2)) == O.ST_SELECTOR_MISMATCH
    assert O.sp1_verify(vk, sel, vkey, pv, pr[:2]) == O.ST_INVALID_PROOF_DATA
    assert O.sp1_verify(vk, sel, vkey, pv, pr[:100]) == O.ST_INVALID_PROOF_DATA
    assert O.sp1_verify(vk, sel, w32(R), pv, pr) == O.ST_VERIFICATION_FAILED          # signal >= R, groth16.rs:32-34
    for i in (4, 90, 150, 259):
        assert O.sp1_verify(vk, sel, vkey, pv, flip(pr, i)) == O.ST_VERIFICATION_FAILED


def test_precompile_semantics_eip196():
    inf = bytes(64)
    assert O.ec_add(G1 + inf) == G1 and O.ec_add(inf + inf) == inf and O.ec_add(b"") == inf      # short input is right-padded
    two = O.ec_add(G1 + G1)
    assert two == O.ec_mul(G1 + w32(2))
    neg = w32(1) + w32(P - 2)
    assert O.ec_add(G1 + neg) == inf
    assert O.ec_mul(G1 + w32(R)) == inf and O.ec_mul(G1 + w32(R + 1)) == G1                       # scalars are not reduced
    assert O.ec_mul(G1 + w32((1 << 256) - 1)) == O.ec_mul(G1 + w32(((1 << 256) - 1) % R))
    assert O.ec_mul(G1 + w32(0)) == inf and O.ec_mul(inf + w32(5)) == inf
    assert O.ec_add(w32(1) + w32(3) + inf) is None                                                # off curve
    assert O.ec_add(w32(P) + w32(2) + inf) is None and O.ec_mul(w32(1) + w32(P + 2) + w32(1)) is None   # coordinate >= p
    # associativity / distributivity spot checks
    a, b = 0x1234567890ABCDEF << 100, 0xFEDCBA987654321 << 50
    assert O.ec_add(O.ec_mul(G1 + w32(a)) + O.ec_mul(G1 + w32(b))) == O.ec_mul(G1 + w32(a + b))


def test_precompile_semantics_eip197(consts):
    from stylus_zkvm_verifiers_b200.synth import G2_GEN, SplitMix64, random_twist_point
    inf1, inf2 = bytes(64), bytes(128)
    one, zero = w32(1), w32(0)
    assert O.ec_pairing(b"") == one                                   # empty product
    assert O.ec_pairing(G1 + inf2) == one and O.ec_pairing(inf1 + G2_GEN) == one
    assert O.ec_pairing(G1 + G2_GEN) == zero
    neg = w32(1) + w32(P - 2)
    assert O.ec_pairing(G1 + G2_GEN + neg + G2_GEN) == one
    assert O.ec_pairing((G1 + G2_GEN)[:-1]) is None                   # length not a multiple of 192
    # bilinearity: e(aP, bQ) e(-abP, Q) = 1
    a, b = 0xA5A5A5A5A5A5A5A5A5A5, 0x5A5A5A5A5A5A5A5A5A5A5A
    aP, bQ = O.g1_mul(G1, a), O.g2_mul(G2_GEN, b)
    abP = O.g1_mul(G1, a * b % R)
    nabP = abP[:32] + w32(P - int.from_bytes(abP[32:], "big"))
    assert O.ec_pairing(aP + bQ + nabP + G2_GEN) == one
    assert O.ec_pairing(aP + bQ + abP + G2_GEN) == zero
    # wrong-subgroup / off-twist / out-of-range G2 make the call fail
    rng = SplitMix64(7)
    assert O.ec_pairing(G1 + random_twist_point(rng)) is None
    bad = bytearray(G2_GEN); bad[127] ^= 1
    assert O.ec_pairing(G1 + bytes(bad)) is None
    assert O.ec_pairing(G1 + w32(P) + G2_GEN[32:]) is None
    # G1 is not subgroup-checked (cofactor 1) but must be on the curve
    assert O.ec_pairing(w32(1) + w32(3) + G2_GEN) is None


def test_negate_g1_quirk(fx):
    """groth16.rs:75-84: Q.wrapping_sub(y) happens before any range check -> A = (0, Q) becomes (0,0) = infinity."""
    r = O.Risc0Oracle(); r.initialize(fx["control_root"], fx["bn254_control_id"])
    seal = fx["seal"]; im, jd = fx["image_id"], fx["journal_digest"]
    a_inf = seal[:4] + bytes(64) + seal[68:]
    a_0q = seal[:4] + w32(0) + w32(P) + seal[68:]
    assert r.verify(a_inf, im, jd) == r.verify(a_0q, im, jd) == O.ST_VERIFICATION_FAILED   # 3-pair product != 1 for this seal
    vk = O.risc0_vk()
    st1, m1, g1 = O.groth16_verify(vk, a_inf[4:], r.signals(O.claim_digest(im, jd)), debug=True)
    st2, m2, g2 = O.groth16_verify(vk, a_0q[4:], r.signals(O.claim_digest(im, jd)), debug=True)
    assert m1 == m2 and g1 == g2 and any(g1)          # both reached the pairing (not an input error) with identical values
    a_x0 = seal[:36] + w32(0) + seal[68:]              # A = (x, 0) -> y' = Q -> rejected as out of range
    st3, m3, g3 = O.groth16_verify(vk, a_x0[4:], r.signals(O.claim_digest(im, jd)), debug=True)
    assert st3 == O.ST_VERIFICATION_FAILED and not any(g3)


@pytest.mark.timeout(600)
def test_python_referee_agrees(fx):
    """Independent slow referee (different Fp12 basis, affine arithmetic, plain pow final exponentiation)."""
    import bn254_py as B
    c = O.constants()
    seal = fx["seal"]
    to_int = lambda h: int(h, 16)
    vk = {k: ([to_int(x) for x in v] if k == "alpha" else [[to_int(x) for x in row] for row in v]) for k, v in c["risc0_vk"].items()}
    r = O.Risc0Oracle(); r.initialize(fx["control_root"], fx["bn254_control_id"])
    sigb = r.signals(O.claim_digest(fx["image_id"], fx["journal_digest"]))
    sig = [int.from_bytes(sigb[32 * i:32 * i + 32], "big") for i in range(5)]
    wv = [int.from_bytes(seal[4 + 32 * i:36 + 32 * i], "big") for i in range(8)]
    assert B.groth16_verify(0, vk, wv[0:2], [wv[2:4], wv[4:6]], wv[6:8], sig) is True
    assert B.groth16_verify(1, vk, wv[0:2], [wv[2:4], wv[4:6]], wv[6:8], sig) is False      # without negating A
    assert B.risc0_selector(fx["control_root"], fx["bn254_control_id"], vk) == seal[:4]
    # GT convention: oracle GT == (canonical pairing)^LAMBDA after basis change
    data = G1 + bytes.fromhex("".join(c["risc0_vk"]["gamma"][0] + c["risc0_vk"]["gamma"][1]))
    ret, m, gt = O.ec_pairing(data, debug=True)
    gt_t = [int.from_bytes(gt[32 * i:32 * i + 32], "big") for i in range(12)]
    Q = B._dec_g2(data[64:])
    e = B.final_exp(B.miller((1, 2), Q))
    assert B.tower_to_poly(gt_t) == B.f12pow(e, B.LAMBDA)


@pytest.mark.timeout(900)
def test_python_referee_agrees_on_every_mutation_class(fx):
    """SURVEY 8c(3): the independent Python referee (affine arithmetic, different Fp12 basis, plain-pow final exponentiation, its own
    restatement of the verifiers' front checks) and the C oracle must return the same status for >= 3 samples of EVERY class of the
    config-4 mix (valid, tampered, off-curve, coordinate >= p incl. the (0, Q) quirk, wrong-subgroup G2, infinity members, malformed),
    for both proof shapes: the reject side of the oracle is pinned by a second implementation family, not only the accept side."""
    import bn254_py as B
    from stylus_zkvm_verifiers_b200 import synth as S

    class OB:
        def g1_mul(self, sc): return [O.g1_mul(S.G1_GEN, s) for s in sc]
        def g2_mul(self, sc): return [O.g2_mul(S.G2_GEN, s) for s in sc]
    be = lambda b: int.from_bytes(b, "big")
    g1 = lambda b: (be(b[:32]), be(b[32:64]))
    g2 = lambda b: ((be(b[0:32]), be(b[32:64])), (be(b[64:96]), be(b[96:128])))
    pyvk = lambda vk: {"alpha": g1(vk.alpha), "beta": g2(vk.beta), "gamma": g2(vk.gamma), "delta": g2(vk.delta), "ic": [g1(p) for p in vk.ic]}
    want_classes = [c for c, _ in S.MIXED_CLASSES]
    seen = {}
    # RISC Zero shape
    vk = S.make_vk(OB(), 0, 6, 0xB2000031)
    ro = O.Risc0Oracle(O.Vk(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)); ro.initialize(fx["control_root"], fx["bn254_control_id"])
    assert B.risc0_selector(fx["control_root"], fx["bn254_control_id"], pyvk(vk)) == ro.selector()
    b = S.make_risc0_batch(OB(), vk, ro.selector(), fx["control_root"], fx["bn254_control_id"], fx["sys0"], 160, 0xB2000032, pool=16)
    S.mutate_risc0(b, OB(), S.SplitMix64(0xB2000033))
    want = ro.verify_batch(b.seals, b.image_ids, b.journals)
    pick = []
    for i, c in enumerate(b.classes):
        if seen.get(("risc0", c), 0) < 3:
            seen[("risc0", c)] = seen.get(("risc0", c), 0) + 1; pick.append(i)
    pv = pyvk(vk)
    for i in pick:
        got = B.risc0_verify_status(pv, ro.selector(), fx["control_root"], fx["bn254_control_id"], b.seals[i], b.image_ids[i], b.journals[i])
        assert got == int(want[i]), ("risc0", b.classes[i], i, got, int(want[i]))
    # SP1 shape
    vk = S.make_vk(OB(), 1, 3, 0xB2000034)
    sb = S.make_sp1_batch(OB(), vk, 160, 0xB2000035, pool=16)
    S.mutate_sp1(sb, OB(), S.SplitMix64(0xB2000036))
    want = O.sp1_verify_batch(O.Vk(1, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic), S.SP1_SELECTOR, sb.vkeys, sb.public_values, sb.proofs)
    pick = []
    for i, c in enumerate(sb.classes):
        if seen.get(("sp1", c), 0) < 3:
            seen[("sp1", c)] = seen.get(("sp1", c), 0) + 1; pick.append(i)
    pv = pyvk(vk)
    for i in pick:
        got = B.sp1_verify_status(pv, S.SP1_SELECTOR, sb.vkeys[i], sb.public_values[i], sb.proofs[i])
        assert got == int(want[i]), ("sp1", sb.classes[i], i, got, int(want[i]))
    for shape in ("risc0", "sp1"):
        for c in want_classes:
            assert seen.get((shape, c), 0) >= 3, (shape, c, seen)


def test_committed_campaign_digests_are_consistent():
    """profiles/r2_campaign_oracle_digests.json (the CPU-oracle half of the >= 10^7-proof exactness campaign): 154 batches of 2^16 proofs, both
    shapes, every mutation class present, only `valid` proofs accepted, histogram and class counts add up."""
    import json, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = json.load(open(os.path.join(root, "profiles", "r2_campaign_oracle_digests.json")))
    assert len(d["batches"]) == 154 and d["batch"] == 1 << 16 and d["classes"][0] == "valid"
    tot = acc = 0
    per = [0] * len(d["classes"])
    for b in d["batches"]:
        assert b["shape"] == ("risc0" if b["k"] % 2 == 0 else "sp1") and len(b["status_sha256"]) == 64
        n = sum(c[0] for c in b["per_class"])
        assert n == d["batch"] == sum(b["status_histogram"].values())
        assert b["accepted"] == b["per_class"][0][1] == b["per_class"][0][0] == b["status_histogram"]["0"]      # every valid proof and nothing else
        assert all(c[1] == 0 for c in b["per_class"][1:])
        tot += n; acc += b["accepted"]
        for i, c in enumerate(b["per_class"]):
            per[i] += c[0]
    assert tot == 10092544 >= 10 ** 7 and all(p > 400000 for p in per) and 0.45 < acc / tot < 0.55
