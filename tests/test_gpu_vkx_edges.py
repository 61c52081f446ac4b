"""The chosen-point proofs of vkx_edges.py on every verification entry point: each status byte against the CPU oracle and the construction
(0 for the accepting proofs, 4 for their twins and random-A variants), vk_x points against the precompile chain, and the pairing / ecAdd /
ecMul services on the edge-point catalogue bit for bit.  Status tests run on a small batch (one chain) and tiled to 2^15 records
(automatic chunking), and on one key with overlap 4 and miller_segments 1 and 7."""
import numpy as np
import pytest

import oracle_lib as O
import vkx_edges as V
from stylus_zkvm_verifiers_b200 import synth as S

pytestmark = pytest.mark.gpu

R = V.R
TILED = 1 << 15


@pytest.fixture(scope="module")
def Z():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import stylus_zkvm_verifiers_b200 as Z
    return Z


def _dev(x):
    import torch
    return torch.from_numpy(np.frombuffer(bytes(x), dtype=np.uint8).copy()).cuda()


def _status(n):
    import torch
    return torch.full((n,), 255, dtype=torch.uint8, device="cuda")


def _tile(seq, n):
    return [seq[i % len(seq)] for i in range(n)]


def _sig_blob(recs):
    return b"".join(O.w32(v) for r in recs for v in r.signals)


# ------------------------------------------------------------------ generic family and key sets
@pytest.fixture(scope="module")
def generic(Z):
    keys, recs, hits = V.generic_cases()
    rng = S.SplitMix64(0xED6E4000)
    n_crafted = len(keys)
    for j in range(3):                                                   # ordinary keys (random multiples of G1) mixed into the set
        keys.append(V.EdgeKey(j % 2, S.G1_GEN, [rng.fr() for _ in range(4 + j)], V.mul(S.G1_GEN, rng.fr()), 0xED6E4010 + j))
        for _ in range(4):
            sig = [rng.fr() for _ in range(3 + j)]
            V.generic_records(recs, "ordinary%d" % j, len(keys) - 1, keys[-1], sig, rng)
    kvs = [k.load(Z) for k in keys]
    want = np.array([r.expect for r in recs], dtype=np.uint8)
    for ki, key in enumerate(keys):                                      # the oracle agrees with the construction
        idx = [i for i, r in enumerate(recs) if r.key == ki]
        st = O.groth16_verify_batch(key.ovk(), b"".join(recs[i].proof for i in idx), _sig_blob([recs[i] for i in idx]), len(idx))
        assert st.tolist() == want[idx].tolist(), ki
    return dict(keys=keys, kvs=kvs, recs=recs, want=want, n_crafted=n_crafted)


def test_vk_x_batch_matches_precompile_chain(Z, generic):
    for ki, (key, kv) in enumerate(zip(generic["keys"], generic["kvs"])):
        rs = [r for r in generic["recs"] if r.key == ki]
        out = Z.vk_x_batch(kv, _sig_blob(rs), key.k, len(rs)).tobytes()
        for i, r in enumerate(rs):
            assert out[64 * i:64 * i + 64] == key.vk_x(r.signals), (r.case, i)
        if ki == 0:
            assert any(out[64 * i:64 * i + 64] == V.INF for i in range(len(rs)))


def test_vk_x_batch_of_risc0_keys(Z):
    """the RISC Zero cases' five signals through the generic vk_x (64 windows each, one addition order) equal the precompile chain"""
    for rc in V.risc0_cases():
        kv = rc.key.load(Z)
        sigs = [S.risc0_signals(rc.cr, rc.cid, S.risc0_claim_digest(im, jr, V.SYS0)) for _, im, jr, _, _ in rc.recs]
        out = Z.vk_x_batch(kv, b"".join(O.w32(v) for s in sigs for v in s), 5, len(sigs)).tobytes()
        for i, s in enumerate(sigs):
            assert out[64 * i:64 * i + 64] == rc.key.vk_x(s), (rc.name, i)


def test_generic_path(Z, generic):
    for ki, (key, kv) in enumerate(zip(generic["keys"], generic["kvs"])):
        idx = [i for i, r in enumerate(generic["recs"]) if r.key == ki]
        rs = [generic["recs"][i] for i in idx]
        got = Z.Groth16Verifier.verify_batch(kv, b"".join(r.proof for r in rs), _sig_blob(rs), key.k, len(rs))
        assert got.tolist() == generic["want"][idx].tolist(), [(r.case, int(g)) for r, g in zip(rs, got) if g != r.expect]


def _keyset_call(Z, ks, recs, device=False):
    key_idx = np.array([r.key for r in recs], dtype=np.uint32)
    if not device:
        return Z.Groth16Verifier.verify_batch_keys(ks, key_idx, [r.proof for r in recs], [r.signals for r in recs])
    import torch
    off = np.zeros(len(recs) + 1, dtype=np.uint64); off[1:] = np.cumsum([len(r.signals) for r in recs])
    d_k, d_p, d_s, d_o = _dev(key_idx.tobytes()), _dev(b"".join(r.proof for r in recs)), _dev(_sig_blob(recs)), _dev(off.tobytes())
    d_st = _status(len(recs))
    Z.Groth16Verifier.verify_batch_keys_device(ks, 0, d_k.data_ptr(), d_p.data_ptr(), d_s.data_ptr(), d_o.data_ptr(), len(recs), d_st.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return d_st.cpu().numpy()


def test_key_set_host_and_device(Z, generic):
    """the crafted keys among ordinary ones in one set: host and device forms, caller order shuffled, and tiled to 2^15 records"""
    ks = Z.VerificationKeySet(generic["kvs"])
    order = np.random.default_rng(7).permutation(len(generic["recs"]))
    recs = [generic["recs"][i] for i in order]
    want = generic["want"][order]
    assert _keyset_call(Z, ks, recs).tolist() == want.tolist()
    assert _keyset_call(Z, ks, recs, device=True).tolist() == want.tolist()
    big = _tile(recs, TILED)
    got = _keyset_call(Z, ks, big)
    assert got.tolist() == _tile(want.tolist(), TILED)


# ------------------------------------------------------------------ SP1
@pytest.fixture(scope="module")
def sp1(Z):
    keys, recs, hits = V.sp1_cases()
    kvs = [k.load(Z) for k in keys]
    return dict(keys=keys, kvs=kvs, recs=recs, want=np.array([r.expect for r in recs], dtype=np.uint8))


def _sp1_host(h, recs, sel):
    return h.verify_batch([r.vkey for r in recs], [r.pv for r in recs], [sel + r.proof for r in recs])


def test_sp1_handle_host_device_and_schedules(Z, sp1):
    """route 0 (the branch targets and the edge points) on one handle: host and device forms, tiled to 2^15, overlap 4, miller_segments 1 / 7"""
    import torch
    h = Z.Sp1Verifier(sp1["kvs"][0])
    sel = h.verifier_hash()[:4]
    idx = [i for i, r in enumerate(sp1["recs"]) if r.route == 0]
    recs, want = [sp1["recs"][i] for i in idx], sp1["want"][idx].tolist()
    ovk = sp1["keys"][0].ovk()
    assert O.sp1_verify_batch(ovk, sel, [r.vkey for r in recs], [r.pv for r in recs], [sel + r.proof for r in recs]).tolist() == want
    assert _sp1_host(h, recs, sel).tolist() == want
    fixed = [i for i, r in enumerate(recs) if len(r.pv) == 96]
    d_st = _status(len(fixed))
    d_v, d_pv, d_p = _dev(b"".join(recs[i].vkey for i in fixed)), _dev(b"".join(recs[i].pv for i in fixed)), _dev(b"".join(sel + recs[i].proof for i in fixed))
    h.verify_batch_device(0, d_v.data_ptr(), d_pv.data_ptr(), 96, d_p.data_ptr(), len(fixed), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert d_st.cpu().numpy().tolist() == [want[i] for i in fixed]
    big, bwant = _tile(recs, TILED), _tile(want, TILED)
    assert _sp1_host(h, big, sel).tolist() == bwant
    segs0 = h.tune("miller_segments")
    try:
        h.tune("overlap", 4)
        assert _sp1_host(h, big, sel).tolist() == bwant
        h.tune("overlap", 0)
        for segs in (1, 7):
            h.tune("miller_segments", segs)
            assert _sp1_host(h, recs, sel).tolist() == want, segs
            assert _sp1_host(h, big, sel).tolist() == bwant, segs
    finally:
        h.tune("overlap", 0); h.tune("miller_segments", segs0)


def test_sp1_gateway(Z, sp1):
    """every SP1 route (the main key and the two crafted t = 0 keys) as a version handle of one gateway: host and device forms"""
    import torch
    hs = [Z.Sp1Verifier(kv, verifier_hash=O.sha256(b"edge sp1 route %d" % j), version="v%d.0.0-edge" % (7 + j)) for j, kv in enumerate(sp1["kvs"])]
    sels = [h.verifier_hash()[:4] for h in hs]
    recs, want = sp1["recs"], sp1["want"]
    for j, key in enumerate(sp1["keys"]):                                    # the oracle of each route agrees with the construction
        idx = [i for i, r in enumerate(recs) if r.route == j]
        st = O.sp1_verify_batch(key.ovk(), sels[j], [recs[i].vkey for i in idx], [recs[i].pv for i in idx], [sels[j] + recs[i].proof for i in idx])
        assert st.tolist() == want[idx].tolist(), j
    gw = Z.Sp1VerifierGateway(hs)
    order = np.random.default_rng(9).permutation(len(recs))
    proofs = [sels[recs[i].route] + recs[i].proof for i in order]
    got = gw.verify_batch([recs[i].vkey for i in order], [recs[i].pv for i in order], proofs)
    assert got.tolist() == want[order].tolist()
    fixed = [i for i in order if len(recs[i].pv) == 96]
    d_st = _status(len(fixed))
    d_v, d_pv, d_p = (_dev(b"".join(recs[i].vkey for i in fixed)), _dev(b"".join(recs[i].pv for i in fixed)),
                      _dev(b"".join(sels[recs[i].route] + recs[i].proof for i in fixed)))
    gw.verify_batch_device(0, d_v.data_ptr(), d_pv.data_ptr(), 96, d_p.data_ptr(), len(fixed), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert d_st.cpu().numpy().tolist() == want[fixed].tolist()


# ------------------------------------------------------------------ RISC Zero handles and router
@pytest.fixture(scope="module")
def risc0(Z):
    cases = V.risc0_cases()
    out = []
    for rc in cases:
        h = Z.RiscZeroVerifier(rc.key.load(Z))
        h.initialize(rc.cr, rc.cid)
        assert h.get_selector() == rc.selector()
        ro = O.Risc0Oracle(rc.key.ovk()); ro.initialize(rc.cr, rc.cid)
        _, ims, jrs, seals, want = zip(*rc.recs)
        assert ro.verify_batch(list(seals), list(ims), list(jrs)).tolist() == list(want), rc.name
        out.append((rc, h))
    return out


def test_risc0_handles(Z, risc0):
    """verify_batch, verify_integrity_batch and verify_batch_device of each handle (K, mid or a claim addition at a special branch)"""
    import torch
    for rc, h in risc0:
        names, ims, jrs, seals, want = (list(x) for x in zip(*rc.recs))
        assert h.verify_batch(seals, ims, jrs).tolist() == want, rc.name
        assert h.verify_integrity_batch(seals, [O.claim_digest(a, b) for a, b in zip(ims, jrs)]).tolist() == want, rc.name
        d_s, d_i, d_j, d_st = _dev(b"".join(seals)), _dev(b"".join(ims)), _dev(b"".join(jrs)), _status(len(seals))
        h.verify_batch_device(0, d_s.data_ptr(), d_i.data_ptr(), d_j.data_ptr(), len(seals), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert d_st.cpu().numpy().tolist() == want, rc.name


def test_risc0_router(Z, risc0):
    """one router over every crafted handle (the 32-window route tables with each folded base): host, integrity and device forms, and
    tiled to 2^15 seals"""
    import torch
    router = Z.RiscZeroVerifierRouter([h for _, h in risc0])
    assert 8 <= len(router) <= 16
    recs = [r for rc, _ in risc0 for r in rc.recs]
    order = np.random.default_rng(13).permutation(len(recs))
    names, ims, jrs, seals, want = (list(x) for x in zip(*[recs[i] for i in order]))
    assert router.verify_batch(seals, ims, jrs).tolist() == want
    assert router.verify_integrity_batch(seals, [O.claim_digest(a, b) for a, b in zip(ims, jrs)]).tolist() == want
    d_s, d_i, d_j, d_st = _dev(b"".join(seals)), _dev(b"".join(ims)), _dev(b"".join(jrs)), _status(len(seals))
    router.verify_batch_device(0, d_s.data_ptr(), d_i.data_ptr(), d_j.data_ptr(), len(seals), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert d_st.cpu().numpy().tolist() == want
    got = router.verify_batch(_tile(seals, TILED), _tile(ims, TILED), _tile(jrs, TILED))
    assert got.tolist() == _tile(want, TILED)


# ------------------------------------------------------------------ services on the edge-point catalogue
def test_ec_add_mul_on_catalogue(Z):
    pts = [p for _, p in V.edge_points()] + [V.INF]
    adds = [a + b for a in pts for b in pts]                                 # includes P + P and P + (-P)
    out, rev = Z.ec_add_batch(b"".join(adds), len(adds)); out = out.tobytes()
    for i, d in enumerate(adds):
        assert rev[i] == 0 and out[64 * i:64 * i + 64] == O.ec_add(d), i
    scal = [0, 1, 2, 3, 16, 15 << 252, R - 1, R, R + 1, (1 << 256) - 1, 0xED6E]
    muls = [p + O.w32(s) for p in pts for s in scal]
    out, rev = Z.ec_mul_batch(b"".join(muls), len(muls)); out = out.tobytes()
    for i, d in enumerate(muls):
        assert rev[i] == 0 and out[64 * i:64 * i + 64] == O.ec_mul(d), i


def test_pairing_services_on_edge_points(Z):
    """pairing4_batch and ec_pairing_batch with every G1 input at an edge point: the accept bit, the Miller value and the GT value bit for
    bit against the oracle; half the instances satisfy the product equation by construction"""
    rng = S.SplitMix64(0xED6E5000)
    ep = [p for _, p in V.edge_points()]
    n = len(ep)
    key = V.EdgeKey(0, S.G1_GEN, [1, 2], S.G1_GEN, 0xED6E5001)
    kv = key.load(Z)
    t = key.trap
    g1s, g2s, expect = [], [], []
    for i in range(2 * n):
        q = rng.fr()
        p0, p1, p2 = ep[i % n], ep[(i + 3) % n], ep[(i + 7) % n]
        if i < n:     # q P0 + beta P1 + gamma P2 + delta P3 = 0
            p3 = V.mul(V.add(V.mul(p0, q), V.mul(p1, t["beta"]), V.mul(p2, t["gamma"])), -pow(t["delta"], -1, R))
        else:
            p3 = ep[(i + 11) % n]
        g1s.append(p0 + p1 + p2 + p3); g2s.append(O.g2_mul(S.G2_GEN, q)); expect.append(1 if i < n else 0)
    ok, gt, ml = Z.pairing4_batch(kv, b"".join(g1s), b"".join(g2s), len(g1s), want_gt=True, want_miller=True)
    blob = b"".join(g[0:64] + q + g[64:128] + key.beta + g[128:192] + key.gamma + g[192:256] + key.delta for g, q in zip(g1s, g2s))
    ook, ogt, oml = O.pairing4_batch(blob, len(g1s), want_gt=True, want_miller=True)
    assert ok.tolist() == ook.tolist() == expect
    assert ml.tobytes() == oml.tobytes() and gt.tobytes() == ogt.tobytes()
    # the general service: three pairs with variable G2 points
    inst = []
    for i in range(n):
        a, b = rng.fr(), rng.fr()
        q1, q2 = O.g2_mul(S.G2_GEN, a), O.g2_mul(S.G2_GEN, b)
        p2 = V.neg(V.add(V.mul(ep[i], a), V.mul(ep[(i + 5) % n], b))) if i % 2 == 0 else ep[(i + 9) % n]
        inst.append(ep[i] + q1 + ep[(i + 5) % n] + q2 + p2 + S.G2_GEN)
    words, rev, ml = Z.ec_pairing_batch(b"".join(inst), 3, n, want_miller=True)
    for i in range(n):
        w, m, _ = O.ec_pairing(inst[i], debug=True)
        assert rev[i] == 0 and bytes(words[32 * i:32 * i + 32]) == w and bytes(ml[384 * i:384 * i + 384]) == m, i
        assert w == O.w32(1 if i % 2 == 0 else 0), i
