"""The single-cause cases of single_cause.py on every verification entry point and on the pairing services: each status byte against the
case's expected status (VERIFICATION_FAILED for a case, OK for its twin), which test_single_cause.py checks against the CPU oracle.

Each case sits beside its twin at lanes 0, 31, 32, 127 and 128, at the last record and at the chunk edges of the schedule, so that a flag
written to a neighbour shows.  The verification path finishes the G2 subgroup test in its last Miller segment (k_g2_target + lz_r_is); the
pairing services run k_g2_check.  About 10 s on one B200 (1000 W power limit)."""
import numpy as np
import pytest

import batch_geometry as BG
import oracle_lib as O
import single_cause as SC

pytestmark = pytest.mark.gpu

TILED = 1 << 15
CHUNK = BG.chunk_size(TILED, 4)          # four pieces: overlap 4, and the automatic schedule at 2^15


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


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _check(got, recs, what):
    want = [r.expect for r in recs]
    got = [int(g) for g in got]
    bad = [(i, recs[i].name, got[i]) for i in range(len(recs)) if got[i] != want[i]]
    assert not bad, "%s: %d of %d wrong, first %s" % (what, len(bad), len(recs), bad[:8])


def _small(units):
    return SC.layout(units, 2 * len(units), SC.anchors(2 * len(units)))


def _tiled(units):
    return SC.layout(units, TILED, SC.anchors(TILED, CHUNK))


def _sig_blob(recs):
    return b"".join(O.w32(v) for r in recs for v in r.signals)


# ------------------------------------------------------------------ generic family and key sets
@pytest.fixture(scope="module")
def generic(Z):
    keys, units, ordinary = SC.generic_cases()
    return dict(keys=keys, kvs=[k.load(Z) for k in keys], units=units, ordinary=ordinary)


SCHEDULES = [("overlap1", dict(overlap=1)), ("overlap4,segs1", dict(overlap=4, miller_segments=1)),
             ("overlap4,segs2", dict(overlap=4, miller_segments=2)), ("overlap4,segs7", dict(overlap=4, miller_segments=7)),
             ("overlap4,segs16", dict(overlap=4, miller_segments=16)), ("overlap4,fe_stages0", dict(overlap=4, final_exp_stages=0)),
             ("overlap4,fe_stages1", dict(overlap=4, final_exp_stages=1))]


def _tuned(h, settings):
    """apply settings to a key or handle; returns the previous values"""
    return {k: h.tune(k, v) for k, v in settings.items()}


def test_generic_verify_batch_small(Z, generic):
    for ki, (key, kv) in enumerate(zip(generic["keys"], generic["kvs"])):
        units = [u for u in generic["units"] if u.case.key == ki]
        recs = _small(units)
        got = Z.Groth16Verifier.verify_batch(kv, b"".join(r.proof for r in recs), _sig_blob(recs), key.k, len(recs))
        _check(got, recs, "key %d" % ki)


@pytest.mark.parametrize("name,settings", SCHEDULES, ids=[s[0] for s in SCHEDULES])
def test_generic_verify_batch_tiled(Z, generic, name, settings):
    for ki, (key, kv) in enumerate(zip(generic["keys"], generic["kvs"])):
        recs = _tiled([u for u in generic["units"] if u.case.key == ki])
        old = _tuned(kv, settings)
        try:
            got = Z.Groth16Verifier.verify_batch(kv, b"".join(r.proof for r in recs), _sig_blob(recs), key.k, len(recs))
        finally:
            _tuned(kv, old)
        _check(got, recs, "key %d, %s" % (ki, name))


def _keyset_call(Z, ks, recs, device):
    key_idx = np.array([r.key for r in recs], dtype=np.uint32)
    if not device:
        return Z.Groth16Verifier.verify_batch_keys(ks, key_idx, [r.proof for r in recs], [r.signals for r in recs])
    import torch
    off = np.zeros(len(recs) + 1, dtype=np.uint64); off[1:] = np.cumsum([len(r.signals) for r in recs])
    d_k, d_p, d_s, d_o = _dev(key_idx.tobytes()), _dev(b"".join(r.proof for r in recs)), _dev(_sig_blob(recs)), _dev(off.tobytes())
    d_st = _status(len(recs))
    Z.Groth16Verifier.verify_batch_keys_device(ks, 0, d_k.data_ptr(), d_p.data_ptr(), d_s.data_ptr(), d_o.data_ptr(), len(recs), d_st.data_ptr(), _stream())
    torch.cuda.synchronize()
    return d_st.cpu().numpy()


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_key_set(Z, generic, device):
    """the case keys (two of them with alpha at infinity) among two ordinary keys in one set, the units interleaved across keys"""
    ks = Z.VerificationKeySet(generic["kvs"])
    order = np.random.default_rng(3).permutation(len(generic["units"]))
    units = [generic["units"][i] for i in order]
    for recs, what in ((_small(units), "small"), (_tiled(units), "2^15")):
        _check(_keyset_call(Z, ks, recs, device), recs, what)


# ------------------------------------------------------------------ RISC Zero handles and router
@pytest.fixture(scope="module")
def risc0(Z):
    hs, units = SC.risc0_cases()
    handles = []
    for h in hs:
        z = Z.RiscZeroVerifier(h.key.load(Z))
        z.initialize(h.cr, h.cid)
        assert z.get_selector() == h.selector() and z.get_bn254_control_id() == h.cid
        handles.append(z)
    return dict(hs=hs, handles=handles, units=units, sels=[z.get_selector() for z in handles])


def _risc0_calls(Z, target, sels, recs, what):
    """verify_batch, verify_integrity_batch and verify_batch_device of a handle or router on recs"""
    import torch
    seals = [sels[r.key] + r.proof for r in recs]
    ims, jrs = [r.im for r in recs], [r.jr for r in recs]
    _check(target.verify_batch(seals, ims, jrs), recs, what + " host")
    _check(target.verify_integrity_batch(seals, [O.claim_digest(a, b) for a, b in zip(ims, jrs)]), recs, what + " integrity")
    d_s, d_i, d_j, d_st = _dev(b"".join(seals)), _dev(b"".join(ims)), _dev(b"".join(jrs)), _status(len(seals))
    target.verify_batch_device(0, d_s.data_ptr(), d_i.data_ptr(), d_j.data_ptr(), len(seals), d_st.data_ptr(), _stream())
    torch.cuda.synchronize()
    _check(d_st.cpu().numpy(), recs, what + " device")


def test_risc0_handles(Z, risc0):
    """each handle on its own records: the B catalogue with A = (0, 0) and (0, p) and the proof-word ranges on handle c (small and 2^15),
    the deep handle, and the control-id handles c + kR and 2R - 1 (all rejected) beside c and R - 1 (all accepted)"""
    from stylus_zkvm_verifiers_b200 import errors as E
    hs, handles, units, sels = risc0["hs"], risc0["handles"], risc0["units"], risc0["sels"]
    for hi, z in enumerate(handles):
        own = [r for r in SC.records(units) if r.key == hi]
        assert own, hs[hi].name
        _risc0_calls(Z, z, sels, own, hs[hi].name)
        same = [u for u in units if u.case.key == hi and u.twin.key == hi]
        if same:
            _risc0_calls(Z, z, sels, _small(same), hs[hi].name + " lanes")
        if hi == 0:
            _risc0_calls(Z, z, sels, _tiled(same), hs[hi].name + " 2^15")
    picked = [u for u in units if u.case.name.startswith(("risc0:A=(0,p)|B=order=l3", "risc0deep:A=(0,0)|B=-order=H2", "risc0:cid=c+5R#0",
                                                         "risc0:cid=2R-1#1", "risc0|w6+"))]
    assert len(picked) >= 5
    for u in picked:
        assert handles[u.twin.key].verify(sels[u.twin.key] + u.twin.proof, u.twin.im, u.twin.jr) is True, u.twin.name
        with pytest.raises(E.VerificationFailed):
            handles[u.case.key].verify(sels[u.case.key] + u.case.proof, u.case.im, u.case.jr)


def test_risc0_router(Z, risc0):
    """every handle as a route of one router: a c + kR route beside its c route, the deep route, host / integrity / device, small and 2^15"""
    router = Z.RiscZeroVerifierRouter(risc0["handles"])
    order = np.random.default_rng(5).permutation(len(risc0["units"]))
    units = [risc0["units"][i] for i in order]
    for recs, what in ((_small(units), "router"), (_tiled(units), "router 2^15")):
        _risc0_calls(Z, router, risc0["sels"], recs, what)


# ------------------------------------------------------------------ SP1 handle and gateway
@pytest.fixture(scope="module")
def sp1(Z):
    keys, units = SC.sp1_cases()
    return dict(keys=keys, kvs=[k.load(Z) for k in keys], units=units)


def _sp1_calls(Z, target, sels, recs, what):
    import torch
    proofs = [sels[r.key] + r.proof for r in recs]
    _check(target.verify_batch([r.vkey for r in recs], [r.pv for r in recs], proofs), recs, what + " host")
    d_st = _status(len(recs))
    d_v, d_pv, d_p = _dev(b"".join(r.vkey for r in recs)), _dev(b"".join(r.pv for r in recs)), _dev(b"".join(proofs))
    target.verify_batch_device(0, d_v.data_ptr(), d_pv.data_ptr(), SC.PV_LEN, d_p.data_ptr(), len(recs), d_st.data_ptr(), _stream())
    torch.cuda.synchronize()
    _check(d_st.cpu().numpy(), recs, what + " device")


def test_sp1_handles(Z, sp1):
    """route 0 (B catalogue with A at infinity, vkey v + kR, R and 2R - 1, proof-word ranges) and the deep route, each on its own handle:
    host and device forms, small and 2^15, and single verify_proof calls"""
    from stylus_zkvm_verifiers_b200 import errors as E
    for route, kv in enumerate(sp1["kvs"]):
        h = Z.Sp1Verifier(kv)
        sels = [h.verifier_hash()[:4]] * len(sp1["kvs"])
        units = [u for u in sp1["units"] if u.case.key == route]
        _sp1_calls(Z, h, sels, _small(units), "route %d" % route)
        _sp1_calls(Z, h, sels, _tiled(units), "route %d 2^15" % route)
        for u in units[::7]:
            assert h.verify_proof(u.twin.vkey, u.twin.pv, sels[0] + u.twin.proof) is None, u.twin.name
            with pytest.raises(E.VerificationFailed):
                h.verify_proof(u.case.vkey, u.case.pv, sels[0] + u.case.proof)


def test_sp1_gateway(Z, sp1):
    hs = [Z.Sp1Verifier(kv, verifier_hash=O.sha256(b"single-cause sp1 route %d" % j), version="v9.%d.0-sc" % j) for j, kv in enumerate(sp1["kvs"])]
    gw = Z.Sp1VerifierGateway(hs)
    sels = [h.verifier_hash()[:4] for h in hs]
    order = np.random.default_rng(11).permutation(len(sp1["units"]))
    units = [sp1["units"][i] for i in order]
    for recs, what in ((_small(units), "gateway"), (_tiled(units), "gateway 2^15")):
        _sp1_calls(Z, gw, sels, recs, what)


# ------------------------------------------------------------------ services (k_g2_check)
@pytest.fixture(scope="module")
def catalogue():
    return SC.outside_catalogue(), SC.member_catalogue()


def test_g2_check_batch_on_catalogue(Z, catalogue):
    outside, members = catalogue
    pts = [b.point for b in outside] + [q for _, q in members]
    got = Z.g2_check_batch(b"".join(pts), len(pts))
    assert got.tolist() == [0] * len(outside) + [1] * len(members), [(b.name, int(g)) for b, g in zip(outside, got) if g]


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_pairing4_outside_b_with_fixed_pairs_at_one(Z, catalogue, device):
    """P0 = infinity, P1..P3 with beta P1 + gamma P2 + delta P3 = 0 (the fixed pairs multiply to 1): Q outside G2 gives ok = 2 (the call
    reverts), the twin with a member Q ok = 1 with the oracle's GT and Miller values"""
    import torch
    import vkx_edges as V
    from stylus_zkvm_verifiers_b200 import synth as S
    outside, members = catalogue
    rng = S.SplitMix64(0x5C0A4000)
    key = V.EdgeKey(0, S.G1_GEN, [1, 2], S.G1_GEN, 0x5C0A4001)
    kv = key.load(Z)
    t = key.trap
    g1s, g2s, want = [], [], []
    for j, b in enumerate(outside):
        p1, p2 = rng.fr(), rng.fr()
        p3 = (-(p1 * t["beta"] + p2 * t["gamma"])) * pow(t["delta"], -1, SC.R) % SC.R
        g1 = SC.INF1 + V.mul(S.G1_GEN, p1) + V.mul(S.G1_GEN, p2) + V.mul(S.G1_GEN, p3)
        g1s += [g1, g1]; g2s += [b.point, members[j % len(members)][1]]; want += [2, 1]
    n = len(g1s)
    if device:
        d1, d2, d_ok, d_gt = _dev(b"".join(g1s)), _dev(b"".join(g2s)), _status(n), torch.zeros(n * 384, dtype=torch.uint8, device="cuda")
        from stylus_zkvm_verifiers_b200 import _native as N
        N.check(N.lib().zkv_pairing4_batch_device(kv._h, 0, d1.data_ptr(), d2.data_ptr(), n, d_ok.data_ptr(), d_gt.data_ptr(), _stream()))
        torch.cuda.synchronize()
        ok, gt, ml = d_ok.cpu().numpy(), d_gt.cpu().numpy(), None
    else:
        ok, gt, ml = Z.pairing4_batch(kv, b"".join(g1s), b"".join(g2s), n, want_gt=True, want_miller=True)
    assert ok.tolist() == want, [(i, int(o)) for i, o in enumerate(ok) if o != want[i]][:8]
    blob = b"".join(g[0:64] + q + g[64:128] + key.beta + g[128:192] + key.gamma + g[192:256] + key.delta for g, q in zip(g1s, g2s))
    ook, ogt, oml = O.pairing4_batch(blob, n, want_gt=True, want_miller=True)
    assert ook.tolist() == want
    acc = [i for i in range(n) if want[i] == 1]
    row = lambda a, i: a[384 * i:384 * i + 384].tobytes()
    assert all(row(gt, i) == row(ogt, i) == O.FP12_ONE for i in acc)
    if ml is not None:
        assert all(row(ml, i) == row(oml, i) for i in acc)


def test_ec_pairing_outside_q_at_every_position(Z, catalogue):
    """k = 1..4 pairs, one of them (infinity, Q outside G2) at each position, the others multiplying to 1: the call reverts; the twin with a
    member Q returns 1.  Through ec_pairing_batch (one call per k) and single ec_pairing calls."""
    import vkx_edges as V
    from stylus_zkvm_verifiers_b200 import synth as S
    outside, members = catalogue
    rng = S.SplitMix64(0x5C0A5000)

    def others(m):
        """m pairs whose product is 1: random (a G1, b G2) pairs closed by (-(sum a b) G1, G2); one pair: (a G1, infinity)"""
        if m == 1:
            return [V.mul(S.G1_GEN, rng.fr()) + SC.INF2]
        ab = [(rng.fr(), rng.fr()) for _ in range(m - 1)]
        return [V.mul(S.G1_GEN, a) + O.g2_mul(S.G2_GEN, b) for a, b in ab] + [V.mul(S.G1_GEN, -sum(a * b for a, b in ab)) + S.G2_GEN]
    j = 0
    for k in range(1, 5):
        inst, want = [], []
        for pos in range(k):
            for _ in range(3):
                b, (mname, m) = outside[j % len(outside)], SC.member_catalogue()[j % 8]
                j += 1
                rest = others(k - 1) if k > 1 else []
                for q, w in ((b.point, None), (m, O.w32(1))):
                    inst.append(b"".join(rest[:pos]) + SC.INF1 + q + b"".join(rest[pos:])); want.append(w)
        for data, w in zip(inst, want):
            assert O.ec_pairing(data) == w
        words, rev = Z.ec_pairing_batch(b"".join(inst), k, len(inst))
        assert rev.tolist() == [1 if w is None else 0 for w in want], k
        assert all(bytes(words[32 * i:32 * i + 32]) == w for i, w in enumerate(want) if w is not None), k
        for data, w in list(zip(inst, want))[:4]:
            assert Z.ec_pairing(data) == w, k
