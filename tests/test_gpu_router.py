"""RiscZeroVerifierRouter / Sp1VerifierGateway (zkv_risc0_router_*, zkv_sp1_gateway_*): records of many verifier versions in one batch, each
routed to the handle whose selector is its first 4 bytes.  Every status must equal the CPU oracle's for the selected route and the route
handle's own batch call on that record; records no route takes get the status every route handle gives them."""
import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
SIZES = [1, 31, 32, 33, 127, 129, 300]           # group sizes of the mixed batch's routes: warp and block edges


@pytest.fixture(scope="module")
def Z():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import stylus_zkvm_verifiers_b200 as Z
    return Z


@pytest.fixture(scope="module")
def S():
    from stylus_zkvm_verifiers_b200 import synth
    return synth


@pytest.fixture(scope="module")
def gpu(Z):
    return Z.GpuBackend(0)


def _load(Z, vk, devices=None):
    return Z.VerificationKey(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, devices=devices)


def _ovk(vk):
    return O.Vk(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)


class R0Route:
    """one RISC Zero route: its synthetic key, the handle (initialised on a control root) and the oracle of the same version"""

    def __init__(self, Z, vk, kv, control_root, control_id):
        self.vk, self.kv, self.cr, self.cid = vk, kv, control_root, control_id
        self.h = Z.RiscZeroVerifier(kv)
        self.h.initialize(control_root, control_id)
        self.sel = self.h.get_selector()
        self.oracle = O.Risc0Oracle(_ovk(vk))
        self.oracle.initialize(control_root, control_id)


def _r0_routes(Z, S, gpu, n_keys, roots_per_key, seed):
    rng = S.SplitMix64(seed)
    cid = O.w32(rng.fr())
    routes = []
    for k in range(n_keys):
        vk = S.make_vk(gpu, 0, 6, seed + 1 + k)
        kv = _load(Z, vk)
        for _ in range(roots_per_key):
            routes.append(R0Route(Z, vk, kv, rng.bytes(32), cid))
    return routes


def _r0_expect(routes, seals, ims, jrs, integrity=False):
    """the oracle of the route each seal selects; a seal no route takes: what every handle returns for it"""
    by_sel = {r.sel: r for r in routes}
    out = np.zeros(len(seals), dtype=np.uint8)
    for i, s in enumerate(seals):
        r = by_sel.get(bytes(s[:4]), routes[0])
        out[i] = r.oracle.verify_integrity(s, O.claim_digest(ims[i], jrs[i])) if integrity else r.oracle.verify(s, ims[i], jrs[i])
    return out


def _r0_own_calls(routes, seals, ims, jrs, integrity=False):
    """each record through the batch call of the handle its selector names (route 0's for a record no route takes)"""
    by_sel = {r.sel: j for j, r in enumerate(routes)}
    which = np.array([by_sel.get(bytes(s[:4]), 0) if len(s) >= 4 else 0 for s in seals])
    out = np.zeros(len(seals), dtype=np.uint8)
    for j, r in enumerate(routes):
        idx = np.nonzero(which == j)[0]
        if len(idx) == 0:
            continue
        if integrity:
            out[idx] = r.h.verify_integrity_batch([seals[i] for i in idx], [O.claim_digest(ims[i], jrs[i]) for i in idx])
        else:
            out[idx] = r.h.verify_batch([seals[i] for i in idx], [ims[i] for i in idx], [jrs[i] for i in idx])
    return out


@pytest.fixture(scope="module")
def mixed(Z, S, gpu, consts):
    """7 routes (4 control roots on one key, 3 other keys) with the group sizes of SIZES, mutated, plus unroutable and cross-routed seals"""
    sys0 = bytes.fromhex(consts["risc0_system_state_zero_digest"])
    routes = _r0_routes(Z, S, gpu, 1, 4, 0x60E000) + _r0_routes(Z, S, gpu, 3, 1, 0x60E100)
    rng = S.SplitMix64(0x60E200)
    seals, ims, jrs = [], [], []
    for j, (r, n) in enumerate(zip(routes, SIZES)):
        b = S.make_risc0_batch(gpu, r.vk, r.sel, r.cr, r.cid, sys0, n, 0x60E300 + j, pool=64)
        S.mutate_risc0(b, gpu, rng)
        seals += b.seals; ims += b.image_ids; jrs += b.journals
    good = S.make_risc0_batch(gpu, routes[0].vk, routes[0].sel, routes[0].cr, routes[0].cid, sys0, 8, 0x60E400, pool=8)
    cross = []
    for k in range(8):                                              # valid seals of route 0 relabelled with another route's selector
        cross.append(len(seals))
        seals.append(routes[1 + k % 6].sel + good.seals[k][4:]); ims.append(good.image_ids[k]); jrs.append(good.journals[k])
    extra = [b"", b"\x01", b"ab", good.seals[0][:3],                # shorter than 4 bytes
             good.seals[0][:259], good.seals[1] + b"\x00",          # routed, lengths 259 and 261
             b"\xde\xad\xbe\xef" + good.seals[2][4:], b"\x00\x00\x00\x00" + good.seals[3][4:], b"\xff\xff\xff\xff"]   # unknown selectors
    for e in extra:
        seals.append(e); ims.append(good.image_ids[0]); jrs.append(good.journals[0])
    seals += good.seals; ims += good.image_ids; jrs += good.journals
    order = np.random.default_rng(3).permutation(len(seals))
    seals, ims, jrs = [seals[i] for i in order], [ims[i] for i in order], [jrs[i] for i in order]
    cross = [int(np.nonzero(order == c)[0][0]) for c in cross]
    want = _r0_expect(routes, seals, ims, jrs)
    assert want.tolist() == _r0_own_calls(routes, seals, ims, jrs).tolist()       # the route handles agree with the oracle
    return dict(routes=routes, router=Z.RiscZeroVerifierRouter([r.h for r in routes]), seals=seals, ims=ims, jrs=jrs, want=want, cross=cross)


def test_mixed_batch_matches_oracle_and_route_calls(Z, mixed):
    got = mixed["router"].verify_batch(mixed["seals"], mixed["ims"], mixed["jrs"])
    want = mixed["want"]
    bad = [(i, int(got[i]), int(want[i])) for i in range(len(want)) if got[i] != want[i]]
    assert not bad, bad[:10]
    for st in (0, 2, 3, 4):
        assert (want == st).sum() >= 4, st
    sel_ok = {r.sel for r in mixed["routes"]}
    assert {bytes(mixed["seals"][i][:4]) for i in np.nonzero(want == 0)[0]} == sel_ok       # every route accepts some of its seals
    assert all(want[c] == 4 for c in mixed["cross"])                                      # cross-routed: VerificationFailed


def test_integrity_matches_oracle_and_route_calls(Z, mixed):
    claims = [O.claim_digest(a, b) for a, b in zip(mixed["ims"], mixed["jrs"])]
    got = mixed["router"].verify_integrity_batch(mixed["seals"], claims)
    want = _r0_expect(mixed["routes"], mixed["seals"], mixed["ims"], mixed["jrs"], integrity=True)
    assert want.tolist() == _r0_own_calls(mixed["routes"], mixed["seals"], mixed["ims"], mixed["jrs"], integrity=True).tolist()
    assert got.tolist() == want.tolist()
    assert (want == 0).sum() >= len(mixed["routes"])


def test_permuted_batch_gives_permuted_statuses(Z, mixed):
    perm = np.random.default_rng(11).permutation(len(mixed["want"]))
    got = mixed["router"].verify_batch([mixed["seals"][i] for i in perm], [mixed["ims"][i] for i in perm], [mixed["jrs"][i] for i in perm])
    assert got.tolist() == mixed["want"][perm].tolist()


def _fixed(mixed):
    """the mixed batch's 260-byte seals (the records the _device forms take)"""
    idx = [i for i, s in enumerate(mixed["seals"]) if len(s) == 260]
    return idx, b"".join(mixed["seals"][i] for i in idx), b"".join(mixed["ims"][i] for i in idx), b"".join(mixed["jrs"][i] for i in idx)


def test_device_form_on_a_side_stream_matches_host_call(Z, mixed):
    import torch
    idx, s, a, b = _fixed(mixed)
    n = len(idx)
    dev = lambda x: torch.from_numpy(np.frombuffer(x, dtype=np.uint8).copy()).cuda()
    d_s, d_a, d_b = dev(s), dev(a), dev(b)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d_st = torch.full((n,), 255, dtype=torch.uint8, device="cuda")
        mixed["router"].verify_batch_device(0, d_s.data_ptr(), d_a.data_ptr(), d_b.data_ptr(), n, d_st.data_ptr(), side.cuda_stream)
    side.synchronize()
    host = mixed["router"].verify_batch([mixed["seals"][i] for i in idx], [mixed["ims"][i] for i in idx], [mixed["jrs"][i] for i in idx])
    assert d_st.cpu().numpy().tolist() == host.tolist() == mixed["want"][idx].tolist()


def test_edge_routes(Z, S, gpu, consts):
    """a route whose control id is >= r and a route whose key has an invalid point fail every routed seal of the right length; length
    errors still give InvalidProofData, as on the route handle alone"""
    sys0 = bytes.fromhex(consts["risc0_system_state_zero_digest"])
    vk = S.make_vk(gpu, 0, 6, 0x60E500)
    kv = _load(Z, vk)
    rng = S.SplitMix64(0x60E501)
    ok = R0Route(Z, vk, kv, rng.bytes(32), O.w32(rng.fr()))
    big_id = R0Route(Z, vk, kv, rng.bytes(32), O.w32(R + 5))
    ic = list(vk.ic); ic[4] = O.w32(1) + O.w32(3)                   # IC4 off the curve
    bad_vk = S.SynthVk(0, vk.trap, vk.alpha, vk.beta, vk.gamma, vk.delta, ic)
    bad_key = R0Route(Z, bad_vk, _load(Z, bad_vk), rng.bytes(32), O.w32(rng.fr()))
    routes = [ok, big_id, bad_key]
    seals, ims, jrs = [], [], []
    for j, r in enumerate(routes):
        b = S.make_risc0_batch(gpu, vk, r.sel, r.cr, r.cid if r is not big_id else ok.cid, sys0, 40, 0x60E510 + j, pool=16)
        b.seals[0] = b.seals[0][:259]; b.seals[1] = b.seals[1] + b"\x07"; b.seals[2] = b.seals[2][:3]
        seals += b.seals; ims += b.image_ids; jrs += b.journals
    want = _r0_expect(routes, seals, ims, jrs)
    assert want.tolist() == _r0_own_calls(routes, seals, ims, jrs).tolist()
    for j in (1, 2):
        w = want[40 * j:40 * j + 40]
        assert w[:2].tolist() == [2, 2] and w[2] == 2 and (w[3:] == 4).all(), (j, w)
    assert (want[3:40] == 0).all()
    got = Z.RiscZeroVerifierRouter([r.h for r in routes]).verify_batch(seals, ims, jrs)
    assert got.tolist() == want.tolist()


def test_sp1_gateway_over_versions(Z, S, gpu, fx):
    """the embedded v5 handle plus handles of other verifier hashes and keys (zkv_sp1_create_version)"""
    v5 = Z.Sp1Verifier()
    routes = [(v5, O.sp1_vk(), None)]
    for k in range(3):
        vk = S.make_vk(gpu, 1, 3, 0x60E600 + k)
        h = O.sha256(b"sp1 verifier version %d" % k)
        handle = Z.Sp1Verifier(_load(Z, vk), verifier_hash=h, version="v%d.0.0-test" % (6 + k))
        assert handle.verifier_hash() == h and handle.version() == "v%d.0.0-test" % (6 + k)
        routes.append((handle, _ovk(vk), vk))
    assert v5.verifier_hash()[:4] == fx["sp1_selector"] and v5.version() == Z.Sp1Verifier().version()
    rng = S.SplitMix64(0x60E700)
    proofs, vkeys, pvs = [], [], []
    for j, (h, ovk, vk) in enumerate(routes):
        if vk is None:                                              # the embedded key: the reference's proof and tampers of it
            b = S.Sp1Batch([fx["sp1_proof"]] * 40, [fx["sp1_vkey"]] * 40, [fx["sp1_public_values"]] * 40, [0] * 40, ["valid"] * 40)
        else:
            b = S.make_sp1_batch(gpu, vk, SIZES[j + 2], 0x60E710 + j, pool=32, selector=h.verifier_hash()[:4])
        S.mutate_sp1(b, gpu, rng)
        proofs += b.proofs; vkeys += b.vkeys; pvs += b.public_values
    proofs += [b"", b"\x01\x02", b"\xde\xad\xbe\xef" + fx["sp1_proof"][4:]]
    vkeys += [fx["sp1_vkey"]] * 3; pvs += [fx["sp1_public_values"]] * 3
    order = np.random.default_rng(5).permutation(len(proofs))
    proofs, vkeys, pvs = [proofs[i] for i in order], [vkeys[i] for i in order], [pvs[i] for i in order]
    by_sel = {h.verifier_hash()[:4]: (h, ovk) for h, ovk, _ in routes}
    want = np.zeros(len(proofs), dtype=np.uint8); own = np.zeros(len(proofs), dtype=np.uint8)
    for i, p in enumerate(proofs):
        h, ovk = by_sel.get(bytes(p[:4]), routes[0][:2]) if len(p) >= 4 else routes[0][:2]
        want[i] = O.sp1_verify(ovk, h.verifier_hash()[:4], vkeys[i], pvs[i], p)
        own[i] = h.verify_batch([vkeys[i]], [pvs[i]], [p])[0]
    assert want.tolist() == own.tolist()
    for st in (0, 2, 3, 4):
        assert (want == st).sum() >= 2, st
    gw = Z.Sp1VerifierGateway([h for h, _, _ in routes])
    assert gw.verify_batch(vkeys, pvs, proofs).tolist() == want.tolist()
    # the device form on the 260-byte records with a fixed public-value length
    import torch
    idx = [i for i, p in enumerate(proofs) if len(p) == 260 and len(pvs[i]) == 96]
    dev = lambda x: torch.from_numpy(np.frombuffer(x, dtype=np.uint8).copy()).cuda()
    d_v, d_pv, d_p = dev(b"".join(vkeys[i] for i in idx)), dev(b"".join(pvs[i] for i in idx)), dev(b"".join(proofs[i] for i in idx))
    d_st = torch.full((len(idx),), 255, dtype=torch.uint8, device="cuda")
    gw.verify_batch_device(0, d_v.data_ptr(), d_pv.data_ptr(), 96, d_p.data_ptr(), len(idx), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert len(idx) > 100 and d_st.cpu().numpy().tolist() == want[idx].tolist()
    # single-proof calls: the route's errors, RouteNotFound without a route
    assert gw.verify_proof(fx["sp1_vkey"], fx["sp1_public_values"], fx["sp1_proof"]) is None
    with pytest.raises(Z.errors.RouteNotFound) as e:
        gw.verify_proof(fx["sp1_vkey"], fx["sp1_public_values"], b"\xde\xad\xbe\xef" + fx["sp1_proof"][4:])
    assert e.value.selector == b"\xde\xad\xbe\xef"
    with pytest.raises(Z.errors.VerificationFailed):
        gw.verify_proof(fx["sp1_vkey"][:31] + bytes([fx["sp1_vkey"][31] ^ 1]), fx["sp1_public_values"], fx["sp1_proof"])
    with pytest.raises(Z.errors.InvalidProofData):
        gw.verify_proof(fx["sp1_vkey"], fx["sp1_public_values"], fx["sp1_proof"][:200])


def test_single_calls_raise_the_route_errors(Z, mixed):
    router, routes = mixed["router"], mixed["routes"]
    i = int(np.nonzero(mixed["want"] == 0)[0][0])
    s, a, b = mixed["seals"][i], mixed["ims"][i], mixed["jrs"][i]
    assert router.verify(s, a, b) is True and router.verify_integrity(s, O.claim_digest(a, b)) is True
    assert router.get_verifier(s[:4]).get_selector() == s[:4]
    with pytest.raises(Z.errors.SelectorUnknown) as e:
        router.verify(b"\xde\xad\xbe\xef" + s[4:], a, b)
    assert e.value.selector == b"\xde\xad\xbe\xef" and e.value.payload[4:8] == b"\xde\xad\xbe\xef"
    with pytest.raises(Z.errors.SelectorUnknown):
        router.get_verifier(b"\xde\xad\xbe\xef")
    with pytest.raises(Z.errors.VerificationFailed):
        router.verify(s, a, bytes(32))
    with pytest.raises(Z.errors.InvalidProofData):
        router.verify(s[:259], a, b)
    with pytest.raises(Z.errors.InvalidProofData):
        router.verify_integrity(s[:2], O.claim_digest(a, b))
    assert len(router) == len(routes)


def test_pinned_and_pageable_inputs_agree(Z, big16):
    router, seals, ims, jrs, _ = big16
    n = 8192
    blob = b"".join(seals[:n]); off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in seals[:n]])
    a, b = b"".join(ims[:n]), b"".join(jrs[:n])
    pageable = router.verify_batch_packed(blob, off, a, b, n)
    pinned = router.verify_batch_packed(Z.pinned_copy(blob), Z.pinned_copy(off), Z.pinned_copy(a), Z.pinned_copy(b), n)
    assert pinned.tobytes() == pageable.tobytes() and 0 < int((pageable == 4).sum()) < n


def test_creation_errors(Z, S, gpu, mixed):
    from stylus_zkvm_verifiers_b200 import _native as N
    import ctypes as C
    hs = [r.h for r in mixed["routes"]]

    def refused(code, make):
        with pytest.raises(Z.ZkvError) as e:
            make()
        assert e.value.code == code

    refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter([]))
    refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter(hs * 37))                                   # 259 handles
    refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter([hs[0], hs[1], hs[0]]))                     # SelectorInUse
    twin = Z.RiscZeroVerifier(mixed["routes"][0].kv); twin.initialize(mixed["routes"][0].cr, mixed["routes"][0].cid)
    refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter([hs[0], twin]))                             # same version: same selector
    sp1 = Z.Sp1Verifier()
    refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter([hs[0], sp1]))                              # handles of different kinds
    refused(N.ZKV_ERR_ARG, lambda: Z.Sp1VerifierGateway([sp1, hs[0]]))
    refused(N.ZKV_ERR_ARG, lambda: Z.Sp1VerifierGateway([sp1, Z.Sp1Verifier()]))                        # two v5 handles
    refused(N.ZKV_ERR_STATE, lambda: Z.RiscZeroVerifierRouter([hs[0], Z.RiscZeroVerifier(mixed["routes"][0].kv)]))   # uninitialised
    refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter(hs, devices=[Z.device_count()]))            # no such device
    if Z.device_count() >= 2:
        refused(N.ZKV_ERR_ARG, lambda: Z.RiscZeroVerifierRouter(hs, devices=[0, 1]))                    # the keys are on device 0 only
    L = N.lib()
    out = C.c_void_p()
    arr = (C.c_void_p * 2)(hs[0]._h, None)
    assert L.zkv_risc0_router_create(arr, 2, None, 0, C.byref(out)) == N.ZKV_ERR_ARG                    # null handle
    assert L.zkv_sp1_gateway_create((C.c_void_p * 2)(sp1._h, None), 2, None, 0, C.byref(out)) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_create(None, 1, None, 0, C.byref(out)) == N.ZKV_ERR_ARG
    assert L.zkv_sp1_create_version(None, None, b"v", None, 0, C.byref(out)) == N.ZKV_ERR_ARG          # null verifier hash
    assert L.zkv_sp1_create_version(None, bytes(32), None, None, 0, C.byref(out)) == N.ZKV_ERR_ARG     # null version
    with pytest.raises(ValueError):
        Z.Sp1Verifier(version="v9")


def test_call_errors_leave_status_untouched(Z, mixed):
    from stylus_zkvm_verifiers_b200 import _native as N
    router, n = mixed["router"], 40
    seals = mixed["seals"][:n]
    blob = b"".join(seals); off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in seals])
    a, b = b"".join(mixed["ims"][:n]), b"".join(mixed["jrs"][:n])
    L = N.lib()
    st = np.full(n, 0xA5, dtype=np.uint8)
    bad = off.copy(); j = int(np.nonzero(np.diff(off) > 0)[0][1]); bad[j + 1] = bad[j] - 1
    assert L.zkv_risc0_router_verify_batch(router._h, N.buf(blob), bad.ctypes.data, N.buf(a), N.buf(b), n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_integrity_batch(router._h, N.buf(blob), bad.ctypes.data, N.buf(a), n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_batch(router._h, None, off.ctypes.data, N.buf(a), N.buf(b), n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_batch(router._h, N.buf(blob), None, N.buf(a), N.buf(b), n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_batch(router._h, N.buf(blob), off.ctypes.data, N.buf(a), None, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_integrity_batch(router._h, N.buf(blob), off.ctypes.data, None, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_batch(None, N.buf(blob), off.ctypes.data, N.buf(a), N.buf(b), n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert (st == 0xA5).all()
    assert L.zkv_risc0_router_verify_batch(router._h, None, None, None, None, 0, None) == 0                        # n == 0: nothing
    assert len(router.verify_batch([], [], [])) == 0
    assert L.zkv_risc0_router_verify_batch_device(router._h, 0, 1, 1, 1, 1 << 24, 1, None) == N.ZKV_ERR_ARG      # over 2^23
    assert L.zkv_risc0_router_verify_batch_device(router._h, Z.device_count(), 1, 1, 1, 1, 1, None) == N.ZKV_ERR_ARG
    assert L.zkv_risc0_router_verify_batch_device(router._h, 0, None, 1, 1, 1, 1, None) == N.ZKV_ERR_ARG
    gw = Z.Sp1VerifierGateway([Z.Sp1Verifier()])
    pv = np.zeros(n + 1, dtype=np.uint64)
    assert L.zkv_sp1_gateway_verify_batch(gw._h, N.buf(a), N.buf(a), pv.ctypes.data, N.buf(blob), bad.ctypes.data, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_sp1_gateway_verify_batch(gw._h, None, N.buf(a), pv.ctypes.data, N.buf(blob), off.ctypes.data, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_sp1_gateway_verify_batch_device(gw._h, 0, 1, 1, 96, 1, 1 << 24, 1, None) == N.ZKV_ERR_ARG
    assert (st == 0xA5).all()


def test_launch_count_per_call(Z, mixed):
    n = 100
    c0 = Z.launch_count()
    mixed["router"].verify_batch(mixed["seals"][:n], mixed["ims"][:n], mixed["jrs"][:n])
    assert Z.launch_count() - c0 == 11


def _tiled(Z, S, gpu, consts, routes, per_route, distinct, seed):
    """per_route seals of each route, tiled from `distinct` generated ones, one in eight with a tampered journal; random caller order"""
    sys0 = bytes.fromhex(consts["risc0_system_state_zero_digest"])
    seals, ims, jrs = [], [], []
    for j, r in enumerate(routes):
        b = S.make_risc0_batch(gpu, r.vk, r.sel, r.cr, r.cid, sys0, distinct, seed + j, pool=distinct)
        idx = np.arange(per_route) % distinct
        seals += [b.seals[i] for i in idx]; ims += [b.image_ids[i] for i in idx]
        jrs += [b.journals[i] if k % 8 != 3 else bytes(32) for k, i in enumerate(idx)]
    order = np.random.default_rng(seed).permutation(len(seals))
    return [seals[i] for i in order], [ims[i] for i in order], [jrs[i] for i in order]


@pytest.fixture(scope="module")
def big16(Z, S, gpu, consts):
    """2^16 seals over 16 routes (4 keys x 4 control roots)"""
    routes = _r0_routes(Z, S, gpu, 4, 4, 0x60E800)
    seals, ims, jrs = _tiled(Z, S, gpu, consts, routes, 4096, 64, 0x60E900)
    return Z.RiscZeroVerifierRouter([r.h for r in routes]), seals, ims, jrs, routes


def test_16_routes_2p16_match_route_calls(Z, big16):
    router, seals, ims, jrs, routes = big16
    c0 = Z.launch_count()
    got = router.verify_batch(seals, ims, jrs)
    assert Z.launch_count() - c0 == 42                                   # one chunked pass
    assert got.tolist() == _r0_own_calls(routes, seals, ims, jrs).tolist()
    assert (got == 4).sum() == (1 << 16) // 8 and (got == 0).sum() == (1 << 16) - (1 << 16) // 8
    first = {}
    for i, s in enumerate(seals):                                        # the oracle on one seal of each route
        first.setdefault(bytes(s[:4]), i)
    for r in routes:
        i = first[r.sel]
        assert got[i] == r.oracle.verify(seals[i], ims[i], jrs[i])


def test_one_route_router_equals_handle_call_at_2p16(Z, S, gpu, consts):
    routes = _r0_routes(Z, S, gpu, 1, 1, 0x60EA00)
    seals, ims, jrs = _tiled(Z, S, gpu, consts, routes, 1 << 16, 512, 0x60EB00)
    single = routes[0].h.verify_batch(seals, ims, jrs)
    got = Z.RiscZeroVerifierRouter([routes[0].h]).verify_batch(seals, ims, jrs)
    assert got.tobytes() == single.tobytes()
    assert (got == 4).sum() == (1 << 16) // 8


def test_router_workspace_growth_under_an_async_device_call(Z, S, gpu, consts):
    """On a fresh router (empty workspace), a small device call and at once, on another stream, a larger one that grows every buffer of the
    router: the second must wait for the first before it frees anything.  Both must give the host call's bytes on a second router."""
    import torch
    routes = _r0_routes(Z, S, gpu, 1, 3, 0x60EC00)
    small, big = _tiled(Z, S, gpu, consts, routes, 40, 16, 0x60EC10), _tiled(Z, S, gpu, consts, routes, 7000, 32, 0x60EC20)
    ref, rt = Z.RiscZeroVerifierRouter([r.h for r in routes]), Z.RiscZeroVerifierRouter([r.h for r in routes])
    dev = lambda a: torch.from_numpy(np.frombuffer(a, dtype=np.uint8).copy()).cuda()
    calls = []
    for seals, ims, jrs in (small, big):
        want = ref.verify_batch(seals, ims, jrs)
        calls.append((want, [dev(b"".join(seals)), dev(b"".join(ims)), dev(b"".join(jrs))], torch.full((len(seals),), 255, dtype=torch.uint8, device="cuda")))
    assert len(big[0]) > 8192 and 0 < int((calls[1][0] == 0).sum()) < len(big[0])
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for (want, d, d_st), st in zip(calls, streams):
        rt.verify_batch_device(0, *[x.data_ptr() for x in d], len(want), d_st.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    for want, _, d_st in calls:
        assert d_st.cpu().numpy().tolist() == want.tolist()


def test_router_over_all_devices_matches_one_device(Z, S, gpu, consts):
    nd = Z.device_count()
    if nd < 2:
        pytest.skip("one CUDA device")
    devs = list(range(nd))
    rng = S.SplitMix64(0x60ED00)
    vk = S.make_vk(gpu, 0, 6, 0x60ED01)
    kv1, kva = _load(Z, vk), _load(Z, vk, devs)
    crs = [rng.bytes(32) for _ in range(3)]
    cid = O.w32(rng.fr())
    one = [R0Route(Z, vk, kv1, cr, cid) for cr in crs]
    alls = [R0Route(Z, vk, kva, cr, cid) for cr in crs]
    seals, ims, jrs = _tiled(Z, S, gpu, consts, one, 4096, 64, 0x60ED10)
    a = Z.RiscZeroVerifierRouter([r.h for r in one]).verify_batch(seals, ims, jrs)
    b = Z.RiscZeroVerifierRouter([r.h for r in alls], devices=devs).verify_batch(seals, ims, jrs)
    assert a.tobytes() == b.tobytes() and (a == 4).sum() == 3 * 512
