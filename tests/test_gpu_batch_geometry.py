"""Batch shapes past the edges the other GPU tests stay inside: host-buffer calls longer than one device pass (MAX_CHUNK = 2^20 records)
with offsets that start past 0 and records whose length changes across the pass edge; the pairing services past their own chunks
(2^18, 2^16) and up to the 64-pair limit; every *_device entry point at its size limit 2^23 (byte offsets past 2^31 and 2^32) and one
above it; the chunk / segment schedule at size; SP1 public values of any length.  Batches are position-coded (tests/batch_geometry.py):
every status byte is checked against the expectation of its position's code, and sampled positions (pass and chunk edges, both ends,
random ones) against the CPU oracle."""
import contextlib
import gc
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import batch_geometry as G
import oracle_lib as O

pytestmark = pytest.mark.gpu

N1 = G.PASS + 5                                   # a second pass of 5 records (one chain)
N2 = 2 * G.PASS + (1 << 18) + 37                  # three passes, the last one cut into pieces
PASS_EDGE = (G.PASS - 1, G.PASS)                  # records with a changed length on both sides of the first pass edge
DEVICE_CLASSES = (G.KEEP, G.TAMPER, G.SELECTOR)
OFF31 = -(-(1 << 31) // 260)                      # first 260-byte record whose byte offset is past 2^31
SEED = 0xB6E0_1000


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


def _load(Z, vk):
    return Z.VerificationKey(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)


def _ovk(vk):
    return O.Vk(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)


def _same(got, want, what=""):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, "%s: %d of %d statuses differ, first (position, got, want): %s" % (
        what, len(bad), len(want), [(int(i), int(got[i]), int(want[i])) for i in bad[:8]])


def _pmap(fn, items):
    with ThreadPoolExecutor(8) as ex:
        return list(ex.map(fn, items))


@contextlib.contextmanager
def _released(*objs):
    """close verifier objects (routers / sets first, keys last) and return the freed device memory before the next large case"""
    import torch
    try:
        yield
    finally:
        for o in objs:
            o.close()
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


# ------------------------------------------------------------------ launch counts (include/zkv.h, test_gpu_parity.py::test_launch_counter_and_wave_size)
def _chunked(Z, slots):
    return slots >= max(8192, Z.wave_proofs(0, 0) // 2)


def _host_launches(Z, n, segs=4, overlap=0):
    """a verifier handle's host-buffer call: per pass 6 launches as one chain, 4 pieces x (4 front + segs Miller + 4 final-exp) when chunked"""
    per = lambda m: 6 if overlap == 1 or not _chunked(Z, m) else 4 * (4 + segs + 4)
    return sum(per(min(G.PASS, n - s)) for s in range(0, n, G.PASS))


def _grouped_launches(Z, n, n_keys, router):
    """a key set's (router's) host-buffer call: per pass 10 (11) as one chain, 41 (42) once the slot bound is chunked"""
    def per(m):
        slots = (m + 31 * min(n_keys, m) + 31) // 32 * 32
        return (41 if _chunked(Z, slots) else 10) + (1 if router else 0)
    return sum(per(min(G.PASS, n - s)) for s in range(0, n, G.PASS))


# ------------------------------------------------------------------ fixtures: keys, handles, oracles, pools
@pytest.fixture(scope="module")
def r0(Z, S, gpu, fx):
    """one RISC Zero handle on a synthetic key and a router over 4 routes (2 keys x 2 control roots), with their oracles and pools"""
    rng = S.SplitMix64(SEED)
    cid = O.w32(rng.fr())
    keys = [S.make_vk(gpu, 0, 6, SEED + 1 + k) for k in range(2)]
    kvs = [_load(Z, vk) for vk in keys]
    routes = []
    for k in range(2):
        for _ in range(2):
            cr = rng.bytes(32)
            h = Z.RiscZeroVerifier(kvs[k]); h.initialize(cr, cid)
            o = O.Risc0Oracle(_ovk(keys[k])); o.initialize(cr, cid)
            assert o.selector() == h.get_selector() and h.get_selector() != G.UNKNOWN_SELECTOR
            routes.append(dict(vk=keys[k], h=h, o=o, cr=cr, cid=cid, sel=h.get_selector()))
    spec = lambda r: (r["vk"], r["sel"], r["cr"], r["cid"])
    return dict(keys=keys, kvs=kvs, routes=routes, h=routes[0]["h"], router=Z.RiscZeroVerifierRouter([r["h"] for r in routes]),
                pool=G.Risc0Pool(gpu, [spec(routes[0])], fx["sys0"], SEED + 10),
                rpool=G.Risc0Pool(gpu, [spec(r) for r in routes], fx["sys0"], SEED + 11))


def _r0_oracle(routes, blob, off, a, b, idx, integrity=False):
    by_sel = {r["sel"]: r["o"] for r in routes}
    seals = G.slices(blob, off, idx)

    def one(t):
        i, s = t
        o = by_sel.get(bytes(s[:4]), routes[0]["o"])
        return o.verify_integrity(s, a[i].tobytes()) if integrity else o.verify(s, a[i].tobytes(), b[i].tobytes())
    return np.array(_pmap(one, list(zip(idx, seals))), dtype=np.uint8)


def _pv_lengths(seed):
    """public-value lengths of an SP1 pool: 0..300 spread over the pool, and a few long ones"""
    L = (np.arange(G.D) * 37 + seed) % 301
    L[[5, 50, 500, 1000]] = (447, 1024, 4096, 4095)
    return L


@pytest.fixture(scope="module")
def sp1(Z, S, gpu):
    """three SP1 verifier versions (own keys and verifier hashes) and their gateway; the handle of version 0 alone"""
    keys = [S.make_vk(gpu, 1, 3, SEED + 20 + k) for k in range(3)]
    kvs = [_load(Z, vk) for vk in keys]
    hs = [Z.Sp1Verifier(kvs[k], verifier_hash=O.sha256(b"geometry version %d" % k), version="v%d-geometry" % k) for k in range(3)]
    routes = [dict(vk=keys[k], h=hs[k], o=_ovk(keys[k]), sel=hs[k].verifier_hash()[:4]) for k in range(3)]
    return dict(keys=keys, kvs=kvs, routes=routes, h=hs[0], gateway=Z.Sp1VerifierGateway(hs),
                pool=G.Sp1Pool(gpu, [(keys[0], routes[0]["sel"])], _pv_lengths(0), SEED + 21),
                gpool=G.Sp1Pool(gpu, [(r["vk"], r["sel"]) for r in routes], _pv_lengths(7), SEED + 22))


def _sp1_oracle(routes, vkeys, pv, pv_off, proofs, proof_off, idx):
    by_sel = {r["sel"]: r for r in routes}
    recs = G.slices(proofs, proof_off, idx)
    pvs = G.slices(pv, pv_off, idx)

    def one(t):
        i, p, v = t
        r = by_sel.get(bytes(p[:4]), routes[0])
        return O.sp1_verify(r["o"], r["sel"], vkeys[i].tobytes(), v, p)
    return np.array(_pmap(one, list(zip(idx, recs, pvs))), dtype=np.uint8)


@pytest.fixture(scope="module")
def generic(Z, S, gpu):
    """five keys of different n_ic and vm in one key set; a single key (n_ic 3) for Groth16Verifier.verify_batch"""
    keys = [S.make_vk(gpu, k % 2, n_ic, SEED + 30 + k) for k, n_ic in enumerate((2, 3, 4, 6, 9))]
    kvs = [_load(Z, vk) for vk in keys]
    one = S.make_vk(gpu, 1, 3, SEED + 40)
    return dict(keys=keys, kvs=kvs, ovks=[_ovk(k) for k in keys], keyset=Z.VerificationKeySet(kvs), pool=G.GenericPool(gpu, keys, SEED + 31),
                one=one, one_kv=_load(Z, one), one_pool=G.GenericPool(gpu, [one], SEED + 41))


# ------------------------------------------------------------------ a) host forms past one pass
def _host_edges(n):
    return G.schedule_edges(n) + list(PASS_EDGE)


@pytest.mark.parametrize("n", [N1, N2])
def test_risc0_handle_host_form_past_one_pass(Z, r0, n):
    cls, sub = G.codes(SEED + n, n, force_length=PASS_EDGE)
    blob, off, ims, jrs = G.risc0_host(r0["pool"], G.tiled(n), cls, sub)
    assert off[0] == G.SEAL_PREFIX and off[G.PASS] - off[G.PASS - 1] != 260
    c0 = Z.launch_count()
    got = r0["h"].verify_batch_packed(blob, off, ims, jrs, n)
    assert Z.launch_count() - c0 == _host_launches(Z, n)
    _same(got, G.STATUS[cls], "risc0 handle n=%d" % n)
    idx = G.samples(n, n, _host_edges(n))
    _same(_r0_oracle(r0["routes"][:1], blob, off, ims, jrs, idx), got[idx], "oracle")
    if n == N2:          # every input page-locked: the in-place upload path
        pinned = r0["h"].verify_batch_packed(Z.pinned_copy(blob), Z.pinned_copy(off), Z.pinned_copy(ims), Z.pinned_copy(jrs), n)
        assert pinned.tobytes() == got.tobytes()
        # d) the schedule at size: one chain per pass, and seven Miller segments per piece, give the same bytes
        h = r0["h"]
        try:
            h.tune("overlap", 1)
            c0 = Z.launch_count()
            assert h.verify_batch_packed(blob, off, ims, jrs, n).tobytes() == got.tobytes()
            assert Z.launch_count() - c0 == _host_launches(Z, n, overlap=1)
            h.tune("overlap", 0)
            h.tune("miller_segments", 7)
            c0 = Z.launch_count()
            assert h.verify_batch_packed(blob, off, ims, jrs, n).tobytes() == got.tobytes()
            assert Z.launch_count() - c0 == _host_launches(Z, n, segs=7)
        finally:
            h.tune("overlap", 0)
            h.tune("miller_segments", 4)


def test_risc0_integrity_host_form_past_one_pass(Z, r0):
    from stylus_zkvm_verifiers_b200 import _native as N
    n = N1
    cls, sub = G.codes(SEED + 2, n, force_length=PASS_EDGE)
    blob, off, claims, _ = G.risc0_host(r0["pool"], G.tiled(n), cls, sub, integrity=True)
    got = np.full(n, 0xEE, dtype=np.uint8)
    N.check(N.lib().zkv_risc0_verify_integrity_batch(r0["h"]._h, N.buf(blob), off.ctypes.data, N.buf(claims), n, got.ctypes.data))
    _same(got, G.STATUS[cls], "risc0 integrity")
    idx = G.samples(n, 2, _host_edges(n))
    _same(_r0_oracle(r0["routes"][:1], blob, off, claims, None, idx, integrity=True), got[idx], "oracle")


@pytest.mark.parametrize("n", [N1, N2])
def test_risc0_router_host_form_past_one_pass(Z, r0, n):
    cls, sub = G.codes(SEED + 3 + n, n, force_length=PASS_EDGE)
    blob, off, ims, jrs = G.risc0_host(r0["rpool"], G.tiled(n), cls, sub)
    c0 = Z.launch_count()
    got = r0["router"].verify_batch_packed(blob, off, ims, jrs, n)
    assert Z.launch_count() - c0 == _grouped_launches(Z, n, len(r0["routes"]), router=True)
    _same(got, G.STATUS[cls], "risc0 router n=%d" % n)
    idx = G.samples(n, 3, _host_edges(n))
    _same(_r0_oracle(r0["routes"], blob, off, ims, jrs, idx), got[idx], "oracle")


@pytest.mark.parametrize("n", [N1, N2])
def test_sp1_handle_host_form_past_one_pass(Z, sp1, n):
    cls, sub = G.codes(SEED + 4 + n, n, force_length=PASS_EDGE)
    vkeys, pv, pv_off, proofs, proof_off = G.sp1_host(sp1["pool"], G.tiled(n), cls, sub)
    c0 = Z.launch_count()
    got = sp1["h"].verify_batch_packed(vkeys, pv, pv_off, proofs, proof_off, n)
    assert Z.launch_count() - c0 == _host_launches(Z, n)
    _same(got, G.STATUS[cls], "sp1 handle n=%d" % n)
    idx = G.samples(n, 4, _host_edges(n))
    _same(_sp1_oracle(sp1["routes"][:1], vkeys, pv, pv_off, proofs, proof_off, idx), got[idx], "oracle")


@pytest.mark.parametrize("n", [N1, N2])
def test_sp1_gateway_host_form_past_one_pass(Z, sp1, n):
    cls, sub = G.codes(SEED + 5 + n, n, force_length=PASS_EDGE)
    vkeys, pv, pv_off, proofs, proof_off = G.sp1_host(sp1["gpool"], G.tiled(n), cls, sub)
    assert pv_off[0] == G.PV_PREFIX and proof_off[0] == G.SEAL_PREFIX
    c0 = Z.launch_count()
    got = sp1["gateway"].verify_batch_packed(vkeys, pv, pv_off, proofs, proof_off, n)
    assert Z.launch_count() - c0 == _grouped_launches(Z, n, len(sp1["routes"]), router=True)
    _same(got, G.STATUS[cls], "sp1 gateway n=%d" % n)
    idx = G.samples(n, 5, _host_edges(n))
    _same(_sp1_oracle(sp1["routes"], vkeys, pv, pv_off, proofs, proof_off, idx), got[idx], "oracle")
    if n == N2:
        pinned = sp1["gateway"].verify_batch_packed(*[Z.pinned_copy(a) for a in (vkeys, pv, pv_off, proofs, proof_off)], n)
        assert pinned.tobytes() == got.tobytes()


@pytest.mark.parametrize("n", [N1, N2])
def test_key_set_host_form_past_one_pass(Z, generic, n):
    nk = len(generic["keys"])
    cls, sub = G.codes(SEED + 6 + n, n, force_length=PASS_EDGE)
    key, proofs, sig, off = G.generic_host(generic["pool"], G.tiled(n), cls, sub, nk)
    assert off[0] == G.SIG_PREFIX and off[G.PASS] - off[G.PASS - 1] != generic["pool"].nsig[(G.PASS - 1) % G.D]
    c0 = Z.launch_count()
    got = Z.Groth16Verifier.verify_batch_keys_packed(generic["keyset"], key, proofs, sig, off)
    assert Z.launch_count() - c0 == _grouped_launches(Z, n, nk, router=False)
    _same(got, G.generic_expect(cls), "key set n=%d" % n)
    idx = G.samples(n, 6, _host_edges(n))
    words = lambda i: sig[int(off[i]) * 32:int(off[i + 1]) * 32].tobytes()
    want = _pmap(lambda i: O.groth16_verify(generic["ovks"][key[i]], proofs[i].tobytes(), words(i)), idx)
    _same(got[idx], want, "oracle")


@pytest.mark.parametrize("n", [N1, N2])
def test_groth16_single_key_host_form_past_one_pass(Z, generic, n):
    cls, sub = G.codes(SEED + 7 + n, n, classes=(G.KEEP, G.TAMPER))
    _, proofs, sig, _ = G.generic_host(generic["one_pool"], G.tiled(n), cls, sub, 1)
    sig = sig[G.SIG_PREFIX * 32:]
    k = generic["one"].k
    assert len(sig) == n * k * 32
    c0 = Z.launch_count()
    got = Z.Groth16Verifier.verify_batch(generic["one_kv"], proofs, sig, k, n)
    assert Z.launch_count() - c0 == _host_launches(Z, n)
    _same(got, G.generic_expect(cls), "groth16 n=%d" % n)
    idx = G.samples(n, 7, G.schedule_edges(n))
    ovk = _ovk(generic["one"])
    want = _pmap(lambda i: O.groth16_verify(ovk, proofs[i].tobytes(), sig[i * k * 32:(i + 1) * k * 32].tobytes()), idx)
    _same(got[idx], want, "oracle")


# ------------------------------------------------------------------ b) the pairing services past their chunks
def test_pairing4_host_past_its_chunks(Z, S, gpu):
    n = G.PAIRING4_CHUNK + (1 << 16) + 3
    vk = S.make_vk(gpu, 0, 2, SEED + 50)
    kv = _load(Z, vk)
    with _released(kv):
        pool = G.PairingPool(gpu, SEED + 51, vk=vk)
        cls, _ = G.codes(SEED + 52, n, classes=DEVICE_CLASSES)
        g1, g2, want = G.pairing4_host(pool, G.tiled(n), cls)
        ok, gt, ml = Z.pairing4_batch(kv, g1, g2, n, want_gt=True, want_miller=True)
        _same(ok, want, "pairing4 ok")
        idx = G.samples(n, 52, G.schedule_edges(n, G.PAIRING4_CHUNK))
        blob = np.ascontiguousarray(G.pairing4_oracle_blob(g1[idx], g2[idx], vk))
        ook, ogt, oml = O.pairing4_batch(blob.ctypes.data, len(idx), want_gt=True, want_miller=True)
        _same(ok[idx], ook, "oracle ok")
        gt, ml = gt.reshape(n, 384), ml.reshape(n, 384)
        assert gt[idx].tobytes() == ogt.tobytes()                     # zeroed where the call reverts
        live = idx[ok[idx] != 2]                                         # the Miller value is defined where it does not
        assert ml[live].tobytes() == oml.reshape(-1, 384)[ok[idx] != 2].tobytes()


def test_ec_pairing_past_its_chunk(Z, gpu):
    n = G.EC_PAIRING_CHUNK + 3
    pool = G.PairingPool(gpu, SEED + 60)
    cls, _ = G.codes(SEED + 61, n, classes=DEVICE_CLASSES)
    x, want = G.ec_pairing_host(pool, G.tiled(n), cls)
    words, rev, ml = Z.ec_pairing_batch(x, 2, n, want_miller=True)
    words = words.reshape(n, 32)
    _same(rev, (want == 2).astype(np.uint8), "reverted")
    _same(words[:, 31], np.where(want == 2, 0, want), "return word")
    assert not words[:, :31].any()
    idx = G.samples(n, 61, [G.EC_PAIRING_CHUNK])
    ml = ml.reshape(n, 384)
    for i, r in zip(idx, _pmap(lambda i: O.ec_pairing(x[i].tobytes(), debug=True), idx)):
        if r is None:
            assert want[i] == 2 and not ml[i].any()
        else:
            assert r[0][31] == words[i, 31] and r[1] == ml[i].tobytes(), i


@pytest.mark.parametrize("k", [7, 16, 33, 64])
def test_ec_pairing_many_pairs_at_the_block_edge(Z, S, gpu, k):
    """k pairs per instance, n around the 128-thread block: products one by bilinearity and not, members at infinity, an invalid pair at
    the first or at the last pair index"""
    rng = S.SplitMix64(SEED + 70 + k)
    pools = S.Pools(gpu, rng, 64)
    for n in (127, 129):
        insts, sums = [], []
        for i in range(n):
            ja, jb = [rng.below(64) for _ in range(k - 1)], [rng.below(64) for _ in range(k - 1)]
            pairs = [pools.A[a] + pools.B[b] for a, b in zip(ja, jb)]
            s = 0
            for t, (a, b) in enumerate(zip(ja, jb)):
                if i % 5 == 1 and t == i % (k - 1):
                    pairs[t] = bytes(64) + pairs[t][64:]                 # G1 member at infinity: the pair contributes one
                elif i % 5 == 2 and t == (i * 3) % (k - 1):
                    pairs[t] = pairs[t][:64] + bytes(128)                # G2 member at infinity
                else:
                    s += pools.a[a] * pools.b[b]
            insts.append(pairs)
            sums.append((-(s + (i % 2))) % S.R)                           # odd instances: product not one
        last = gpu.g1_mul(sums)
        for i in range(n):
            insts[i].append(last[i] + S.G2_GEN)
            if i % 11 == 3:
                insts[i][0] = G.BAD_G1 + insts[i][0][64:]
            elif i % 11 == 4:
                insts[i][k - 1] = G.BAD_G1 + insts[i][k - 1][64:]
        data = b"".join(b"".join(p) for p in insts)
        words, rev, ml = Z.ec_pairing_batch(data, k, n, want_miller=True)
        words, ml = words.reshape(n, 32), ml.reshape(n, 384)
        want = _pmap(lambda i: O.ec_pairing(b"".join(insts[i]), debug=True), range(n))
        for i, r in enumerate(want):
            if r is None:
                assert rev[i] == 1 and not words[i].any() and not ml[i].any(), (k, n, i)
            else:
                assert rev[i] == 0 and words[i].tobytes() == r[0] and ml[i].tobytes() == r[1], (k, n, i)
        assert {int(words[i, 31]) for i in range(n) if not rev[i]} == {0, 1}
        assert rev[3] == rev[4] == 1 and words[0, 31] == 1 and words[1, 31] == 0


def test_ec_pairing_refuses_more_than_64_pairs(Z, gpu):
    from stylus_zkvm_verifiers_b200 import _native as N
    pair = gpu.g1_mul([5])[0] + gpu.g2_mul([7])[0]
    with pytest.raises(Z.ZkvError) as e:
        Z.ec_pairing(pair * 65)
    assert e.value.code == N.ZKV_ERR_ARG
    with pytest.raises(Z.ZkvError) as e:
        Z.ec_pairing_batch(pair * 65, 65, 1)
    assert e.value.code == N.ZKV_ERR_ARG
    assert Z.ec_pairing(pair * 64) == O.ec_pairing(pair * 64)


# ------------------------------------------------------------------ c) device forms at the size limit
def _device_samples(n, seed):
    return G.samples(n, seed, G.schedule_edges(n, n) + [OFF31, n // 2])


def _status(n):
    import torch
    return torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")


def _refuses_one_more(fn, ptrs):
    """n = 2^23 + 1 returns ZKV_ERR_ARG and leaves the status buffer alone"""
    import torch
    from stylus_zkvm_verifiers_b200 import _native as N
    st = torch.full((64,), 0xA5, dtype=torch.uint8, device="cuda")
    assert fn(*ptrs, G.DEVICE_MAX + 1, st.data_ptr(), None) == N.ZKV_ERR_ARG
    torch.cuda.synchronize()
    assert (st == 0xA5).all()


@pytest.mark.parametrize("n", [G.DEVICE_MAX, 3 * G.PASS + 77])
def test_risc0_handle_device_form_at_the_limit(Z, r0, n):
    import torch
    from stylus_zkvm_verifiers_b200 import _native as N
    kv = _load(Z, r0["keys"][0])
    r = r0["routes"][0]
    h = Z.RiscZeroVerifier(kv)
    h.initialize(r["cr"], r["cid"])
    with _released(h, kv):
        cls, sub = G.codes(SEED + 80 + n, n, classes=DEVICE_CLASSES)
        seals, ims, jrs = G.risc0_device(r0["pool"], *G.device_codes(cls, sub))
        st = _status(n)
        h.verify_batch_device(0, seals.data_ptr(), ims.data_ptr(), jrs.data_ptr(), n, st.data_ptr())
        torch.cuda.synchronize()
        got = st.cpu().numpy()
        _same(got, G.STATUS[cls], "risc0 device n=%d" % n)
        idx = _device_samples(n, 80)
        blob, off, a, b = G.risc0_host(r0["pool"], idx % G.D, cls[idx], sub[idx])
        ti = torch.from_numpy(idx).cuda()
        assert seals[ti].cpu().numpy().tobytes() == blob[G.SEAL_PREFIX:].tobytes() and jrs[ti].cpu().numpy().tobytes() == b.tobytes()
        _same(_r0_oracle(r0["routes"][:1], blob, off, a, b, np.arange(len(idx))), got[idx], "oracle")
        if n == G.DEVICE_MAX:
            _refuses_one_more(lambda *p: N.lib().zkv_risc0_verify_batch_device(h._h, 0, *p), (seals.data_ptr(), ims.data_ptr(), jrs.data_ptr()))


def test_risc0_router_device_form_at_the_limit(Z, r0):
    import torch
    from stylus_zkvm_verifiers_b200 import _native as N
    n = G.DEVICE_MAX
    router = Z.RiscZeroVerifierRouter([r["h"] for r in r0["routes"]])
    with _released(router):
        cls, sub = G.codes(SEED + 81, n, classes=DEVICE_CLASSES)
        seals, ims, jrs = G.risc0_device(r0["rpool"], *G.device_codes(cls, sub))
        st = _status(n)
        router.verify_batch_device(0, seals.data_ptr(), ims.data_ptr(), jrs.data_ptr(), n, st.data_ptr())
        torch.cuda.synchronize()
        got = st.cpu().numpy()
        _same(got, G.STATUS[cls], "risc0 router device")
        idx = _device_samples(n, 81)
        blob, off, a, b = G.risc0_host(r0["rpool"], idx % G.D, cls[idx], sub[idx])
        _same(_r0_oracle(r0["routes"], blob, off, a, b, np.arange(len(idx))), got[idx], "oracle")
        _refuses_one_more(lambda *p: N.lib().zkv_risc0_router_verify_batch_device(router._h, 0, *p), (seals.data_ptr(), ims.data_ptr(), jrs.data_ptr()))


def _sp1_device_check(routes, pool, n, stride, seed, run, raw):
    import torch
    cls, sub = G.codes(seed, n, classes=DEVICE_CLASSES)
    vkeys, pv, proofs = G.sp1_device(pool, *G.device_codes(cls, sub), stride)
    st = _status(n)
    run(vkeys.data_ptr(), pv.data_ptr(), stride, proofs.data_ptr(), n, st.data_ptr())
    torch.cuda.synchronize()
    got = st.cpu().numpy()
    _same(got, G.STATUS[cls], "sp1 device n=%d stride=%d" % (n, stride))
    idx = _device_samples(n, seed) if n > 1000 else np.arange(n)
    hv, hpv, hp = G.sp1_fixed_host(pool, idx % G.D, cls[idx], sub[idx], stride)
    m = len(idx)
    pv_off = (np.arange(m + 1) * stride).astype(np.uint64)
    proof_off = (np.arange(m + 1) * 260).astype(np.uint64)
    flat = np.ascontiguousarray(hpv).reshape(-1)
    _same(_sp1_oracle(routes, hv, flat, pv_off, hp.reshape(-1), proof_off, np.arange(m)), got[idx], "oracle")
    if stride and n > 1000:
        ti = torch.from_numpy(idx).cuda()
        assert pv[ti].cpu().numpy().tobytes() == flat.tobytes()
    if raw is not None:
        _refuses_one_more(lambda *p: raw(p[0], p[1], stride, p[2], *p[3:]), (vkeys.data_ptr(), pv.data_ptr(), proofs.data_ptr()))


@pytest.fixture(scope="module")
def sp1_520(sp1, gpu):
    """pools of 520-byte public values: n x 520 bytes passes 2^32 at n = 2^23"""
    return (G.Sp1Pool(gpu, [(sp1["keys"][0], sp1["routes"][0]["sel"])], [520] * G.D, SEED + 90),
            G.Sp1Pool(gpu, [(r["vk"], r["sel"]) for r in sp1["routes"]], [520] * G.D, SEED + 91))


def test_sp1_handle_device_form_at_the_limit(Z, sp1, sp1_520):
    from stylus_zkvm_verifiers_b200 import _native as N
    r = sp1["routes"][0]
    kv = _load(Z, r["vk"])
    h = Z.Sp1Verifier(kv, verifier_hash=r["h"].verifier_hash(), version="v0-geometry")
    with _released(h, kv):
        _sp1_device_check(sp1["routes"][:1], sp1_520[0], G.DEVICE_MAX, 520, SEED + 92,
                          lambda *p: h.verify_batch_device(0, *p), lambda *p: N.lib().zkv_sp1_verify_batch_device(h._h, 0, *p))


def test_sp1_gateway_device_form_at_the_limit(Z, sp1, sp1_520):
    from stylus_zkvm_verifiers_b200 import _native as N
    gw = Z.Sp1VerifierGateway([r["h"] for r in sp1["routes"]])
    with _released(gw):
        _sp1_device_check(sp1["routes"], sp1_520[1], G.DEVICE_MAX, 520, SEED + 93,
                          lambda *p: gw.verify_batch_device(0, *p), lambda *p: N.lib().zkv_sp1_gateway_verify_batch_device(gw._h, 0, *p))


def test_key_set_device_form_at_the_limit(Z, generic):
    import torch
    from stylus_zkvm_verifiers_b200 import _native as N
    n, nk = G.DEVICE_MAX, len(generic["keys"])
    ks = Z.VerificationKeySet(generic["kvs"])
    with _released(ks):
        cls, sub = G.codes(SEED + 94, n, classes=DEVICE_CLASSES)
        key, proofs, sig, off = G.generic_device(generic["pool"], *G.device_codes(cls, sub), nk)
        st = _status(n)
        Z.Groth16Verifier.verify_batch_keys_device(ks, 0, key.data_ptr(), proofs.data_ptr(), sig.data_ptr(), off.data_ptr(), n, st.data_ptr())
        torch.cuda.synchronize()
        got = st.cpu().numpy()
        _same(got, G.generic_expect(cls), "key set device")
        idx = _device_samples(n, 94)
        hk, hp, hs = G.generic_fixed_host(generic["pool"], idx % G.D, cls[idx], sub[idx], nk)
        want = _pmap(lambda t: O.groth16_verify(generic["ovks"][t[0]], t[1].tobytes(), t[2]) if t[0] < nk else O.ST_VERIFICATION_FAILED,
                     list(zip(hk, hp, hs)))
        _same(got[idx], want, "oracle")
        _refuses_one_more(lambda *p: N.lib().zkv_groth16_verify_batch_keys_device(ks._h, 0, *p),
                          (key.data_ptr(), proofs.data_ptr(), sig.data_ptr(), off.data_ptr()))


def test_pairing4_device_form_at_the_limit(Z, S, gpu):
    import torch
    from stylus_zkvm_verifiers_b200 import _native as N
    n = G.DEVICE_MAX
    vk = S.make_vk(gpu, 0, 2, SEED + 95)
    kv = _load(Z, vk)
    with _released(kv):
        pool = G.PairingPool(gpu, SEED + 96, vk=vk)
        cls, sub = G.codes(SEED + 97, n, classes=DEVICE_CLASSES)
        g1, g2 = G.pairing4_device(pool, G.device_codes(cls, sub)[0])
        ok = _status(n)
        gt = torch.empty((n, 384), dtype=torch.uint8, device="cuda")
        N.check(N.lib().zkv_pairing4_batch_device(kv._h, 0, g1.data_ptr(), g2.data_ptr(), n, ok.data_ptr(), gt.data_ptr(), None))
        torch.cuda.synchronize()
        _same(ok.cpu().numpy(), G.pairing_expect(pool, G.tiled(n), cls), "pairing4 device ok")
        idx = G.samples(n, 97, G.schedule_edges(n, n) + [(1 << 31) // 384 + 1, n // 2])
        hg1, hg2, _ = G.pairing4_host(pool, idx % G.D, cls[idx])
        blob = np.ascontiguousarray(G.pairing4_oracle_blob(hg1, hg2, vk))
        _, ogt, _ = O.pairing4_batch(blob.ctypes.data, len(idx), want_gt=True)
        assert gt[torch.from_numpy(idx).cuda()].cpu().numpy().tobytes() == ogt.tobytes()
        st = torch.full((64,), 0xA5, dtype=torch.uint8, device="cuda")
        assert N.lib().zkv_pairing4_batch_device(kv._h, 0, g1.data_ptr(), g2.data_ptr(), n + 1, st.data_ptr(), None, None) == N.ZKV_ERR_ARG
        torch.cuda.synchronize()
        assert (st == 0xA5).all()


# ------------------------------------------------------------------ e) SP1 public values of any length
LONG = (447, 448, 511, 512, 1000, 1023, 1024, 4095, 4096, 65536, 1 << 20)
STRIDES = (0, 1, 55, 56, 63, 64, 65, 119, 120, 127, 128, 129, 200, 1000, 4096)


def test_sp1_public_values_of_any_length(Z, S, gpu, sp1):
    """every length 0..300 and the long ones, each a valid record with its own proof and a tampered twin, on the handle and the gateway"""
    r = sp1["routes"][0]
    lengths = list(range(301)) + list(LONG)
    rng = S.SplitMix64(SEED + 100)
    vkeys = [b"\0" + rng.bytes(31) for _ in lengths]
    pvs = [G.random_bytes(SEED + 101 + L, L) for L in lengths]
    proofs = [r["sel"] + p for p in S.make_proofs(gpu, r["vk"], [S.sp1_signals(v, p) for v, p in zip(vkeys, pvs)], rng, S.Pools(gpu, rng, 64))]
    twin_v = [v if len(p) else v[:31] + bytes([v[31] ^ 1]) for v, p in zip(vkeys, pvs)]
    twin_p = [p[:len(p) // 2] + bytes([p[len(p) // 2] ^ 0x80]) + p[len(p) // 2 + 1:] if len(p) else p for p in pvs]
    V, P, R = vkeys + twin_v, pvs + twin_p, proofs + proofs
    want = np.array([0] * len(lengths) + [4] * len(lengths), dtype=np.uint8)
    oracle = _pmap(lambda i: O.sp1_verify(r["o"], r["sel"], V[i], P[i], R[i]), range(len(V)))
    _same(oracle, want, "oracle")
    _same(r["h"].verify_batch(V, P, R), want, "handle")
    _same(sp1["gateway"].verify_batch(V, P, R), want, "gateway")
    for i, L in enumerate(lengths):
        if L in LONG:
            assert r["h"].verify_proof(vkeys[i], pvs[i], proofs[i]) is None
            assert sp1["gateway"].verify_proof(vkeys[i], pvs[i], proofs[i]) is None
            for v in (r["h"], sp1["gateway"]):
                with pytest.raises(Z.errors.VerificationFailed):
                    v.verify_proof(twin_v[i], twin_p[i], proofs[i])


@pytest.mark.parametrize("stride", STRIDES)
def test_sp1_device_form_public_value_strides(Z, gpu, sp1, stride):
    """fixed-stride public values at every SHA-256 block edge, n = 300 (past two 128-thread blocks), on the handle and the gateway"""
    pool = G.Sp1Pool(gpu, [(sp1["keys"][0], sp1["routes"][0]["sel"])], [stride] * G.D, SEED + 110 + stride)
    h, gw = sp1["h"], sp1["gateway"]
    _sp1_device_check(sp1["routes"][:1], pool, 300, stride, SEED + 111 + stride, lambda *p: h.verify_batch_device(0, *p), None)
    _sp1_device_check(sp1["routes"], pool, 300, stride, SEED + 112 + stride, lambda *p: gw.verify_batch_device(0, *p), None)
