"""Groth16Verifier.verify_batch_keys / zkv_groth16_verify_batch_keys: N verify_proof_with_key calls (common/groth16.rs:23-49) under up to
256 keys in one batch, against the CPU oracle (per key) and against zkv_groth16_verify_batch on each key alone."""
import numpy as np
import pytest

import oracle_lib as O
from conftest import oracle_vk

pytestmark = pytest.mark.gpu

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
SHAPES = [(0, 2), (1, 3), (0, 6), (1, 16), (0, 16), (1, 2), (0, 3), (1, 6)]     # (vm, n_ic) of the mixed batch's keys
SIZES = [1, 31, 32, 33, 127, 129, 300, 45]                                      # their group sizes: warp and block edges


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


def _add(word, d, mod):
    return w32((int.from_bytes(word, "big") + d) % mod)


def _tamper(S, vk, pr, sg, cls, rng):
    """one of the bad-proof classes; returns (proof, signals)"""
    pr = bytearray(pr); sg = list(sg)
    if cls == 0:
        sg[0] = (sg[0] + 1) % R                              # another statement
    elif cls == 1:
        sg[-1] = sg[-1] + R                                  # signal >= R (groth16.rs:32-34)
    elif cls == 2:
        sg = sg[:-1] if rng.below(2) else sg + [rng.fr()]    # wrong signal count (groth16.rs:32)
    elif cls == 3:
        pr[32:64] = _add(pr[32:64], 1, P)                    # A off the curve
    elif cls == 4:
        pr[224:256] = _add(pr[224:256], 1, P)                # C off the curve
    elif cls == 5:
        pr[160:192] = _add(pr[160:192], 1, P)                # B off the twist
    elif cls == 6:
        pr[64:192] = S.random_twist_point(S.SplitMix64(rng.next()))     # B on the twist, outside G2
    elif cls == 7:
        a, b = [(0, 64), (64, 192), (192, 256)][rng.below(3)]
        pr[a:b] = bytes(b - a)                               # A, B or C at infinity
    else:
        pr[0:64] = w32(0) + w32(P)                           # A = (0, Q): the RISC Zero negation quirk (groth16.rs:75-84)
    return bytes(pr), sg


def _group(S, gpu, vk, n, rng, bad=True):
    sigs = [[rng.fr() for _ in range(vk.k)] for _ in range(n)]
    prs = S.make_proofs(gpu, vk, sigs, rng, S.Pools(gpu, rng, 8))
    if bad:
        for i in range(n):
            if rng.below(2):
                prs[i], sigs[i] = _tamper(S, vk, prs[i], sigs[i], rng.below(9), rng)
    return prs, sigs


def _expect(vk, prs, sigs):
    """oracle statuses of one key's proofs; a wrong signal count is VERIFICATION_FAILED"""
    out = np.full(len(prs), 4, dtype=np.uint8)
    ok = [i for i in range(len(prs)) if len(sigs[i]) == vk.k]
    if ok:
        out[ok] = O.groth16_verify_batch(oracle_vk(vk), b"".join(prs[i] for i in ok), b"".join(w32(v) for i in ok for v in sigs[i]), len(ok))
    return out


def _own_call(Z, kv, vk, prs, sigs):
    """zkv_groth16_verify_batch on the key alone (wrong-count proofs: VERIFICATION_FAILED, as it returns for a call with that count)"""
    out = np.full(len(prs), 4, dtype=np.uint8)
    ok = [i for i in range(len(prs)) if len(sigs[i]) == vk.k]
    if ok:
        out[ok] = Z.Groth16Verifier.verify_batch(kv, b"".join(prs[i] for i in ok), b"".join(w32(v) for i in ok for v in sigs[i]), vk.k, len(ok))
    return out


def _interleave(groups, seed):
    """groups: [(prs, sigs, expect)] -> caller-order key_idx, proofs, signals, expect (a seeded random interleaving)"""
    key_idx = np.concatenate([np.full(len(g[0]), k, dtype=np.uint32) for k, g in enumerate(groups)])
    pos = np.concatenate([np.arange(len(g[0])) for g in groups])
    order = np.random.default_rng(seed).permutation(len(key_idx))
    key_idx, pos = key_idx[order], pos[order]
    prs = [groups[k][0][j] for k, j in zip(key_idx, pos)]
    sigs = [groups[k][1][j] for k, j in zip(key_idx, pos)]
    want = np.array([groups[k][2][j] for k, j in zip(key_idx, pos)], dtype=np.uint8)
    return key_idx, prs, sigs, want


@pytest.fixture(scope="module")
def mixed(Z, S, gpu):
    rng = S.SplitMix64(0x5E7001)
    vks = [S.make_vk(gpu, vm, nic, 0x5E7100 + j) for j, (vm, nic) in enumerate(SHAPES)]
    kvs = [_load(Z, vk) for vk in vks]
    groups = []
    for vk, kv, n in zip(vks, kvs, SIZES):
        prs, sigs = _group(S, gpu, vk, n, rng)
        want = _expect(vk, prs, sigs)
        assert want.tolist() == _own_call(Z, kv, vk, prs, sigs).tolist()       # the single-key entry point agrees with the oracle
        groups.append((prs, sigs, want))
    key_idx, prs, sigs, want = _interleave(groups, 1)
    return dict(vks=vks, kvs=kvs, ks=Z.VerificationKeySet(kvs), key_idx=key_idx, prs=prs, sigs=sigs, want=want)


def test_mixed_batch_matches_oracle_and_per_key_calls(Z, mixed):
    got = Z.Groth16Verifier.verify_batch_keys(mixed["ks"], mixed["key_idx"], mixed["prs"], mixed["sigs"])
    want = mixed["want"]
    bad = [(i, int(mixed["key_idx"][i]), int(got[i]), int(want[i])) for i in range(len(want)) if got[i] != want[i]]
    assert not bad, bad[:10]
    assert (want == 0).sum() > len(want) // 3 and (want == 4).sum() > len(want) // 3
    assert set(int(k) for k in mixed["key_idx"][want == 0]) == set(range(len(SHAPES)))      # every key accepts some of its proofs


def test_order_independence(Z, mixed):
    n = len(mixed["want"])
    perm = np.random.default_rng(7).permutation(n)
    got = Z.Groth16Verifier.verify_batch_keys(mixed["ks"], mixed["key_idx"][perm], [mixed["prs"][i] for i in perm], [mixed["sigs"][i] for i in perm])
    assert got.tolist() == mixed["want"][perm].tolist()


def test_device_form_on_a_side_stream_matches_host_path(Z, mixed):
    import torch
    n = len(mixed["want"])
    off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in mixed["sigs"]])
    blob = b"".join(w32(v) for s in mixed["sigs"] for v in s)
    host = Z.Groth16Verifier.verify_batch_keys_packed(mixed["ks"], mixed["key_idx"], b"".join(mixed["prs"]), blob, off)
    dev = lambda a: torch.from_numpy(np.frombuffer(a, dtype=np.uint8).copy()).cuda()
    d_k, d_p, d_s, d_o = dev(mixed["key_idx"].tobytes()), dev(b"".join(mixed["prs"])), dev(blob), dev(off.tobytes())
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d_st = torch.full((n,), 255, dtype=torch.uint8, device="cuda")
        Z.Groth16Verifier.verify_batch_keys_device(mixed["ks"], 0, d_k.data_ptr(), d_p.data_ptr(), d_s.data_ptr(), d_o.data_ptr(), n, d_st.data_ptr(), side.cuda_stream)
    side.synchronize()
    assert d_st.cpu().numpy().tolist() == host.tolist() == mixed["want"].tolist()


def test_set_workspace_growth_under_an_async_device_call(Z, S, gpu):
    """On a fresh set (empty workspace), a small device call and at once, on another stream, a chunked one that grows every buffer of the
    set: the second must wait for the first before it frees anything.  Both must give the host path's bytes, taken on a second set of the
    same keys (its own workspace)."""
    import torch
    vks = [S.make_vk(gpu, k % 2, 3 + k, 0x5E7600 + k) for k in range(3)]
    kvs = [_load(Z, vk) for vk in vks]
    small, big = _tiled(S, gpu, vks, 100, 32, 0x5E7601), _tiled(S, gpu, vks, 3000, 64, 0x5E7602)
    ref, ks = Z.VerificationKeySet(kvs), Z.VerificationKeySet(kvs)
    dev = lambda a: torch.from_numpy(np.frombuffer(a, dtype=np.uint8).copy()).cuda()
    calls = []
    for key_idx, prs, sigs, _ in (small, big):
        n = len(key_idx)
        off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in sigs])
        blob = b"".join(w32(v) for s in sigs for v in s)
        want = Z.Groth16Verifier.verify_batch_keys_packed(ref, key_idx, b"".join(prs), blob, off)
        calls.append((want, [dev(key_idx.tobytes()), dev(b"".join(prs)), dev(blob), dev(off.tobytes())], torch.full((n,), 255, dtype=torch.uint8, device="cuda")))
    assert len(big[0]) > 8192 and 0 < int((calls[1][0] == 0).sum()) < len(big[0])
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for (want, d, d_st), st in zip(calls, streams):
        Z.Groth16Verifier.verify_batch_keys_device(ks, 0, *[x.data_ptr() for x in d], len(want), d_st.data_ptr(), st.cuda_stream)
    torch.cuda.synchronize()
    for want, _, d_st in calls:
        assert d_st.cpu().numpy().tolist() == want.tolist()


def test_argument_errors_leave_status_untouched(Z, mixed):
    from stylus_zkvm_verifiers_b200 import _native as N
    ks, n = mixed["ks"], 40
    key_idx = mixed["key_idx"][:n].copy(); prs = b"".join(mixed["prs"][:n])
    off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in mixed["sigs"][:n]])
    blob = b"".join(w32(v) for s in mixed["sigs"][:n] for v in s)

    def call(ki, of, sig=blob):
        st = np.full(n, 0xA5, dtype=np.uint8)
        with pytest.raises(Z.ZkvError) as e:
            Z.Groth16Verifier.verify_batch_keys_packed(ks, ki, prs, sig, of, status_out=st)
        assert e.value.code == N.ZKV_ERR_ARG and (st == 0xA5).all()

    bad_k = key_idx.copy(); bad_k[n // 2] = len(ks)
    call(bad_k, off)                                                     # key index >= n_keys
    bad_o = off.copy(); bad_o[3], bad_o[4] = bad_o[4], bad_o[3]
    if bad_o[3] != bad_o[4]:
        call(key_idx, bad_o)                                             # decreasing offsets
    call(key_idx, off, b"")                                              # signals missing (null pointer)
    st = np.full(n, 0xA5, dtype=np.uint8)
    L = N.lib()
    assert L.zkv_groth16_verify_batch_keys(ks._h, None, N.buf(prs), N.buf(blob), off.ctypes.data, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_groth16_verify_batch_keys(ks._h, key_idx.ctypes.data, None, N.buf(blob), off.ctypes.data, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_groth16_verify_batch_keys(ks._h, key_idx.ctypes.data, N.buf(prs), N.buf(blob), None, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert L.zkv_groth16_verify_batch_keys(None, key_idx.ctypes.data, N.buf(prs), N.buf(blob), off.ctypes.data, n, st.ctypes.data) == N.ZKV_ERR_ARG
    assert (st == 0xA5).all()
    assert len(Z.Groth16Verifier.verify_batch_keys(ks, [], b"", [])) == 0                # n == 0: nothing to do
    for keys in ([], [mixed["kvs"][0]] * 257):                                           # n_keys outside 1..256
        with pytest.raises(Z.ZkvError) as e:
            Z.VerificationKeySet(keys)
        assert e.value.code == N.ZKV_ERR_ARG
    with pytest.raises(Z.ZkvError) as e:
        Z.VerificationKeySet(mixed["kvs"], devices=[Z.device_count()])                   # no such device
    assert e.value.code == N.ZKV_ERR_ARG
    if Z.device_count() >= 2:
        with pytest.raises(Z.ZkvError) as e:
            Z.VerificationKeySet(mixed["kvs"], devices=[0, 1])                           # the keys are loaded on device 0 only
        assert e.value.code == N.ZKV_ERR_ARG


def test_launch_count_per_call(Z, mixed):
    n = 100
    c0 = Z.launch_count()
    Z.Groth16Verifier.verify_batch_keys(mixed["ks"], mixed["key_idx"][:n], mixed["prs"][:n], mixed["sigs"][:n])
    assert Z.launch_count() - c0 == 10


def test_edge_keys_in_a_set(Z, S, gpu):
    """keys with an invalid point fail every proof; keys with a point at infinity give their own call's statuses (and the oracle's)"""
    rng = S.SplitMix64(0x5E7200)
    base = S.make_vk(gpu, 0, 4, 0x5E7201)
    variants = [(base, base, False)]                                      # (key, key whose trapdoor makes the proofs, every proof fails)
    for mod in ("ic", "gamma", "alpha"):                                  # invalid points
        ic, gamma, alpha = list(base.ic), base.gamma, base.alpha
        if mod == "ic":
            ic[2] = w32(1) + w32(3)
        elif mod == "gamma":
            gamma = S.random_twist_point(S.SplitMix64(4))
        else:
            alpha = w32(P) + w32(1)
        variants.append((S.SynthVk(0, base.trap, alpha, base.beta, gamma, base.delta, ic), base, True))
    for vm in (0, 1):                                                     # points at infinity: a zero trapdoor value keeps the proofs valid
        for pt in ("alpha", "beta", "gamma", "delta"):                    # (except for delta: those proofs are the base key's)
            t = {k: v for k, v in base.trap.items() if k != "delta_inv"}
            pts = dict(alpha=base.alpha, beta=base.beta, gamma=base.gamma, delta=base.delta)
            pts[pt] = bytes(64 if pt == "alpha" else 128)
            t[pt] = 0
            vk = S.SynthVk(vm, t, pts["alpha"], pts["beta"], pts["gamma"], pts["delta"], list(base.ic))
            variants.append((vk, base if pt == "delta" else vk, False))
    kvs = [_load(Z, vk) for vk, _, _ in variants]
    groups = []
    for j, ((vk, src, all_fail), kv) in enumerate(zip(variants, kvs)):
        prs, sigs = _group(S, gpu, src, 40, rng)
        want = _expect(vk, prs, sigs)
        assert want.tolist() == _own_call(Z, kv, vk, prs, sigs).tolist(), j
        assert (want == 4).all() if all_fail else True, j
        groups.append((prs, sigs, want))
    assert all((g[2] == 0).any() for (vk, src, _), g in zip(variants, groups) if src is vk)
    key_idx, prs, sigs, want = _interleave(groups, 2)
    got = Z.Groth16Verifier.verify_batch_keys(Z.VerificationKeySet(kvs), key_idx, prs, sigs)
    assert got.tolist() == want.tolist()


def _tiled(S, gpu, vks, per_key, distinct, seed):
    """per_key proofs of each key, tiled from `distinct` generated ones, one in eight with a tampered signal; random caller order"""
    rng = S.SplitMix64(seed)
    groups = []
    for vk in vks:
        prs, sigs = _group(S, gpu, vk, distinct, rng, bad=False)
        idx = np.arange(per_key) % distinct
        gp = [prs[i] for i in idx]; gs = [list(sigs[i]) for i in idx]
        for j in range(3, per_key, 8):
            gs[j][0] = (gs[j][0] + 1) % R
        groups.append((gp, gs, np.zeros(per_key, dtype=np.uint8)))
    return _interleave(groups, seed)


def test_one_key_set_equals_single_key_call_at_2p16(Z, S, gpu):
    vk = S.make_vk(gpu, 0, 6, 0x5E7300)
    kv = _load(Z, vk)
    key_idx, prs, sigs, _ = _tiled(S, gpu, [vk], 1 << 16, 512, 0x5E7301)
    single = Z.Groth16Verifier.verify_batch(kv, b"".join(prs), b"".join(w32(v) for s in sigs for v in s), vk.k, len(prs))
    ks = Z.VerificationKeySet([kv])
    c0 = Z.launch_count()
    got = Z.Groth16Verifier.verify_batch_keys(ks, key_idx, prs, sigs)
    assert Z.launch_count() - c0 == 41                                   # one chunked pass
    assert got.tobytes() == single.tobytes()
    assert (got == 4).sum() == (1 << 16) // 8 and (got == 0).sum() == (1 << 16) - (1 << 16) // 8


def test_64_keys_2p17_match_per_key_calls(Z, S, gpu):
    vks = [S.make_vk(gpu, k % 2, 2 + k % 15, 0x5E7400 + k) for k in range(64)]
    kvs = [_load(Z, vk) for vk in vks]
    key_idx, prs, sigs, _ = _tiled(S, gpu, vks, 2048, 64, 0x5E7401)
    got = Z.Groth16Verifier.verify_batch_keys(Z.VerificationKeySet(kvs), key_idx, prs, sigs)
    for k, (vk, kv) in enumerate(zip(vks, kvs)):
        sel = np.nonzero(key_idx == k)[0]
        own = _own_call(Z, kv, vk, [prs[i] for i in sel], [sigs[i] for i in sel])
        assert got[sel].tolist() == own.tolist(), k
    assert (got == 4).sum() == 64 * 256


def test_set_over_all_devices_matches_one_device(Z, S, gpu):
    nd = Z.device_count()
    if nd < 2:
        pytest.skip("one CUDA device")
    devs = list(range(nd))
    vks = [S.make_vk(gpu, k % 2, 3 + k, 0x5E7500 + k) for k in range(4)]
    key_idx, prs, sigs, _ = _tiled(S, gpu, vks, 4096, 128, 0x5E7501)
    one = Z.Groth16Verifier.verify_batch_keys(Z.VerificationKeySet([_load(Z, vk) for vk in vks]), key_idx, prs, sigs)
    allv = Z.Groth16Verifier.verify_batch_keys(Z.VerificationKeySet([_load(Z, vk, devs) for vk in vks], devices=devs), key_idx, prs, sigs)
    assert one.tobytes() == allv.tobytes()
    assert (one == 4).sum() == 4 * 512
