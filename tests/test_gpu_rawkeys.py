"""RawKeyVerifier / zkv_groth16_verify_batch_rawkeys: N verify_proof_with_key calls (common/groth16.rs:23-49) with every key passed as bytes in
the call, against the CPU oracle under the same raw key, against the loaded-key and key-set paths, and across batch geometries and call forms."""

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
INF1, INF2 = bytes(64), bytes(128)
SHAPES = [(0, 2), (1, 3), (0, 6), (1, 16), (0, 16), (1, 2), (0, 3), (1, 6), (0, 9), (1, 11)]
SIZES = [1, 31, 32, 33, 127, 129, 300, 45, 3, 64]


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


@pytest.fixture(scope="module")
def rv(Z):
    return Z.RawKeyVerifier()


def key_of(vk):
    return (vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, list(vk.ic))


def oracle(key, prs, sigs):
    vm, alpha, beta, gamma, delta, ic = key
    ovk = O.Vk(vm, alpha, beta, gamma, delta, ic)
    out = np.full(len(prs), 4, dtype=np.uint8)
    for i, (pr, sg) in enumerate(zip(prs, sigs)):
        if len(sg) == len(ic) - 1:
            out[i] = O.groth16_verify(ovk, pr, b"".join(w32(v) for v in sg))
    return out


def _add(word, d, mod):
    return w32((int.from_bytes(word, "big") + d) % mod)


def tamper(S, pr, sg, cls, rng):
    """the bad-proof classes of the key-set tests"""
    pr = bytearray(pr); sg = list(sg)
    if cls == 0:
        sg[0] = (sg[0] + 1) % R
    elif cls == 1:
        sg[-1] = sg[-1] + R
    elif cls == 2:
        sg = sg[:-1] if rng.below(2) else sg + [rng.fr()]
    elif cls == 3:
        pr[32:64] = _add(pr[32:64], 1, P)
    elif cls == 4:
        pr[224:256] = _add(pr[224:256], 1, P)
    elif cls == 5:
        pr[160:192] = _add(pr[160:192], 1, P)
    elif cls == 6:
        pr[64:192] = S.random_twist_point(S.SplitMix64(rng.next()))
    elif cls == 7:
        a, b = [(0, 64), (64, 192), (192, 256)][rng.below(3)]
        pr[a:b] = bytes(b - a)
    else:
        pr[0:64] = w32(0) + w32(P)
    return bytes(pr), sg


def group(S, gpu, vk, n, rng, bad=True):
    sigs = [[rng.fr() for _ in range(vk.k)] for _ in range(n)]
    prs = S.make_proofs(gpu, vk, sigs, rng, S.Pools(gpu, rng, 8))
    if bad:
        for i in range(n):
            if rng.below(2):
                prs[i], sigs[i] = tamper(S, prs[i], sigs[i], rng.below(9), rng)
    return prs, sigs


def interleave(groups, seed):
    key_idx = np.concatenate([np.full(len(g[0]), k, dtype=np.uint32) for k, g in enumerate(groups)])
    pos = np.concatenate([np.arange(len(g[0])) for g in groups])
    order = np.random.default_rng(seed).permutation(len(key_idx))
    key_idx, pos = key_idx[order], pos[order]
    return (key_idx, [groups[k][0][j] for k, j in zip(key_idx, pos)], [groups[k][1][j] for k, j in zip(key_idx, pos)],
            np.array([groups[k][2][j] for k, j in zip(key_idx, pos)], dtype=np.uint8))


@pytest.fixture(scope="module")
def mixed(Z, S, gpu):
    rng = S.SplitMix64(0x4A3001)
    vks = [S.make_vk(gpu, vm, nic, 0x4A3100 + j) for j, (vm, nic) in enumerate(SHAPES)]
    groups = []
    for vk, n in zip(vks, SIZES):
        prs, sigs = group(S, gpu, vk, n, rng)
        groups.append((prs, sigs, oracle(key_of(vk), prs, sigs)))
    key_idx, prs, sigs, want = interleave(groups, 3)
    return dict(vks=vks, keys=[key_of(v) for v in vks], key_idx=key_idx, prs=prs, sigs=sigs, want=want)


def test_mixed_batch_matches_oracle(Z, rv, mixed):
    got = rv.verify_batch(mixed["keys"], mixed["key_idx"], mixed["prs"], mixed["sigs"])
    want = mixed["want"]
    bad = [(i, int(mixed["key_idx"][i]), int(got[i]), int(want[i])) for i in range(len(want)) if got[i] != want[i]]
    assert not bad, bad[:10]
    assert (want == 0).sum() > len(want) // 4 and (want == 4).sum() > len(want) // 4
    assert set(int(k) for k in mixed["key_idx"][want == 0]) >= set(k for k, n in enumerate(SIZES) if n >= 31)


def test_mixed_batch_matches_key_set(Z, rv, mixed):
    kvs = [Z.VerificationKey(v.vm, v.alpha, v.beta, v.gamma, v.delta, v.ic) for v in mixed["vks"]]
    ks = Z.VerificationKeySet(kvs)
    want = Z.Groth16Verifier.verify_batch_keys(ks, mixed["key_idx"], mixed["prs"], mixed["sigs"])
    got = rv.verify_batch(mixed["keys"], mixed["key_idx"], mixed["prs"], mixed["sigs"])
    assert got.tolist() == want.tolist() == mixed["want"].tolist()


def test_statuses_equal_key_set_64_keys_2p17(Z, S, gpu, rv):
    """64 loaded keys (both vm types, n_ic 2..16), 2^17 proofs with the tamper classes: the raw-key statuses are byte-identical to one
    key-set call's"""
    rng = S.SplitMix64(0x4A3F00)
    vks = [S.make_vk(gpu, j % 2, 2 + j % 15, 0x4A3F10 + j) for j in range(64)]
    base = []
    for k, vk in enumerate(vks):
        prs, sigs = group(S, gpu, vk, 32, rng)
        base += [(k, p, sg) for p, sg in zip(prs, sigs)]
    n = 1 << 17
    order = np.random.default_rng(5).integers(0, len(base), n)
    ki = np.array([base[j][0] for j in order], dtype=np.uint32)
    prs, sigs = [base[j][1] for j in order], [base[j][2] for j in order]
    ks = Z.VerificationKeySet([Z.VerificationKey(v.vm, v.alpha, v.beta, v.gamma, v.delta, v.ic) for v in vks])
    want = Z.Groth16Verifier.verify_batch_keys(ks, ki, prs, sigs)
    got = rv.verify_batch([key_of(v) for v in vks], ki, prs, sigs)
    assert got.tolist() == want.tolist()
    assert n // 4 < int((want == 0).sum()) < 3 * n // 4


def test_single_proof_with_raw_key(Z, S, gpu):
    vk = S.make_vk(gpu, 0, 4, 0x4A3200)
    rng = S.SplitMix64(5)
    sg = [rng.fr() for _ in range(3)]
    pr = S.make_proofs(gpu, vk, [sg], rng, S.Pools(gpu, rng, 2))[0]
    word = lambda o: int.from_bytes(pr[o:o + 32], "big")
    a, b, c = [word(0), word(32)], [[word(64), word(96)], [word(128), word(160)]], [word(192), word(224)]
    assert Z.Groth16Verifier.verify_proof_with_raw_key(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, a, b, c, sg) is True
    assert Z.Groth16Verifier.verify_proof_with_raw_key(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, a, b, c, [sg[0] + 1] + sg[1:]) is False
    assert Z.Groth16Verifier.verify_proof_with_raw_key(1, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, a, b, c, sg) is False   # no negation of A


def _variant(S, vk, trap=None, **pts):
    t = dict(vk.trap)
    t.pop("delta_inv", None)
    t.update(trap or {})
    v = S.SynthVk(vk.vm, t, vk.alpha, vk.beta, vk.gamma, vk.delta, list(vk.ic))
    for k, val in pts.items():
        if k.startswith("ic"):
            v.ic[int(k[2:])] = val
        else:
            setattr(v, k, val)
    return v


def test_key_level_faults_fail_only_their_proofs(Z, S, gpu, rv):
    rng = S.SplitMix64(0x4A3300)
    base = [S.make_vk(gpu, vm, 4, 0x4A3400 + vm) for vm in (0, 1)]
    twist = S.random_twist_point(S.SplitMix64(9))
    keys, groups = [], []
    for vk in base:
        a, b = vk.alpha, vk.beta
        faults = [_variant(S, vk, alpha=a[:32] + _add(a[32:], 1, P)), _variant(S, vk, alpha=w32(int.from_bytes(a[:32], "big") + P) + a[32:]),
                  _variant(S, vk, ic0=vk.ic[0][:32] + _add(vk.ic[0][32:], 1, P)), _variant(S, vk, ic2=w32(P) + vk.ic[2][32:]),
                  _variant(S, vk, ic3=w32(0) + w32(1))]
        for name in ("beta", "gamma", "delta"):
            g = getattr(vk, name)
            faults += [_variant(S, vk, **{name: g[:96] + _add(g[96:], 1, P)}), _variant(S, vk, **{name: w32(P) + g[32:]}),
                       _variant(S, vk, **{name: twist}), _variant(S, vk, **{name: INF2})]
        faults += [_variant(S, vk, alpha=INF1), _variant(S, vk, ic1=INF1), _variant(S, vk, ic0=INF1)]
        # trapdoor-crafted keys with a point at infinity whose proofs are accepted: alpha = inf (e(alpha, beta) = 1), gamma = inf
        faults += [_variant(S, vk, trap={"alpha": 0}, alpha=INF1), _variant(S, vk, trap={"gamma": 0}, gamma=INF2),
                   _variant(S, vk, trap={"beta": 0}, beta=INF2)]
        for v in [vk] + faults:
            prs, sigs = group(S, gpu, v, 6, rng, bad=False)
            t = v.trap
            # vk_x = infinity: the last signal solves IC_0 + sum s_j IC_j = 0 through the trapdoor
            s = [rng.fr() for _ in range(v.k)]
            partial = (t["ic"][0] + sum(x * c for x, c in zip(s[:-1], t["ic"][1:-1]))) % R
            s[-1] = (-partial) * pow(t["ic"][-1], -1, R) % R
            prs += S.make_proofs(gpu, v, [s], rng, S.Pools(gpu, rng, 2)); sigs.append(s)
            prs.append(prs[0]); sigs.append(sigs[0][:-1])                                    # wrong signal count
            prs.append(prs[0]); sigs.append(sigs[0][:-1] + [sigs[0][-1] + R])                # signal >= r
            keys.append(key_of(v))
            groups.append((prs, sigs, oracle(keys[-1], prs, sigs)))
    key_idx, prs, sigs, want = interleave(groups, 11)
    got = rv.verify_batch(keys, key_idx, prs, sigs)
    bad = [(i, int(key_idx[i]), int(got[i]), int(want[i])) for i in range(len(want)) if got[i] != want[i]]
    assert not bad, bad[:10]
    per_key = [g[2] for g in groups]                                             # statuses in group order: 6 valid proofs, vk_x = inf, 2 bad
    assert sum(int((w == 0).all()) for w in per_key) == 0                       # every key has failing proofs (the crafted ones)
    assert sum(int((w[:6] == 0).all()) for w in per_key) >= 2 * 4              # base keys and the three crafted accepts of each vm
    assert sum(int((w == 4).all()) for w in per_key) >= 2 * 15                 # the faulty keys fail all their proofs


def test_vk_x_hook_equals_oracle_chain(Z, S, gpu, rv):
    rng = S.SplitMix64(0x4A3500)
    vks = [S.make_vk(gpu, vm, nic, 0x4A3600 + nic) for vm, nic in ((0, 2), (1, 6), (0, 16))]
    keys = [key_of(v) for v in vks]
    nA = O.g1_mul(w32(1) + w32(2), R - 1)
    keys.append((0, vks[0].alpha, vks[0].beta, vks[0].gamma, vks[0].delta, [w32(1) + w32(2), nA, INF1]))       # partial sums at infinity
    keys.append((0, vks[0].alpha, vks[0].beta, vks[0].gamma, vks[0].delta, [w32(1) + w32(2), w32(1) + w32(3)]))  # invalid IC_1
    key_idx, sigs = [], []
    for k, key in enumerate(keys):
        for s in ([0] * (len(key[5]) - 1), [1] * (len(key[5]) - 1), [R - 1] * (len(key[5]) - 1), [rng.fr() for _ in range(len(key[5]) - 1)],
                  [rng.u256() for _ in range(len(key[5]) - 1)]):
            key_idx.append(k); sigs.append(s)
    pts, failed = rv.vk_x_batch(keys, key_idx, sigs)
    for i, (k, s) in enumerate(zip(key_idx, sigs)):
        ic = keys[k][5]
        acc = ic[0]
        for p, v in zip(ic[1:], s):
            t = O.ec_mul(p + w32(v))
            acc = None if (t is None or acc is None) else O.ec_add(acc + t)
        assert (acc is None) == bool(failed[i]), i
        assert pts[i] == (acc if acc is not None else INF1), i


def _batch(S, gpu, n, seed, n_keys=3):
    """n proofs over n_keys keys tiled from a small mixed pool, with the oracle's statuses"""
    rng = S.SplitMix64(seed)
    vks = [S.make_vk(gpu, j % 2, 2 + 3 * j, seed + j) for j in range(n_keys)]
    keys = [key_of(v) for v in vks]
    base = []
    for k, vk in enumerate(vks):
        prs, sigs = group(S, gpu, vk, 24, rng)
        base += [(k, p, s, w) for p, s, w in zip(prs, sigs, oracle(keys[k], prs, sigs))]
    order = np.random.default_rng(seed).integers(0, len(base), n)
    return keys, [base[j] for j in order]


def _packed(Z, keys, recs):
    kb = b"".join(Z.raw_key_bytes(*k[1:]) for k in keys)
    ko = np.zeros(len(keys) + 1, dtype=np.uint64); ko[1:] = np.cumsum([448 + 64 * len(k[5]) for k in keys])
    kv = np.array([k[0] for k in keys], dtype=np.uint8)
    ki = np.array([r[0] for r in recs], dtype=np.uint32)
    pr = np.frombuffer(b"".join(r[1] for r in recs), dtype=np.uint8)
    so = np.zeros(len(recs) + 1, dtype=np.uint64); so[1:] = np.cumsum([len(r[2]) for r in recs])
    sb = np.frombuffer(b"".join(w32(v) for r in recs for v in r[2]), dtype=np.uint8)
    want = np.array([r[3] for r in recs], dtype=np.uint8)
    return kb, ko, kv, ki, pr, sb, so, want


@pytest.mark.parametrize("n", [1, 127, 128, 129, "wave+129"])
def test_batch_geometry(Z, S, gpu, rv, n):
    if n == "wave+129":
        n = Z.wave_proofs(0, 0) + 129
    keys, recs = _batch(S, gpu, n, 0x4A3700 + (n % 1000))
    kb, ko, kv, ki, pr, sb, so, want = _packed(Z, keys, recs)
    assert rv.verify_batch_packed(kb, ko, kv, ki, pr, sb, so).tolist() == want.tolist()


def test_one_pass_plus_one_page_locked(Z, S, gpu, rv):
    n = (1 << 20) + 1
    keys, recs = _batch(S, gpu, 4096, 0x4A3800)
    kb, ko, kv, ki, pr, sb, so, want = _packed(Z, keys, recs)
    reps = -(-n // 4096)
    ki2 = np.tile(ki, reps)[:n]; want2 = np.tile(want, reps)[:n]
    pr2 = np.tile(pr.reshape(4096, 256), (reps, 1))[:n].reshape(-1)
    cnt = np.diff(so).astype(np.uint64)
    cnt2 = np.tile(cnt, reps)[:n]
    so2 = np.zeros(n + 1, dtype=np.uint64); so2[1:] = np.cumsum(cnt2)
    words = sb.reshape(-1, 32)
    starts = so[:-1]
    idx = np.concatenate([np.arange(int(starts[j]), int(starts[j] + cnt[j])) for j in range(4096)])
    sb2 = np.tile(words[idx], (reps, 1))[:int(so2[-1])].reshape(-1)
    got = rv.verify_batch_packed(kb, ko, kv, ki2, pr2, sb2, so2)
    assert got.tolist() == want2.tolist()
    # the same from page-locked arrays (uploaded in place)
    pins = []
    def pinned(a):
        a = np.ascontiguousarray(a)
        p = Z.pinned_copy(a) if hasattr(Z, "pinned_copy") else a
        pins.append(p)
        return p
    got2 = rv.verify_batch_packed(pinned(np.frombuffer(kb, dtype=np.uint8)), pinned(ko), pinned(kv), pinned(ki2[:1 << 16]), pinned(pr2[:256 << 16]),
                                  pinned(sb2[:int(so2[1 << 16]) * 32]), pinned(so2[:(1 << 16) + 1]))
    assert got2.tolist() == want2[:1 << 16].tolist()


def test_agreement_with_loaded_key(Z, S, gpu, rv):
    """one key, 2^16 proofs: byte-identical to zkv_groth16_verify_batch under the loaded key"""
    rng = S.SplitMix64(0x4A3900)
    vk = S.make_vk(gpu, 0, 6, 0x4A3901)
    prs, sigs = group(S, gpu, vk, 2048, rng)
    keep = [i for i in range(len(prs)) if len(sigs[i]) == vk.k]
    prs = [prs[i] for i in keep] * 40; sigs = [sigs[i] for i in keep] * 40
    n = 1 << 16
    prs, sigs = prs[:n], sigs[:n]
    kv = Z.VerificationKey(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    want = Z.Groth16Verifier.verify_batch(kv, b"".join(prs), b"".join(w32(v) for s in sigs for v in s), vk.k, n)
    got = rv.verify_batch([key_of(vk)], np.zeros(n, dtype=np.uint32), prs, sigs)
    assert got.tolist() == want.tolist() and 0 < int((want == 0).sum()) < n


def test_device_form_side_stream_and_growth(Z, S, gpu):
    import torch
    rv = Z.RawKeyVerifier()          # a fresh handle: its workspace is empty, so the second call below really reallocates it
    keys, recs = _batch(S, gpu, 20000, 0x4A3A00)
    kb, ko, kv, ki, pr, sb, so, want = _packed(Z, keys, recs)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).cuda()
    d = [dev(np.frombuffer(kb, dtype=np.uint8)), dev(ko), dev(kv), dev(ki), dev(pr), dev(sb), dev(so)]
    small = torch.zeros(300, dtype=torch.uint8, device="cuda")
    big = torch.zeros(len(recs), dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        # a small call, then a larger one that grows the workspace while the first may still run
        rv.verify_batch_device(0, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), len(keys), d[3].data_ptr(), d[4].data_ptr(), d[5].data_ptr(),
                               d[6].data_ptr(), 300, small.data_ptr(), s.cuda_stream)
        rv.verify_batch_device(0, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), len(keys), d[3].data_ptr(), d[4].data_ptr(), d[5].data_ptr(),
                               d[6].data_ptr(), len(recs), big.data_ptr(), s.cuda_stream)
    s.synchronize()
    assert small.cpu().numpy().tolist() == want[:300].tolist()
    assert big.cpu().numpy().tolist() == want.tolist()
    # on the device a bad key index or a malformed key fails only that proof
    ki_bad = ki.copy(); ki_bad[5] = len(keys)
    kv_bad = kv.copy(); kv_bad[1] = 7
    d[3] = dev(ki_bad); d[2] = dev(kv_bad)
    rv.verify_batch_device(0, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), len(keys), d[3].data_ptr(), d[4].data_ptr(), d[5].data_ptr(),
                           d[6].data_ptr(), len(recs), big.data_ptr(), None)
    torch.cuda.synchronize()
    w2 = want.copy(); w2[5] = 4; w2[ki_bad == 1] = 4
    assert big.cpu().numpy().tolist() == w2.tolist()


def test_argument_errors_leave_status_untouched(Z, S, gpu, rv):
    keys, recs = _batch(S, gpu, 16, 0x4A3B00)
    kb, ko, kv, ki, pr, sb, so, want = _packed(Z, keys, recs)
    st = np.full(16, 0xAB, dtype=np.uint8)
    cases = []
    k2 = ki.copy(); k2[3] = len(keys); cases.append((kb, ko, kv, k2, so))
    v2 = kv.copy(); v2[0] = 2; cases.append((kb, ko, v2, ki, so))
    o2 = ko.copy(); o2[1] += 1; cases.append((kb, o2, kv, ki, so))                     # key length not 448 + 64 n_ic
    o3 = ko.copy(); o3[1], o3[2] = o3[2], o3[1]; cases.append((kb, o3, kv, ki, so))   # decreasing key offsets
    s2 = so.copy(); s2[4], s2[5] = s2[5], s2[4]; cases.append((kb, ko, kv, ki, s2))   # decreasing signal offsets
    for kb_, ko_, kv_, ki_, so_ in cases:
        with pytest.raises(Z.ZkvError) as e:
            rv.verify_batch_packed(kb_, ko_, kv_, ki_, pr, sb, so_, status_out=st)
        assert e.value.code == -1 and (st == 0xAB).all()
    with pytest.raises(Z.ZkvError) as e:
        rv.verify_batch_packed(b"", np.zeros(1, dtype=np.uint64), np.zeros(0, dtype=np.uint8), ki, pr, sb, so, status_out=st)
    assert e.value.code == -1 and (st == 0xAB).all()
    assert rv.verify_batch_packed(kb, ko, kv, ki[:0], pr[:0], sb[:0], so[:1]).tolist() == []


def test_launch_count_does_not_depend_on_keys(Z, S, gpu, rv):
    counts = []
    for n_keys in (1, 4096):
        keys, recs = _batch(S, gpu, 1 << 16, 0x4A3C00, n_keys=1)
        keys = keys * n_keys
        recs = [(i % n_keys, p, s, w) for i, (_, p, s, w) in enumerate(recs)]
        kb, ko, kv, ki, pr, sb, so, want = _packed(Z, keys, recs)
        c0 = Z.launch_count()
        got = rv.verify_batch_packed(kb, ko, kv, ki, pr, sb, so)
        counts.append(Z.launch_count() - c0)
        assert got.tolist() == want.tolist()
    assert counts[0] == counts[1] == 34


def test_multi_device_split(Z, S, gpu):
    if Z.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    keys, recs = _batch(S, gpu, 20000, 0x4A3D00)
    kb, ko, kv, ki, pr, sb, so, want = _packed(Z, keys, recs)
    rv2 = Z.RawKeyVerifier(devices=[0, 1])
    assert rv2.verify_batch_packed(kb, ko, kv, ki, pr, sb, so).tolist() == want.tolist()


# ------------------------------------------------------------------ G2 points outside the order-r subgroup as the only fault
def _solve_inf(t, rng, k):
    """signals whose vk_x is infinity under the trapdoor IC scalars t["ic"]"""
    s = [rng.fr() for _ in range(k)]
    rest = (t["ic"][0] + sum(x * c for x, c in zip(s[:-1], t["ic"][1:-1]))) % R
    s[-1] = (-rest) * pow(t["ic"][-1], -1, R) % R
    return s


@pytest.fixture(scope="module")
def outside_units(S, gpu):
    """For each twist point outside G2 of the single-cause catalogue and both vm types, four records in which that point is the only fault,
    each beside its twin with a member of G2 in its place (accepted):
      (1) a key with alpha at infinity (trapdoor alpha = 0) and beta = the point;
      (2) a key with gamma = the point, under signals whose vk_x is infinity;
      (3) a key with delta = the point, the proof's C at infinity (A and B solved for it);
      (4) the proof's B = the point with A at infinity and C solved.
    Every pair that holds the point is skipped (a member at infinity), so only the order-r test of the Miller loop's last segment can fail
    it.  Returns (keys, records of (key index, proof, signals, expected status, name))."""
    import single_cause as SC
    rng = S.SplitMix64(0x4A3E00)
    outside = SC.outside_catalogue()
    members = [m for _, m in SC.member_catalogue() if m != INF2]
    pools = S.Pools(gpu, rng, 4)
    keys, recs = [], []

    def rec(v, pr, sg, st, name):
        keys.append(key_of(v))
        recs.append((len(keys) - 1, pr, sg, st, name))

    for vm in (0, 1):
        base = S.make_vk(gpu, vm, 4, 0x4A3E10 + vm)
        t = base.trap
        for j, b in enumerate(outside):
            for pt, st, tag in ((b.point, 4, b.name), (members[j % len(members)], 0, "member")):
                v = _variant(S, base, trap={"alpha": 0}, alpha=INF1, beta=pt)
                sg = [rng.fr() for _ in range(v.k)]
                rec(v, S.make_proofs(gpu, v, [sg], rng, pools)[0], sg, st, "vm%d|alpha=inf,beta=%s" % (vm, tag))
                v = _variant(S, base, gamma=pt)
                sg = _solve_inf(t, rng, v.k)
                rec(v, S.make_proofs(gpu, v, [sg], rng, pools)[0], sg, st, "vm%d|vk_x=inf,gamma=%s" % (vm, tag))
                v = _variant(S, base, delta=pt)
                sg = [rng.fr() for _ in range(v.k)]
                bb = rng.fr()
                ab = (t["alpha"] * t["beta"] + v.x_of(sg) * t["gamma"]) * pow(bb, -1, R) % R      # c = 0: a b = alpha beta + x gamma (vm 0)
                aa = ab if vm == 0 else (-ab) % R                                                  # vm 1: a b + alpha beta + x gamma = 0
                rec(v, gpu.g1_mul([aa])[0] + gpu.g2_mul([bb])[0] + INF1, sg, st, "vm%d|C=inf,delta=%s" % (vm, tag))
                sg = [rng.fr() for _ in range(base.k)]
                c = S.solve_c(base, 0, 0, base.x_of(sg))
                rec(base, INF1 + pt + gpu.g1_mul([c])[0], sg, st, "vm%d|A=inf,B=%s" % (vm, tag))
    for k, pr, sg, st, name in recs:                       # the construction is what the reference decides
        assert oracle(keys[k], [pr], [sg])[0] == st, name
    return keys, recs


def test_outside_g2_is_the_only_fault(Z, rv, outside_units):
    keys, recs = outside_units
    got = rv.verify_batch(keys, [r[0] for r in recs], [r[1] for r in recs], [r[2] for r in recs])
    bad = [(r[4], int(g), r[3]) for r, g in zip(recs, got) if g != r[3]]
    assert not bad, bad[:10]
    assert sum(r[3] == 4 for r in recs) >= 4 * 2 * 20


def test_outside_g2_only_fault_in_a_chunked_pass(Z, rv, outside_units):
    """the same records scattered over a pass of 40 000 proofs (four chunks: the targets, flags and skip bytes at every chunk offset)"""
    keys, recs = outside_units
    n = 40000
    order = np.random.default_rng(17).integers(0, len(recs), n)
    order[:len(recs)] = np.random.default_rng(18).permutation(len(recs))          # every record at least once
    order = np.random.default_rng(19).permutation(order)
    got = rv.verify_batch(keys, [recs[j][0] for j in order], [recs[j][1] for j in order], [recs[j][2] for j in order])
    assert got.tolist() == [recs[j][3] for j in order]
