"""The G2 subgroup test finished by the shared-memory Miller kernels (k_g2_target + the last segment of k_miller_lz / k_miller_lz_keys)
against the CPU oracle: 2^16 proofs under a RISC Zero-shape and an SP1-shape key, a part of them with B on the twist but outside G2
(random points, G2 + small-order points, small-order points), some of those with A or vk_x at infinity, through the single chain, the
chunked schedule and the key-set calls (host buffers and device form)."""
import numpy as np
import pytest

import oracle_lib as O
from conftest import oracle_vk

pytestmark = pytest.mark.gpu

R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
U = 4965661367192848881
P = 36 * U**4 + 36 * U**3 + 24 * U**2 + 6 * U + 1
H2 = 2 * P - R
SMALL = 10069
w32 = O.w32
PER_KEY = 1 << 15
DISTINCT = 384


@pytest.fixture(scope="module")
def Z():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import stylus_zkvm_verifiers_b200 as Z
    return Z


def _outside_points(S, rng, G2_GEN):
    """B values on the twist and outside G2: random twist points, G2 + an order-10069 point, order-10069 points"""
    small = []
    while len(small) < 4:
        q = O.g2_mul(O.g2_mul(S.random_twist_point(rng), R), H2 // SMALL)
        if q != bytes(128):
            small.append(q)
    mixed = [O.g2_add(O.g2_mul(G2_GEN, rng.fr()), q) for q in small]
    return [S.random_twist_point(rng) for _ in range(8)] + mixed + small


def _key_batch(S, gpu, vk, rng, outside):
    """DISTINCT proofs of one key with their oracle statuses, and how many have B outside G2"""
    sigs = [[rng.fr() for _ in range(vk.k)] for _ in range(DISTINCT)]
    for i in range(0, DISTINCT, 7):                 # vk_x = infinity: IC0 + sum s_j IC_j = 0
        t = vk.trap["ic"]
        rest = (t[0] + sum(s * c for s, c in zip(sigs[i][:-1], t[1:-1]))) % R
        sigs[i][-1] = (-rest) * pow(t[-1], -1, R) % R
        assert vk.x_of(sigs[i]) == 0
    prs = [bytearray(p) for p in S.make_proofs(gpu, vk, sigs, rng, S.Pools(gpu, rng, 8))]
    n_out = 0
    for i in range(DISTINCT):
        cls = rng.below(8)
        if cls < 3:                                  # B outside G2
            prs[i][64:192] = outside[rng.below(len(outside))]
            n_out += 1
            if cls == 1:
                prs[i][0:64] = bytes(64)             # ... and A at infinity
        elif cls == 3:
            sigs[i][0] = (sigs[i][0] + 1) % R        # another statement
        elif cls == 4:
            prs[i][0:64] = bytes(64)                 # A at infinity, B in G2
    prs = [bytes(p) for p in prs]
    want = O.groth16_verify_batch(oracle_vk(vk), b"".join(prs), b"".join(w32(v) for s in sigs for v in s), DISTINCT)
    return prs, sigs, want, n_out


@pytest.fixture(scope="module")
def batch(Z):
    from stylus_zkvm_verifiers_b200 import synth as S
    gpu = Z.GpuBackend(0)
    rng = S.SplitMix64(0x6F2E0001)
    outside = _outside_points(S, rng, S.G2_GEN)
    keys = []
    for vm, nic, seed in ((0, 6, 0x6F2E0010), (1, 3, 0x6F2E0011)):         # RISC Zero and SP1 shapes
        vk = S.make_vk(gpu, vm, nic, seed)
        prs, sigs, want, n_out = _key_batch(S, gpu, vk, rng, outside)
        assert n_out > DISTINCT // 4 and (want == 0).sum() > DISTINCT // 4 and set(want.tolist()) <= {0, 4}
        idx = np.arange(PER_KEY) % DISTINCT
        keys.append(dict(vk=vk, prs=[prs[i] for i in idx], sigs=[sigs[i] for i in idx], want=want[idx]))
    return keys


def _load(Z, vk):
    return Z.VerificationKey(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)


def _single(Z, kv, key):
    vk = key["vk"]
    return Z.Groth16Verifier.verify_batch(kv, b"".join(key["prs"]), b"".join(w32(v) for s in key["sigs"] for v in s), vk.k, len(key["prs"]))


@pytest.mark.parametrize("overlap,layout", [(1, 1), (4, 1), (0, 1)])
def test_single_key_paths(Z, batch, overlap, layout):
    """overlap 1: one chain (k_g2_target, one Miller launch); 4 / 0 (automatic at 2^15): four chunks, four Miller segments each"""
    for key in batch:
        kv = _load(Z, key["vk"])
        kv.tune("overlap", overlap)
        kv.tune("layout", layout)
        assert _single(Z, kv, key).tolist() == key["want"].tolist()


def _set_inputs(batch):
    key_idx = np.concatenate([np.full(PER_KEY, k, dtype=np.uint32) for k in range(len(batch))])
    order = np.random.default_rng(7).permutation(len(key_idx))
    pos = np.concatenate([np.arange(PER_KEY)] * len(batch))[order]
    key_idx = key_idx[order]
    prs = [batch[k]["prs"][j] for k, j in zip(key_idx, pos)]
    sigs = [batch[k]["sigs"][j] for k, j in zip(key_idx, pos)]
    want = np.array([batch[k]["want"][j] for k, j in zip(key_idx, pos)], dtype=np.uint8)
    return key_idx, prs, sigs, want


def test_key_set_host_and_device(Z, batch):
    import torch
    ks = Z.VerificationKeySet([_load(Z, key["vk"]) for key in batch])
    key_idx, prs, sigs, want = _set_inputs(batch)
    n = len(want)
    assert n == 1 << 16
    assert Z.Groth16Verifier.verify_batch_keys(ks, key_idx, prs, sigs).tolist() == want.tolist()
    small = 300                                                                     # one chain, not chunked
    assert Z.Groth16Verifier.verify_batch_keys(ks, key_idx[:small], prs[:small], sigs[:small]).tolist() == want[:small].tolist()
    off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in sigs])
    blob = b"".join(w32(v) for s in sigs for v in s)
    dev = lambda a: torch.from_numpy(np.frombuffer(a, dtype=np.uint8).copy()).cuda()
    d_k, d_p, d_s, d_o = dev(key_idx.tobytes()), dev(b"".join(prs)), dev(blob), dev(off.tobytes())
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d_st = torch.full((n,), 255, dtype=torch.uint8, device="cuda")
        Z.Groth16Verifier.verify_batch_keys_device(ks, 0, d_k.data_ptr(), d_p.data_ptr(), d_s.data_ptr(), d_o.data_ptr(), n, d_st.data_ptr(), side.cuda_stream)
    side.synchronize()
    assert d_st.cpu().numpy().tolist() == want.tolist()
