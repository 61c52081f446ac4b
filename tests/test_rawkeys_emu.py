"""The raw-key verification path's arithmetic on a CPU-only box: csrc/bn254.cuh g1_vkx_var (the variable-base vk_x) and the four-variable-pair
Miller loop of csrc/lazy.cuh with its fused order-r test (lz_gen_subgroup_ok), compiled as plain C++ (tests/host_emu/rawkeys.cpp), against the
oracle's chain of ecMul / ecAdd calls and its ecPairing."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest

import oracle_lib as O
from stylus_zkvm_verifiers_b200.synth import G2_GEN, SplitMix64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
G1 = w32(1) + w32(2)
INF1, INF2 = bytes(64), bytes(128)


@pytest.fixture(scope="module")
def emu():
    out = tempfile.mkdtemp(prefix="zkv_rawkeys_emu_")
    so = os.path.join(out, "librawkeys_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "host_emu", "rawkeys.cpp")])
    return C.CDLL(so)


def chain(ic, scalars):
    """compute_vk_x (groth16.rs:51-58) as precompile calls: None where an ecMul / ecAdd call fails"""
    acc = ic[0]
    for p, s in zip(ic[1:], scalars):
        t = O.ec_mul(p + w32(s))
        if t is None:
            return None
        acc = O.ec_add(acc + t)
        if acc is None:
            return None
    return acc


def vkx(emu, ic, scalars):
    out = C.create_string_buffer(64)
    r = emu.emu_vkx_var(b"".join(ic), len(ic), b"".join(w32(s) for s in scalars), out)
    return r, out.raw


def check(emu, ic, scalars):
    want = chain(ic, scalars)
    r, got = vkx(emu, ic, scalars)
    if want is None:
        assert r == 2 and got == INF1
    else:
        assert got == want and r == (1 if want == INF1 else 0)
    return r


def test_random_keys_every_width(emu):
    rng = SplitMix64(101)
    for n_ic in range(2, 17):
        for _ in range(2):
            ic = [O.g1_mul(G1, rng.fr()) for _ in range(n_ic)]
            assert check(emu, ic, [rng.fr() for _ in range(n_ic - 1)]) == 0


def test_edge_scalars(emu):
    rng = SplitMix64(102)
    ic = [O.g1_mul(G1, rng.fr()) for _ in range(6)]
    edges = [0, 1, 2, 7, 8, 9, 15, 16, 17, R - 1, R - 2, R - 8, (1 << 253) - 1, 1 << 253, (R - 1) // 2, 0x7777777777777777, 0x9999999999999999]
    for s in edges:
        check(emu, ic, [s, 1, R - 1, 0, s])
    for s in (R, R + 1, 2 * R - 1, (1 << 256) - 1, 5 * R + 3):      # ecMul takes any 256-bit scalar
        check(emu, ic, [s, rng.fr(), s, 0, 1])
    assert check(emu, ic, [0] * 5) == 0                              # vk_x = IC_0


def test_exceptional_additions(emu):
    """IC_j at infinity, equal to or the negation of another IC point or of a partial sum, vk_x = infinity"""
    rng = SplitMix64(103)
    a, b = rng.fr(), rng.fr()
    A, B = O.g1_mul(G1, a), O.g1_mul(G1, b)
    nA = O.g1_mul(G1, R - a)
    cases = [
        ([A, INF1, B], [rng.fr(), rng.fr()]),                 # IC_1 at infinity
        ([INF1, A, B], [rng.fr(), rng.fr()]),                 # IC_0 at infinity
        ([INF1, INF1, INF1], [5, 7]),                         # everything at infinity
        ([A, A, A], [1, 1]),                                  # P + P along the chain
        ([A, nA, A], [1, 1]),                                 # partial sum at infinity, then P
        ([A, nA], [1]),                                       # vk_x = infinity
        ([A, A], [R - 1]),                                    # IC_0 + (r - 1) IC_0 = infinity
        ([A, B, A], [3, R - 3]),                              # the two scalar multiples cancel
        ([A, G1, G1], [b, R - b]),
        ([O.g1_mul(G1, 5), G1, G1], [R - 5, 0]),              # IC_0 = -s IC_1: infinity after the first ecAdd
        ([O.g1_mul(G1, 3), G1, G1, G1], [1, 1, R - 5]),       # 3 + 1 = 4 (P + P step at the partial sum), then -5 ... = -1
        ([A, G1, O.g1_mul(G1, 2)], [2, 3]),                   # digit additions that hit equal points inside the sum
    ]
    for ic, s in cases:
        check(emu, ic, s)
    assert check(emu, [A, nA], [1]) == 1


def test_invalid_ic_points(emu):
    rng = SplitMix64(104)
    ic = [O.g1_mul(G1, rng.fr()) for _ in range(4)]
    s = [rng.fr() for _ in range(3)]
    for j in range(4):
        for mutate in (lambda p: p[:32] + w32((int.from_bytes(p[32:], "big") + 1) % P),     # off the curve
                       lambda p: w32(int.from_bytes(p[:32], "big") + P) + p[32:],           # x >= p
                       lambda p: p[:32] + w32(P),                                           # y = p
                       lambda p: w32(0) + w32(1)):                                          # (0, 1): off the curve
            bad = list(ic); bad[j] = mutate(ic[j])
            assert check(emu, bad, s) == 2
            assert check(emu, bad, [0] * 3) == 2                                            # whatever the scalar: the call fails


def _pairs_data(pairs):
    return b"".join(g1 + g2 for g1, g2 in pairs)


def _accepts(g2):
    """the oracle's verdict on a G2 point: a pairing with it and a finite G1 point does not revert"""
    return O.ec_pairing(G1 + g2) is not None


def test_fused_four_point_subgroup_test_matches_oracle(emu):
    """Each of the four G2 points in turn is a multiple of the generator, a twist point from g2_from_x (almost always outside G2) or
    infinity, paired with a G1 point at infinity and with a finite one, beside three members; 1 and 3 segments."""
    rng = SplitMix64(105)
    members = [O.g2_mul(G2_GEN, k) for k in (1, 2, 3, R - 1, rng.fr(), rng.fr())]
    twist = []
    x = 1
    while len(twist) < 6:
        q = O.g2_from_x(x, rng.u256() % P)
        if q is not None:
            twist.append(q)
        x += 1
    out = C.create_string_buffer(384)
    outside = 0
    for cand in members + twist + [INF2]:
        want = 1 if (cand == INF2 or _accepts(cand)) else 0
        outside += want == 0
        for slot in range(4):
            for g1 in (INF1, O.g1_mul(G1, rng.fr())):
                pairs = [(O.g1_mul(G1, rng.fr()), members[(slot + t) % len(members)]) for t in range(4)]
                pairs[slot] = (g1, cand)
                for nseg in (1, 3):
                    assert emu.emu_rawkeys_miller4(_pairs_data(pairs), nseg, out) == want, (cand.hex()[:16], slot, g1 == INF1, nseg)
    assert outside >= 4


def test_four_pair_miller_value_is_the_oracles(emu):
    """With every point in G2 the loop's value is the oracle's Miller value bit for bit, pairs with a member at infinity contributing 1."""
    rng = SplitMix64(106)
    out = C.create_string_buffer(384)
    for mask in (0, 1, 2, 4, 8, 6, 15):
        pairs = []
        for j in range(4):
            g1, g2 = O.g1_mul(G1, rng.fr()), O.g2_mul(G2_GEN, rng.fr())
            if (mask >> j) & 1:
                if rng.below(2):
                    g1 = INF1
                else:
                    g2 = INF2
            pairs.append((g1, g2))
        assert emu.emu_rawkeys_miller4(_pairs_data(pairs), 4, out) == 1
        kept = [p for j, p in enumerate(pairs) if not (mask >> j) & 1]
        want = O.ec_pairing(_pairs_data(kept), debug=True)[1] if kept else w32(1) + bytes(352)
        assert out.raw == want, mask


def test_no_device_no_fallback():
    """without a CUDA device the raw-key handle cannot be created: ZKV_ERR_CUDA, never a CPU path"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import stylus_zkvm_verifiers_b200 as Z
    with pytest.raises(Z.ZkvError) as e:
        Z.RawKeyVerifier()
    assert e.value.code == Z._native.ZKV_ERR_CUDA
    L = Z._native.lib()                                        # a call without a handle is an argument error
    assert L.zkv_groth16_verify_batch_rawkeys(None, None, None, None, 0, None, None, None, None, 1, None) == Z._native.ZKV_ERR_ARG
    assert L.zkv_groth16_verify_batch_rawkeys_device(None, 0, None, None, None, 0, None, None, None, None, 1, None, None) == Z._native.ZKV_ERR_ARG
    assert L.zkv_vk_x_rawkeys_batch(None, None, None, 0, None, None, None, 1, None, None) == Z._native.ZKV_ERR_ARG
