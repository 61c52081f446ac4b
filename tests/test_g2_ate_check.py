"""The G2 subgroup test that the verification Miller loop finishes (csrc/lazy.cuh: lz_miller_norm_seg leaves R = [6u+2]B + psi(B) - psi^2(B),
lz_r_is compares it with -psi^3(B)).  The number theory behind its accept set, and the kernel's own code compiled as plain C++
(tests/host_emu/g2_ate.cpp) against the oracle's [r]B = infinity on members, non-members, mixed-order and small-order points and infinity."""
import ctypes as C
import math
import os
import subprocess

import pytest

import oracle_lib as O
from stylus_zkvm_verifiers_b200.synth import G2_GEN, SplitMix64, random_twist_point

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 4965661367192848881
P = 36 * U**4 + 36 * U**3 + 24 * U**2 + 6 * U + 1
R = 36 * U**4 + 36 * U**3 + 18 * U**2 + 6 * U + 1
T = 6 * U * U + 1                     # trace of Frobenius: psi^2 - T psi + P = 0 on the twist
H2 = 2 * P - R                        # cofactor of G2 in E'(Fp2)
SMALL = 10069                         # the small prime factor of H2
INF = bytes(128)


def alpha():
    """alpha = 6u+2 + psi - psi^2 + psi^3 as a0 + a1 psi in Z[psi] / (psi^2 - T psi + P)"""
    # psi^2 = T psi - P, psi^3 = (T^2 - P) psi - T P
    return 6 * U + 2 + P - T * P, 1 - T + T * T - P


def norm(a0, a1):
    return a0 * a0 + a0 * a1 * T + a1 * a1 * P


def test_constants():
    assert P == 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
    assert R == 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001


def test_congruence():
    assert (6 * U + 2 + P - P * P + P**3) % R == 0


def test_alpha_norm_is_prime_to_the_cofactor():
    n = norm(*alpha())
    assert n % R == 0
    assert math.gcd(n, H2) == 1          # alpha has no kernel in the cofactor part of E'(Fp2)
    assert math.gcd(R, H2) == 1          # E'(Fp2) = G2 x (cofactor group)
    assert H2 % 2 == 1                   # no 2-torsion: doubling never meets Y = 0
    assert H2 % SMALL == 0 and (H2 // SMALL) % SMALL != 0


def add_prefixes():
    """R = [k]B before each addition of the loop, as integers: the NAF additions, then the two Frobenius additions ([6u+2] + psi(B),
    then - psi^2(B)); returned as (k, the multiple of B added) with psi standing for P on G2"""
    naf = O.ate_naf()
    k, out = 1, []
    for d in range(len(naf) - 2, -1, -1):
        k *= 2
        if naf[d]:
            out.append((k, naf[d]))
            k += naf[d]
    assert k == 6 * U + 2
    out.append((k, P))
    out.append((k + P, -P * P))
    return out


def test_no_exceptional_step_for_members():
    """For B in G2 the homogeneous formulas meet none of their exceptional cases: no doubling of O (no prefix = 0) and no addition of
    +-(the added point) (prefix = +-added, mod r)."""
    for k, a in add_prefixes():
        assert k % R != 0
        assert (k - a) % R != 0 and (k + a) % R != 0


def test_naf_prefixes_modulo_the_small_factor():
    """For a point of order 10069, no NAF addition meets R = +-B or R = O (so those points exercise the Frobenius steps and the final
    comparison, not an early collapse)."""
    for k, a in add_prefixes()[:-2]:
        assert k % SMALL not in (0, 1, SMALL - 1)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    d = os.path.join(ROOT, "tests", "host_emu")
    so = str(tmp_path_factory.mktemp("g2ate") / "libg2ate.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(d, "g2_ate.cpp")])
    lib = C.CDLL(so)
    lib.emu_ate_g2_check.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p]
    return lib


def fused(emu, q, nseg=1, var_off=0):
    out = C.create_string_buffer(192)
    return emu.emu_ate_g2_check(q, nseg, var_off, out), out.raw


def oracle_member(q):
    return q == INF or O.g2_mul(q, R) == INF


def small_point(rng):
    while True:
        q = O.g2_mul(O.g2_mul(random_twist_point(rng), R), H2 // SMALL)
        if q != INF:
            assert O.g2_mul(q, SMALL) == INF
            return q


def check(emu, q, want, **kw):
    assert oracle_member(q) == want
    got, _ = fused(emu, q, **kw)
    assert got == (1 if want else 0)


def test_members(emu):
    rng = SplitMix64(21)
    check(emu, G2_GEN, True)
    for j in range(4):
        check(emu, O.g2_mul(G2_GEN, rng.u256() % R), True, nseg=(1, 3, 4)[j % 3], var_off=j & 1)
    check(emu, O.g2_mul(G2_GEN, R - 1), True)


def test_infinity(emu):
    assert fused(emu, INF)[0] == 1
    assert fused(emu, INF, nseg=4, var_off=1)[0] == 1


def test_random_twist_points(emu):
    rng = SplitMix64(22)
    for j in range(5):
        check(emu, random_twist_point(rng), False, nseg=(1, 4)[j % 2], var_off=j & 1)


def test_member_plus_small_order(emu):
    rng = SplitMix64(23)
    for _ in range(3):
        q = O.g2_add(O.g2_mul(G2_GEN, rng.u256() % R), small_point(rng))
        check(emu, q, False)


def test_small_order(emu):
    """Pure order-10069 points, their multiples and negatives, including any multiple for which a Frobenius addition of the loop meets
    R = +-(the added point) or R = O (read back from R's Z coordinate)."""
    rng = SplitMix64(24)
    q = small_point(rng)
    zero_z = 0
    for m in (1, 2, SMALL - 1, 1 + rng.below(SMALL - 1), 1 + rng.below(SMALL - 1)):
        qm = O.g2_mul(q, m)
        got, r = fused(emu, qm, nseg=4)
        assert oracle_member(qm) is False and got == 0
        zero_z += r[128:] == bytes(64)
    # whether an exceptional case occurs here depends on psi's eigenvalue on the order-10069 subgroup, which is the same for every such point
    assert zero_z in (0, 5)


def test_order_r_multiple_of_a_non_member(emu):
    """[h'] Q is always in G2, [r] Q (Q off G2) never: both agree with the oracle."""
    rng = SplitMix64(25)
    q = random_twist_point(rng)
    check(emu, O.g2_mul(O.g2_mul(q, SMALL), H2 // SMALL), True)
    check(emu, O.g2_mul(q, R), False)
