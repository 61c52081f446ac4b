"""CPU-side check of the arithmetic the kernels are built from: csrc/bn254.cuh compiled as plain C++
(tests/host_emu/emu.cpp) against the oracle, and the PTX instruction lists of csrc/fp_ptx.cuh simulated
against Python integers (tools/gen_fp_ptx.py --check)."""
import ctypes as C
import os
import subprocess
import sys

import pytest

import oracle_lib as O
from stylus_zkvm_verifiers_b200.synth import G2_GEN, SplitMix64, random_twist_point

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
w32 = O.w32
G1 = w32(1) + w32(2)


@pytest.fixture(scope="module")
def emu():
    d = os.path.join(ROOT, "tests", "host_emu")
    so = os.path.join(d, "libzkv_emu.so")
    srcs = [os.path.join(d, "emu.cpp"), os.path.join(d, "lazy_leaf_host.h")] + [os.path.join(ROOT, "stylus_zkvm_verifiers_b200", "csrc", f) for f in ("bn254.cuh", "bn254_consts.cuh", "lazy.cuh", "lazy_gen.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, srcs[0]])
    return C.CDLL(so)


def rand_f12(rng):
    return b"".join(w32(rng.u256() % P) for _ in range(12))


def test_ptx_instruction_lists_simulate_correctly():
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "gen_fp_ptx.py"), "--check"])


def test_generated_header_is_current():
    """csrc/fp_ptx.cuh must be exactly what the (verified) generator emits."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_fp_ptx", os.path.join(ROOT, "tools", "gen_fp_ptx.py"))
    g = importlib.util.module_from_spec(spec); spec.loader.exec_module(g)
    assert open(os.path.join(ROOT, "stylus_zkvm_verifiers_b200", "csrc", "fp_ptx.cuh")).read() == g.render()


def test_fp_and_fp12_ops(emu):
    rng = SplitMix64(11)
    out = C.create_string_buffer(384)
    for _ in range(50):
        a, b = rng.u256() % P, rng.u256() % P
        emu.emu_fp_mul(w32(a), w32(b), out); assert out.raw[:32] == w32(a * b % P)
        emu.emu_fp_inv(w32(a), out); assert out.raw[:32] == w32(pow(a, -1, P))
    for _ in range(10):
        x, y = rand_f12(rng), rand_f12(rng)
        emu.emu_f12_mul(x, y, out); assert out.raw == O.fp12_mul(x, y)
        emu.emu_f12_sqr(x, out); assert out.raw == O.fp12_mul(x, x)
        emu.emu_f12_inv(x, out); inv = out.raw
        one = w32(1) + bytes(352)
        assert O.fp12_mul(x, inv) == one


def test_safegcd_inversion_equals_fermat_and_pow(emu):
    """fp_inv (constant-time safegcd, 20 x 30 division steps) against the Fermat inversion it replaced and Python's pow, on edge values
    (0 -> 0, 1, p - 1, small, powers of two, values around 2^k) and random ones."""
    rng = SplitMix64(77)
    out, ref = C.create_string_buffer(32), C.create_string_buffer(32)
    vals = [0, 1, 2, 3, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, 1 << 253, (1 << 253) - 1, (1 << 128), (1 << 128) + 1, (1 << 30), (1 << 30) - 1, (1 << 60) + 5]
    vals += [(1 << k) % P for k in range(0, 256, 17)] + [rng.fr() % P for _ in range(400)]
    for a in vals:
        emu.emu_fp_inv(w32(a), out); emu.emu_fp_inv_fermat(w32(a), ref)
        want = pow(a, -1, P) if a else 0
        assert out.raw[:32] == w32(want) == ref.raw[:32], hex(a)


def test_final_exp_and_cyclotomic(emu):
    rng = SplitMix64(12)
    out = C.create_string_buffer(384)
    for _ in range(3):
        m = rand_f12(rng)
        emu.emu_final_exp(m, out); gt = out.raw
        assert gt == O.final_exp(m)
        emu.emu_f12_cyc_sqr(gt, out)                                  # GT is in the cyclotomic subgroup
        assert out.raw == O.fp12_mul(gt, gt) == O.fp12_cyc_sqr(gt)


def test_staged_final_exp_equals_single(emu):
    rng = SplitMix64(21)
    a, b = C.create_string_buffer(384), C.create_string_buffer(384)
    for _ in range(3):
        x = rand_f12(rng)
        emu.emu_final_exp(x, a); emu.emu_final_exp_staged(x, b)
        assert a.raw == b.raw == O.final_exp(x)


def test_g2_subgroup_test_matches_oracle(emu):
    rng = SplitMix64(13)
    for k in (1, 2, 3, R - 1, rng.fr(), rng.fr()):
        assert emu.emu_g2_check(O.g2_mul(G2_GEN, k)) == 1
    for _ in range(6):
        q = random_twist_point(rng)
        assert O.ec_pairing(G1 + q) is None                           # oracle: [r]Q != inf -> revert
        assert emu.emu_g2_check(q) == 0
        # small-order component: add a subgroup point; still outside G2
        assert emu.emu_g2_check(O.g2_add(q, O.g2_mul(G2_GEN, rng.fr()))) == 0
    bad = bytearray(G2_GEN); bad[100] ^= 4
    assert emu.emu_g2_check(bytes(bad)) == 2


def test_pairing_values_bit_exact(emu, consts):
    rng = SplitMix64(14)
    h = bytes.fromhex
    vkj = consts["risc0_vk"]
    fixed = b"".join(h(vkj[n][i][j]) for n in ("beta", "gamma", "delta") for i in range(2) for j in range(2))
    mo, go, m3 = C.create_string_buffer(384), C.create_string_buffer(384), C.create_string_buffer(384)
    for _ in range(3):
        g1s = b"".join(O.g1_mul(G1, rng.fr()) for _ in range(4))
        q = O.g2_mul(G2_GEN, rng.fr())
        data = g1s[0:64] + q + g1s[64:128] + fixed[0:128] + g1s[128:192] + fixed[128:256] + g1s[192:256] + fixed[256:384]
        ret, m, gt = O.ec_pairing(data, debug=True)
        ok = emu.emu_pairing4(g1s, q, fixed, mo, go)
        assert mo.raw == m and go.raw == gt and ok == ret[31]
        emu.emu_pairing3_pre(g1s, q, fixed, m3)                        # 3-pair loop x precomputed Miller(alpha, beta): same field element
        assert m3.raw == m
        # verification path (normalised gamma / delta lines): different Miller value, the SAME final-exponentiation output
        assert emu.emu_verify_norm_gt(g1s, q, fixed, 0, go) == ret[31] and go.raw == gt
        # pairs switched off (a member at infinity contributes 1): compare with the oracle on the remaining pairs
        for mask, keep in ((2, (0, 1, 3)), (4, (0, 1, 2)), (1, (1, 2, 3)), (6, (0, 1))):
            g2s = (q, fixed[0:128], fixed[128:256], fixed[256:384])
            d2 = b"".join(g1s[64 * j:64 * j + 64] + g2s[j] for j in keep)
            r2, _, gt2 = O.ec_pairing(d2, debug=True)
            assert emu.emu_verify_norm_gt(g1s, q, fixed, mask, go) == r2[31] and go.raw == gt2, mask


def test_lazy_generator_bounds_and_current_header():
    """tools/gen_lazy.py proves every bound of the lazily reduced routines and checks their values; csrc/lazy_gen.cuh is what it emits."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_lazy", os.path.join(ROOT, "tools", "gen_lazy.py"))
    g = importlib.util.module_from_spec(spec); spec.loader.exec_module(g)
    assert open(os.path.join(ROOT, "stylus_zkvm_verifiers_b200", "csrc", "lazy_gen.cuh")).read() == g.render()


def test_two_lane_generator_bounds_and_current_header():
    """tools/gen_lazy2.py (two lanes per proof, the measured alternative layout of DESIGN.md section 5) proves the bounds of its routines for
    both lanes and checks their values against plain modular arithmetic; csrc/lazy2_gen.cuh is what it emits."""
    import importlib.util
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    spec = importlib.util.spec_from_file_location("gen_lazy2", os.path.join(ROOT, "tools", "gen_lazy2.py"))
    g = importlib.util.module_from_spec(spec); spec.loader.exec_module(g)
    assert open(os.path.join(ROOT, "stylus_zkvm_verifiers_b200", "csrc", "lazy2_gen.cuh")).read() == g.render()


def test_lazy_tower_on_slots_matches_round1_tower(emu):
    """csrc/lazy.cuh (shared-memory slots, lazily reduced Fp6 routines) against the round-1 tower and the oracle, including all-(p-1),
    all-zero and mixed-extreme operands; the portable leaves abort on any carry, borrow or reduction-range violation."""
    import random
    rnd = random.Random(5)

    def rv(n, mode):
        if mode == 0: return [P - 1] * n
        if mode == 1: return [0] * n
        if mode == 2: return [rnd.choice([0, P - 1, 1, P - 2]) for _ in range(n)]
        return [rnd.randrange(P) for _ in range(n)]
    out, ref, o12 = C.create_string_buffer(192), C.create_string_buffer(192), C.create_string_buffer(384)
    for it in range(120):
        m = it % 4 if it < 40 else 3
        a = b"".join(w32(x) for x in rv(6, m)); b = b"".join(w32(x) for x in rv(6, (m + it // 4) % 4 if it < 40 else 3))
        for sp in (0, 1):
            emu.emu_lz_f6mul(a, b, sp, out, ref); assert out.raw == ref.raw, (it, sp)
    for it in range(40):
        x = b"".join(w32(v) for v in rv(12, it % 4 if it < 20 else 3))
        emu.emu_lz_f12sqr(x, o12); assert o12.raw == O.fp12_mul(x, x), it


def test_lazy_fp12_routines_match_oracle(emu):
    """The Fp12-level routines of csrc/lazy.cuh on slots, over the operand classes of oracle_lib.fp12_operand_classes (all p - 1, zero,
    one, -1, edge words, subfield elements, c0 = 0, c1 = 0, b = a, b = conj(a)): lz_f12mul_g plain and conjugated against the oracle and the
    round-1 tower, lz_f12inv by its product with the operand (inv(0) = 0), lz_frob against the round-1 Frobenius and, on some operands,
    against a^(p^k) by square-and-multiply, lz_cyc_sqr on cyclotomic elements only, the staged lz_final_exp_stage against the oracle."""
    mul, mulc, inv, csq, rmulc, fe = (C.create_string_buffer(384) for _ in range(6))
    fr, rfr = C.create_string_buffer(3 * 384), C.create_string_buffer(3 * 384)
    firsts = {}
    for name, a, b in O.fp12_operand_classes(31):
        emu.emu_lz_f12_ops(a, b, mul, mulc, inv, csq, fr)
        emu.emu_f12_misc(a, b, rmulc, rfr)
        assert mul.raw == O.fp12_mul(a, b), name
        assert mulc.raw == rmulc.raw == O.fp12_mul(a, O.fp12_conj(b)), name
        if a == bytes(384):
            assert inv.raw == bytes(384), name
        else:
            assert O.fp12_mul(a, inv.raw) == O.FP12_ONE, name
        assert fr.raw == rfr.raw, name
        firsts.setdefault(a, (name.split("|")[0], fr.raw))
    for a, (name, frs) in list(firsts.items())[::2]:
        x = a
        for k in range(3):
            x = O.fp12_frob(x, 1)
            assert frs[384 * k:384 * k + 384] == x, (name, k + 1)
    for a, (name, _) in firsts.items():
        emu.emu_lz_final_exp(a, fe)
        assert fe.raw == O.final_exp(a), name
    for name, g in O.fp12_cyclotomic_operands(31):
        emu.emu_lz_f12_ops(g, g, mul, mulc, inv, csq, fr)
        assert csq.raw == O.fp12_cyc_sqr(g) == O.fp12_mul(g, g), name
        assert mulc.raw == O.FP12_ONE, name                          # g * conj(g) = 1 on the cyclotomic subgroup


def test_lazy_miller_loop_bit_exact_with_round1_loop(emu, consts):
    """lz_miller_norm_seg (one and several segments, pairs switched off) reproduces miller_loop_norm's Fp12 value bit for bit."""
    rng = SplitMix64(21)
    h = bytes.fromhex
    vkj = consts["risc0_vk"]
    fixed = b"".join(h(vkj[n][i][j]) for n in ("beta", "gamma", "delta") for i in range(2) for j in range(2))
    a, b = C.create_string_buffer(384), C.create_string_buffer(384)
    for k, (mask, nseg) in enumerate(((0, 1), (0, 8), (1, 3), (2, 1), (4, 5), (7, 2))):
        g1s = b"".join(O.g1_mul(G1, rng.fr()) for _ in range(4))
        q = O.g2_mul(G2_GEN, rng.fr())
        assert emu.emu_lz_miller_norm(g1s, q, fixed, mask, nseg, a, b) == 0
        assert a.raw == b.raw, (mask, nseg)


def test_g1_scalar_mul(emu):
    rng = SplitMix64(15)
    out = C.create_string_buffer(64)
    for k in (0, 1, 2, R - 1, R, R + 5, (1 << 256) - 1, rng.u256(), rng.u256()):
        emu.emu_g1_mul(G1, w32(k), out)
        assert out.raw == O.ec_mul(G1 + w32(k))


def test_routines_with_large_temporaries_stay_out_of_line():
    """Source rule from DESIGN.md section 5: nvcc's optimiser merged the stack slots of an INLINED routine's temporaries with live values
    of the Miller loop.  The routines below hold Fp2-and-larger temporaries and are called from frames that keep values across the call,
    so they must remain out of line; the Frobenius operands of the Miller loops must be computed inside the loop that uses them."""
    src = open(os.path.join(ROOT, "stylus_zkvm_verifiers_b200", "csrc", "bn254.cuh")).read()
    for name in ("f12_mul_line_at", "f12_mul_nline_at", "f12_mul_line", "f12_mul_line1", "miller_loop", "miller_loop_norm", "miller_loop_norm_seg", "g2_precompute_lines",
                 "g2_normalise_lines", "g1_slopes2", "line_dbl", "line_add", "f12_sqr", "f12_mul", "f6_mul", "f6_mul_01", "f12_pow_u", "final_exp"):
        decl = [l for l in src.split("\n") if (" " + name + "(") in l and l.startswith("ZKV_HD")]
        assert decl and all("ZKV_NOINLINE" in l for l in decl), name
    for loop in ("miller_loop", "miller_loop_norm", "miller_loop_norm_seg"):
        body = src[src.index("void " + loop + "("):]
        body = body[:body.index("\n}\n")]
        tail = body[body.index("for (int s = 1; s <= 2; s++)"):]
        assert "g2_frob_affine(xs, ys, s)" in tail and "fp2 x2" not in body, loop
