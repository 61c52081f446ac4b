"""The single-cause cases of single_cause.py on the CPU: the catalogue's orders, every case rejected and every twin accepted by the C oracle,
the Python referee on a sample, and the host emulation of the fused G2 subgroup test (tests/host_emu/g2_ate.cpp) on every catalogue point."""
import ctypes as C
import os
import subprocess

import pytest

import oracle_lib as O
import single_cause as SC
import vkx_edges as V
from stylus_zkvm_verifiers_b200 import synth as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P, R, H2, ELL = SC.P, SC.R, SC.H2, SC.ELL


def _is_prime(n):
    """Miller-Rabin with the first 20 primes as bases (deterministic far beyond the sizes here, and a strong test at 178 bits)"""
    bases = (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37, 41, 43, 47, 53, 59, 61, 67, 71)
    if n in bases:
        return True
    if n < 2 or any(n % b == 0 for b in bases):
        return False
    d, s = n - 1, 0
    while d % 2 == 0:
        d //= 2; s += 1
    for a in bases:
        x = pow(a, d, n)
        if x in (1, n - 1):
            continue
        for _ in range(s - 1):
            x = x * x % n
            if x == n - 1:
                break
        else:
            return False
    return True


@pytest.fixture(scope="module")
def outside():
    return SC.outside_catalogue()


@pytest.fixture(scope="module")
def members():
    return SC.member_catalogue()


@pytest.fixture(scope="module")
def generic():
    return SC.generic_cases()


@pytest.fixture(scope="module")
def sp1():
    return SC.sp1_cases()


@pytest.fixture(scope="module")
def risc0():
    return SC.risc0_cases()


def test_cofactor_factors():
    assert H2 == ELL[0] * ELL[1] * ELL[2] * ELL[3] and len(set(ELL)) == 4
    assert all(_is_prime(l) for l in ELL) and ELL[3].bit_length() == 178
    assert all(H2 % (l * l) for l in ELL)                                   # square-free: [r]Q of order H2 has a point of each order l | H2


def test_catalogue_orders(outside, members):
    """[r]B != infinity for every outside point; where an order is stated, [order]B = infinity and [order / l]B != infinity for each of its
    prime factors l (the order is exact); members: [r]B = infinity"""
    assert len({b.point for b in outside}) == len(outside)
    for b in outside:
        assert b.point != SC.INF2 and O.g2_mul(b.point, R) != SC.INF2, b.name
        if b.order is None:
            continue
        assert SC.g2_mul_all(b.point, b.order) == SC.INF2, b.name
        for i in range(len(b.order)):
            assert SC.g2_mul_all(b.point, b.order[:i] + b.order[i + 1:]) != SC.INF2, (b.name, b.order[i])
    orders = {b.order for b in outside}
    assert all((l,) in orders and (R, l) in orders for l in ELL) and ELL in orders
    assert sum(1 for o in orders if o and len(o) == 2 and R not in o) >= 3
    assert sum(1 for b in outside if b.name.startswith("-")) >= 4
    for b in outside:                                                        # negations are the negated points
        if b.name.startswith("-"):
            assert O.g2_add(b.point, next(c.point for c in outside if c.name == b.name[1:])) == SC.INF2
    for name, q in members:
        assert q == SC.INF2 or O.g2_mul(q, R) == SC.INF2, name
    by = dict(members)
    assert by["inf"] == SC.INF2 and by["-G2"] == by["[r-1]G2"]               # the negation by its coordinates and by its scalar
    assert len({q for _, q in members}) == len(members) - 1


def _generic_status(keys, recs):
    out = []
    for r in recs:
        out.append(int(O.groth16_verify_batch(keys[r.key].ovk(), r.proof, b"".join(O.w32(v) for v in r.signals), 1)[0]))
    return out


def test_generic_cases_oracle(generic):
    keys, units, _ = generic
    recs = SC.records(units)
    assert _generic_status(keys, recs) == [r.expect for r in recs], [r.name for r, s in zip(recs, _generic_status(keys, recs)) if s != r.expect]
    causes = {(u.case.key, u.cause) for u in units}
    assert {(0, "g2"), (1, "g2"), (2, "g2"), (3, "g2"), (0, "range"), (1, "range"), (4, "range"), (5, "range")} <= causes
    assert keys[2].alpha == SC.INF1 and keys[3].alpha == SC.INF1
    for u in units:                                                          # the twin differs from the case in one input only
        assert u.case.key == u.twin.key and u.case.signals == u.twin.signals
        diff = [i for i in range(8) if SC.word(u.case.proof, i) != SC.word(u.twin.proof, i)]
        assert diff and (diff[0] in (2, 3, 4, 5) if u.cause == "g2" else len(diff) == 1), u.case.name


def test_sp1_cases_oracle(sp1):
    keys, units = sp1
    for route, key in enumerate(keys):
        rs = [r for r in SC.records(units) if r.key == route]
        st = O.sp1_verify_batch(key.ovk(), S.SP1_SELECTOR, [r.vkey for r in rs], [r.pv for r in rs], [S.SP1_SELECTOR + r.proof for r in rs])
        assert st.tolist() == [r.expect for r in rs], [r.name for r, s in zip(rs, st) if s != r.expect]
    vk = {int.from_bytes(u.case.vkey, "big") for u in units}
    v = int.from_bytes(next(u.twin.vkey for u in units if u.case.name == "sp1:vkey=v+1R"), "big")
    assert {v + k * R for k in range(1, 6)} <= vk and R in vk and 2 * R - 1 in vk
    assert v + 5 * R < 1 << 256 <= v + 6 * R or v + 6 * R < 1 << 256      # every k that fits, up to 5
    assert all(len(r.pv) == SC.PV_LEN for r in SC.records(units))


def test_risc0_cases_oracle(risc0):
    hs, units = risc0
    ros = [h.oracle() for h in hs]
    assert len({ro.selector() for ro in ros}) == len(hs)                    # each handle is its own route
    for hi, ro in enumerate(ros):
        rs = [r for r in SC.records(units) if r.key == hi]
        assert rs, hs[hi].name
        st = ro.verify_batch([ro.selector() + r.proof for r in rs], [r.im for r in rs], [r.jr for r in rs])
        assert st.tolist() == [r.expect for r in rs], [r.name for r, s in zip(rs, st) if s != r.expect]
        assert [ro.verify_integrity(ro.selector() + r.proof, O.claim_digest(r.im, r.jr)) for r in rs] == [r.expect for r in rs]
    c = int.from_bytes(hs[0].cid, "big")
    assert [int.from_bytes(h.cid, "big") for h in hs[1:8]] == [c + k * R for k in range(1, 6)] + [R - 1, 2 * R - 1]
    for u in units:                                                          # a control-id case is its twin's proof on another route
        if u.case.key != u.twin.key:
            assert u.case.proof == u.twin.proof and (u.case.im, u.case.jr) == (u.twin.im, u.twin.jr)
            assert int.from_bytes(hs[u.case.key].cid, "big") % R == int.from_bytes(hs[u.twin.key].cid, "big")


def test_python_referee_on_a_sample(generic, sp1, risc0):
    """the independent Python restatement agrees on a B-outside case of each family with its twin, a deep case, a proof-word range case and
    the control-id and vkey ranges"""
    import bn254_py as PY

    def vkd(k):
        g2 = lambda b: ((int.from_bytes(b[0:32], "big"), int.from_bytes(b[32:64], "big")), (int.from_bytes(b[64:96], "big"), int.from_bytes(b[96:128], "big")))
        return dict(alpha=V.coords(k.alpha), beta=g2(k.beta), gamma=g2(k.gamma), delta=g2(k.delta), ic=[V.coords(p) for p in k.ic])
    words = lambda pr: [SC.word(pr, i) for i in range(8)]
    def pick(units, *names):
        out = [u for u in units if any(u.case.name.startswith(n) for n in names)]
        assert len(out) >= len(names), names
        return out
    keys, units, _ = generic
    for u in pick(units, "generic0:A=(0,p)|B=order=l2", "deep3:A=(0,0)|B=G2m+order=l4", "generic1|w3+1p"):
        for r in (u.case, u.twin):
            w = words(r.proof)
            assert PY.groth16_verify(keys[r.key].vm, vkd(keys[r.key]), w[0:2], [w[2:4], w[4:6]], w[6:8], r.signals) == (r.expect == SC.OK), r.name
    keys, units = sp1
    for u in pick(units, "sp1:vkey=v+5R", "sp1deep:A=(0,0)|B=order=H2"):
        for r in (u.case, u.twin):
            st = PY.sp1_verify_status(vkd(keys[r.key]), S.SP1_SELECTOR, r.vkey, r.pv, S.SP1_SELECTOR + r.proof)
            assert st == r.expect, r.name
    hs, units = risc0
    for u in pick(units, "risc0:cid=c+1R#0", "risc0deep:A=(0,p)|B=random1", "risc0|A.y=y_w-1p"):
        for r in (u.case, u.twin):
            h = hs[r.key]
            st = PY.risc0_verify_status(vkd(h.key), h.selector(), h.cr, h.cid, h.selector() + r.proof, r.im, r.jr)
            assert st == r.expect, r.name


def test_layout():
    units = [SC.Unit("g2", SC.Rec("c%d" % i, 0, b"", SC.FAIL), SC.Rec("t%d" % i, 0, b"", SC.OK)) for i in range(5)]
    for n, chunk in ((40, None), (130, None), (300, None), (1 << 12, 1024)):
        lanes = SC.anchors(n, chunk)
        recs = SC.layout(units, n, lanes)
        assert len(recs) == n and all(r is not None for r in recs)
        for a in lanes:                     # a case beside its twin (at n = 130, lane 128 holds the twin of the last record's case)
            other = ("t" if recs[a].expect == SC.FAIL else "c") + recs[a].name[1:]
            assert recs[a].expect == SC.FAIL or (n, a) == (130, 128), (n, a)
            assert any(recs[b].name == other for b in (a - 1, a + 1) if 0 <= b < n), (n, a)
        assert recs[n - 1].expect == SC.FAIL
        assert {0, 31, 32, n - 1} <= set(lanes) and (chunk is None or {chunk - 1, chunk, 3 * chunk} <= set(lanes))


# ------------------------------------------------------------------ host emulation of the fused subgroup test
@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    d = os.path.join(ROOT, "tests", "host_emu")
    so = str(tmp_path_factory.mktemp("g2ate_sc") / "libg2ate.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(d, "g2_ate.cpp")])
    lib = C.CDLL(so)
    lib.emu_ate_g2_check.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p]
    return lib


@pytest.mark.parametrize("nseg", [1, 4, 7, 16])
def test_host_emulation_on_catalogue(emu, outside, members, nseg):
    """the kernel's Miller loop with the variable pair switched off (as for A at infinity) and its final comparison: 0 on every outside
    point (each cofactor prime's order, their products, H2, members plus them), 1 on every member and on infinity"""
    out = C.create_string_buffer(192)
    for b in outside:
        assert emu.emu_ate_g2_check(b.point, nseg, 1, out) == 0, b.name
    for name, q in members:
        assert emu.emu_ate_g2_check(q, nseg, 1, out) == 1, name
