"""CPU side of the chosen-point proofs of vkx_edges.py: the edge-point catalogue, the proof synthesis against synth.solve_c, every
accepting proof accepted and every twin rejected by the C oracle (and a sample by the Python referee), and the model's branch coverage of
every verification entry-point family."""
import pytest

import oracle_lib as O
import vkx_edges as V
from stylus_zkvm_verifiers_b200 import synth as S

P, R = V.P, V.R


@pytest.fixture(scope="module")
def generic():
    return V.generic_cases()


@pytest.fixture(scope="module")
def sp1():
    return V.sp1_cases()


@pytest.fixture(scope="module")
def risc0():
    return V.risc0_cases()


def test_edge_catalogue():
    import bn254_py as PY
    edges = V.edge_points()
    assert len(edges) == 20 and len({p for _, p in edges}) == 20
    for (name, p), (nname, q) in zip(edges[::2], edges[1::2]):
        assert nname == "-" + name and V.on_curve(p) and V.on_curve(q) and PY.g1_on_curve(V.coords(p))
        assert V.coords(q) == (V.coords(p)[0], P - V.coords(p)[1])
    by = dict(edges)
    x = lambda n: V.coords(by[n])[0]
    y = lambda n: V.coords(by[n])[1]
    assert x("x=p-1") == P - 1 and y("x=p-1") ** 2 % P == 2
    assert by["G1"] == S.G1_GEN and [x(n) for n in ("G1", "x=2", "x=3", "x=5")] == [1, 2, 3, 5]
    assert [x for x in range(6) if V.sqrt_p(x ** 3 + 3) is not None] == [1, 2, 3, 5]          # the smallest x on the curve
    for n, m in (("2", 2), ("4", 4), ("p-1", P - 1), ("p-2", P - 2)):
        assert V.mont(x("mont(x)=" + n)) == m and V.mont(x("-mont(x)=" + n)) == m
    assert V.mont(y("mont(y)=2")) == 2 and V.mont(y("-mont(y)=2")) == P - 2
    # residue 1 has no point: x = 2^-256 is not an x-coordinate, and y = +-2^-256 gives x^3 = y^2 - 3, a cubic non-residue
    assert V.point_at_x(V.MONT_INV) is None and V._cube_root(V.MONT_INV ** 2 - 3) is None


def test_catalogue_point_arithmetic_matches_python_referee():
    """ecAdd / ecMul of the oracle on the catalogue (doubling, P + (-P), multiples around r) against the independent Python referee"""
    import bn254_py as PY
    pts = [p for _, p in V.edge_points()] + [V.INF]
    for a in pts:
        for b in pts:
            assert O.ec_add(a + b) == PY.ec_add(a + b)
        for k in (0, 1, 2, 3, 16, R - 1, R, R + 1, (1 << 256) - 1):
            assert O.ec_mul(a + O.w32(k)) == PY.ec_mul(a + O.w32(k))
        assert V.add(a, a) == V.mul(a, 2) and V.add(a, V.neg(a)) == V.INF and V.mul(a, R - 1) == V.neg(a)


@pytest.mark.parametrize("vm", [0, 1])
def test_point_solved_proofs_equal_synth_solve_c(vm, oracle_backend):
    """with alpha and the IC points as known multiples of G1, C (and A) solved with point arithmetic equal synth.solve_c's scalars"""
    rng = S.SplitMix64(0xED6E3000 + vm)
    coefs = [rng.fr() for _ in range(4)]
    alpha = rng.fr()
    key = V.EdgeKey(vm, S.G1_GEN, coefs, V.mul(S.G1_GEN, alpha), 0xED6E3010 + vm)
    trap = dict(key.trap, alpha=alpha, ic=coefs)
    svk = S.SynthVk(vm, trap, key.alpha, key.beta, key.gamma, key.delta, key.ic)
    for _ in range(3):
        sig = [rng.fr() for _ in range(3)]
        a, b = rng.fr(), rng.fr()
        pr = key.prove(key.vk_x(sig), rng, A=V.mul(S.G1_GEN, a), b=b)
        c = S.solve_c(svk, a, b, svk.x_of(sig))
        assert pr == V.mul(S.G1_GEN, a) + O.g2_mul(S.G2_GEN, b) + V.mul(S.G1_GEN, c)
        assert key.prove(key.vk_x(sig), rng, C=V.mul(S.G1_GEN, c), b=b) == pr                      # A solved for the chosen C
        st = O.groth16_verify_batch(key.ovk(), pr + V.random_a(pr, rng), b"".join(O.w32(v) for v in sig) * 2, 2)
        assert st.tolist() == [0, 4]


def _generic_statuses(keys, recs):
    got = {}
    for ki, key in enumerate(keys):
        rs = [r for r in recs if r.key == ki]
        st = O.groth16_verify_batch(key.ovk(), b"".join(r.proof for r in rs), b"".join(O.w32(v) for r in rs for v in r.signals), len(rs))
        for r, s in zip(rs, st):
            got[id(r)] = int(s)
    return [got[id(r)] for r in recs]


def test_generic_cases_oracle(generic):
    keys, recs, _ = generic
    got = _generic_statuses(keys, recs)
    bad = [(r.case, g, r.expect) for r, g in zip(recs, got) if g != r.expect]
    assert not bad, bad[:10]
    assert sum(r.expect == 0 for r in recs) >= 50


def test_sp1_cases_oracle(sp1):
    keys, recs, _ = sp1
    for route, key in enumerate(keys):
        rs = [r for r in recs if r.route == route]
        st = O.sp1_verify_batch(key.ovk(), S.SP1_SELECTOR, [r.vkey for r in rs], [r.pv for r in rs], [S.SP1_SELECTOR + r.proof for r in rs])
        assert st.tolist() == [r.expect for r in rs], [r.case for r, s in zip(rs, st) if s != r.expect]
        assert all(int.from_bytes(r.vkey, "big") < R for r in rs)


def test_risc0_cases_oracle(risc0):
    for rc in risc0:
        ro = O.Risc0Oracle(rc.key.ovk()); ro.initialize(rc.cr, rc.cid)
        _, ims, jrs, seals, want = zip(*rc.recs)
        assert ro.verify_batch(list(seals), list(ims), list(jrs)).tolist() == list(want), rc.name
        assert [ro.verify_integrity(s, O.claim_digest(a, b)) for s, a, b in zip(seals, ims, jrs)] == list(want), rc.name
    assert len({rc.selector() for rc in risc0}) == len(risc0)                                        # one route each in a router


def test_python_referee_on_a_sample(generic, risc0):
    """the slow, independent Python restatement agrees on a branch case, an edge-point case and a RISC Zero case with their twins"""
    import bn254_py as PY
    keys, recs, _ = generic

    def vkd(k):
        g2 = lambda b: ((int.from_bytes(b[0:32], "big"), int.from_bytes(b[32:64], "big")), (int.from_bytes(b[64:96], "big"), int.from_bytes(b[96:128], "big")))
        return dict(alpha=V.coords(k.alpha), beta=g2(k.beta), gamma=g2(k.gamma), delta=g2(k.delta), ic=[V.coords(p) for p in k.ic])
    words = lambda pr: [int.from_bytes(pr[32 * i:32 * i + 32], "big") for i in range(8)]
    picked = [r for r in recs if r.case.startswith("generic:acc=inf")][:3] + [r for r in recs if r.case.startswith("edge:vk_x=mont(y)=2")][:3]
    assert len(picked) == 6 and picked[0].expect == 0 and picked[3].expect == 0
    for r in picked:
        w = words(r.proof)
        ok = PY.groth16_verify(keys[r.key].vm, vkd(keys[r.key]), w[0:2], [w[2:4], w[4:6]], w[6:8], r.signals)
        assert ok == (r.expect == 0), r.case
    rc = next(c for c in risc0 if c.name == "risc0:mid=inf")
    for name, im, jr, seal, want in rc.recs[:2]:
        st = PY.risc0_verify_status(vkd(rc.key), rc.selector(), rc.cr, rc.cid, seal, im, jr)
        assert st == want, name


def _families(generic, sp1, risc0):
    """entry-point family -> [(case, branch)] of the model's special-branch hits (key sets reuse the generic cases, routes the handles')"""
    fam = {"generic": [], "key set": [], "sp1": [], "risc0 handle": [], "risc0 route": []}
    for name, hits in generic[2].items():
        for *_, b in hits:
            fam["generic"].append((name, b)); fam["key set"].append((name, b))
    for name, hits in sp1[2].items():
        fam["sp1"] += [(name, b) for *_, b in hits]
    for rc in risc0:
        for where, hits in (("per-proof", rc.hits), ("K", rc.k_hits), ("mid", rc.mid_hits)):
            for *_, b in hits:
                fam["risc0 handle"].append((rc.name + ":" + where, b)); fam["risc0 route"].append((rc.name + ":" + where, b))
    return fam


def test_every_family_reaches_every_branch(generic, sp1, risc0):
    fam = _families(generic, sp1, risc0)
    for f, hits in fam.items():
        for b in V.BRANCHES:
            assert any(h == b for _, h in hits), (f, b)
    names = {rc.name: rc for rc in risc0}
    assert names["risc0:K=inf"].K == 0 and names["risc0:mid=inf"].mid == 0
    for rc in risc0:                                                    # every per-proof accumulation under the 32-window tables
        assert all(w < 32 for _, w, _, _ in rc.hits)
    # a cancellation in the middle of the sum followed by a restart, at t >= 1, in each family with signals
    mid_restart = lambda hits: any(b == V.BR_INF and t >= 1 for t, _, _, b in hits)
    assert any(mid_restart(h) for h in generic[2].values()) and any(mid_restart(h) for h in sp1[2].values())
    assert any(mid_restart(rc.hits) for rc in risc0)
