"""Rejected proofs with exactly one cause, each beside an accepting twin that differs from it in that one input (test helpers of
test_single_cause.py and test_gpu_single_cause.py).

Most rejected proofs elsewhere in the suite fail for two reasons at once: a B swapped for a twist point outside G2 still sits next to the A
and C made for the old B, and an SP1 vkey or RISC Zero control id pushed to v + R still comes with a proof made for another statement.  The
status byte then cannot show whether the check under test fired.  Here:

  * B outside G2 with the equation otherwise holding: A is at infinity (the pair (A, B) contributes 1 whatever B is) and C is solved for the
    statement, so the twin with B in G2 is accepted and the subgroup test is the only cause.  RISC Zero keys get both encodings of A at
    infinity, (0, 0) and (0, p) (the negation quirk maps the latter to (0, 0)).  The "deep" variant takes a key with alpha at infinity and
    signals solved so that vk_x is infinity, with C at infinity: every pair is skipped and only R's run through the Miller loop and the
    final comparison decide the status.
  * Inputs at or above the modulus whose reduced value is accepted: an SP1 vkey v + kR beside v, a RISC Zero control id c + kR beside c,
    each proof word w + kp beside w, and the RISC Zero A.y word in the form y_w - kp (mod 2^256) that the negation quirk turns into y + kp.

The B catalogue covers the cofactor group of E'(Fp2): H2 = 2p - r = l1 l2 l3 l4 (four distinct primes), so every twist point is a member plus
a point whose order divides H2.  Points are built by clearing factors of a random twist point Q: [r]Q has order H2, [H2 / l][r]Q order l."""
import oracle_lib as O
import vkx_edges as V
from stylus_zkvm_verifiers_b200 import synth as S

P, R = S.P, S.R
H2 = 2 * P - R                                       # cofactor of G2 in E'(Fp2)
ELL = (10069, 5864401, 1875725156269, H2 // (10069 * 5864401 * 1875725156269))     # its prime factors (the last one has 178 bits)
G1, G2 = S.G1_GEN, S.G2_GEN
INF1, INF2 = bytes(64), bytes(128)
A_INF_R0 = O.w32(0) + O.w32(P)                       # RISC Zero's second encoding of A at infinity: negate_g1 maps (0, p) to (0, 0)
OK, FAIL = S.ST_OK, S.ST_VERIFICATION_FAILED
PV_LEN = 96                                          # every SP1 record's public values (the device forms take one stride)


# ------------------------------------------------------------------ the B catalogue
def g2_neg(q):
    """-Q in wire order (x_im, x_re, y_im, y_re); infinity stays infinity"""
    if q == INF2:
        return q
    return q[:64] + b"".join(O.w32((P - int.from_bytes(q[i:i + 32], "big")) % P) for i in (64, 96))


def g2_mul_all(q, factors):
    for f in factors:
        q = O.g2_mul(q, f)
    return q


class BPoint:
    """a twist point with its name and, where it is known, its exact order as a tuple of prime factors (None: a random twist point, of
    which only [r]B != infinity is claimed)"""

    def __init__(self, name, point, order):
        self.name, self.point, self.order = name, point, order


def outside_catalogue(seed=0x5C0A0001):
    """twist points outside G2: random ones; order l for each of the four cofactor primes; order l_i l_j; order H2; a random member plus
    an order-l point for each l; and negations of some of these"""
    rng = S.SplitMix64(seed)

    def cofactor_point():
        """[r]Q of a random twist point Q, kept when its order is all of H2"""
        while True:
            q = O.g2_mul(S.random_twist_point(rng), R)
            if all(O.g2_mul(q, H2 // l) != INF2 for l in ELL):
                return q
    out = [BPoint("random%d" % j, S.random_twist_point(rng), None) for j in range(3)]
    h = cofactor_point()
    for i, l in enumerate(ELL):
        out.append(BPoint("order=l%d" % (i + 1), O.g2_mul(h, H2 // l), (l,)))
    for i, j in ((0, 1), (1, 2), (0, 3), (2, 3)):
        out.append(BPoint("order=l%d*l%d" % (i + 1, j + 1), O.g2_mul(h, H2 // (ELL[i] * ELL[j])), (ELL[i], ELL[j])))
    out.append(BPoint("order=H2", h, ELL))
    h2 = cofactor_point()
    for i, l in enumerate(ELL):
        out.append(BPoint("G2m+order=l%d" % (i + 1), O.g2_add(O.g2_mul(G2, rng.fr()), O.g2_mul(h2, H2 // l)), (R, l)))
    for b in [out[0], out[3], out[6], out[11], out[-1]]:               # random0, order l1, order l4, order H2, member + order l4
        out.append(BPoint("-" + b.name, g2_neg(b.point), b.order))
    return out


def member_catalogue(seed=0x5C0A0002):
    """(name, point) members of G2 and infinity: the accepting twins' B"""
    rng = S.SplitMix64(seed)
    return [("G2", G2), ("-G2", g2_neg(G2)), ("[2]G2", O.g2_mul(G2, 2)), ("[r-1]G2", O.g2_mul(G2, R - 1)),
            ("[(r+1)/2]G2", O.g2_mul(G2, (R + 1) // 2)), ("member0", O.g2_mul(G2, rng.fr())), ("member1", O.g2_mul(G2, rng.fr())),
            ("inf", INF2)]


# ------------------------------------------------------------------ records and units
class Rec:
    """one record: key / handle / route index, the 256-byte proof (no selector) and the statement (generic signals, SP1 vkey and public
    values, or RISC Zero image id and journal digest); expect is the status the construction gives it"""

    def __init__(self, name, key, proof, expect, signals=None, vkey=None, pv=None, im=None, jr=None):
        self.name, self.key, self.proof, self.expect = name, key, proof, expect
        self.signals, self.vkey, self.pv, self.im, self.jr = signals, vkey, pv, im, jr

    def but(self, name, expect, **kw):
        d = dict(signals=self.signals, vkey=self.vkey, pv=self.pv, im=self.im, jr=self.jr, key=self.key, proof=self.proof)
        d.update(kw)
        return Rec(name, d.pop("key"), d.pop("proof"), expect, **d)


class Unit:
    """a rejected record whose only cause is `cause` ("g2" or "range") and its accepting twin"""

    def __init__(self, cause, case, twin):
        self.cause, self.case, self.twin = cause, case, twin
        assert case.expect == FAIL and twin.expect == OK


def with_b(proof, b):
    return proof[:64] + b + proof[192:]


def with_a(proof, a):
    return a + proof[64:]


def word(proof, i):
    return int.from_bytes(proof[32 * i:32 * i + 32], "big")


def with_word(proof, i, v):
    assert 0 <= v < 1 << 256
    return proof[:32 * i] + O.w32(v) + proof[32 * i + 32:]


def kmax(v, m):
    """the largest k with v + k m < 2^256"""
    return ((1 << 256) - 1 - v) // m


def b_units(out, base, outside, members, tag):
    """one unit per outside point: `base` (an accepted record with A at infinity) with B replaced, beside the same record with a member B"""
    for j, b in enumerate(outside):
        name, m = members[j % len(members)]
        out.append(Unit("g2", base.but("%s|B=%s" % (tag, b.name), FAIL, proof=with_b(base.proof, b.point)),
                        base.but("%s|B=%s" % (tag, name), OK, proof=with_b(base.proof, m))))


def range_units(out, base, vm, tag, words=range(8)):
    """each proof word w of an accepted record as w + kp (k = 1 and the largest k that fits); for RISC Zero also A.y as y_w - kp mod 2^256,
    which the negation quirk turns into y + kp.  The twin is the record itself."""
    for i in words:
        w = word(base.proof, i)
        for k in sorted({1, kmax(w, P)}):
            out.append(Unit("range", base.but("%s|w%d+%dp" % (tag, i, k), FAIL, proof=with_word(base.proof, i, w + k * P)), base))
    if vm == 0:
        y = (P - word(base.proof, 1)) % (1 << 256)                  # the A.y the verifier uses
        for k in sorted({1, kmax(y, P)}):
            out.append(Unit("range", base.but("%s|A.y=y_w-%dp" % (tag, k), FAIL, proof=with_word(base.proof, 1, (P - y - k * P) % (1 << 256))), base))


def solve_last_for_inf(key, signals):
    """signals with the last one replaced so that vk_x = IC0 + sum s_t IC_t is infinity"""
    c = key.coefs
    rest = (c[0] + sum(s * ct for s, ct in zip(signals[:-1], c[1:-1]))) % R
    return list(signals[:-1]) + [(-rest) * pow(c[-1], -1, R) % R]


# ------------------------------------------------------------------ generic family and key sets
def generic_cases(seed=0x5C0A1000):
    """(keys, units, ordinary): EdgeKeys over G1 (0: RISC Zero convention, 5 signals; 1: SP1 convention, 2 signals; 2, 3: the same with
    alpha at infinity, the deep variant) and their units; `ordinary` is the index of the first of two ordinary keys whose units are
    range cases only (for mixing into key sets)"""
    rng = S.SplitMix64(seed)
    outside, members = outside_catalogue(), member_catalogue()
    keys = []
    for vm, nic, alpha in ((0, 6, V.mul(G1, rng.fr())), (1, 3, V.mul(G1, rng.fr())), (0, 6, INF1), (1, 3, INF1),
                           (0, 4, V.mul(G1, rng.fr())), (1, 5, V.mul(G1, rng.fr()))):
        keys.append(V.EdgeKey(vm, G1, [rng.fr() for _ in range(nic)], alpha, seed + len(keys)))
    units = []
    for ki in (0, 1):
        k = keys[ki]
        encs = (("A=(0,0)", INF1), ("A=(0,p)", A_INF_R0)) if k.vm == 0 else (("A=(0,0)", INF1),)
        for aname, a in encs:
            sig = [rng.fr() for _ in range(k.k)]
            pr = with_a(k.prove(k.vk_x(sig), rng, A=INF1), a)
            b_units(units, Rec("", ki, pr, OK, signals=sig), outside, members, "generic%d:%s" % (ki, aname))
        sig = [rng.fr() for _ in range(k.k)]
        range_units(units, Rec("generic%d:range" % ki, ki, k.prove(k.vk_x(sig), rng), OK, signals=sig), k.vm, "generic%d" % ki)
    for ki in (2, 3):                                                  # deep: alpha, vk_x, A and C at infinity
        k = keys[ki]
        sig = solve_last_for_inf(k, [rng.fr() for _ in range(k.k)])
        assert k.vk_x(sig) == INF1
        pr = k.prove(INF1, rng, A=INF1)
        assert pr[:64] == INF1 and pr[192:] == INF1
        encs = (("A=(0,0)", INF1), ("A=(0,p)", A_INF_R0)) if k.vm == 0 else (("A=(0,0)", INF1),)
        for aname, a in encs:
            b_units(units, Rec("", ki, with_a(pr, a), OK, signals=sig), outside, members, "deep%d:%s" % (ki, aname))
    for ki in (4, 5):
        k = keys[ki]
        sig = [rng.fr() for _ in range(k.k)]
        range_units(units, Rec("ordinary%d" % ki, ki, k.prove(k.vk_x(sig), rng), OK, signals=sig), k.vm, "ordinary%d" % ki, words=(0, 5))
    return keys, units, 4


# ------------------------------------------------------------------ SP1
def sp1_cases(seed=0x5C0A2000):
    """(keys, units): route 0 an SP1 key (B catalogue with A at infinity, vkey ranges, proof-word ranges), route 1 the deep variant (alpha
    at infinity, the vkey solved so that vk_x is infinity)"""
    rng = S.SplitMix64(seed)
    outside, members = outside_catalogue(), member_catalogue()
    keys = [V.EdgeKey(1, G1, [rng.fr() for _ in range(3)], V.mul(G1, rng.fr()), seed + 1), V.EdgeKey(1, G1, [rng.fr() for _ in range(3)], INF1, seed + 2)]
    k = keys[0]
    units = []

    def rec(name, vkey, pv, A=None):
        return Rec(name, 0, k.prove(k.vk_x(S.sp1_signals(vkey, pv)), rng, A=A), OK, vkey=vkey, pv=pv)
    b_units(units, rec("", b"\0" + rng.bytes(31), rng.bytes(PV_LEN), A=INF1), outside, members, "sp1:A=(0,0)")
    v = rng.fr() >> 3                                                  # v + 5R < 2^256
    base = rec("sp1:vkey=v", O.w32(v), rng.bytes(PV_LEN))
    for kk in range(1, 6):
        assert v + kk * R < 1 << 256
        units.append(Unit("range", base.but("sp1:vkey=v+%dR" % kk, FAIL, vkey=O.w32(v + kk * R)), base))
    zero = rec("sp1:vkey=0", O.w32(0), rng.bytes(PV_LEN))
    units.append(Unit("range", zero.but("sp1:vkey=R", FAIL, vkey=O.w32(R)), zero))
    top = rec("sp1:vkey=R-1", O.w32(R - 1), rng.bytes(PV_LEN))
    units.append(Unit("range", top.but("sp1:vkey=2R-1", FAIL, vkey=O.w32(2 * R - 1)), top))
    range_units(units, rec("sp1:range", b"\0" + rng.bytes(31), rng.bytes(PV_LEN)), 1, "sp1")
    d = keys[1]
    pv = rng.bytes(PV_LEN)
    s1 = S.sp1_signals(bytes(32), pv)[1]
    vkey = O.w32((-(d.coefs[0] + s1 * d.coefs[2])) * pow(d.coefs[1], -1, R) % R)
    assert d.vk_x(S.sp1_signals(vkey, pv)) == INF1
    pr = d.prove(INF1, rng, A=INF1)
    b_units(units, Rec("", 1, pr, OK, vkey=vkey, pv=pv), outside, members, "sp1deep:A=(0,0)")
    return keys, units


# ------------------------------------------------------------------ RISC Zero handles and routes
class Handle:
    """one initialised RISC Zero verifier: key, control root, control id (32 bytes)"""

    def __init__(self, name, key, cr, cid):
        self.name, self.key, self.cr, self.cid = name, key, cr, cid

    def oracle(self):
        ro = O.Risc0Oracle(self.key.ovk())
        ro.initialize(self.cr, self.cid)
        return ro

    def selector(self):
        return self.oracle().selector()

    def prove(self, im, jr, rng, A=None):
        """a 256-byte proof of the claim (im, jr) under this handle's control root and control id"""
        sig = S.risc0_signals(self.cr, self.cid, S.risc0_claim_digest(im, jr, V.SYS0))
        return self.key.prove(self.key.vk_x(sig), rng, A=A)


def risc0_cases(seed=0x5C0A3000):
    """(handles, units).  Handle 0: a key with control id c (B catalogue with both encodings of A at infinity, proof-word ranges);
    handles 1..5: the same key and control root with control id c + kR; handle 6: control id R - 1, handle 7: 2R - 1; handle 8: the deep
    variant (alpha at infinity, the control id solved so that vk_x is infinity for one claim).  The control-id units pair a record of
    handle c + kR (or 2R - 1) with the same proof under handle c (R - 1): in a router they are two routes."""
    rng = S.SplitMix64(seed)
    outside, members = outside_catalogue(), member_catalogue()
    key = V.EdgeKey(0, G1, [rng.fr() for _ in range(6)], V.mul(G1, rng.fr()), seed + 1)
    cr = rng.bytes(32)
    c = rng.fr() >> 3
    hs = [Handle("risc0:cid=c", key, cr, O.w32(c))]
    hs += [Handle("risc0:cid=c+%dR" % k, key, cr, O.w32(c + k * R)) for k in range(1, 6)]
    hs += [Handle("risc0:cid=R-1", key, cr, O.w32(R - 1)), Handle("risc0:cid=2R-1", key, cr, O.w32(2 * R - 1))]
    units = []
    h0 = hs[0]
    for aname, a in (("A=(0,0)", INF1), ("A=(0,p)", A_INF_R0)):
        im, jr = rng.bytes(32), rng.bytes(32)
        pr = with_a(h0.prove(im, jr, rng, A=INF1), a)
        b_units(units, Rec("", 0, pr, OK, im=im, jr=jr), outside, members, "risc0:" + aname)
    im, jr = rng.bytes(32), rng.bytes(32)
    range_units(units, Rec("risc0:range", 0, h0.prove(im, jr, rng), OK, im=im, jr=jr), 0, "risc0")
    for hi, twin_hi in [(k, 0) for k in range(1, 6)] + [(7, 6)]:
        for j in range(2):
            im, jr = rng.bytes(32), rng.bytes(32)
            t = Rec("%s#%d" % (hs[twin_hi].name, j), twin_hi, hs[twin_hi].prove(im, jr, rng), OK, im=im, jr=jr)
            units.append(Unit("range", t.but("%s#%d" % (hs[hi].name, j), FAIL, key=hi), t))
    dkey = V.EdgeKey(0, G1, [rng.fr() for _ in range(6)], INF1, seed + 2)
    dcr, im, jr = rng.bytes(32), rng.bytes(32), rng.bytes(32)
    sig = solve_last_for_inf(dkey, S.risc0_signals(dcr, bytes(32), S.risc0_claim_digest(im, jr, V.SYS0)))
    hs.append(Handle("risc0deep", dkey, dcr, O.w32(sig[-1])))
    assert dkey.vk_x(sig) == INF1
    pr = dkey.prove(INF1, rng, A=INF1)
    for aname, a in (("A=(0,0)", INF1), ("A=(0,p)", A_INF_R0)):
        b_units(units, Rec("", len(hs) - 1, with_a(pr, a), OK, im=im, jr=jr), outside, members, "risc0deep:" + aname)
    return hs, units


# ------------------------------------------------------------------ placement in a batch
def anchors(n, chunk=None):
    """lanes where a case goes with its twin beside it: 0, 31, 32, 127, 128, the last record, and (chunk given) every chunk edge and the
    record before it"""
    a = {0, 31, 32, 127, 128, n - 1}
    if chunk:
        for e in range(chunk, n, chunk):
            a |= {e - 1, e}
    return sorted(x for x in a if 0 <= x < n)


def layout(units, n, lanes):
    """n records: at each lane of `lanes` a case with its twin in a neighbouring record that is not such a lane where there is one (lanes
    are taken from the last down, so when three lanes are consecutive, as 127, 128, 129 at n = 130, the middle one holds the last lane's
    twin); the other records alternate case, twin, case, ... through the units in order"""
    recs, lset, u = [None] * n, set(lanes), 0
    for a in sorted(lanes, reverse=True):
        if recs[a] is not None:
            continue
        free = [t for t in (a + 1, a - 1) if 0 <= t < n and recs[t] is None]
        t = ([t for t in free if t not in lset] or free)[0]
        recs[a], recs[t] = units[u % len(units)].case, units[u % len(units)].twin
        u += 1
    k = 0
    for i in range(n):
        if recs[i] is None:
            unit = units[(k // 2) % len(units)]
            recs[i] = unit.twin if k % 2 else unit.case
            k += 1
    return recs


def records(units):
    return [r for u in units for r in (u.case, u.twin)]
