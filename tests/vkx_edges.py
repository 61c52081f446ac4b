"""Accepting Groth16 proofs built around chosen G1 points (test helpers of test_vkx_edges.py and test_gpu_vkx_edges.py).

synth.make_proofs draws A, C and vk_x as multiples of G1 with random discrete logs, so two kinds of input never reach the verification
kernels inside a proof that should be accepted:

  * the special branches of the vk_x accumulation (vkx_one in csrc/kernels.cuh adds the 4-bit window entries d 16^w IC_t to a Jacobian
    accumulator with g1_add_affine, which restarts from the entry when the accumulator is at infinity, doubles when it equals the entry and
    gives infinity when it equals minus the entry);
  * G1 points whose coordinates sit at the edges of the field arithmetic (x = p - 1, small x, Montgomery residues 2, p - 1, p - 2).

Here a key's G2 points have known scalars beta, gamma, delta, while its G1 points (alpha, IC_t) are arbitrary points; every IC_t is a known
multiple of one base point P (an edge point, whose discrete log nobody knows), so the vk_x accumulation can be modelled exactly over the
multipliers mod r.  The missing proof element is solved with point arithmetic on the CPU oracle (ecAdd / ecMul):

    RISC Zero (vm 0, the verifier negates A):        -b A + beta alpha + gamma X + delta C = 0
    SP1 (vm 1, the stored beta, gamma, delta are the negated ones):  b A + beta alpha + gamma X + delta C = 0

with X = vk_x and B = b G2.  Every accepting proof has twins that must be rejected: one signal + 1 (or one journal / public-value bit
flipped) and a random A."""
import oracle_lib as O
from stylus_zkvm_verifiers_b200 import synth as S

P, R = S.P, S.R
G1, G2 = S.G1_GEN, S.G2_GEN
INF = bytes(64)
MONT_INV = pow(1 << 256, -1, P)                  # 2^-256 mod p: x MONT_INV has Montgomery residue x
BR_INF, BR_DBL, BR_NEG = "acc=inf", "acc=entry", "acc=-entry"
BRANCHES = (BR_INF, BR_DBL, BR_NEG)
SYS0 = bytes.fromhex("a3acc27117418996340b84e5a90f3ef4c49d22c79e44aad822ec9c313e1eb8e2")   # risc0 SystemState zero digest


# ------------------------------------------------------------------ points as 64-byte EVM words
def pt(x, y):
    return O.w32(x) + O.w32(y)


def coords(p):
    return int.from_bytes(p[:32], "big"), int.from_bytes(p[32:64], "big")


def neg(p):
    x, y = coords(p)
    return INF if p == INF else pt(x, (P - y) % P)


def add(*ps):
    acc = INF
    for p in ps:
        acc = O.ec_add(acc + p)
    return acc


def mul(p, k):
    return O.ec_mul(p + O.w32(k % R))


def on_curve(p):
    x, y = coords(p)
    return x < P and y < P and (y * y - x ** 3 - 3) % P == 0


def sqrt_p(a):
    """square root mod p (p = 3 mod 4: one power), None for a non-residue"""
    y = pow(a % P, (P + 1) // 4, P)
    return y if y * y % P == a % P else None


def point_at_x(x):
    y = sqrt_p(x ** 3 + 3)
    return None if y is None else pt(x, min(y, P - y))


def mont(v):
    return v * (1 << 256) % P


def _cube_root(a):
    """a cube root of a mod p, or None (Adleman-Manders-Miller for p - 1 = 3^s t)"""
    a %= P
    if a == 0:
        return 0
    if pow(a, (P - 1) // 3, P) != 1:
        return None
    s, t = 0, P - 1
    while t % 3 == 0:
        s += 1; t //= 3
    z = 2
    while pow(z, (P - 1) // 3, P) == 1:                 # a cubic non-residue
        z += 1
    r0 = pow(a, pow(3, -1, t), P)                       # r0^3 = a times an element of the 3^s-torsion
    c = pow(z, t, P)                                    # generator of the 3^s-torsion (s = 2 for this p): try its powers
    for j in range(3 ** s):
        r = r0 * pow(c, j, P) % P
        if pow(r, 3, P) == a:
            return r
    return None


def edge_points():
    """[(name, point)]: about 20 G1 points at the edges of the field arithmetic, each followed by its negation ('-name')"""
    out = []

    def put(name, p):
        assert p is not None and on_curve(p), name
        out.append((name, p))
        out.append(("-" + name, neg(p)))
    put("x=p-1", point_at_x(P - 1))                     # y = +-sqrt(2)
    put("G1", G1)                                       # x = 1, the smallest x on the curve
    for x in (2, 3, 5):
        put("x=%d" % x, point_at_x(x))
    for m, name in ((2, "2"), (4, "4"), (P - 1, "p-1"), (P - 2, "p-2")):
        put("mont(x)=" + name, point_at_x(m * MONT_INV % P))
    y = 2 * MONT_INV % P
    put("mont(y)=2", pt(_cube_root(y * y - 3), y))      # its negation has mont(y) = p - 2
    return out


# ------------------------------------------------------------------ the vk_x accumulation of vkx_one, over multipliers mod r
def vkx_model(base, coefs, scalars, nwin):
    """vkx_one (csrc/kernels.cuh) over discrete logs to a common point: the accumulator starts at `base` (0 = infinity), then for
    t = 0, 1, .., for w = 0 .. nwin - 1 with digit d = (scalars[t] >> 4 w) & 15 != 0 the entry d 16^w coefs[t] is added (an entry at
    infinity, coefs[t] = 0, is skipped as the kernel skips zeroed table entries).  Returns (final accumulator, [(t, w, d, branch)]) with
    branch the special case of g1_add_affine the addition takes: BR_INF (accumulator at infinity), BR_DBL (accumulator = entry) or BR_NEG
    (accumulator = -entry)."""
    acc, hits = base % R, []
    for t, (c, s) in enumerate(zip(coefs, scalars)):
        if c % R == 0:
            continue
        for w in range(nwin):
            d = (s >> (4 * w)) & 15
            if not d:
                continue
            e = d * pow(16, w, R) * c % R
            if acc == 0:
                hits.append((t, w, d, BR_INF)); acc = e
            elif acc == e:
                hits.append((t, w, d, BR_DBL)); acc = 2 * e % R
            elif acc == (R - e) % R:
                hits.append((t, w, d, BR_NEG)); acc = 0
            else:
                acc = (acc + e) % R
    return acc, hits


def acc_before(base, coefs, scalars, t, w):
    """the accumulator (mod r) just before the addition of window w of scalars[t]"""
    return (base + sum(scalars[u] * coefs[u] for u in range(t)) + (scalars[t] % (16 ** w)) * coefs[t]) % R


def target_acc(branch, e):
    return {BR_INF: 0, BR_DBL: e % R, BR_NEG: (-e) % R}[branch]


def entry(coefs, scalars, t, w):
    d = (scalars[t] >> (4 * w)) & 15
    assert d, "window %d of scalar %d is zero" % (w, t)
    return d * pow(16, w, R) * coefs[t] % R


def nonzero_window(s, at_least, nwin=64):
    """the first window >= at_least of s with a nonzero digit (the last nonzero one below it if there is none)"""
    for w in list(range(at_least, nwin)) + list(range(at_least - 1, -1, -1)):
        if (s >> (4 * w)) & 15:
            return w
    raise ValueError("zero scalar")


def top_window(s):
    return max(w for w in range(64) if (s >> (4 * w)) & 15)


# ------------------------------------------------------------------ keys with arbitrary G1 points and proofs solved around them
class EdgeKey:
    """A key whose IC_t = coefs[t] * base (coefs[t] = 0: IC_t at infinity) and whose alpha is any point; beta, gamma, delta are known
    multiples of G2 (for vm 1 they play the role of the stored, negated constants)."""

    def __init__(self, vm, base, coefs, alpha, seed):
        rng = S.SplitMix64(seed)
        self.vm, self.base, self.coefs, self.alpha = vm, base, [c % R for c in coefs], alpha
        self.trap = {"beta": rng.fr(), "gamma": rng.fr(), "delta": rng.fr()}
        self.beta, self.gamma, self.delta = (O.g2_mul(G2, self.trap[k]) for k in ("beta", "gamma", "delta"))
        self.ic = [mul(base, c) for c in self.coefs]

    @property
    def k(self):
        return len(self.ic) - 1

    def ovk(self):
        return O.Vk(self.vm, self.alpha, self.beta, self.gamma, self.delta, self.ic)

    def load(self, Z):
        return Z.VerificationKey(self.vm, self.alpha, self.beta, self.gamma, self.delta, self.ic)

    def vk_x(self, signals):
        """compute_vk_x as the reference does it: k ecMul + k ecAdd precompile calls"""
        acc = self.ic[0]
        for s, ic in zip(signals, self.ic[1:]):
            acc = O.ec_add(acc + O.ec_mul(ic + O.w32(s)))
        return acc

    def model(self, signals):
        return vkx_model(self.coefs[0], self.coefs[1:], signals, 64)

    def prove(self, X, rng, A=None, C=None, b=None):
        """a 256-byte proof (A, B, C) for vk_x = X and B = b G2 (b random by default): C solved for a chosen (or random) A, or A solved for
        a chosen C"""
        t = self.trap
        b = b if b is not None else rng.fr()
        B = O.g2_mul(G2, b)
        if C is None:
            A = A if A is not None else mul(G1, rng.fr())
            if self.vm == 0:
                C = mul(add(mul(A, b), neg(mul(self.alpha, t["beta"])), neg(mul(X, t["gamma"]))), pow(t["delta"], -1, R))
            else:
                C = mul(add(mul(A, b), mul(self.alpha, t["beta"]), mul(X, t["gamma"])), -pow(t["delta"], -1, R))
        else:
            s = add(mul(self.alpha, t["beta"]), mul(X, t["gamma"]), mul(C, t["delta"]))
            A = mul(s, pow(b, -1, R) if self.vm == 0 else -pow(b, -1, R))
        return A + B + C


def random_a(proof, rng):
    return mul(G1, rng.fr()) + proof[64:]


def bump(signals, keycoefs):
    """the twin's signals: the first signal whose IC point is not at infinity, + 1 (- 1 at r - 1)"""
    s = list(signals)
    j = next(i for i in range(len(s)) if keycoefs[i + 1])
    s[j] = s[j] + 1 if s[j] + 1 < R else s[j] - 1
    return s


# ------------------------------------------------------------------ generic / key-set cases
class Rec:
    """one record of a generic or key-set batch: key index, proof, signals, the status the construction gives it"""

    def __init__(self, case, key, proof, signals, expect):
        self.case, self.key, self.proof, self.signals, self.expect = case, key, proof, list(signals), expect


def generic_records(out, name, ki, key, signals, rng, A=None, C=None):
    """the accepting proof, its twin (one signal + 1) and the same proof with a random A"""
    pr = key.prove(key.vk_x(signals), rng, A=A, C=C)
    out.append(Rec(name, ki, pr, signals, 0))
    out.append(Rec(name + "|twin", ki, pr, bump(signals, key.coefs), 4))
    out.append(Rec(name + "|random_a", ki, random_a(pr, rng), signals, 4))


def generic_cases(seed=0xED6E0000):
    """(keys, records, hits): keys of the generic family (5 signals unless stated) and records that reach every special branch of vk_x,
    plus one small key per edge point with vk_x, A, C and alpha at edge points.  hits[name] = the model's branch hits of that case."""
    rng = S.SplitMix64(seed)
    edges = edge_points()
    ep = [p for _, p in edges]
    keys, recs, hits = [], [], {}

    def key(vm, base, coefs, alpha):
        keys.append(EdgeKey(vm, base, coefs, alpha, seed + len(keys)))
        return len(keys) - 1

    def case(name, ki, signals, branch=None, where=None, A=None, C=None):
        k = keys[ki]
        acc, h = k.model(signals)
        assert mul(k.base, acc) == k.vk_x(signals), name                     # the model's vk_x is the precompile chain's
        if branch is not None:
            assert any(b == branch and (where is None or (t, w) == where) for t, w, _, b in h), (name, h)
        hits[name] = h
        generic_records(recs, name, ki, k, signals, rng, A=A, C=C)

    # one ordinary-looking key over an edge base point: branches at t >= 1 by solving an earlier signal mod r
    main = key(0, ep[0], [rng.fr() for _ in range(6)], ep[3])
    c = keys[main].coefs
    for branch, t, w0, free in ((BR_DBL, 3, 7, 1), (BR_NEG, 2, 11, 0), (BR_INF, 4, 21, 2), (BR_DBL, 1, 0, 0), (BR_NEG, 4, None, 3),
                                (BR_INF, 2, 0, 1)):
        s = [rng.fr() for _ in range(5)]
        if w0 is None:                                                     # the top window of a signal close to r
            s[t] = R - 1 - rng.below(1 << 200)
        w = nonzero_window(s[t], w0) if w0 is not None else top_window(s[t])
        e = entry(c[1:], s, t, w)
        s[free] = 0
        rest = acc_before(c[0], c[1:], s, t, w)
        s[free] = (target_acc(branch, e) - rest) * pow(c[1 + free], -1, R) % R
        case("generic:%s@t%dw%d" % (branch, t, w), main, s, branch, (t, w))
    s = [rng.fr() for _ in range(5)]                                        # vk_x = infinity after the last window
    s[0] = (-(c[0] + sum(a * b for a, b in zip(s[1:], c[2:])))) * pow(c[1], -1, R) % R
    case("generic:vk_x=inf", main, s, BR_NEG)
    case("generic:zero_signals", main, [0] * 5)                             # vk_x = IC0 = the edge base point
    # t = 0: crafted keys
    d = 9
    s = [d + 16 * rng.below(1 << 60)] + [rng.fr() for _ in range(4)]
    k1 = rng.fr()
    case("generic:ic0=-d.ic1", key(0, ep[4], [-d * k1, k1] + [rng.fr() for _ in range(4)], ep[5]), s, BR_NEG, (0, 0))
    case("generic:ic0=+d.ic1", key(0, ep[6], [d * k1, k1] + [rng.fr() for _ in range(4)], ep[7]), s, BR_DBL, (0, 0))
    case("generic:ic0=inf", key(0, ep[8], [0] + [rng.fr() for _ in range(5)], ep[9]), [rng.fr() for _ in range(5)], BR_INF, (0, 0))
    ki = key(0, ep[10], [rng.fr(), rng.fr(), 0, rng.fr(), 0, rng.fr()], ep[11])          # IC2 and IC4 at infinity
    case("generic:ic2,ic4=inf", ki, [rng.fr() for _ in range(5)])
    case("generic:ic2,ic4=inf,zero_others", ki, [0, rng.fr(), 0, rng.fr(), 0])          # vk_x = IC0 with entries of IC2 / IC4 only
    k1 = rng.fr()
    case("generic:ic2=ic1", key(0, ep[12], [0, k1, k1, rng.fr(), rng.fr(), rng.fr()], ep[13]), [5, 5, 0, 0, 0], BR_DBL, (1, 0))
    case("generic:ic2=16.ic1", key(0, ep[14], [0, k1, 16 * k1, rng.fr(), rng.fr(), rng.fr()], ep[15]), [7 * 16, 7, 1, 2, 3], BR_DBL, (1, 0))
    # SP1-convention key of the same family, with branch targets
    sk = key(1, ep[16], [rng.fr() for _ in range(6)], ep[17])
    c = keys[sk].coefs
    for branch in BRANCHES:
        s = [rng.fr() for _ in range(5)]
        w = nonzero_window(s[2], 30)
        e = entry(c[1:], s, 2, w)
        s[1] = 0
        s[1] = (target_acc(branch, e) - acc_before(c[0], c[1:], s, 2, w)) * pow(c[2], -1, R) % R
        case("generic_vm1:%s@t2w%d" % (branch, w), sk, s, branch, (2, w))
    # one small key per edge point: vk_x = the point (zero signals), A and C at other edge points, alpha at an edge point
    n = len(ep)
    for i, (name, q) in enumerate(edges):
        ki = key(i % 2, q, [1, rng.fr(), rng.fr()], ep[(i + 1) % n])
        case("edge:vk_x=%s,A=%s" % (name, edges[(i + 2) % n][0]), ki, [0, 0], A=ep[(i + 2) % n])
        case("edge:C=%s" % edges[(i + 3) % n][0], ki, [rng.fr(), rng.fr()], C=ep[(i + 3) % n])
    return keys, recs, hits


# ------------------------------------------------------------------ SP1 cases
def sp1_signals(vkey, pv):
    return S.sp1_signals(vkey, pv)


class Sp1Rec:
    def __init__(self, case, route, vkey, pv, proof, expect):
        self.case, self.route, self.vkey, self.pv, self.proof, self.expect = case, route, vkey, pv, proof, expect


def sp1_cases(seed=0xED6E1000):
    """(keys, records, hits): SP1 keys (route 0 is the main key; routes 1, 2 are crafted for t = 0) and records whose vkey is solved mod r
    so that an addition of the public-value hash's windows takes each special branch; edge points as A and C."""
    rng = S.SplitMix64(seed)
    edges = edge_points()
    ep = [p for _, p in edges]
    keys, recs, hits = [], [], {}
    c = [rng.fr() for _ in range(3)]
    keys.append(EdgeKey(1, ep[2], c, ep[6], seed))

    def case(name, route, vkey, pv, branch=None, where=None, A=None, C=None):
        k = keys[route]
        sig = sp1_signals(vkey, pv)
        acc, h = k.model(sig)
        assert mul(k.base, acc) == k.vk_x(sig), name
        if branch is not None:
            assert any(b == branch and (where is None or (t, w) == where) for t, w, _, b in h), (name, h)
        hits[name] = h
        pr = k.prove(k.vk_x(sig), rng, A=A, C=C)
        recs.append(Sp1Rec(name, route, vkey, pv, pr, 0))
        flip = bytearray(pv); flip[rng.below(len(pv))] ^= 1 << rng.below(8)
        recs.append(Sp1Rec(name + "|twin", route, vkey, bytes(flip), pr, 4))
        recs.append(Sp1Rec(name + "|random_a", route, vkey, pv, random_a(pr, rng), 4))

    for j, branch in enumerate(BRANCHES * 2):
        pv = rng.bytes(33 if j == 1 else 96)
        s1 = sp1_signals(bytes(32), pv)[1]
        w = nonzero_window(s1, (0, 17, 40, 1, 25, 60)[j])
        e = entry(c[1:], [0, s1], 1, w)
        s0 = (target_acc(branch, e) - acc_before(c[0], c[1:], [0, s1], 1, w)) * pow(c[1], -1, R) % R
        case("sp1:%s@t1w%d" % (branch, w), 0, O.w32(s0), pv, branch, (1, w))
    pv = rng.bytes(64)
    s1 = sp1_signals(bytes(32), pv)[1]
    case("sp1:vk_x=inf", 0, O.w32((-(c[0] + s1 * c[2])) * pow(c[1], -1, R) % R), pv, BR_NEG)
    for i, (name, q) in enumerate(edges):
        vkey = bytes([0]) + rng.bytes(31)
        case("sp1:A=%s" % name if i % 2 == 0 else "sp1:C=%s" % name, 0, vkey, rng.bytes(96), A=q if i % 2 == 0 else None, C=q if i % 2 else None)
    # t = 0 on crafted keys: IC0 = -+d IC1 with d the vkey's lowest digit
    for route, (sign, branch) in enumerate(((-1, BR_NEG), (1, BR_DBL)), start=1):
        vkey = bytes([0]) + rng.bytes(31)
        d = vkey[31] & 15 or 1
        vkey = vkey[:31] + bytes([(vkey[31] & 0xF0) | d])
        k1 = rng.fr()
        keys.append(EdgeKey(1, ep[7 + route], [sign * d * k1, k1, rng.fr()], ep[11 + route], seed + route))
        case("sp1:ic0=%sd.ic1" % ("-" if sign < 0 else "+"), route, vkey, rng.bytes(96), branch, (0, 0))
    return keys, recs, hits


# ------------------------------------------------------------------ RISC Zero cases: one handle (key, control root, control id) each
class R0Case:
    """One initialised RISC Zero verifier: key, control root and bn254_control_id, chosen so that K (the folded base IC0 + c0 IC1 + c1 IC2
    + id IC5), the intermediate mid = IC0 + c0 IC1 + c1 IC2, or an addition against the claim halves of (image_id, journal) takes a
    special branch.  recs: (case, image_id, journal, seal, expect)."""

    def __init__(self, name, key, control_root, control_id, image_id, journal):
        self.name, self.key, self.cr, self.cid, self.image_id, self.journal = name, key, control_root, control_id, image_id, journal
        c = key.coefs
        c0, c1 = S.split_digest(control_root)
        idv = int.from_bytes(control_id, "big")
        self.mid, self.mid_hits = vkx_model(c[0], c[1:3], [c0, c1], 64)
        self.K, self.k_hits = vkx_model(self.mid, [c[5]], [idv], 64)
        lo, hi = S.split_digest(S.risc0_claim_digest(image_id, journal, SYS0))
        self.acc, self.hits = vkx_model(self.K, c[3:5], [lo, hi], 32)
        sig = S.risc0_signals(control_root, control_id, S.risc0_claim_digest(image_id, journal, SYS0))
        assert mul(key.base, self.acc) == key.vk_x(sig), name
        self.recs = []

    def selector(self):
        ro = O.Risc0Oracle(self.key.ovk()); ro.initialize(self.cr, self.cid)
        return ro.selector()

    def add_records(self, rng, extra):
        """the targeted proof, its twin (one journal bit flipped) and a random A; then `extra` proofs of other claims with A or C at edge points"""
        sel = self.selector()
        k = self.key

        def seal_for(im, jr, A=None, C=None):
            sig = S.risc0_signals(self.cr, self.cid, S.risc0_claim_digest(im, jr, SYS0))
            return sel + k.prove(k.vk_x(sig), rng, A=A, C=C)
        s = seal_for(self.image_id, self.journal)
        flip = bytearray(self.journal); flip[rng.below(32)] ^= 1 << rng.below(8)
        self.recs += [(self.name, self.image_id, self.journal, s, 0), (self.name + "|twin", self.image_id, bytes(flip), s, 4),
                      (self.name + "|random_a", self.image_id, self.journal, s[:4] + random_a(s[4:], rng), 4)]
        for name, q in extra:
            im, jr = rng.bytes(32), rng.bytes(32)
            use_a = rng.below(2) == 0
            self.recs.append((self.name + (":A=" if use_a else ":C=") + name, im, jr, seal_for(im, jr, A=q if use_a else None, C=None if use_a else q), 0))


def risc0_cases(seed=0xED6E2000):
    """RISC Zero handles whose K, mid or per-proof accumulation takes each special branch under the 32-window claim tables, plus one whose
    vk_x is the edge base point itself; every case gets a few proofs with A or C at edge points."""
    rng = S.SplitMix64(seed)
    edges = edge_points()
    ep = [p for _, p in edges]
    cases = []

    def claim_halves(im, jr):
        return S.split_digest(S.risc0_claim_digest(im, jr, SYS0))

    def id_for_K(c, cr, K):
        c0, c1 = S.split_digest(cr)
        mid = (c[0] + c0 * c[1] + c1 * c[2]) % R
        return O.w32((K - mid) * pow(c[5], -1, R) % R)

    for j, (branch, t, w0) in enumerate(((BR_DBL, 0, 5), (BR_NEG, 0, 20), (BR_INF, 0, 9), (BR_DBL, 1, 0), (BR_NEG, 1, 31), (BR_INF, 1, 14))):
        base = ep[(3 * j) % len(ep)]
        key = EdgeKey(0, base, [rng.fr() for _ in range(6)], ep[(3 * j + 1) % len(ep)], seed + j)
        c = key.coefs
        cr, im, jr = rng.bytes(32), rng.bytes(32), rng.bytes(32)
        lo, hi = claim_halves(im, jr)
        s = [lo, hi]
        w = nonzero_window(s[t], w0, 32) if w0 < 31 else top_window(s[t])
        if branch == BR_INF and t == 0 and w == nonzero_window(lo, 0):
            w = nonzero_window(lo, w + 1, 32)                                  # not the first addition: that is the K = infinity case
        e = entry(c[3:5], s, t, w)
        K = (target_acc(branch, e) - acc_before(0, c[3:5], s, t, w)) % R
        rc = R0Case("risc0:%s@%s,w%d" % (branch, ("lo", "hi")[t], w), key, cr, id_for_K(c, cr, K), im, jr)
        assert any(b == branch and (tt, ww) == (t, w) for tt, ww, _, b in rc.hits), (rc.name, rc.hits)
        cases.append(rc)
    # K = infinity: the per-proof accumulation starts from infinity (the folding's last addition cancels)
    key = EdgeKey(0, ep[1], [rng.fr() for _ in range(6)], ep[2], seed + 10)
    cr = rng.bytes(32)
    rc = R0Case("risc0:K=inf", key, cr, id_for_K(key.coefs, cr, 0), rng.bytes(32), rng.bytes(32))
    assert rc.K == 0 and rc.hits[0][3] == BR_INF and any(b == BR_NEG for *_, b in rc.k_hits), rc.name
    cases.append(rc)
    # mid = infinity: IC0 = -(c0 IC1 + c1 IC2) for the chosen control root; the second folding call starts from a base at infinity
    cr = rng.bytes(32)
    c0, c1 = S.split_digest(cr)
    c = [rng.fr() for _ in range(6)]
    c[0] = (-(c0 * c[1] + c1 * c[2])) % R
    key = EdgeKey(0, ep[5], c, ep[9], seed + 11)
    rc = R0Case("risc0:mid=inf", key, cr, O.w32(rng.fr()), rng.bytes(32), rng.bytes(32))
    assert rc.mid == 0 and rc.k_hits[0][3] == BR_INF and any(b == BR_NEG for *_, b in rc.mid_hits), rc.name
    cases.append(rc)
    # K and mid both at infinity on the same key as above, another control id
    rc = R0Case("risc0:mid=inf,K=inf", key, cr, O.w32(0), rng.bytes(32), rng.bytes(32))
    assert rc.mid == 0 and rc.K == 0 and rc.hits[0][3] == BR_INF, rc.name
    cases.append(rc)
    # vk_x = the edge base point itself (K solved for a per-proof total of 1)
    key = EdgeKey(0, ep[15], [rng.fr() for _ in range(6)], ep[16], seed + 12)
    cr, im, jr = rng.bytes(32), rng.bytes(32), rng.bytes(32)
    lo, hi = claim_halves(im, jr)
    rc = R0Case("risc0:vk_x=base", key, cr, id_for_K(key.coefs, cr, 1 - lo * key.coefs[3] - hi * key.coefs[4]), im, jr)
    assert rc.acc == 1, rc.name
    cases.append(rc)
    for j, rc in enumerate(cases):
        rc.add_records(rng, [edges[(2 * j + i) % len(edges)] for i in range(3)])
    return cases
