"""ctypes binding of the CPU oracle (oracle/libzkv_oracle.so).  TEST INFRASTRUCTURE ONLY:
imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs."""
import ctypes as C
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
SO = os.path.join(ORACLE_DIR, "libzkv_oracle.so")

ST_OK, ST_INVALID_INITIALIZATION, ST_INVALID_PROOF_DATA, ST_SELECTOR_MISMATCH, ST_VERIFICATION_FAILED = range(5)


def build(force=False):
    src = [os.path.join(ORACLE_DIR, f) for f in ("zkv_oracle.c", "bn254.h")]
    if force or not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(SO)
        _lib.zkvo_vk_sizeof.restype = C.c_size_t
        _lib.zkvo_risc0_sizeof.restype = C.c_size_t
        for name in ("zkvo_ec_add", "zkvo_ec_mul", "zkvo_ec_pairing"):
            getattr(_lib, name).argtypes = [C.c_char_p, C.c_size_t, C.c_char_p]
        _lib.zkvo_ec_pairing_debug.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_char_p]
        _lib.zkvo_sha256.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p]
        _lib.zkvo_risc0_verify.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p]
        _lib.zkvo_risc0_verify_integrity.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.c_char_p]
        _lib.zkvo_sp1_verify.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]
        _lib.zkvo_sp1_hash_public_values.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p]
        _lib.zkvo_groth16_verify_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_long, C.c_void_p]
        _lib.zkvo_risc0_verify_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        _lib.zkvo_risc0_verify_integrity_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        _lib.zkvo_sp1_verify_batch.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        _lib.zkvo_pairing4_batch.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p]
    return _lib


def w32(v):
    return int(v).to_bytes(32, "big")


class Vk:
    """Packed verification key (common/types.rs:17-23). Points in wire order: G2 = (x[0],x[1],y[0],y[1])."""

    def __init__(self, vm, alpha, beta, gamma, delta, ic):
        self.vm, self.alpha, self.beta, self.gamma, self.delta, self.ic = vm, alpha, beta, gamma, delta, list(ic)
        L = lib()
        self.buf = C.create_string_buffer(L.zkvo_vk_sizeof())
        L.zkvo_vk_pack(self.buf, vm, alpha, beta, gamma, delta, b"".join(self.ic), len(self.ic))

    @property
    def k(self):
        return len(self.ic) - 1


def vk_from_json(d, vm):
    g1 = lambda p: bytes.fromhex(p[0]) + bytes.fromhex(p[1])
    g2 = lambda q: b"".join(bytes.fromhex(q[i][j]) for i in range(2) for j in range(2))
    return Vk(vm, g1(d["alpha"]), g2(d["beta"]), g2(d["gamma"]), g2(d["delta"]), [g1(p) for p in d["ic"]])


_consts = None


def constants():
    global _consts
    if _consts is None:
        _consts = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_constants.json")))
    return _consts


def risc0_vk():
    return vk_from_json(constants()["risc0_vk"], 0)


def sp1_vk():
    return vk_from_json(constants()["sp1_vk"], 1)


def ec_add(data):
    out = C.create_string_buffer(64)
    return bytes(out.raw) if lib().zkvo_ec_add(data, len(data), out) == 0 else None


def ec_mul(data):
    out = C.create_string_buffer(64)
    return bytes(out.raw) if lib().zkvo_ec_mul(data, len(data), out) == 0 else None


def ec_pairing(data, debug=False):
    out = C.create_string_buffer(32)
    if not debug:
        return bytes(out.raw) if lib().zkvo_ec_pairing(data, len(data), out) == 0 else None
    m, gt = C.create_string_buffer(384), C.create_string_buffer(384)
    rc = lib().zkvo_ec_pairing_debug(data, len(data), out, m, gt)
    return (bytes(out.raw), bytes(m.raw), bytes(gt.raw)) if rc == 0 else None


def g1_mul(pt, k):
    out = C.create_string_buffer(64)
    assert lib().zkvo_g1_mul(pt, w32(k), out) == 0
    return bytes(out.raw)


def g2_mul(pt, k):
    out = C.create_string_buffer(128)
    assert lib().zkvo_g2_mul(pt, w32(k), out) == 0
    return bytes(out.raw)


def g2_add(a, b):
    out = C.create_string_buffer(128)
    assert lib().zkvo_g2_add(a, b, out) == 0
    return bytes(out.raw)


def g2_from_x(x_im, x_re):
    out = C.create_string_buffer(128)
    return bytes(out.raw) if lib().zkvo_g2_from_x(w32(x_im) + w32(x_re), out) == 0 else None


def sha256(msg):
    out = C.create_string_buffer(32)
    lib().zkvo_sha256(msg, len(msg), out)
    return bytes(out.raw)


def final_exp(m):
    out = C.create_string_buffer(384)
    assert lib().zkvo_final_exp(m, out) == 0
    return bytes(out.raw)


def fp12_mul(a, b):
    out = C.create_string_buffer(384)
    assert lib().zkvo_fp12_mul(a, b, out) == 0
    return bytes(out.raw)


def fp12_cyc_sqr(a):
    out = C.create_string_buffer(384)
    assert lib().zkvo_fp12_cyc_sqr(a, out) == 0
    return bytes(out.raw)


P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
FP12_ONE = w32(1) + bytes(352)


def fp12_words(a):
    return [int.from_bytes(a[32 * i:32 * i + 32], "big") for i in range(12)]


def fp12_from_words(ws):
    return b"".join(w32(x) for x in ws)


def fp12_conj(a):
    """a^(p^6): c1 -> -c1 (the inverse of a unitary element)"""
    ws = fp12_words(a)
    return fp12_from_words(ws[:6] + [(P - x) % P for x in ws[6:]])


def fp12_pow(a, e):
    """a^e by left-to-right square-and-multiply over the oracle's Fp12 product (independent of every Frobenius routine)"""
    r = FP12_ONE
    for bit in bin(e)[2:]:
        r = fp12_mul(r, r)
        if bit == "1":
            r = fp12_mul(r, a)
    return r


def fp12_frob(a, k):
    """a^(p^k), k = 1, 2, 3, as k successive p-th powers"""
    for _ in range(k):
        a = fp12_pow(a, P)
    return a


# Fp words where lazily reduced arithmetic can go wrong: 0, 1, 2, p - 2, p - 1, (p -+ 1) / 2 and 2^256 mod p (the Montgomery radix)
EDGE_WORDS = (0, 1, 2, P - 2, P - 1, (P - 1) // 2, (P + 1) // 2, (1 << 256) % P)


def fp12_operand_classes(seed):
    """(name, a, b) operand pairs of 12 x BE-32 Fp12 elements at the edges of the tower arithmetic, shared by the GPU and host-emulation
    tests of csrc/lazy.cuh: all words p - 1, zero, one, -1, words drawn from EDGE_WORDS, Fp2 / Fp4 / Fp6 subfield elements, c0 = 0, c1 = 0,
    and a second operand equal to the first or to its conjugate.  Every class appears with a random partner and with an edge partner."""
    import random
    rnd = random.Random(seed)
    rand = lambda: [rnd.randrange(P) for _ in range(12)]
    edge = lambda: [rnd.choice(EDGE_WORDS) for _ in range(12)]
    keep = lambda ws, idx: [w if i in idx else 0 for i, w in enumerate(ws)]
    e = fp12_from_words
    firsts = [
        ("all_p-1", e([P - 1] * 12)),
        ("zero", bytes(384)),
        ("one", FP12_ONE),
        ("minus_one", e([P - 1] + [0] * 11)),
        ("edge_words_a", e(edge())),
        ("edge_words_b", e(edge())),
        ("edge_words_c", e(edge())),
        ("fp2_subfield", e(keep(rand(), (0, 1)))),
        ("fp2_subfield_edge", e(keep([P - 1] * 12, (0, 1)))),
        ("fp4_subfield", e(keep(rand(), (0, 1, 8, 9)))),            # c0.c0 + c1.c1 (v w = w^3)
        ("fp6_subfield", e(keep(edge(), range(6)))),
        ("c0_zero", e(keep(rand(), range(6, 12)))),
        ("c0_zero_edge", e(keep([P - 1] * 12, range(6, 12)))),
        ("c1_zero", e(keep(rand(), range(6)))),
        ("random", e(rand())),
    ]
    out = []
    for name, a in firsts:
        out.append((name + "|random", a, e(rand())))
        out.append((name + "|all_p-1", a, e([P - 1] * 12)))
        out.append((name + "|same", a, a))
        out.append((name + "|conj", a, fp12_conj(a)))
    out.append(("random|edge_words", e(rand()), e(edge())))
    out.append(("random|zero", e(rand()), bytes(384)))
    out.append(("random|one", e(rand()), FP12_ONE))
    out.append(("random|c0_zero", e(rand()), e(keep(rand(), range(6, 12)))))
    return out


def fp12_cyclotomic_operands(seed, nfrob=2):
    """(name, g) elements of the cyclotomic subgroup, the only inputs the Granger-Scott squaring is defined on: one, the final-exponentiation
    outputs of the nonzero operand classes (the subfield ones map to one), their conjugates, and Frobenius images of `nfrob` of them"""
    seen, out = {FP12_ONE}, [("one", FP12_ONE)]

    def add(name, g):
        if g not in seen:
            seen.add(g); out.append((name, g))
    gts = []
    for name, a, _ in fp12_operand_classes(seed):
        if a != bytes(384):
            g = final_exp(a)
            if g not in seen:
                gts.append((name.split("|")[0], g))
            add("final_exp(%s)" % name.split("|")[0], g)
    for name, g in gts:
        add("conj(final_exp(%s))" % name, fp12_conj(g))
    for name, g in gts[-nfrob:]:
        for k in (1, 2, 3):
            add("final_exp(%s)^(p^%d)" % (name, k), fp12_frob(g, k))
    return out


def ate_naf():
    buf = (C.c_int8 * 80)()
    n = lib().zkvo_ate_naf(buf, 80)
    return [buf[i] for i in range(n)]


def groth16_verify(vk, proof, signals, debug=False):
    k = len(signals) // 32
    if not debug:
        return lib().zkvo_groth16_verify(vk.buf, proof, signals, k)
    m, gt = C.create_string_buffer(384), C.create_string_buffer(384)
    st = lib().zkvo_groth16_verify_debug(vk.buf, proof, signals, k, m, gt)
    return st, bytes(m.raw), bytes(gt.raw)


class Risc0Oracle:
    """risc0/verifier.rs storage + methods (statuses instead of revert payloads)."""

    def __init__(self, vk=None):
        self.vk = vk or risc0_vk()
        self.h = C.create_string_buffer(lib().zkvo_risc0_sizeof())
        lib().zkvo_risc0_new(self.h, self.vk.buf)

    def initialize(self, control_root, bn254_control_id):
        return lib().zkvo_risc0_initialize(self.h, control_root, bn254_control_id)

    def selector(self):
        out = C.create_string_buffer(4); lib().zkvo_risc0_get_selector(self.h, out); return bytes(out.raw)

    def vk_digest(self):
        out = C.create_string_buffer(32); lib().zkvo_risc0_get_vk_digest(self.h, out); return bytes(out.raw)

    def signals(self, claim):
        out = C.create_string_buffer(160); lib().zkvo_risc0_signals(self.h, claim, out); return bytes(out.raw)

    def verify(self, seal, image_id, journal):
        return lib().zkvo_risc0_verify(self.h, seal, len(seal), image_id, journal)

    def verify_integrity(self, seal, claim):
        return lib().zkvo_risc0_verify_integrity(self.h, seal, len(seal), claim)

    def verify_batch(self, seals, image_ids, journals):
        import numpy as np
        n = len(seals)
        off = np.zeros(n + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in seals])
        blob = b"".join(seals) or b"\0"
        st = np.zeros(n, dtype=np.uint8)
        lib().zkvo_risc0_verify_batch(self.h, blob, off.ctypes.data, b"".join(image_ids), b"".join(journals), n, st.ctypes.data)
        return st


def claim_digest(image_id, journal):
    out = C.create_string_buffer(32); lib().zkvo_risc0_claim_digest(image_id, journal, out); return bytes(out.raw)


def sp1_hash_public_values(pv):
    out = C.create_string_buffer(32); lib().zkvo_sp1_hash_public_values(pv, len(pv), out); return bytes(out.raw)


def sp1_verify(vk, selector, vkey, pv, proof):
    return lib().zkvo_sp1_verify(vk.buf, selector, vkey, pv, len(pv), proof, len(proof))


def sp1_verify_batch(vk, selector, vkeys, pvs, proofs):
    import numpy as np
    n = len(proofs)
    po = np.zeros(n + 1, dtype=np.uint64); po[1:] = np.cumsum([len(s) for s in proofs])
    vo = np.zeros(n + 1, dtype=np.uint64); vo[1:] = np.cumsum([len(s) for s in pvs])
    st = np.zeros(n, dtype=np.uint8)
    lib().zkvo_sp1_verify_batch(vk.buf, selector, b"".join(vkeys), (b"".join(pvs) or b"\0"), vo.ctypes.data,
                                (b"".join(proofs) or b"\0"), po.ctypes.data, n, st.ctypes.data)
    return st


def pairing4_batch(blob, n, want_gt=False, want_miller=False):
    import numpy as np
    ok = np.zeros(n, dtype=np.uint8)
    gt = np.zeros(n * 384, dtype=np.uint8) if want_gt else None
    ml = np.zeros(n * 384, dtype=np.uint8) if want_miller else None
    lib().zkvo_pairing4_batch(blob, n, ok.ctypes.data, gt.ctypes.data if want_gt else None, ml.ctypes.data if want_miller else None)
    return ok, gt, ml


def groth16_verify_batch(vk, proofs, signals, n):
    import numpy as np
    st = np.zeros(n, dtype=np.uint8)
    lib().zkvo_groth16_verify_batch(vk.buf, proofs, signals, vk.k, n, st.ctypes.data)
    return st


def max_threads():
    return lib().zkvo_max_threads()
