"""Position-coded batches for the shape tests of the batch entry points (tests/test_batch_geometry.py, tests/test_gpu_batch_geometry.py).

A batch tiled from one record hides most shape bugs: a status written to the wrong slot still looks right.  Here record i is pool[i mod D],
one of D distinct valid records, altered by a code c(i) = SplitMix64(seed, i) that picks a class, and its expected status is a function
of that class alone:

    KEEP     -> OK
    TAMPER   -> VerificationFailed      (a journal / claim / public-value byte, or a signal, changed)
    SELECTOR -> SelectorMismatch        (a selector no handle or route has)
    LENGTH   -> InvalidProofData        (host forms: the seal or proof one byte longer or shorter)

A status copied to the wrong pass, slot or chunk, or a record read at a wrong base, then mismatches at about half of the positions it
touches.  D is an odd prime, so the tiling period shares no factor with a pass, chunk, block or warp size.  Host forms are built with
numpy, device forms gathered and altered with torch on the GPU from the uploaded pool; `samples` names the positions to compare one to
one with the CPU oracle (pass and chunk edges, both ends, random ones)."""
import numpy as np

from stylus_zkvm_verifiers_b200 import synth as S

D = 1021                     # pool size (prime)
PASS = 1 << 20               # MAX_CHUNK of csrc/zkv.cu: records per device pass of a host-buffer call
DEVICE_MAX = PASS * 8        # the largest n a *_device entry point accepts
PAIRING4_CHUNK = 1 << 18     # zkv_pairing4_batch cuts host batches here
EC_PAIRING_CHUNK = 1 << 16   # zkv_ec_pairing_batch cuts here
HTPB = 128                   # block size of the heavy kernels: chunk sizes are multiples of it

KEEP, TAMPER, SELECTOR, LENGTH = range(4)
STATUS = np.array([S.ST_OK, S.ST_VERIFICATION_FAILED, S.ST_SELECTOR_MISMATCH, S.ST_INVALID_PROOF_DATA], dtype=np.uint8)
UNKNOWN_SELECTOR = b"\xde\xad\xbe\xef"
BAD_G1 = S.w32(1) + S.w32(3)                   # off the curve: the pairing call reverts
SEAL_PREFIX, PV_PREFIX, SIG_PREFIX = 13, 7, 3  # junk in front of the first record: offsets start there, not at 0
_M64 = 0xFFFFFFFFFFFFFFFF
DEVICE = "cuda"                                # where the device forms are built


def splitmix(seed, n):
    """The first n outputs of synth.SplitMix64(seed), vectorised: output i mixes the state seed + (i + 1) * 0x9E3779B97F4A7C15."""
    i = np.arange(1, n + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed & _M64) + i * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def random_bytes(seed, n):
    return splitmix(seed, (n + 7) // 8).astype(">u8").tobytes()[:n]


def codes(seed, n, classes=(KEEP, TAMPER, SELECTOR, LENGTH), force_length=()):
    """(cls, sub) per position: the class (top 4 bits of c(i): 8/16 KEEP, 4/16 TAMPER, 2/16 SELECTOR, 2/16 LENGTH; a class the form has
    not becomes TAMPER) and 16 more bits that pick the altered byte or the direction of a length change.  Positions in force_length get
    LENGTH (records around a pass edge, so the blob offsets shift across it)."""
    z = splitmix(seed, n)
    v = (z >> np.uint64(60)).astype(np.uint8)
    cls = np.select([v < 8, v < 12, v < 14], [KEEP, TAMPER, SELECTOR], LENGTH).astype(np.uint8)
    for c in (SELECTOR, LENGTH):
        if c not in classes:
            cls[cls == c] = TAMPER
    for p in force_length:
        if p < n:
            cls[p] = LENGTH
    sub = ((z >> np.uint64(8)) & np.uint64(0xFFFF)).astype(np.int64)
    return cls, sub


def tiled(n):
    return np.arange(n, dtype=np.int64) % D


def _rows(items):
    return np.frombuffer(b"".join(items), dtype=np.uint8).reshape(len(items), -1).copy()


def _routes_of(n_routes):
    """pool entry j belongs to route j mod n_routes"""
    return [list(range(r, D, n_routes)) for r in range(n_routes)]


# ------------------------------------------------------------------ pools
class Risc0Pool:
    """D valid RISC Zero records; entry j is a seal of route j mod len(routes).  routes: (synth key, selector, control root, control id)."""

    def __init__(self, backend, routes, sys0, seed):
        seals, ims, jrs = [None] * D, [None] * D, [None] * D
        for r, ((vk, sel, cr, cid), idx) in enumerate(zip(routes, _routes_of(len(routes)))):
            b = S.make_risc0_batch(backend, vk, sel, cr, cid, sys0, len(idx), seed + r, pool=64)
            for t, j in enumerate(idx):
                seals[j], ims[j], jrs[j] = b.seals[t], b.image_ids[t], b.journals[t]
        self.seals, self.ims, self.jrs = _rows(seals), _rows(ims), _rows(jrs)
        self.claims = _rows([S.risc0_claim_digest(a, b, sys0) for a, b in zip(ims, jrs)])


class Sp1Pool:
    """D valid SP1 records with public values of the given D lengths; entry j is a proof of route j mod len(routes).
    routes: (synth key, selector)."""

    def __init__(self, backend, routes, lengths, seed):
        rng = S.SplitMix64(seed)
        self.pv_len = np.asarray(lengths, dtype=np.int64)
        assert len(self.pv_len) == D
        vkeys = [b"\0" + rng.bytes(31) for _ in range(D)]
        pvs = [random_bytes(seed * 7919 + j, int(L)) for j, L in enumerate(self.pv_len)]
        proofs = [None] * D
        for (vk, sel), idx in zip(routes, _routes_of(len(routes))):
            ps = S.make_proofs(backend, vk, [S.sp1_signals(vkeys[j], pvs[j]) for j in idx], rng, S.Pools(backend, rng, 64))
            for j, p in zip(idx, ps):
                proofs[j] = sel + p
        self.vkeys, self.proofs = _rows(vkeys), _rows(proofs)
        self.pv_off = np.concatenate([[0], np.cumsum(self.pv_len)]).astype(np.int64)
        self.pv_blob = np.frombuffer(b"".join(pvs), dtype=np.uint8).copy()


class GenericPool:
    """D valid Groth16 proofs under `keys` (synth keys of different n_ic): entry j under key j mod len(keys), with its signals as
    32-byte words."""

    def __init__(self, backend, keys, seed):
        rng = S.SplitMix64(seed)
        self.key = np.arange(D, dtype=np.int64) % len(keys)
        sigs = [[rng.fr() for _ in range(keys[k].k)] for k in self.key]
        proofs = [None] * D
        for k, idx in enumerate(_routes_of(len(keys))):
            ps = S.make_proofs(backend, keys[k], [sigs[j] for j in idx], rng, S.Pools(backend, rng, 64))
            for j, p in zip(idx, ps):
                proofs[j] = p
        self.proofs = _rows(proofs)
        self.nsig = np.array([len(s) for s in sigs], dtype=np.int64)
        self.sig_off = np.concatenate([[0], np.cumsum(self.nsig)]).astype(np.int64)           # in words
        self.sig_blob = np.frombuffer(b"".join(S.w32(v) for s in sigs for v in s), dtype=np.uint8).copy()


class PairingPool:
    """D instances of the pairing services.  pairing4 (vk given): 4 G1 points + 1 G2 point, about half of them with product one
    (synth.make_pairing4_batch).  Otherwise 2-pair ecPairing instances (A, B) (C, G2) with C = -(a b) G1 (product one) or -(a b + 1) G1."""

    def __init__(self, backend, seed, vk=None):
        if vk is not None:
            g1s, g2s, ok = S.make_pairing4_batch(backend, vk, D, seed, pool=64)
            self.g1, self.g2, self.ok = _rows(g1s), _rows(g2s), np.array(ok, dtype=np.uint8)
            return
        rng = S.SplitMix64(seed)
        pools = S.Pools(backend, rng, 64)
        ja = [rng.below(64) for _ in range(D)]
        jb = [rng.below(64) for _ in range(D)]
        self.ok = np.array([rng.below(2) for _ in range(D)], dtype=np.uint8)
        cs = backend.g1_mul([(-(pools.a[ja[j]] * pools.b[jb[j]] + (1 - int(self.ok[j])))) % S.R for j in range(D)])
        self.pairs = _rows([pools.A[ja[j]] + pools.B[jb[j]] + cs[j] + S.G2_GEN for j in range(D)])      # D x 384


# ------------------------------------------------------------------ host forms (numpy)
def _fixed_records(recs, j, cls, sub, sel=UNKNOWN_SELECTOR, prefix=SEAL_PREFIX):
    """260-byte records recs[j], SELECTOR -> `sel`, LENGTH -> one byte shorter or longer; (blob with `prefix` junk bytes in front, n+1 offsets)"""
    n = len(j)
    rows = np.empty((n, 261), dtype=np.uint8)
    rows[:, :260] = recs[j]
    rows[:, 260] = 0xA5
    rows[cls == SELECTOR, :4] = np.frombuffer(sel, dtype=np.uint8)
    ln = np.full(n, 260, dtype=np.int64)
    lc = cls == LENGTH
    ln[lc] = np.where(sub[lc] & 1, 261, 259)
    blob = np.concatenate([np.full(prefix, 0x5C, dtype=np.uint8), rows[np.arange(261)[None, :] < ln[:, None]]])
    off = np.empty(n + 1, dtype=np.uint64)
    off[0] = prefix
    off[1:] = prefix + np.cumsum(ln)
    return blob, off


def _flip(a, cls, sub, width):
    """flip the low bit of byte sub mod width of every TAMPER row of a (n x width)"""
    t = np.nonzero(cls == TAMPER)[0]
    a[t, sub[t] % width] ^= 1
    return a


def risc0_host(pool, j, cls, sub, integrity=False):
    """(seal blob, seal offsets, image ids or claims, journals or None): TAMPER flips a journal byte (a claim byte with integrity)"""
    blob, off = _fixed_records(pool.seals, j, cls, sub)
    if integrity:
        return blob, off, _flip(pool.claims[j].copy(), cls, sub, 32), None
    return blob, off, pool.ims[j].copy(), _flip(pool.jrs[j].copy(), cls, sub, 32)


def _gather(blob, off, j, prefix):
    """the pool segments blob[off[j] : off[j + 1]] for every j, concatenated behind `prefix` junk bytes (tiled j: np.tile)"""
    head = np.full(prefix, 0x3E, dtype=np.uint8)
    n = len(j)
    if n >= D and np.array_equal(j, tiled(n)):
        return np.concatenate([head, np.tile(blob, n // D), blob[:off[n % D]]])
    return np.concatenate([head] + [blob[off[k]:off[k + 1]] for k in j])


def sp1_host(pool, j, cls, sub):
    """(vkeys, pv blob, pv offsets, proof blob, proof offsets): TAMPER flips a public-value byte (the vkey's last byte for empty ones)"""
    proofs, proof_off = _fixed_records(pool.proofs, j, cls, sub)
    vkeys = pool.vkeys[j].copy()
    ln = pool.pv_len[j]
    pv_off = np.empty(len(j) + 1, dtype=np.uint64)
    pv_off[0] = PV_PREFIX
    pv_off[1:] = PV_PREFIX + np.cumsum(ln)
    pv = _gather(pool.pv_blob, pool.pv_off, j, PV_PREFIX)
    t = np.nonzero(cls == TAMPER)[0]
    tp, tv = t[ln[t] > 0], t[ln[t] == 0]
    pv[pv_off[tp].astype(np.int64) + sub[tp] % ln[tp]] ^= 1
    vkeys[tv, 31] ^= 1
    return vkeys, pv, pv_off, proofs, proof_off


def generic_host(pool, j, cls, sub, n_keys):
    """(key_idx, proofs, signal blob, signal word offsets) of a key-set call: TAMPER flips the low bit of the first signal (signal +- 1),
    SELECTOR names the next key (a wrong key), LENGTH drops the last signal or adds one: all VerificationFailed"""
    n = len(j)
    key = pool.key[j].copy()
    sc = cls == SELECTOR
    key[sc] = (key[sc] + 1) % n_keys
    cnt = pool.nsig[j].copy()
    lc = cls == LENGTH
    cnt[lc] += np.where(sub[lc] & 1, 1, -1)
    width = int(pool.nsig.max()) + 1
    words = np.zeros((n, width, 32), dtype=np.uint8)
    src = pool.sig_blob.reshape(-1, 32)
    for w in range(width - 1):                      # word w of every record that has one in the pool
        has = pool.nsig[j] > w
        words[has, w] = src[pool.sig_off[j[has]] + w]
    add = np.nonzero(lc & (sub & 1 == 1))[0]
    words[add, pool.nsig[j[add]]] = 0x11            # the added signal: 0x1111...11 < r
    t = np.nonzero(cls == TAMPER)[0]
    words[t, 0, 31] ^= 1
    sig = np.concatenate([np.full(SIG_PREFIX * 32, 0x2B, dtype=np.uint8), words[np.arange(width)[None, :] < cnt[:, None]].reshape(-1)])
    off = np.empty(n + 1, dtype=np.uint64)
    off[0] = SIG_PREFIX
    off[1:] = SIG_PREFIX + np.cumsum(cnt)
    return key.astype(np.uint32), pool.proofs[j].copy(), sig, off


def generic_expect(cls):
    return np.where(cls == KEEP, S.ST_OK, S.ST_VERIFICATION_FAILED).astype(np.uint8)


def pairing4_host(pool, j, cls):
    """(g1s n x 256, g2s n x 128, expected ok bytes): TAMPER puts P1 off the curve (reverts: 2), SELECTOR makes P0 the point at infinity
    (the product of the other three pairs is not one: 0)"""
    g1, g2 = pool.g1[j].copy(), pool.g2[j].copy()
    g1[cls == TAMPER, 64:128] = np.frombuffer(BAD_G1, dtype=np.uint8)
    g1[cls == SELECTOR, 0:64] = 0
    return g1, g2, pairing_expect(pool, j, cls)


def pairing_expect(pool, j, cls):
    return np.where(cls == KEEP, pool.ok[j], np.where(cls == TAMPER, 2, 0)).astype(np.uint8)


def ec_pairing_host(pool, j, cls):
    """(n x 384 instances, expected: 1 / 0 / 2 = reverts): TAMPER puts the second pair's G1 point off the curve, SELECTOR makes the first
    pair's G1 point infinity"""
    x = pool.pairs[j].copy()
    x[cls == TAMPER, 192:256] = np.frombuffer(BAD_G1, dtype=np.uint8)
    x[cls == SELECTOR, 0:64] = 0
    return x, pairing_expect(pool, j, cls)


def pairing4_oracle_blob(g1, g2, vk):
    """the oracle's 768-byte form of pairing4 instances: P0 Q | P1 beta | P2 gamma | P3 delta"""
    n = len(g1)
    fixed = [np.broadcast_to(np.frombuffer(q, dtype=np.uint8), (n, 128)) for q in (vk.beta, vk.gamma, vk.delta)]
    return np.concatenate([g1[:, 0:64], g2, g1[:, 64:128], fixed[0], g1[:, 128:192], fixed[1], g1[:, 192:256], fixed[2]], axis=1)


# ------------------------------------------------------------------ device forms (torch, on the GPU)
def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEVICE)


def device_codes(cls, sub):
    return _cuda(cls), _cuda(sub.astype(np.int32))


def _tiled_rows(rows, n):
    import torch
    return _cuda(rows)[torch.arange(n, device=DEVICE) % D]


def _flip_device(a, cls, sub, width):
    import torch
    t = torch.nonzero(cls == TAMPER).squeeze(1)
    col = (sub[t] % width).long()
    a[t, col] ^= 1
    return a


def _selector_device(recs, cls):
    import torch
    sel = torch.tensor(list(UNKNOWN_SELECTOR), dtype=torch.uint8, device=DEVICE)
    recs[:, :4] = torch.where((cls == SELECTOR)[:, None], sel[None, :], recs[:, :4])
    return recs


def risc0_device(pool, cls, sub):
    """(seals n x 260, image ids, journals) on the GPU: the records risc0_host builds for tiled positions, without LENGTH"""
    n = len(cls)
    return _selector_device(_tiled_rows(pool.seals, n), cls), _tiled_rows(pool.ims, n), _flip_device(_tiled_rows(pool.jrs, n), cls, sub, 32)


def sp1_device(pool, cls, sub, stride):
    """(vkeys, public values n x stride, proofs n x 260) on the GPU from a pool whose public values are all `stride` bytes long"""
    n = len(cls)
    assert (pool.pv_len == stride).all()
    vkeys = _tiled_rows(pool.vkeys, n)
    if stride:
        pv = _flip_device(_tiled_rows(pool.pv_blob.reshape(D, stride), n), cls, sub, stride)
    else:
        import torch
        pv = torch.zeros(1, dtype=torch.uint8, device=DEVICE)
        vkeys[:, 31] ^= (cls == TAMPER).to(vkeys.dtype)
    return vkeys, pv, _selector_device(_tiled_rows(pool.proofs, n), cls)


def sp1_fixed_host(pool, j, cls, sub, stride):
    """the host counterpart of sp1_device for the records j: (vkeys, pv n x stride, proofs n x 260)"""
    vkeys = pool.vkeys[j].copy()
    if stride:
        pv = _flip(pool.pv_blob.reshape(D, stride)[j].copy(), cls, sub, stride)
    else:
        pv = np.zeros((len(j), 0), dtype=np.uint8)
        vkeys[cls == TAMPER, 31] ^= 1
    proofs = pool.proofs[j].copy()
    proofs[cls == SELECTOR, :4] = np.frombuffer(UNKNOWN_SELECTOR, dtype=np.uint8)
    return vkeys, pv, proofs


def generic_device(pool, cls, sub, n_keys):
    """(key_idx uint32 as int32, proofs, signal words, word offsets uint64 as int64) on the GPU: TAMPER flips the first signal's low bit,
    SELECTOR sets the key index to n_keys (out of range: that proof fails)"""
    import torch
    n = len(cls)
    j = torch.arange(n, device=DEVICE) % D
    key = _cuda(pool.key.astype(np.int32))[j]
    key = torch.where(cls == SELECTOR, torch.full_like(key, n_keys), key)
    cnt = _cuda(pool.nsig)[j]
    off = torch.zeros(n + 1, dtype=torch.int64, device=DEVICE)
    off[1:] = torch.cumsum(cnt, 0)
    reps, rem = n // D, n % D
    src = _cuda(pool.sig_blob)
    sig = torch.cat([src.repeat(reps), src[:int(pool.sig_off[rem]) * 32]]).reshape(-1, 32)
    t = torch.nonzero(cls == TAMPER).squeeze(1)
    sig[off[t], 31] ^= 1
    return key, _tiled_rows(pool.proofs, n), sig, off


def generic_fixed_host(pool, j, cls, sub, n_keys):
    """the host counterpart of generic_device for the records j: (key indices, proofs, per-record signal words)"""
    key = pool.key[j].copy()
    key[cls == SELECTOR] = n_keys
    sigs = []
    for k, c in zip(j, cls):
        w = bytearray(pool.sig_blob[pool.sig_off[k] * 32:pool.sig_off[k + 1] * 32].tobytes())
        if c == TAMPER:
            w[31] ^= 1
        sigs.append(bytes(w))
    return key, pool.proofs[j].copy(), sigs


def pairing4_device(pool, cls):
    import torch
    n = len(cls)
    g1, g2 = _tiled_rows(pool.g1, n), _tiled_rows(pool.g2, n)
    bad = torch.tensor(list(BAD_G1), dtype=torch.uint8, device=DEVICE)
    g1[:, 64:128] = torch.where((cls == TAMPER)[:, None], bad[None, :], g1[:, 64:128])
    g1[:, 0:64] = torch.where((cls == SELECTOR)[:, None], torch.zeros_like(g1[:, 0:64]), g1[:, 0:64])
    return g1, g2


# ------------------------------------------------------------------ positions for the oracle
def chunk_size(m, chunks=4):
    """csrc/zkv.cu chunk_size: records per piece when m records are cut into `chunks` (a multiple of the heavy kernels' block size)"""
    per = (m + chunks - 1) // chunks
    return (per + HTPB - 1) // HTPB * HTPB


def schedule_edges(n, pass_size=PASS, chunks=4):
    """the first record of every pass of `pass_size` and of every piece of a pass cut into `chunks` (csrc/zkv.cu host_pass / run_verify)"""
    out = []
    for s0 in range(0, n, pass_size):
        m = min(pass_size, n - s0)
        out += [s0 + o for o in range(0, m, chunk_size(m, chunks))]
    return out


def samples(n, seed, edges=(), count=300):
    """sorted positions: both ends (64 each), edges +- 2, and `count` random positions"""
    s = set(range(min(64, n))) | set(range(max(0, n - 64), n))
    for e in edges:
        s |= {p for p in range(e - 2, e + 3) if 0 <= p < n}
    s |= set(np.random.default_rng(seed).integers(0, n, count).tolist())
    return np.array(sorted(s), dtype=np.int64)


def slices(blob, off, idx):
    """the records blob[off[i] : off[i + 1]] for i in idx, as bytes"""
    return [blob[int(off[i]):int(off[i + 1])].tobytes() for i in idx]
