"""The position-coded batches of tests/batch_geometry.py checked against the CPU oracle, without a GPU: for a small tiled batch (every pool
entry three times, every class present) the expectation built from the codes must equal the oracle's status record by record, for every
shape the GPU tests send; the codes and pools must be deterministic; the public-value hash must match the oracle at every length."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import batch_geometry as G
import oracle_lib as O
from stylus_zkvm_verifiers_b200 import synth as S

N = 3 * G.D + 5
SEED = 0xB6E0_0001
# every public-value length the GPU tests hash: 0..300, the long host-form lengths, and the device-form strides
PV_LENGTHS = sorted(set(range(301)) | {447, 448, 511, 512, 520, 1000, 1023, 1024, 4095, 4096, 65536, 1 << 20}
                    | {0, 1, 55, 56, 63, 64, 65, 119, 120, 127, 128, 129, 200, 1000, 4096})


def _ovk(vk):
    return O.Vk(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)


@pytest.fixture(scope="module")
def risc0(oracle_backend, fx):
    vk = S.make_vk(oracle_backend, 0, 6, SEED + 1)
    ro = O.Risc0Oracle(_ovk(vk))
    ro.initialize(fx["control_root"], fx["bn254_control_id"])
    return ro, G.Risc0Pool(oracle_backend, [(vk, ro.selector(), fx["control_root"], fx["bn254_control_id"])], fx["sys0"], SEED + 2)


def test_codes_are_splitmix64_and_cover_every_class():
    rng = S.SplitMix64(SEED)
    assert G.splitmix(SEED, 40).tolist() == [rng.next() for _ in range(40)]
    cls, sub = G.codes(SEED, N)
    counts = np.bincount(cls, minlength=4) / N
    assert abs(counts[G.KEEP] - 0.5) < 0.05 and all(0.05 < counts[c] for c in (G.TAMPER, G.SELECTOR, G.LENGTH))
    assert sub.min() >= 0 and sub.max() < 1 << 16 and len(set((sub & 1).tolist())) == 2
    again, _ = G.codes(SEED, N)
    assert np.array_equal(cls, again) and not np.array_equal(cls, G.codes(SEED + 1, N)[0])
    dev, _ = G.codes(SEED, N, classes=(G.KEEP, G.TAMPER), force_length=(5, 7))
    assert set(dev.tolist()) == {G.KEEP, G.TAMPER, G.LENGTH} and dev[5] == dev[7] == G.LENGTH
    keep = cls == G.KEEP
    keep[[5, 7]] = False
    assert (dev[keep] == G.KEEP).all() and (dev[(cls == G.SELECTOR) | (cls == G.TAMPER)] != G.KEEP).all()
    # the tiling covers every pool entry in every class
    j = G.tiled(1 << 16)
    c16, _ = G.codes(SEED, 1 << 16)
    for c in range(4):
        assert len(set(j[c16 == c].tolist())) > G.D // 2


def test_pool_is_deterministic(oracle_backend, fx):
    vk = S.make_vk(oracle_backend, 0, 6, SEED + 1)
    route = [(vk, b"\x01\x02\x03\x04", fx["control_root"], fx["bn254_control_id"])]
    a = G.Risc0Pool(oracle_backend, route, fx["sys0"], SEED + 9)
    b = G.Risc0Pool(oracle_backend, route, fx["sys0"], SEED + 9)
    assert a.seals.shape == (G.D, 260) and len({r.tobytes() for r in a.seals}) == G.D            # D distinct records
    for x, y in ((a.seals, b.seals), (a.ims, b.ims), (a.jrs, b.jrs), (a.claims, b.claims)):
        assert np.array_equal(x, y)
    assert not np.array_equal(a.jrs, G.Risc0Pool(oracle_backend, route, fx["sys0"], SEED + 10).jrs)


def test_risc0_expectation_matches_oracle(risc0):
    ro, pool = risc0
    cls, sub = G.codes(SEED + 3, N, force_length=(G.D - 1, G.D))
    blob, off, ims, jrs = G.risc0_host(pool, G.tiled(N), cls, sub)
    assert off[0] == G.SEAL_PREFIX and off[-1] == len(blob)
    st = np.zeros(N, dtype=np.uint8)
    O.lib().zkvo_risc0_verify_batch(ro.h, blob.ctypes.data, off.ctypes.data, ims.ctypes.data, jrs.ctypes.data, N, st.ctypes.data)
    assert st.tolist() == G.STATUS[cls].tolist()
    assert set(st.tolist()) == {0, 2, 3, 4}
    blob, off, claims, _ = G.risc0_host(pool, G.tiled(N), cls, sub, integrity=True)
    st = np.zeros(N, dtype=np.uint8)
    O.lib().zkvo_risc0_verify_integrity_batch(ro.h, blob.ctypes.data, off.ctypes.data, claims.ctypes.data, N, st.ctypes.data)
    assert st.tolist() == G.STATUS[cls].tolist()


def _sp1_oracle(vk, sel, vkeys, pv, pv_off, proofs, proof_off):
    n = len(vkeys)
    st = np.zeros(n, dtype=np.uint8)
    O.lib().zkvo_sp1_verify_batch(vk.buf, sel, vkeys.ctypes.data, pv.ctypes.data, pv_off.ctypes.data, proofs.ctypes.data, proof_off.ctypes.data,
                                  n, st.ctypes.data)
    return st


def test_sp1_expectation_matches_oracle(oracle_backend):
    vk = S.make_vk(oracle_backend, 1, 3, SEED + 4)
    lengths = [(7 * j) % 300 for j in range(G.D)]
    lengths[:4] = [0, 447, 1024, 4096]
    pool = G.Sp1Pool(oracle_backend, [(vk, S.SP1_SELECTOR)], lengths, SEED + 5)
    cls, sub = G.codes(SEED + 6, N, force_length=(G.D - 1, G.D))
    vkeys, pv, pv_off, proofs, proof_off = G.sp1_host(pool, G.tiled(N), cls, sub)
    assert pv_off[0] == G.PV_PREFIX and pv_off[-1] == len(pv) and proof_off[-1] == len(proofs)
    st = _sp1_oracle(_ovk(vk), S.SP1_SELECTOR, vkeys, pv, pv_off, proofs, proof_off)
    assert st.tolist() == G.STATUS[cls].tolist()
    # the same records rebuilt one by one (the path the GPU tests take for sampled positions of a large batch)
    idx = np.array([0, 1, 2, 3, G.D - 1, G.D, N - 1])
    v2, pv2, pvo2, pr2, pro2 = G.sp1_host(pool, idx % G.D, cls[idx], sub[idx])
    assert G.slices(pv2, pvo2, range(len(idx))) == G.slices(pv, pv_off, idx)
    assert G.slices(pr2, pro2, range(len(idx))) == G.slices(proofs, proof_off, idx) and np.array_equal(v2, vkeys[idx])


def test_sp1_fixed_stride_expectation_matches_oracle(oracle_backend):
    vk = S.make_vk(oracle_backend, 1, 3, SEED + 4)
    for stride in (0, 520):
        pool = G.Sp1Pool(oracle_backend, [(vk, S.SP1_SELECTOR)], [stride] * G.D, SEED + 7)
        cls, sub = G.codes(SEED + 8, N, classes=(G.KEEP, G.TAMPER, G.SELECTOR))
        vkeys, pv, proofs = G.sp1_fixed_host(pool, G.tiled(N), cls, sub, stride)
        pv_off = (np.arange(N + 1) * stride).astype(np.uint64)
        proof_off = (np.arange(N + 1) * 260).astype(np.uint64)
        st = _sp1_oracle(_ovk(vk), S.SP1_SELECTOR, vkeys, np.ascontiguousarray(pv).reshape(-1) if stride else np.zeros(1, np.uint8), pv_off,
                         proofs, proof_off)
        assert st.tolist() == G.STATUS[cls].tolist()


@pytest.fixture(scope="module")
def generic(oracle_backend):
    keys = [S.make_vk(oracle_backend, k % 2, n_ic, SEED + 20 + n_ic) for k, n_ic in enumerate((2, 3, 4, 6, 9))]
    return keys, G.GenericPool(oracle_backend, keys, SEED + 11)


def test_key_set_expectation_matches_oracle(generic):
    keys, pool = generic
    ovks = [_ovk(k) for k in keys]
    cls, sub = G.codes(SEED + 12, N, force_length=(G.D - 1, G.D))
    key, proofs, sig, off = G.generic_host(pool, G.tiled(N), cls, sub, len(keys))
    assert off[0] == G.SIG_PREFIX and int(off[-1]) * 32 == len(sig)
    words = lambda i: sig[int(off[i]) * 32:int(off[i + 1]) * 32].tobytes()
    with ThreadPoolExecutor(8) as ex:
        st = list(ex.map(lambda i: O.groth16_verify(ovks[key[i]], proofs[i].tobytes(), words(i)), range(N)))
    assert st == G.generic_expect(cls).tolist()
    # the device form's host counterpart (out-of-range key index for SELECTOR: checked as the kernel checks it, a failed proof)
    idx = np.arange(0, N, 7)
    cls, sub = G.codes(SEED + 12, N, classes=(G.KEEP, G.TAMPER, G.SELECTOR))
    key2, proofs2, sigs2 = G.generic_fixed_host(pool, idx % G.D, cls[idx], sub[idx], len(keys))
    got = [O.groth16_verify(ovks[k], p.tobytes(), s) if k < len(keys) else O.ST_VERIFICATION_FAILED for k, p, s in zip(key2, proofs2, sigs2)]
    want = np.where(cls[idx] == G.KEEP, 0, 4)
    assert got == want.tolist()


def test_pairing4_expectation_matches_oracle(oracle_backend):
    vk = S.make_vk(oracle_backend, 0, 2, SEED + 13)
    pool = G.PairingPool(oracle_backend, SEED + 14, vk=vk)
    cls, _ = G.codes(SEED + 15, N, classes=(G.KEEP, G.TAMPER, G.SELECTOR))
    g1, g2, want = G.pairing4_host(pool, G.tiled(N), cls)
    blob = np.ascontiguousarray(G.pairing4_oracle_blob(g1, g2, vk))
    ok, _, _ = O.pairing4_batch(blob.ctypes.data, N)
    assert ok.tolist() == want.tolist() and set(want.tolist()) == {0, 1, 2}


def test_ec_pairing_expectation_matches_oracle(oracle_backend):
    pool = G.PairingPool(oracle_backend, SEED + 16)
    cls, _ = G.codes(SEED + 17, N, classes=(G.KEEP, G.TAMPER, G.SELECTOR))
    x, want = G.ec_pairing_host(pool, G.tiled(N), cls)
    with ThreadPoolExecutor(8) as ex:
        got = list(ex.map(lambda i: O.ec_pairing(x[i].tobytes()), range(N)))
    assert [2 if g is None else g[31] for g in got] == want.tolist() and set(want.tolist()) == {0, 1, 2}


def test_sp1_signals_match_oracle_hash_at_every_length():
    vkey = bytes(1) + bytes(range(31))
    for L in PV_LENGTHS:
        pv = G.random_bytes(L + 1, L)
        assert len(pv) == L
        assert S.sp1_signals(vkey, pv)[1] == int.from_bytes(O.sp1_hash_public_values(pv), "big"), L


def test_sample_positions_cover_the_schedule():
    n = (1 << 21) + (1 << 18) + 37
    edges = G.schedule_edges(n)
    assert [e for e in edges if e % G.PASS == 0] == [0, 1 << 20, 1 << 21]
    assert len(edges) == 12 and all(e % G.HTPB == 0 for e in edges)
    assert G.chunk_size((1 << 18) + 37, 4) == 65664 and (1 << 21) + 3 * 65664 in edges
    s = G.samples(n, 1, edges)
    for e in edges[1:]:
        assert all(p in s for p in range(e - 2, e + 3))
    assert all(p in s for p in range(64)) and all(p in s for p in range(n - 64, n)) and len(s) > 300 + 128
