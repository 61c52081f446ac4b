"""Throughput of the key-set entry point (zkv_groth16_verify_batch_keys) against one zkv_groth16_verify_batch call per key, on device 0.

  (a) 2^16 proofs spread evenly over K in {1, 8, 64} keys: one set call against K single-key calls;
  (b) one key at 2^16 and 2^20: the set call against the single-key call (what grouping and padding cost);
  (c) the set's end-to-end rate (host arrays) over its device-resident rate (the _device form on inputs already in HBM).

Host clock around calls that end synchronised; host inputs in page-locked memory (pinned_copy), so both entry points upload them in place;
every status of every call is checked against the generator's expectation (one proof in eight carries a tampered signal).  The two forms
are alternated call by call.  One JSON line per measurement; the first names the GPU and its power limit, read in the same run.

    python tools/keyset_bench.py --out profiles/r3_keyset_bench.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
SHAPES = [(0, 6), (1, 3), (0, 2), (1, 4), (0, 5), (1, 6), (0, 3), (1, 2)]      # (vm, n_ic), cycled over the keys


def gpu_info():
    import torch
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                  # noqa: BLE001 - reported, not hidden
        pl = "unavailable (%s)" % e
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": pl}


def workload(Z, S, gpu, K, n, distinct, seed):
    """n proofs over K keys (n / K each, tiled from `distinct` generated proofs per key), caller order a seeded random interleaving"""
    w = lambda v: v.to_bytes(32, "big")
    rng = S.SplitMix64(seed)
    per = n // K
    keys, kvs, per_key = [], [], []
    for k in range(K):
        vm, nic = SHAPES[k % len(SHAPES)]
        vk = S.make_vk(gpu, vm, nic, seed + 1 + k)
        sigs = [[rng.fr() for _ in range(vk.k)] for _ in range(distinct)]
        prs = S.make_proofs(gpu, vk, sigs, rng, S.Pools(gpu, rng, 16))
        good = np.frombuffer(b"".join(w(v) for s in sigs for v in s), dtype=np.uint8).reshape(distinct, vk.k * 32)
        bad = good.copy()
        bad[:, :32] = np.frombuffer(b"".join(w((s[0] + 1) % R) for s in sigs), dtype=np.uint8).reshape(distinct, 32)
        j = np.arange(per)
        tam = (j % 8) == 3
        pk = np.frombuffer(b"".join(prs), dtype=np.uint8).reshape(distinct, 256)[j % distinct]
        sk = np.where(tam[:, None], bad[j % distinct], good[j % distinct])
        keys.append(vk); kvs.append(Z.VerificationKey(vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic))
        per_key.append((pk, sk, np.where(tam, 4, 0).astype(np.uint8)))
    key_idx = np.repeat(np.arange(K, dtype=np.uint32), per)
    pos = np.concatenate([np.arange(per)] * K)
    order = np.random.default_rng(seed).permutation(len(key_idx))
    key_idx, pos = key_idx[order], pos[order]
    proofs = np.empty((len(key_idx), 256), dtype=np.uint8)
    expect = np.empty(len(key_idx), dtype=np.uint8)
    counts = np.array([keys[k].k for k in key_idx], dtype=np.uint64)
    sig_off = np.zeros(len(key_idx) + 1, dtype=np.uint64); sig_off[1:] = np.cumsum(counts)
    sig = np.empty(int(sig_off[-1]) * 32, dtype=np.uint8)
    for k in range(K):
        sel = np.nonzero(key_idx == k)[0]
        proofs[sel] = per_key[k][0][pos[sel]]
        expect[sel] = per_key[k][2][pos[sel]]
        rows = per_key[k][1][pos[sel]]
        starts = (sig_off[sel] * 32).astype(np.int64)
        idx = starts[:, None] + np.arange(keys[k].k * 32)[None, :]
        sig[idx.ravel()] = rows.ravel()
    P = Z.pinned_copy
    single = [(kvs[k], P(per_key[k][0]), P(per_key[k][1]), keys[k].k, per_key[k][2]) for k in range(K)]
    return dict(kvs=kvs, key_idx=P(key_idx), proofs=P(proofs), sig=P(sig), sig_off=P(sig_off), expect=expect, single=single)


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON-lines output file")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    import stylus_zkvm_verifiers_b200 as Z
    from stylus_zkvm_verifiers_b200 import synth as S
    G = Z.Groth16Verifier
    gpu = Z.GpuBackend(0)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    out = open(args.out, "w")

    def emit(d):
        print(json.dumps(d), flush=True); out.write(json.dumps(d) + "\n"); out.flush()

    emit(dict(gpu_info(), what="device 0 of the run below"))
    for part, K, n, reps in [("a", 1, 1 << 16, args.reps), ("a", 8, 1 << 16, args.reps), ("a", 64, 1 << 16, args.reps), ("b", 1, 1 << 20, 3)]:
        W = workload(Z, S, gpu, K, n, 256, 0x4B5E7000 + K * 7 + n)
        ks = Z.VerificationKeySet(W["kvs"])
        st = np.zeros(n, dtype=np.uint8)

        def set_call():
            G.verify_batch_keys_packed(ks, W["key_idx"], W["proofs"], W["sig"], W["sig_off"], status_out=st)

        def single_calls():
            for kv, pk, sk, k, e in W["single"]:
                got = G.verify_batch(kv, pk, sk, k, len(pk))
                assert got.tobytes() == e.tobytes(), "single-key statuses differ from the expectation"

        set_call(); assert st.tobytes() == W["expect"].tobytes(), "set statuses differ from the expectation"
        single_calls()
        t_set, t_single = [], []
        for _ in range(reps):                          # alternate the two forms
            t_set += timed(set_call, 1); assert st.tobytes() == W["expect"].tobytes()
            t_single += timed(single_calls, 1)
        ms, mk = float(np.median(t_set)), float(np.median(t_single))
        emit({"part": ("a+b" if n == 1 << 16 else "a") if K == 1 and part == "a" else part, "keys": K, "n": n, "set_s": t_set, "per_key_calls_s": t_single,
              "set_verifies_per_s": n / ms, "per_key_calls_verifies_per_s": n / mk, "set_over_per_key": mk / ms,
              "what": "one zkv_groth16_verify_batch_keys call vs %d zkv_groth16_verify_batch calls (median of %d, alternated)" % (K, reps)})
        if K in (1, 64) or n == 1 << 20:                # (c): the same set, inputs already in HBM
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()
            d_k, d_p, d_s, d_o = t(W["key_idx"]), t(W["proofs"]), t(W["sig"]), t(W["sig_off"])
            d_st = torch.empty(n, dtype=torch.uint8, device="cuda")
            s = torch.cuda.current_stream()

            def dev_call():
                G.verify_batch_keys_device(ks, 0, d_k.data_ptr(), d_p.data_ptr(), d_s.data_ptr(), d_o.data_ptr(), n, d_st.data_ptr(), s.cuda_stream)
                torch.cuda.synchronize()

            dev_call(); assert d_st.cpu().numpy().tobytes() == W["expect"].tobytes()
            t_dev = timed(dev_call, reps)
            assert d_st.cpu().numpy().tobytes() == W["expect"].tobytes()
            md = float(np.median(t_dev))
            emit({"part": "c", "keys": K, "n": n, "device_s": t_dev, "device_verifies_per_s": n / md, "end_to_end_verifies_per_s": n / ms,
                  "end_to_end_over_device": md / ms, "what": "set call on host arrays vs its _device form on inputs in HBM (median of %d)" % reps})
        ks.close()
        del W
    out.close()


if __name__ == "__main__":
    main()
