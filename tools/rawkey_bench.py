"""Throughput of Groth16 verification under keys passed as bytes (RawKeyVerifier, zkv_groth16_verify_batch_rawkeys) against the two ways to
get the same statuses without it: (b) zkv_vk_load of the K keys plus one key-set call (K <= 256; the load time reported separately), and
(c) the host composition of the precompile services (ecMul / ecAdd per signal, A negated on the host for RISC Zero keys, one 4-pair ecPairing).
2^16 proofs under K = 1 / 64 / 4096 distinct synthetic keys (RISC Zero- and SP1-shaped, alternating), and 2^20 under one key.  Page-locked
inputs, a warm-up call of each, then medians of alternated calls (a, b, c in turn; c also with its min / max), every status checked (all
proofs are valid).  One JSON line per run.  --kernel-split: GPU time per kernel instead (torch.profiler, a run of its own)."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import stylus_zkvm_verifiers_b200 as Z  # noqa: E402
from stylus_zkvm_verifiers_b200 import synth as S  # noqa: E402

P = S.P


def build(gpu, n, K, seed):
    rng = S.SplitMix64(seed)
    vks = [S.make_vk(gpu, j % 2, 6 if j % 2 == 0 else 3, seed + 1 + j) for j in range(K)]     # RISC Zero: 5 signals, SP1: 2
    pools = S.Pools(gpu, rng, 64)
    key_idx = np.arange(n, dtype=np.uint32) % K
    base_n = min(n, 1 << 16)
    prs, sigs = [None] * base_n, [None] * base_n
    for k, vk in enumerate(vks):
        idx = list(range(k, base_n, K))
        if not idx:
            continue
        s = [[rng.fr() for _ in range(vk.k)] for _ in idx]
        for i, p, sg in zip(idx, S.make_proofs(gpu, vk, s, rng, pools), s):
            prs[i], sigs[i] = p, sg
    reps = n // base_n
    prs, sigs = prs * reps, sigs * reps
    return vks, key_idx, prs, sigs


def pinned(a):
    return Z.pinned_copy(np.ascontiguousarray(a))


def med(ts):
    return statistics.median(ts)


def compose(vks, key_idx, prs, sigs):
    """(c): k rounds of ecMul + ecAdd batches, A negated on the host for RISC Zero keys, one 4-pair ecPairing batch"""
    n = len(prs)
    acc = np.frombuffer(b"".join(vks[k].ic[0] for k in key_idx), dtype=np.uint8).reshape(n, 64).copy()
    kmax = max(v.k for v in vks)
    for j in range(kmax):
        rows = [i for i in range(n) if j < len(sigs[i])]
        if not rows:
            break
        mul_in = b"".join(vks[key_idx[i]].ic[j + 1] + S.w32(sigs[i][j]) for i in rows)
        t, rev = Z.ec_mul_batch(mul_in, len(rows))
        t = np.frombuffer(bytes(t), dtype=np.uint8).reshape(len(rows), 64)
        add_in = np.concatenate([acc[rows], t], axis=1).tobytes()
        a2, rev2 = Z.ec_add_batch(add_in, len(rows))
        acc[rows] = np.frombuffer(bytes(a2), dtype=np.uint8).reshape(len(rows), 64)
    pairs = []
    for i in range(n):
        vk, pr = vks[key_idx[i]], prs[i]
        a = pr[0:64]
        if vk.vm == 0 and a != bytes(64):
            a = a[:32] + S.w32((P - int.from_bytes(a[32:], "big")) % (1 << 256))
        pairs.append(a + pr[64:192] + vk.alpha + vk.beta + acc[i].tobytes() + vk.gamma + pr[192:256] + vk.delta)
    out, rev = Z.ec_pairing_batch(b"".join(pairs), 4, n)
    return np.where((rev == 0) & (out.reshape(n, 32)[:, 31] == 1), 0, 4).astype(np.uint8)


def run(gpu, rv, n, K, reps, seed):
    vks, key_idx, prs, sigs = build(gpu, n, K, seed)
    keys = [(v.vm, v.alpha, v.beta, v.gamma, v.delta, list(v.ic)) for v in vks]
    kb = b"".join(Z.raw_key_bytes(*k[1:]) for k in keys)
    ko = np.zeros(K + 1, dtype=np.uint64); ko[1:] = np.cumsum([448 + 64 * len(k[5]) for k in keys])
    kv = np.array([k[0] for k in keys], dtype=np.uint8)
    so = np.zeros(n + 1, dtype=np.uint64); so[1:] = np.cumsum([len(s) for s in sigs])
    sb = np.frombuffer(b"".join(S.w32(v) for s in sigs for v in s), dtype=np.uint8)
    pr = np.frombuffer(b"".join(prs), dtype=np.uint8)
    args = [pinned(np.frombuffer(kb, dtype=np.uint8)), pinned(ko), pinned(kv), pinned(key_idx), pinned(pr), pinned(sb), pinned(so)]
    st = pinned(np.zeros(n, dtype=np.uint8))
    rec = {"n": n, "keys": K, "device": gpu_name()}
    ta, tb = [], []
    ks = None
    if K <= 256:
        t0 = time.perf_counter()
        kvs = [Z.VerificationKey(v.vm, v.alpha, v.beta, v.gamma, v.delta, v.ic) for v in vks]
        rec["b_vk_load_ms"] = (time.perf_counter() - t0) * 1e3
        ks = Z.VerificationKeySet(kvs)
    # warm-up of all three (every status checked), then `reps` rounds of a, b, c in turn
    rv.verify_batch_packed(*args, status_out=st); assert (st == 0).all(), "rawkeys: %d rejected" % int((st != 0).sum())
    if ks is not None:
        st2 = Z.Groth16Verifier.verify_batch_keys_packed(ks, args[3], args[4], args[5], args[6])
        assert (st2 == 0).all()
    sc = compose(vks, key_idx, prs, sigs); assert (sc == 0).all(), "composition: %d rejected" % int((sc != 0).sum())
    tc = []
    for _ in range(reps):
        t0 = time.perf_counter(); rv.verify_batch_packed(*args, status_out=st); ta.append(time.perf_counter() - t0)
        assert (st == 0).all()
        if ks is not None:
            t0 = time.perf_counter(); st2 = Z.Groth16Verifier.verify_batch_keys_packed(ks, args[3], args[4], args[5], args[6]); tb.append(time.perf_counter() - t0)
            assert (st2 == 0).all()
        t0 = time.perf_counter(); sc = compose(vks, key_idx, prs, sigs); tc.append(time.perf_counter() - t0)
        assert (sc == 0).all()
    rec["a_rawkeys_ms"] = med(ta) * 1e3
    rec["a_rawkeys_verifies_per_s"] = n / med(ta)
    if tb:
        rec["b_keyset_ms"] = med(tb) * 1e3
        rec["b_keyset_verifies_per_s"] = n / med(tb)
        rec["a_over_b_rate"] = med(tb) / med(ta)
        rec["b_with_load_ms"] = rec["b_keyset_ms"] + rec["b_vk_load_ms"]
    rec["c_compose_ms"] = med(tc) * 1e3
    rec["c_compose_ms_range"] = [min(tc) * 1e3, max(tc) * 1e3]
    rec["a_over_c_speedup"] = rec["c_compose_ms"] / rec["a_rawkeys_ms"]
    return rec


def kernel_split(gpu, rv, n, K, seed):
    """GPU time per kernel of one raw-key call and one key-set call (torch.profiler, CUDA activities), summed by kernel name over the call's
    streams: where the raw-key path spends its time against the loaded-key path.  A run of its own: tracing slows the host."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    vks, key_idx, prs, sigs = build(gpu, n, K, seed)
    keys = [(v.vm, v.alpha, v.beta, v.gamma, v.delta, list(v.ic)) for v in vks]
    kb = b"".join(Z.raw_key_bytes(*k[1:]) for k in keys)
    ko = np.zeros(K + 1, dtype=np.uint64); ko[1:] = np.cumsum([448 + 64 * len(k[5]) for k in keys])
    kv = np.array([k[0] for k in keys], dtype=np.uint8)
    so = np.zeros(n + 1, dtype=np.uint64); so[1:] = np.cumsum([len(s) for s in sigs])
    sb = np.frombuffer(b"".join(S.w32(v) for s in sigs for v in s), dtype=np.uint8)
    pr = np.frombuffer(b"".join(prs), dtype=np.uint8)
    ks = Z.VerificationKeySet([Z.VerificationKey(v.vm, v.alpha, v.beta, v.gamma, v.delta, v.ic) for v in vks])
    out = {"n": n, "keys": K, "device": gpu_name()}
    for name, call in (("rawkeys", lambda: rv.verify_batch_packed(kb, ko, kv, key_idx, pr, sb, so)),
                       ("keyset", lambda: Z.Groth16Verifier.verify_batch_keys_packed(ks, key_idx, pr, sb, so))):
        assert (call() == 0).all()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            assert (call() == 0).all()
            torch.cuda.synchronize()
        per, other = {}, set()
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            m = re.match(r"_ZN3zkv(\d+)", e.name)              # mangled zkv::<kernel>: the name's length, then the name
            d = re.search(r"zkv::(\w+)\(", e.name) or re.match(r"(\w+)\(", e.name)   # demangled
            kname = e.name[m.end():m.end() + int(m.group(1))] if m else d.group(1) if d else None
            if kname is None:
                other.add(e.name[:60])
                continue
            per[kname] = per.get(kname, 0.0) + e.device_time_total / 1e3
        out[name + "_kernel_ms"] = {k: round(v, 3) for k, v in sorted(per.items(), key=lambda x: -x[1])}
        out[name + "_other_events"] = sorted(other)[:10]
    return out


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_rawkey_bench.jsonl"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="2^12 proofs per run (smoke)")
    ap.add_argument("--kernel-split", metavar="FILE", help="instead: GPU time per kernel of one raw-key and one key-set call (2^16, 64 keys) to FILE")
    a = ap.parse_args()
    gpu = Z.GpuBackend(0)
    rv = Z.RawKeyVerifier()
    if a.kernel_split:
        rec = kernel_split(gpu, rv, 1 << 16, 64, 0x7A0040)
        print(json.dumps(rec), flush=True)
        with open(a.kernel_split, "w") as f:
            f.write(json.dumps(rec) + "\n")
        return
    runs = [(1 << 16, 1), (1 << 16, 64), (1 << 16, 4096), (1 << 20, 1)]
    if a.small:
        runs = [(1 << 12, 1), (1 << 12, 64)]
    with open(a.out, "w") as f:
        for n, K in runs:
            rec = run(gpu, rv, n, K, a.reps if n <= (1 << 16) else 3, 0x7A0000 + K)
            print(json.dumps(rec), flush=True)
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
