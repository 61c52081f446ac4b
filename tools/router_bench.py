"""Throughput of the routers (zkv_risc0_router_*, zkv_sp1_gateway_*) against one batch call per route handle, on device 0.

  (a) 2^16 RISC Zero-shape seals spread evenly over K in {1, 4, 16} routes: one router call against K handle calls.  Odd routes are
      distinct control roots on the embedded key (their seals come from a synthetic key of the same shape, so every one of them runs the
      whole verification and fails), even routes synthetic keys with their own control roots;
  (b) one route at 2^16 and 2^20: the router call against zkv_risc0_verify_batch (what routing, grouping and padding cost);
  (c) the SP1 gateway at K in {1, 4} over the embedded v5 handle and zkv_sp1_create_version handles of synthetic keys, 2^16 proofs;
  (d) the router's end-to-end rate (host arrays) over its device-resident rate (the _device form on inputs already in HBM).

Host clock around calls that end synchronised; host inputs in page-locked memory (pinned_copy), so every entry point uploads them in place.
Every status of every router call is compared with the per-handle calls' statuses (one seal in eight of a synthetic route carries a
tampered journal or public value).  The two forms are alternated call by call and the median of --reps is reported.  One JSON line per
measurement; the first names the GPU and its power limit, read in the same run.

    python tools/router_bench.py --out profiles/r3_router_bench.jsonl
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


def gpu_info():
    import torch
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                  # noqa: BLE001 - reported, not hidden
        pl = "unavailable (%s)" % e
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": pl}


def _tile(rows, per, distinct):
    return np.ascontiguousarray(rows[np.arange(per) % distinct])


def risc0_workload(Z, S, gpu, sys0, K, n, distinct, seed):
    """n seals over K routes (n / K each, tiled from `distinct` generated seals per route), caller order a seeded random interleaving"""
    rng = S.SplitMix64(seed)
    per = n // K
    embedded = Z.VerificationKey.risc0()
    cid = S.w32(rng.fr())
    handles, per_route = [], []
    for k in range(K):
        gen = S.make_vk(gpu, 0, 6, seed + 1 + k)
        kv = embedded if k % 2 else Z.VerificationKey(0, gen.alpha, gen.beta, gen.gamma, gen.delta, gen.ic)
        h = Z.RiscZeroVerifier(kv)
        cr = rng.bytes(32)
        h.initialize(cr, cid)
        b = S.make_risc0_batch(gpu, gen, h.get_selector(), cr, cid, sys0, distinct, seed + 100 + k, pool=min(distinct, 64))
        seals = _tile(np.frombuffer(b"".join(b.seals), dtype=np.uint8).reshape(distinct, 260), per, distinct)
        ims = _tile(np.frombuffer(b"".join(b.image_ids), dtype=np.uint8).reshape(distinct, 32), per, distinct)
        jrs = _tile(np.frombuffer(b"".join(b.journals), dtype=np.uint8).reshape(distinct, 32), per, distinct)
        jrs[3::8] = 0                                             # one in eight: another journal
        handles.append((h, kv))
        per_route.append((seals, ims, jrs))
    which = np.repeat(np.arange(K), per)
    pos = np.concatenate([np.arange(per)] * K)
    order = np.random.default_rng(seed).permutation(len(which))
    which, pos = which[order], pos[order]
    seals = np.empty((len(which), 260), dtype=np.uint8); ims = np.empty((len(which), 32), dtype=np.uint8); jrs = np.empty_like(ims)
    for k in range(K):
        sel = np.nonzero(which == k)[0]
        seals[sel], ims[sel], jrs[sel] = per_route[k][0][pos[sel]], per_route[k][1][pos[sel]], per_route[k][2][pos[sel]]
    P = Z.pinned_copy
    off = np.arange(len(which) + 1, dtype=np.uint64) * 260
    single = [(h, P(s), P(np.arange(per + 1, dtype=np.uint64) * 260), P(a), P(j)) for (h, _), (s, a, j) in zip(handles, per_route)]
    return dict(handles=handles, which=which, pos=pos, seals=P(seals), off=P(off), ims=P(ims), jrs=P(jrs), single=single)


def sp1_workload(Z, S, gpu, fx_proof, fx_vkey, fx_pv, K, n, distinct, seed):
    """n proofs over K gateway routes: route 0 the embedded v5 handle (the reference's proof, one in eight with another vkey), the others
    zkv_sp1_create_version handles of synthetic keys; public values of the reference proof's length throughout"""
    per = n // K
    handles, per_route = [], []
    for k in range(K):
        if k == 0:
            h = Z.Sp1Verifier(); kv = None
            pr = np.frombuffer(fx_proof, dtype=np.uint8)[None, :].repeat(distinct, 0)
            vkeys = np.frombuffer(fx_vkey, dtype=np.uint8)[None, :].repeat(distinct, 0)
            pvs = np.frombuffer(fx_pv, dtype=np.uint8)[None, :].repeat(distinct, 0)
        else:
            gen = S.make_vk(gpu, 1, 3, seed + 1 + k)
            kv = Z.VerificationKey(1, gen.alpha, gen.beta, gen.gamma, gen.delta, gen.ic)
            h = Z.Sp1Verifier(kv, verifier_hash=bytes([k]) * 32, version="bench-%d" % k)
            b = S.make_sp1_batch(gpu, gen, distinct, seed + 100 + k, pv_len=len(fx_pv), pool=min(distinct, 64), selector=h.verifier_hash()[:4])
            pr = np.frombuffer(b"".join(b.proofs), dtype=np.uint8).reshape(distinct, 260)
            vkeys = np.frombuffer(b"".join(b.vkeys), dtype=np.uint8).reshape(distinct, 32)
            pvs = np.frombuffer(b"".join(b.public_values), dtype=np.uint8).reshape(distinct, len(fx_pv))
        pr, vkeys, pvs = _tile(pr, per, distinct), _tile(vkeys, per, distinct), _tile(pvs, per, distinct)
        vkeys[3::8, 31] ^= 1                                      # one in eight: another program key
        handles.append((h, kv))
        per_route.append((pr, vkeys, pvs))
    which = np.repeat(np.arange(K), per)
    pos = np.concatenate([np.arange(per)] * K)
    order = np.random.default_rng(seed).permutation(len(which))
    which, pos = which[order], pos[order]
    L = len(fx_pv)
    pr = np.empty((len(which), 260), dtype=np.uint8); vk = np.empty((len(which), 32), dtype=np.uint8); pv = np.empty((len(which), L), dtype=np.uint8)
    for k in range(K):
        sel = np.nonzero(which == k)[0]
        pr[sel], vk[sel], pv[sel] = per_route[k][0][pos[sel]], per_route[k][1][pos[sel]], per_route[k][2][pos[sel]]
    P = Z.pinned_copy
    offs = lambda m, w: P(np.arange(m + 1, dtype=np.uint64) * w)
    single = [(h, P(v), P(p), offs(per, L), P(q), offs(per, 260)) for (h, _), (q, v, p) in zip(handles, per_route)]
    return dict(handles=handles, which=which, pos=pos, proofs=P(pr), vkeys=P(vk), pvs=P(pv), pv_off=offs(len(which), L), proof_off=offs(len(which), 260), single=single, L=L)


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return ts


def alternate(a, b, reps):
    ta, tb = [], []
    for _ in range(reps):
        ta += timed(a, 1); tb += timed(b, 1)
    return ta, tb


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON-lines output file")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    import stylus_zkvm_verifiers_b200 as Z
    from stylus_zkvm_verifiers_b200 import synth as S
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    c = O.constants()
    h = bytes.fromhex
    sys0 = h(c["risc0_system_state_zero_digest"])
    fx = c["sp1_fixture"]
    gpu = Z.GpuBackend(0)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    out = open(args.out, "w")

    def emit(d):
        print(json.dumps(d), flush=True); out.write(json.dumps(d) + "\n"); out.flush()

    emit(dict(gpu_info(), what="device 0 of the run below"))
    for part, K, n, reps in [("a+b", 1, 1 << 16, args.reps), ("a", 4, 1 << 16, args.reps), ("a", 16, 1 << 16, args.reps), ("b", 1, 1 << 20, 3)]:
        W = risc0_workload(Z, S, gpu, sys0, K, n, 256, 0x52700000 + K * 7 + n)
        rt = Z.RiscZeroVerifierRouter([hh for hh, _ in W["handles"]])
        st = np.zeros(n, dtype=np.uint8)

        def router_call():
            rt.verify_batch_packed(W["seals"], W["off"], W["ims"], W["jrs"], n, status_out=st)

        singles = []

        def handle_calls():
            singles.clear()
            for hh, s, o, a, j in W["single"]:
                singles.append(hh.verify_batch_packed(s, o, a, j, len(a)))

        handle_calls(); router_call()
        assert same_as_handles(W, st, singles), "router statuses differ from the handle calls"
        t_r, t_h = alternate(router_call, handle_calls, reps)
        assert same_as_handles(W, st, singles)
        mr, mh = float(np.median(t_r)), float(np.median(t_h))
        emit({"part": part, "shape": "risc0", "routes": K, "n": n, "router_s": t_r, "per_handle_calls_s": t_h, "router_verifies_per_s": n / mr,
              "per_handle_calls_verifies_per_s": n / mh, "router_over_per_handle": mh / mr, "accepted": int((st == 0).sum()),
              "what": "one zkv_risc0_router_verify_batch call vs %d zkv_risc0_verify_batch calls (median of %d, alternated)" % (K, reps)})
        if K in (1, 16) and n == 1 << 16:                         # (d): the same router, inputs already in HBM
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()
            d_s, d_a, d_b = t(W["seals"]), t(W["ims"]), t(W["jrs"])
            d_st = torch.empty(n, dtype=torch.uint8, device="cuda")
            s = torch.cuda.current_stream()

            def dev_call():
                rt.verify_batch_device(0, d_s.data_ptr(), d_a.data_ptr(), d_b.data_ptr(), n, d_st.data_ptr(), s.cuda_stream)
                torch.cuda.synchronize()

            dev_call(); assert d_st.cpu().numpy().tobytes() == st.tobytes()
            t_d, t_r2 = alternate(dev_call, router_call, reps)
            assert d_st.cpu().numpy().tobytes() == st.tobytes()
            md, mr2 = float(np.median(t_d)), float(np.median(t_r2))
            emit({"part": "d", "shape": "risc0", "routes": K, "n": n, "device_s": t_d, "router_s": t_r2, "device_verifies_per_s": n / md,
                  "end_to_end_verifies_per_s": n / mr2, "end_to_end_over_device": md / mr2,
                  "what": "router call on host arrays vs its _device form on inputs in HBM (median of %d, alternated)" % reps})
        rt.close()
        del W
    for K in (1, 4):
        n = 1 << 16
        W = sp1_workload(Z, S, gpu, h(fx["proof"]), h(fx["vkey"]), h(fx["public_values"]), K, n, 256, 0x5B100000 + K)
        gw = Z.Sp1VerifierGateway([hh for hh, _ in W["handles"]])
        st = np.zeros(n, dtype=np.uint8)
        singles = []

        def gw_call():
            gw.verify_batch_packed(W["vkeys"], W["pvs"], W["pv_off"], W["proofs"], W["proof_off"], n, status_out=st)

        def handle_calls_sp1():
            singles.clear()
            for hh, v, p, po, q, qo in W["single"]:
                singles.append(hh.verify_batch_packed(v, p, po, q, qo, len(v)))

        gw_call(); handle_calls_sp1()
        assert same_as_handles(W, st, singles), "gateway statuses differ from the handle calls"
        t_g, t_h = alternate(gw_call, handle_calls_sp1, args.reps)
        assert same_as_handles(W, st, singles)
        mg, mh = float(np.median(t_g)), float(np.median(t_h))
        emit({"part": "c", "shape": "sp1", "routes": K, "n": n, "gateway_s": t_g, "per_handle_calls_s": t_h, "gateway_verifies_per_s": n / mg,
              "per_handle_calls_verifies_per_s": n / mh, "gateway_over_per_handle": mh / mg, "accepted": int((st == 0).sum()),
              "what": "one zkv_sp1_gateway_verify_batch call vs %d zkv_sp1_verify_batch calls (median of %d, alternated)" % (K, args.reps)})
        gw.close()
        del W
    out.close()


def same_as_handles(W, st, singles):
    """caller record i is row pos[i] of route which[i]'s arrays, i.e. record pos[i] of that route handle's own call"""
    want = np.empty_like(st)
    for k, got in enumerate(singles):
        sel = W["which"] == k
        want[sel] = got[W["pos"][sel]]
    return st.tobytes() == want.tobytes()


if __name__ == "__main__":
    main()
