#!/usr/bin/env python3
"""Headline benchmark: Groth16 verifies/sec on synthetic RISC Zero-shape proofs (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N ...            # the CPU restatement of the reference path (oracle port)

One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE); proofs are independent, so ranks shard by
contiguous proof ranges with no data-path collective ("weak" scaling: 2^16 proofs per GPU per step).  A step is one
pass of the whole verification path over one batch.  `value` is measured with the batch resident in HBM (CUDA events
on the launching stream, L2 flushed between steps); `e2e` goes through the reference-facing C-ABI batch call with HOST
buffers, host<->device copies inside the timed region.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

M_MAC32 = 136                      # one 8-limb Montgomery multiplication = 64 + 8 + 64 MAC32 (SURVEY.md 8d)
# Fp-multiplication counts per proof (DESIGN.md section 5).  The verify path runs a 3-pair Miller loop (A/B variable, vk_x/gamma and
# C/delta from line tables) times the per-key constant Miller(alpha, beta); the pairing service (config 5) runs all 4 pairs.
W_MILLER3_M = 65 * (36 + 20 + 3 * 43) + 21 * (37 + 3 * 43) + 2 * (37 + 3 * 43) + 54
W_MILLER4_M = 65 * (36 + 20 + 4 * 43) + 21 * (37 + 4 * 43) + 2 * (37 + 4 * 43)
W_FINALEXP_M = 8410
W_RISC0_M = W_MILLER3_M + W_FINALEXP_M + 1800 + 40 + 1000
W_SP1_M = W_MILLER3_M + W_FINALEXP_M + 1800 + 40 + 1700
DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs: at most this much in all, .npy headers included


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array (all of one length n) as out_dir/<name>.npy in float32, so that two builds can be compared output for
    output.  Past DUMP_BYTES in all, every array keeps the same fixed, seeded sample of indices, written as sample_index.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    per = 4 * len(arrays)
    index_path = os.path.join(out_dir, "sample_index.npy")
    if n * per + 4096 > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(n, (DUMP_BYTES - 4096) // (per + 8), replace=False))
        np.save(index_path, idx.astype(np.float64))
        arrays = {k: a[idx] for k, a in arrays.items()}
    elif os.path.exists(index_path):
        os.remove(index_path)          # left by an earlier, sampled dump into the same directory
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.asarray(a, dtype=np.float32))


def ncu_summary(kernel):
    """The committed ncu --set full summary of one launch of `kernel` at this workload (profiles/r2_ncu_summary.json for the shared-memory
    kernels, profiles/r1_ncu_summary.json for the round-1 kernels): DRAM traffic per launch, EXECUTED IMAD.WIDE per proof and the pipe
    counters.  None if absent."""
    for name in ("r2_ncu_summary.json", "r1_ncu_summary.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            for k in d["kernels"]:
                if k["kernel"] == kernel and "source_page" in k:
                    sp = k["source_page"]
                    per_proof = sp.get("executed_imad_wide_per_proof") or round(sp["executed_warp_instructions"] * sp["opcode_share"].get("IMAD.WIDE", 0) * 32 / k["proofs"])
                    return {"traffic": {"bytes_per_launch": k["dram_bytes_read"] + k["dram_bytes_write"], "proofs_per_launch": k["proofs"], "source": "profiles/" + name},
                            "executed_imad_wide_per_proof": per_proof,
                            "ncu_fmaheavy_pct": k.get("sm__pipe_fmaheavy_cycles_active.avg.pct_of_peak_sustained_active [%]"),
                            "ncu_executed_imad_wide_frac": sp.get("executed_imad_wide_frac_of_issue_peak")}
        except Exception:
            pass
    return None


def workload_config(shape, n):
    """`config` of the JSON line: the workload only, shared verbatim by this repo's arm and the --impl reference arm"""
    return {"workload": "%s: 2^%d synthetic %s-shape Groth16 proofs per GPU per step (%d public inputs, fixed random vk, trapdoor-simulated; a seeded half "
                        "carries one flipped bit of its %s and is rejected after the full verification path)" %
            ("configs[1]" if shape == "risc0" else "configs[2] shape", n.bit_length() - 1, "RISC Zero" if shape == "risc0" else "SP1 v5", 5 if shape == "risc0" else 2,
             "journal digest" if shape == "risc0" else "public values"),
            "proofs_per_gpu": n, "sharding": "contiguous proof ranges, no collective"}


def tamper_half(S, batch, shape, seed):
    """Flips one bit of the journal digest (RISC Zero) or of the public values (SP1) of a fixed, seeded half of the proofs, in place, and
    sets their expected status to VerificationFailed.  Such a proof changes only a hashed public input: it runs the whole verification
    path at the cost of a valid one (decode, hashing, vk_x, G2 check, Miller loop, final exponentiation) and is rejected by the final
    comparison, so the per-proof statuses depend on every stage of the computation."""
    import numpy as np
    field = batch.journals if shape == "risc0" else batch.public_values
    for i in np.flatnonzero(np.random.default_rng(seed).random(len(field)) < 0.5):
        b = bytearray(field[i]); b[-1] ^= 1; field[i] = bytes(b)
        batch.expect[i] = S.ST_VERIFICATION_FAILED


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.15)

    def __enter__(self):
        self.th.start(); return self

    def __exit__(self, *a):
        self.stop.set(); self.th.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(self.rows)}


def make_workload(Z, S, consts, device, n, shape, seed):
    """Synthetic proofs for one rank, generated with the library's own GPU ecMul / G2 services (no oracle)."""
    h = bytes.fromhex
    gpu = Z.GpuBackend(device)
    r = consts["risc0_fixture"]
    if shape == "risc0":
        vk = S.make_vk(gpu, 0, 6, 0xB2000001)
        kv = Z.VerificationKey(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, devices=[device])
        v = Z.RiscZeroVerifier(kv, devices=[device])
        v.initialize(h(r["control_root"]), h(r["bn254_control_id"]))
        b = S.make_risc0_batch(gpu, vk, v.get_selector(), h(r["control_root"]), h(r["bn254_control_id"]), h(consts["risc0_system_state_zero_digest"]), n, seed, pool=4096)
    else:
        vk = S.make_vk(gpu, 1, 3, 0xB2000003)
        kv = Z.VerificationKey(1, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic, devices=[device])
        v = Z.Sp1Verifier(kv, devices=[device])
        b = S.make_sp1_batch(gpu, vk, n, seed, pool=4096)
    tamper_half(S, b, shape, seed)
    return v, kv, vk, b


def cpu_baseline(O, shape, vk, batch, consts, target_s=12.0):
    """The oracle port of the reference path under OpenMP on all host cores, on a bounded prefix of the same batch."""
    import numpy as np
    h = bytes.fromhex
    cores = O.max_threads()
    ovk = O.Vk(vk.vm, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic)
    if shape == "risc0":
        ro = O.Risc0Oracle(ovk); ro.initialize(h(consts["risc0_fixture"]["control_root"]), h(consts["risc0_fixture"]["bn254_control_id"]))
        run = lambda m: ro.verify_batch(batch.seals[:m], batch.image_ids[:m], batch.journals[:m])
    else:
        run = lambda m: O.sp1_verify_batch(ovk, h(consts["sp1_verifier_hash"])[:4], batch.vkeys[:m], batch.public_values[:m], batch.proofs[:m])
    m0 = min(len(batch.expect), 4 * cores)
    t0 = time.perf_counter(); st = run(m0); t1 = time.perf_counter()
    rate0 = m0 / (t1 - t0)
    m = int(min(len(batch.expect), max(m0, rate0 * target_s)))
    t0 = time.perf_counter(); st = run(m); t1 = time.perf_counter()
    assert np.asarray(st).tolist() == batch.expect[:m], "oracle status differs from the synthetic batch's expectation"
    return {"value": m / (t1 - t0), "unit": "verifies/s", "cores": cores, "kind": "port",
            "sample": "first %d proofs of the same batch, oracle/zkv_oracle.c under OpenMP schedule(dynamic), %.1f s" % (m, t1 - t0)}, st


def run_reference(args, rank, world):
    """--impl reference: the reference path's CPU restatement (oracle port; the Rust reference cannot be built here), all host threads."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers; this arm is the CPU implementation on ALL host threads, and libgomp reads the
    # variable when the oracle library is loaded
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle_lib as O
    from stylus_zkvm_verifiers_b200 import synth as S
    consts = O.constants()
    h = bytes.fromhex

    class OB:
        def g1_mul(self, sc): return [O.g1_mul(S.G1_GEN, s) for s in sc]
        def g2_mul(self, sc): return [O.g2_mul(S.G2_GEN, s) for s in sc]
    cores = O.max_threads()
    vk = S.make_vk(OB(), 0, 6, 0xB2000001)
    ro = O.Risc0Oracle(O.Vk(0, vk.alpha, vk.beta, vk.gamma, vk.delta, vk.ic))
    r = consts["risc0_fixture"]
    ro.initialize(h(r["control_root"]), h(r["bn254_control_id"]))
    m = 4096                            # bounded sample per step: the first 4096 proofs of the same seeded workload (about 1 s on 16 threads)
    b = S.make_risc0_batch(OB(), vk, ro.selector(), h(r["control_root"]), h(r["bn254_control_id"]), h(consts["risc0_system_state_zero_digest"]), m, 0xB2000001, pool=256)
    tamper_half(S, b, "risc0", 0xB2000001)
    for _ in range(args.warmup):
        ro.verify_batch(b.seals, b.image_ids, b.journals)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st = ro.verify_batch(b.seals, b.image_ids, b.journals)
    dt = time.perf_counter() - t0
    assert np.asarray(st).tolist() == b.expect
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"status": np.asarray(st)})
    val = m * args.steps / dt
    line = {"impl": "reference", "metric": "groth16_verifies_per_sec", "value": val, "unit": "verifies/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u256 (4x64-bit Montgomery)",
            "data": "synthetic", "config": workload_config("risc0", args.n),
            "cpu_baseline": {"value": val, "unit": "verifies/s", "cores": cores, "kind": "port",
                             "sample": "each step = a bounded sample of %d proofs of the configured workload (same key seed, same generator), %d steps; oracle/zkv_oracle.c (C restatement of the "
                                       "reference path; the Rust reference cannot be built here) under OpenMP on all %d host threads" % (m, args.steps, cores)},
            "e2e": {"value": val, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="risc0", choices=["risc0", "sp1"])
    ap.add_argument("--n", type=int, default=1 << 16, help="proofs per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exact-lines", action="store_true", help="verification path with the unscaled gamma / delta lines (A/B measurement)")
    ap.add_argument("--fe-stages", type=int, default=-1, help="staged final exponentiation for chunked batches: 1 on, 0 off (-1 = library default)")
    ap.add_argument("--segments", type=int, default=0, help="Miller loop segments per chunk (0 = library default)")
    ap.add_argument("--chunks", type=int, default=0, help="stream-overlap chunks per device batch (0 = library default)")
    ap.add_argument("--layout", type=int, default=-1, help="1 = shared-memory-resident lazily reduced kernels (default), 0 = the round-1 thread-stack kernels (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the per-proof status bytes of the last step as DIR/<name>.npy "
                                                          "(float32; status = device-resident path, e2e_status = host-buffer path; rank 0 only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, local_rank, world = dist_env()
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import numpy as np
    import torch
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    import stylus_zkvm_verifiers_b200 as Z
    from stylus_zkvm_verifiers_b200 import synth as S
    consts = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_constants.json")))
    dev = local_rank
    torch.cuda.set_device(dev)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    n = args.n
    v, kv, vk, batch = make_workload(Z, S, consts, dev, n, args.shape, 0xB2000001 + 7919 * rank)

    # ---- device-resident inputs
    t8 = lambda blobs: torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()
    if args.shape == "risc0":
        d_a, d_b, d_c = t8(batch.seals), t8(batch.image_ids), t8(batch.journals)
        launch = lambda st, stream, m=n: v.verify_batch_device(dev, d_a.data_ptr(), d_b.data_ptr(), d_c.data_ptr(), m, st.data_ptr(), stream)
        # e2e inputs live in page-locked host memory (the contract's "pinned host memory"): the library uploads such arrays in place
        h_blob = Z.pinned_copy(np.frombuffer(b"".join(batch.seals), dtype=np.uint8)); h_off = Z.pinned_copy(np.arange(n + 1, dtype=np.uint64) * 260)
        h_b = Z.pinned_copy(np.frombuffer(b"".join(batch.image_ids), dtype=np.uint8)); h_c = Z.pinned_copy(np.frombuffer(b"".join(batch.journals), dtype=np.uint8))
        e2e_call = lambda out: v.verify_batch_packed(h_blob, h_off, h_b, h_c, n, out)
        h2d = h_blob.nbytes + h_off.nbytes + h_b.nbytes + h_c.nbytes      # seals (260 B each), their offsets, image ids, journal digests
        W_M = W_RISC0_M
    else:
        d_a, d_b, d_c = t8(batch.proofs), t8(batch.vkeys), t8(batch.public_values)
        launch = lambda st, stream, m=n: v.verify_batch_device(dev, d_b.data_ptr(), d_c.data_ptr(), 96, d_a.data_ptr(), m, st.data_ptr(), stream)
        h_blob = Z.pinned_copy(np.frombuffer(b"".join(batch.proofs), dtype=np.uint8)); h_off = Z.pinned_copy(np.arange(n + 1, dtype=np.uint64) * 260)
        h_b = Z.pinned_copy(np.frombuffer(b"".join(batch.vkeys), dtype=np.uint8)); h_c = Z.pinned_copy(np.frombuffer(b"".join(batch.public_values), dtype=np.uint8))
        h_voff = Z.pinned_copy(np.arange(n + 1, dtype=np.uint64) * 96)
        e2e_call = lambda out: v.verify_batch_packed(h_b, h_c, h_voff, h_blob, h_off, n, out)
        h2d = h_blob.nbytes + h_off.nbytes + h_b.nbytes + h_c.nbytes + h_voff.nbytes
        W_M = W_SP1_M
    d_st = torch.full((n,), 255, dtype=torch.uint8, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")          # > 126 MB L2
    stream = torch.cuda.Stream()                 # a real (non-null) stream: the library enqueues its kernels on the stream it is given
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    assert sp != 0

    def barrier():
        torch.cuda.synchronize()
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    if args.exact_lines:
        v.tune("normalised_lines", 0)
    if args.fe_stages >= 0:
        v.tune("final_exp_stages", args.fe_stages)
    if args.segments:
        v.tune("miller_segments", args.segments)
    if args.chunks:
        v.tune("overlap", args.chunks)
    if args.layout >= 0:
        v.tune("layout", args.layout)
    chunks, layout = v.tune("overlap"), v.tune("layout")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    n_chunks = chunks if chunks else (1 if n < sms * 128 else 4)      # automatic policy of csrc/zkv.cu chunk_count
    for _ in range(max(args.warmup, 3)):
        launch(d_st, sp)
    torch.cuda.synchronize()
    expect = torch.tensor(batch.expect, dtype=torch.uint8, device="cuda")
    assert bool((d_st == expect).all()), "a status differs from the synthetic batch's expectation"
    imad_peak, fpmul_peak = Z.imad_peak(dev)

    # per-kernel durations for the roofline: one chain on one stream (no overlap between chunks), CUDA events around every stage
    stage_sum, stage_reps = {}, 3
    v.tune("overlap", 1)
    launch(d_st, sp); torch.cuda.synchronize()
    for k in range(stage_reps):
        flush_ = torch.empty(256 << 20, dtype=torch.uint8, device="cuda").fill_(k); del flush_
        launch(d_st, sp); torch.cuda.synchronize()
        for name, ms in v.stage_ms(dev).items():
            stage_sum[name] = stage_sum.get(name, 0.0) + ms / stage_reps
    # roofline launches: a whole number of waves of the kernel in question (prefix of the same batch), so that the figure is the kernel's
    # rate and not the batch's tail: a serial chain over all n proofs pays for a full last wave whatever its fill
    def whole_waves(kernel):
        w = Z.wave_proofs(dev, kernel)
        return (n // w) * w if n >= w else n
    wave_ms, wave_n = {}, {}
    for name, kernel in (("miller", 0 if layout else 2), ("final_exp", 1 if layout else 3)):
        m = whole_waves(kernel); wave_n[name] = m; acc = 0.0
        launch(d_st, sp, m); torch.cuda.synchronize()
        for k in range(stage_reps):
            flush_ = torch.empty(256 << 20, dtype=torch.uint8, device="cuda").fill_(k); del flush_
            launch(d_st, sp, m); torch.cuda.synchronize()
            acc += v.stage_ms(dev)[name] / stage_reps
        wave_ms[name] = acc
    v.tune("overlap", chunks)
    launch(d_st, sp); torch.cuda.synchronize()

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    launches0 = Z.launch_count()
    with ClockSampler(dev) as clocks:
        for k in range(args.steps):
            flush.fill_(k)                                    # evict L2 between timed steps (not timed)
            d_st.fill_(255)                                   # each step must write every status itself (not timed)
            ev[k][0].record(stream)
            launch(d_st, sp)
            ev[k][1].record(stream)
            ev[k][1].synchronize()
        barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = Z.launch_count() - launches0          # counted by the library at its launch sites (all chunks, Miller segments, final-exp stages)
    assert bool((d_st == expect).all())

    # ---- end to end through the C-ABI with host buffers
    out = np.zeros(n, dtype=np.uint8)
    for _ in range(2):
        e2e_call(out)
    barrier()
    out.fill(255)                                     # the timed calls must write every status themselves
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_call(out)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert out.tolist() == batch.expect
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"status": d_st.cpu().numpy(), "e2e_status": out})

    t = torch.tensor([dev_ms, e2e_s], dtype=torch.float64, device="cuda")
    if use_dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s = float(t[0].item()), float(t[1].item())
    total = n * world * args.steps
    value = total / (dev_ms * 1e-3)
    miller_ms, miller_n = wave_ms["miller"], wave_n["miller"]
    fe_ms, fe_n = wave_ms["final_exp"], wave_n["final_exp"]
    mac_miller = miller_n * W_MILLER3_M * M_MAC32
    serial_miller_ms = stage_sum.get("miller", 0.0)
    miller_kernel = "k_miller" if args.exact_lines else ("k_miller_lz" if layout else "k_miller_norm")    # verification path: normalised gamma / delta lines by default
    ncu = ncu_summary(miller_kernel) or {}
    ncu_fe = ncu_summary("k_final_exp_lz" if layout else "k_final_exp") or {}
    exec_pp, exec_fe_pp = ncu.get("executed_imad_wide_per_proof"), ncu_fe.get("executed_imad_wide_per_proof")
    line = {
        "metric": "groth16_verifies_per_sec", "value": value, "unit": "verifies/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u256 (8x32-bit Montgomery limbs, IMAD.WIDE.U32)", "data": "synthetic",
        "config": workload_config(args.shape, n),
        "execution": {"l2": "flushed between timed steps (256 MiB fill)", "layout": "shared-memory-resident lazily reduced kernels" if layout else "round-1 thread-stack kernels",
                      "overlap": "%d chunks per device batch on side streams%s (stage_ms: serial single-chain pass over all proofs; roofline: serial single-chain launches of a whole number of waves)" % (n_chunks, "" if chunks else " (automatic; front kernels first, then per chunk 4 Miller segment + 4 final-exponentiation stage kernels)")},
        "e2e": {"value": total / e2e_s, "unit": "verifies/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": n},
        "gpu_launches": launches,
        "stage_ms": stage_sum,
        "roofline": {"bound": "imad", "bound_note": "integer-multiply (IMAD.WIDE) issue rate; neither HBM nor the tensor cores bound this path (SURVEY 8d)", "kernel": miller_kernel, "achieved": mac_miller / (miller_ms * 1e-3) / 1e12 if miller_ms else None, "peak": imad_peak / 1e12,
                     "unit": "TMAC32/s", "frac": (mac_miller / (miller_ms * 1e-3)) / imad_peak if miller_ms else None, "traffic": ncu.get("traffic"),
                     "frac_note": "frac = SURVEY 8d's FIXED work per proof (136 MAC32 per Fp multiplication, no credit taken away for algorithmic savings) / time / peak; executed_frac = IMAD.WIDE "
                                  "instructions actually executed per proof (ncu source page of the same kernel, profiles/) x proofs / time / peak = the multiplier pipe's issue utilisation",
                     "executed_imad_wide_per_proof": exec_pp,
                     "executed_frac": (miller_n * exec_pp / (miller_ms * 1e-3)) / imad_peak if (miller_ms and exec_pp) else None,
                     "final_exp_executed_imad_wide_per_proof": exec_fe_pp,
                     "final_exp_executed_frac": (fe_n * exec_fe_pp / (fe_ms * 1e-3)) / imad_peak if (fe_ms and exec_fe_pp) else None,
                     "ncu_fmaheavy_pct": {"miller": ncu.get("ncu_fmaheavy_pct"), "final_exp": ncu_fe.get("ncu_fmaheavy_pct")},
                     "peak_source": "IMAD.WIDE.U32 issue rate measured live on this GPU (zkv_imad_peak); MEASURED_PEAKS.json holds no integer figure",
                     "fpmul_chain_per_s": fpmul_peak,
                     "whole_path_frac": value / world * W_M * M_MAC32 / imad_peak,
                     "final_exp_frac": (fe_n * W_FINALEXP_M * M_MAC32 / (fe_ms * 1e-3)) / imad_peak if fe_ms else None,
                     "launch": {"proofs": miller_n, "ms": miller_ms, "note": "one " + miller_kernel + " launch over a whole number of its waves (prefix of the batch), serial chain, CUDA events on the launching stream"},
                     "final_exp_launch": {"proofs": fe_n, "ms": fe_ms},
                     "frac_serial_all_proofs": (n * W_MILLER3_M * M_MAC32 / (serial_miller_ms * 1e-3)) / imad_peak if serial_miller_ms else None},
        "clocks": clocks.summary(),
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        line["cpu_baseline"], _ = cpu_baseline(O, args.shape, vk, batch, consts)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if use_dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
