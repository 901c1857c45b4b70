#!/usr/bin/env python
"""bench.py — headline benchmark of the Lasso prover hot path on B200 (contract in the task prompt).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload prove|msm] [--log-s 20]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic lookups:
    DensifiedRepresentation::from_lookup_indices -> commit -> SparsePolynomialEvaluationProof::prove
for the XOR subtable strategy, C = 4, M = 2^16, 2^20 lookups, G = curve25519 (BASELINE.json configs[1]).

  value : lookups/s with the densified representation already resident in HBM (commit + prove timed)
  e2e   : lookups/s through the C-ABI with HOST buffers (densify incl. the host->device upload of the
          index / counter arrays, commit, prove incl. every device->host transfer of round messages and
          the proof bytes)
  roofline     : the bind kernel (K1) timed alone with CUDA events on the library's stream
  cpu_baseline : the CPU oracle port on this box's host cores, the same 2^20 workload (rank 0, N = 1 only)
  configs      : BASELINE.json configs 2-4 (XOR 2^20, LT C=8 2^22, RangeCheck<40> C=4 2^24), ONE proof each:
                 N = 1 on one GPU; N > 1 the same proof SHARDED over the N GPUs (csrc/comm.cu), with the SHA-256 of
                 the proof bytes compared with a single-GPU proof of the same inputs made in the same run and with the
                 oracle-generated golden hash (tests/golden/big_proofs.json)

N > 1: one process per GPU under torchrun; the headline numbers are N independent proofs (one per rank, weak scaling,
no data-path collective — proofs of different lookup batches are independent objects): value = N * s / max_t.
--impl reference: the reference's own CPU implementation of the path = the oracle port (the Rust crate cannot
be built in this image: no cargo/rustc, crates not vendored), all host threads, rank 0 only, the SAME 2^20 workload.
--workload msm: BASELINE.json configs[4], the VariableBaseMSM-only sweep (tools/msm_bench.py holds the details).
--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned to its caller (see
dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared file by file.

The benchmark writes nothing into the source tree (it may be read-only): no bytecode, no generator cache.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import workloads as wl  # noqa: E402

METRIC = "Lasso prove lookups/sec (2^20 lookups, C=4, M=2^16)"
UNIT = "lookups/s"
KIND_XOR = 2
make_inputs = wl.make_inputs


def golden_cases():
    p = os.path.join(ROOT, "tests", "golden", "big_proofs.json")
    return json.load(open(p))["cases"] if os.path.exists(p) else {}


def dump_outputs(d, commitment, proof, challenges):
    """--dump-outputs: what commit + prove hand their caller, byte for byte, as float32 arrays (one value 0..255 per
    byte): DIR/commitment.npy and DIR/proof.npy (the serialized bytes) and DIR/challenges.npy (one row of 32 bytes,
    the four Montgomery limbs, per Fiat-Shamir challenge).  The library's output caps (4 MiB commitment, 4 MiB proof,
    2^14 challenges) bound the three files to 34 MiB."""
    os.makedirs(d, exist_ok=True)
    chal = np.ascontiguousarray(challenges, dtype=np.uint64)
    arrays = {"commitment": np.frombuffer(commitment, dtype=np.uint8),
              "proof": np.frombuffer(proof, dtype=np.uint8),
              "challenges": chal.view(np.uint8).reshape(chal.shape[0], 32)}
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a.astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Samples before this point (warm-up, process start-up) are dropped: only the loaded region counts."""
        self.first = len(self.lines)

    def count(self):
        return len(self.lines) - getattr(self, "first", 0)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines[getattr(self, "first", 0):]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def generator_stream(lb, need):
    """The first `need` points of the b"gens_sparse_poly" stream: a cached file of the oracle's sampler (the same
    bytes: tests/test_gpu_kernels.py checks the library's sampler against it) or sampled here."""
    d = os.path.join(ROOT, "oracle", "_build")
    have = []
    if os.path.isdir(d):
        for f in os.listdir(d):
            if f.startswith("gens_gens_sparse_poly_") and f.endswith(".npy"):
                have.append(int(f[len("gens_gens_sparse_poly_"):-4]))
    for cand in sorted(have):
        if cand >= need:
            return np.ascontiguousarray(np.load(os.path.join(d, "gens_gens_sparse_poly_%d.npy" % cand))[:need])
    return lb.sample_generators(b"gens_sparse_poly", need)


def best_threads(C=4, log_m=16, log_probe=14):
    """The oracle port (like the reference's rayon path) has long serial sections (Bulletproofs generator folding,
    serial binds), and an OpenMP team larger than the cores this container may use is disastrous (measured on the
    GPU box: 2^18 lookups take 2.1 s on 16-32 threads, 2.7 s on 64, 16.6 s on 128).  Probe a small instance and keep
    the fastest team size, so the CPU arm is the best the port can do on this box."""
    import oracle_lib as ol

    ncpu = os.cpu_count() or 8
    cands = sorted({t for t in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8) if 1 <= t <= ncpu}, reverse=True)
    idx, r, seed = make_inputs(log_probe, C, log_m, 4242)
    gens = ol.generators(max((1 << ((log_probe + 3) - (log_probe + 3) // 2)) + 2, 600), persist=False)
    best, best_t = None, None
    ol.lib().orc_set_num_threads(int(max(1, min(16, ncpu // 2))))
    ol.prove(KIND_XOR, C, log_m, 0, idx, r, gens, seed, flags=0)  # untimed: fault the heap in
    for t in cands:
        ol.lib().orc_set_num_threads(int(t))
        t0 = time.perf_counter()
        ol.prove(KIND_XOR, C, log_m, 0, idx, r, gens, seed, flags=0)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, best_t = dt, t
    ol.lib().orc_set_num_threads(int(best_t))
    return best_t, ncpu


def cpu_workload(log_s, C=4, log_m=16):
    """The bench workload itself (seed BENCH_SEED, rank 0) for the CPU arm."""
    import oracle_lib as ol

    idx, r, seed = make_inputs(log_s, C, log_m, wl.BENCH_SEED)
    gens = np.ascontiguousarray(ol.generators(wl.gens_needed(C, log_s, C, log_m), persist=False))
    return ol, idx, r, seed, gens


def run_reference(args):
    """--impl reference: the reference's own CPU path = oracle port, all host threads it can use, rank 0 only, the
    SAME workload as the GPU arm (XOR C=4 M=2^16, 2^20 lookups per step, the same seed)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    C, log_m, log_s = 4, 16, args.log_s
    nthreads, ncpu = best_threads()
    ol, idx, r, seed, gens = cpu_workload(log_s, C, log_m)
    cores = ol.lib().orc_num_threads()
    res = None
    for _ in range(max(1, args.warmup)):
        res = ol.prove(KIND_XOR, C, log_m, 0, idx, r, gens, seed, flags=0)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = ol.prove(KIND_XOR, C, log_m, 0, idx, r, gens, seed, flags=0)
        assert res["rc"] == 0
    dt = time.perf_counter() - t0
    val = args.steps * (1 << log_s) / dt
    sha = hashlib.sha256(res["proof"]).hexdigest()
    gold = golden_cases().get("xor_c4_s20", {}) if log_s == 20 else {}
    sample = ("XOR C=4 M=2^16, 2^%d lookups per step = the whole workload of the GPU arm (same seed), densify+commit+prove; "
              "OpenMP team = fastest of a probe over team sizes (%d of %d logical CPUs)" % (log_s, nthreads, ncpu))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64x4 Montgomery (CPU)", "data": "synthetic",
        "config": {"workload": "Lasso XOR subtable, C=4, M=2^16, 2^%d lookups per step, G=curve25519: densify + commit + prove" % log_s,
                   "note": "restated CPU baseline (C++/OpenMP oracle port), not the Rust binary",
                   "proof_sha256": sha, "golden_match": (sha == gold.get("proof_sha256")) if gold else None,
                   "spans_ms": {k: round(v, 1) for k, v in res["spans"].items()}},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res["commitment"], res["proof"], res["challenges"])
    print(json.dumps(line))


def prove_config(lb, ctx, name, steps, stream_cache, sync=lambda: None):
    """ONE proof of a BASELINE configuration on `ctx` (single GPU, or sharded when the context has a communicator):
    1 warm-up, then `steps` timed end-to-end runs (densify + commit + prove, host buffers); returns the timings of the
    library's own spans and the hashes of the bytes."""
    kind, C, log_m, log_r, log_s, idx, r, tape_seed = wl.config_inputs(name)
    S = lb.Strategy(kind, C, log_m, log_r)
    s = 1 << log_s
    need = lb.gens_points_needed(C, s, S.num_memories, log_m)
    if need not in stream_cache:
        stream_cache[need] = generator_stream(lb, need)
    t0 = time.perf_counter()
    gens = lb.SparsePolyCommitmentGens.new(ctx, b"gens_sparse_poly", C, s, S.num_memories, log_m, stream=stream_cache[need])
    setup_ms = 1e3 * (time.perf_counter() - t0)
    best = None
    com = proof = None
    for it in range(1 + steps):
        t0 = time.perf_counter()
        dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, idx, log_m)
        sync()  # the upload and the sort are asynchronous; sharded: every rank starts the commitment together
        t1 = time.perf_counter()
        com = dense.commit(gens)
        t2 = time.perf_counter()
        proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=tape_seed)
        t3 = time.perf_counter()
        del dense
        cur = {"densify_ms": 1e3 * (t1 - t0), "commit_ms": 1e3 * (t2 - t1), "prove_ms": 1e3 * (t3 - t2)}
        if it >= 1 and (best is None or cur["commit_ms"] + cur["prove_ms"] < best["commit_ms"] + best["prove_ms"]):
            best = cur
    del gens
    out = {"name": name, "lookups": s, "setup_ms": round(setup_ms, 1)}
    out.update({k: round(v, 3) for k, v in best.items()})
    out["ms_per_proof"] = round(best["commit_ms"] + best["prove_ms"], 3)  # device-resident: commit + prove
    out["e2e_ms_per_proof"] = round(best["densify_ms"] + best["commit_ms"] + best["prove_ms"], 3)
    out["proof_sha256"] = hashlib.sha256(proof.bytes).hexdigest()
    out["commitment_sha256"] = hashlib.sha256(com).hexdigest()
    return out


def run_msm(args):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import msm_bench

    msm_bench.main(args)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="prove", choices=["prove", "msm"])
    ap.add_argument("--log-s", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-configuration block (configs 2-4, one proof each)")
    ap.add_argument("--configs", default="xor_c4_s20,lt_c8_s22,rc40_c4_s24")
    ap.add_argument("--msm-max-log", type=int, default=24)
    ap.add_argument("--batch", type=int, default=4, help="proofs in flight for the throughput_batched block (N = 1)")
    ap.add_argument("--no-batched", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not pin the host threads to the GPU's NUMA node")
    ap.add_argument("--no-sampler", action="store_true", help="diagnosis: no nvidia-smi clock sampler during the run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the commitment, proof and challenges of the last timed step to DIR/*.npy (prove workload)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload != "prove":
        ap.error("--dump-outputs applies to the prove workload")
    if args.workload == "msm":
        run_msm(args)
        return
    if args.impl == "reference":
        run_reference(args)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    import lasso_b200 as lb
    from lasso_b200 import parallel

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if world > 1:
        # the first collective sets the NCCL communicator up (connections, proxy threads, buffers): do that here, not
        # in the barrier that opens the timed region
        dist.barrier()
        torch.cuda.synchronize()
    C, log_m, log_s = 4, 16, args.log_s
    s = 1 << log_s
    S = lb.Strategy(lb.XOR, C, log_m)
    # independent proofs: each rank its own batch
    idx, r, tape_seed = make_inputs(log_s, C, log_m, wl.BENCH_SEED + rank)
    ctx = lb.Context(local_rank)
    numa_node = -1
    need = lb.gens_points_needed(C, s, S.num_memories, log_m)
    streams = {need: generator_stream(lb, need)}
    free0 = torch.cuda.mem_get_info()[0]
    t0 = time.perf_counter()
    gens = lb.SparsePolyCommitmentGens.new(ctx, b"gens_sparse_poly", C, s, S.num_memories, log_m, stream=streams[need])
    setup_ms = 1e3 * (time.perf_counter() - t0)
    tables_gb = (free0 - torch.cuda.mem_get_info()[0]) / 1e9

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_e2e():
        dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, idx, log_m)
        com = dense.commit(gens)
        proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=tape_seed)
        return dense, com, proof

    def step_resident(dense, g=None):
        com = dense.commit(g or gens)
        proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, g or gens, tape_seed=tape_seed)
        return com, proof

    # ---- warm-up (>= 3): also produces the resident densified representation.  The clock sampler (one streaming
    # nvidia-smi process, a line every 100 ms) is started first so that it is already emitting when the timed
    # region begins; only its samples from the loaded region on are used.
    sampler = ClockSampler(local_rank)
    if not args.no_sampler:
        sampler.start()
    # one process per GPU: the proving thread gets a dedicated core of the GPU's NUMA node, helper threads the rest of
    # the node (after every other thread of the process exists: they keep their affinity)
    if world > 1 and not args.no_numa_bind:
        numa_node = ctx.bind_host_threads()
    dense = None
    for _ in range(args.warmup):
        dense, com0, proof0 = step_e2e()
    proof_bytes, com_bytes = len(proof0.bytes), len(com0)
    proof_sha = hashlib.sha256(proof0.bytes).hexdigest()

    # ---- timed: device-resident (value)
    barrier()
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launches
    ev0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step_resident(dense)
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    t_res = ev0.elapsed_time(ev1) / 1e3
    launches = ctx.launches - l0
    # ---- timed: end to end through the C-ABI with host buffers (e2e)
    barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    dens_ms = 0.0
    for _ in range(args.steps):
        step_e2e()
        dens_ms += ctx.last_timings_ms()["densify"]
    ev3.record()
    barrier()
    t_e2e = ev2.elapsed_time(ev3) / 1e3
    # the timed region can be shorter than the sampling period: keep the same load running (untimed) until the
    # sampler has seen the GPU under it at least twice
    t_guard = time.perf_counter()
    while sampler.proc and sampler.count() < 2 and time.perf_counter() - t_guard < 3.0:
        step_resident(dense)
    clocks = sampler.stop()

    print("rank %d: resident %.3f ms/step, e2e %.3f ms/step, proving thread on CPUs %s" % (
        rank, 1e3 * t_res / args.steps, 1e3 * t_e2e / args.steps,
        sorted(os.sched_getaffinity(0)) if len(os.sched_getaffinity(0)) <= 8 else "%d CPUs" % len(os.sched_getaffinity(0))),
        file=sys.stderr, flush=True)
    if world > 1:
        t_res, t_e2e = parallel.max_over_ranks([t_res, t_e2e])

    # ---- the same step without the digit-multiples tables: the Pippenger-bucket path the north star names
    no_tables = None
    if world == 1:
        os.environ["LASSO_B200_NO_MULTIPLES"] = "1"
        try:
            g2 = lb.SparsePolyCommitmentGens.new(ctx, b"gens_sparse_poly", C, s, S.num_memories, log_m, stream=streams[need])
            com2, proof2 = step_resident(dense, g2)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                step_resident(dense, g2)
            torch.cuda.synchronize()
            no_tables = {"ms_per_step": round(1e3 * (time.perf_counter() - t0) / args.steps, 3),
                         "same_bytes_as_table_path": bool(proof2.bytes == proof0.bytes and com2 == com0)}
            del g2
        finally:
            del os.environ["LASSO_B200_NO_MULTIPLES"]

    # ---- K proofs in flight on the one GPU (a context = stream + scratch + host transcript thread per proof, the
    # generator tables shared): a single proof leaves the GPU idle while the host hashes, and most of its rounds
    # occupy a few SMs.  Throughput mode; the single-proof latency above stays the headline.
    batched = None
    if world == 1 and not args.no_batched:
        try:
            K = args.batch
            ctxs = [lb.Context(local_rank) for _ in range(K)]
            inputs = [make_inputs(log_s, C, log_m, wl.BENCH_SEED + 100 + k) for k in range(K)]
            denses = [lb.DensifiedRepresentation.from_lookup_indices(ctxs[k], inputs[k][0], log_m) for k in range(K)]
            shas = [None] * K

            def worker(k, reps):
                for _ in range(reps):
                    com_k = denses[k].commit(gens)
                    pr = lb.SparsePolynomialEvaluationProof.prove(ctxs[k], S, denses[k], inputs[k][1], gens, tape_seed=inputs[k][2])
                shas[k] = (hashlib.sha256(com_k).hexdigest(), hashlib.sha256(pr.bytes).hexdigest())

            def run_all(reps):
                th = [threading.Thread(target=worker, args=(k, reps)) for k in range(K)]
                for t in th:
                    t.start()
                for t in th:
                    t.join()

            run_all(1)  # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run_all(args.steps)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            # every proof of the batch must be the proof the single-context path produces for the same inputs
            solo = [hashlib.sha256(lb.SparsePolynomialEvaluationProof.prove(ctx, S, denses[k], inputs[k][1], gens,
                                                                            tape_seed=inputs[k][2]).bytes).hexdigest() for k in range(K)]
            batched = {"proofs_in_flight": K, "value": K * args.steps * s / dt, "unit": UNIT,
                       "ms_per_proof_amortised": round(1e3 * dt / (K * args.steps), 3),
                       "ms_per_batch": round(1e3 * dt / args.steps, 3),
                       "same_bytes_as_single_context": bool(all(shas[k][1] == solo[k] for k in range(K)))}
            del denses
            for cx in ctxs:
                cx.close()
        except Exception as e:
            batched = {"error": repr(e)}

    # ---- roofline of the bind kernel (K1), timed alone with CUDA events on the library's stream:
    # 5 polynomials x 2^22 elements (640 MiB > 126 MB L2), 96 algorithmic bytes per output element
    bind_len, bind_np = 1 << 22, 5
    ms = ctx.bench_bind(bind_len, bind_np, 20)
    alg_bytes = 96.0 * (bind_len // 2) * bind_np
    achieved = alg_bytes / (ms * 1e-3) / 1e9
    peak, peak_src = measured_peak_hbm()

    # ---- BASELINE configs 2-4, ONE proof each: single GPU at N = 1, the SAME proof sharded over the N GPUs otherwise
    gold = golden_cases()
    config_rows = []
    if not args.no_configs:
        del dense, gens
        names = [n for n in args.configs.split(",") if n]
        single = {}
        if world > 1:
            # reference bytes for the sharded proofs: a single-GPU proof of the same inputs, made by rank 0 right here
            if rank == 0:
                for n in names:
                    single[n] = prove_config(lb, ctx, n, 2, streams, torch.cuda.synchronize)
            dist.barrier()
            sctx = lb.Context(local_rank)
            sctx.init_comm(rank, world)
            if not args.no_numa_bind:
                sctx.bind_host_threads()
        for n in names:
            row = prove_config(lb, sctx if world > 1 else ctx, n, max(1, min(args.steps, 3)), streams, barrier)
            row["mode"] = "one proof sharded over %d GPUs (low index bits)" % world if world > 1 else "one proof on one GPU"
            if world > 1:
                tm = parallel.max_over_ranks([row["ms_per_proof"], row["e2e_ms_per_proof"]])
                row["ms_per_proof"], row["e2e_ms_per_proof"] = round(tm[0], 3), round(tm[1], 3)
                if rank == 0:
                    row["single_gpu_ms_per_proof"] = single[n]["ms_per_proof"]
                    row["matches_single_gpu"] = bool(row["proof_sha256"] == single[n]["proof_sha256"] and
                                                     row["commitment_sha256"] == single[n]["commitment_sha256"])
            g = gold.get(n)
            row["golden_match"] = bool(g and g["proof_sha256"] == row["proof_sha256"] and
                                       g["commitment_sha256"] == row["commitment_sha256"]) if g else None
            config_rows.append(row)
        if world > 1:
            sctx.close()

    line = None
    if rank == 0:
        h2d = 4 * s * C  # the index matrix narrowed to u32 (the timestamps are derived on the device)
        g20 = gold.get("xor_c4_s20") if log_s == 20 else None
        line = {
            "metric": METRIC, "value": world * args.steps * s / t_res, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_res / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 (8-limb 256-bit Montgomery)",
            "data": "synthetic",
            "config": {"workload": "Lasso XOR subtable, C=4, M=2^16, 2^%d lookups per GPU, G=curve25519: commit + prove "
                                   "(densify in e2e)" % log_s,
                       "l2": "inputs larger than L2 (>= 128 MiB per polynomial set)",
                       "parallelism": "independent proof per GPU (weak scaling, no data-path collective); the `configs` block "
                                      "holds ONE proof per BASELINE configuration, sharded over the GPUs when N > 1",
                       "proof_bytes": proof_bytes, "commitment_bytes": com_bytes, "wall_s_resident": wall,
                       "proof_sha256": proof_sha,
                       "golden_match": bool(g20 and g20["proof_sha256"] == proof_sha) if g20 else None,
                       "golden": "tests/golden/big_proofs.json (CPU oracle, verifier accepted), rank 0's inputs",
                       "setup_ms": round(setup_ms, 1), "tables_gb": round(tables_gb, 2),
                       "setup": "SparsePolyCommitmentGens.new equivalent: generator stream -> window table + digit-multiples "
                                "tables, outside the timed region like the reference's gens (bench.rs:54-57)",
                       "no_tables": no_tables, "numa_node": numa_node},
            "e2e": {"value": world * args.steps * s / t_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": proof_bytes + com_bytes, "ms_per_step": 1e3 * t_e2e / args.steps,
                    "densify_ms_per_step": dens_ms / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"kernel": "bind_top2_kernel (K1: bound_poly_var_top, two outputs per thread)", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch of this exact shape, from the
                         # ncu --set full capture in profiles/r02_bind_top2_kernel_ncu_full.txt (671.1 MB + 294.3 MB)
                         "traffic": 965458176,
                         "peak_source": peak_src, "ms_per_launch": ms,
                         "alg_bytes_per_launch": alg_bytes},
            "throughput_batched": batched,
            "configs": config_rows,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                nthreads, ncpu = best_threads()
                ol, cidx, cr, cseed, cgens = cpu_workload(log_s, C, log_m)
                cores = ol.lib().orc_num_threads()
                ol.prove(KIND_XOR, C, log_m, 0, cidx, cr, cgens, cseed, flags=0)  # warm-up
                t0 = time.perf_counter()
                res = ol.prove(KIND_XOR, C, log_m, 0, cidx, cr, cgens, cseed, flags=0)
                dt = time.perf_counter() - t0
                line["cpu_baseline"] = {"value": (1 << log_s) / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                        "sample": "the whole workload: XOR C=4 M=2^16, 2^%d lookups, same inputs as the GPU arm, "
                                                  "densify+commit+prove, 1 timed run after 1 warm-up (oracle C++/OpenMP port; not "
                                                  "the Rust binary); OpenMP team = fastest of a probe (%d of %d logical CPUs)"
                                                  % (log_s, nthreads, ncpu),
                                        "same_bytes_as_gpu": bool(res["proof"] == proof0.bytes),
                                        "spans_ms": {k: round(v, 1) for k, v in res["spans"].items()}}
            except Exception as e:  # the checker failing must not hide the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": "failed: %r" % e}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last[0], last[1].bytes, last[1].challenges)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
