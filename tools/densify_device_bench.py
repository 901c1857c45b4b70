"""Densify + commit + prove on one GPU with the lookup indices given as a host numpy array (lasso_densify: host threads
narrow and range-check them into pinned staging, then upload) and as a CUDA int64 tensor already on the device
(lasso_densify_device), both row-major and as one column expanded to C columns (stride 0).  Each step ends in the proof
bytes on the host, so the wall time of a step is synchronised.  The inputs alternate within every step, the median over
the timed steps is reported, and every step's proof must hash to tests/golden/big_proofs.json.
usage: python tools/densify_device_bench.py OUT_DIR [--steps 10] [--warmup 2] [--configs xor_c4_s20,lt_c8_s22,rc40_c4_s24]
Writes OUT_DIR/densify_device_bench.json."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import lasso_b200 as lb  # noqa: E402
import oracle_lib as ol  # noqa: E402
import workloads as wl  # noqa: E402


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--configs", default="xor_c4_s20,lt_c8_s22,rc40_c4_s24")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "big_proofs.json")))["cases"]
    dev = torch.device("cuda", 0)
    doc = {"gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0), "steps": args.steps,
           "warmup": args.warmup, "timing": "host wall clock of densify + commit + prove (ends in host bytes); median",
           "configs": {}}
    print("GPU: %s, power limit %s W" % (doc["gpu"], doc["power_limit_w"]), flush=True)
    ctx = lb.Context(0)
    for name in args.configs.split(","):
        kind, C_, log_m, log_r, log_s, idx, r, tape_seed = wl.config_inputs(name)
        g = golden[name]
        S = lb.Strategy(kind, C_, log_m, log_r)
        s = 1 << log_s
        stream = np.ascontiguousarray(ol.generators(lb.gens_points_needed(C_, s, S.num_memories, log_m)))
        gens = lb.SparsePolyCommitmentGens.new(ctx, b"gens_sparse_poly", C_, s, S.num_memories, log_m, stream=stream)
        row = torch.from_numpy(idx.astype(np.int64)).to(dev)
        inputs = {"numpy": idx, "cuda_int64_row_major": row,
                  "cuda_int64_expand": torch.from_numpy(idx[:, :1].astype(np.int64)).to(dev).expand(idx.shape[0], C_)}
        assert (inputs["cuda_int64_expand"] == row).all()
        torch.cuda.synchronize()
        times = {k: [] for k in inputs}
        phases = {k: [] for k in inputs}
        golden_ok = {k: [] for k in inputs}
        for step in range(args.warmup + args.steps):
            for key, x in inputs.items():
                t0 = time.perf_counter()
                dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, x, log_m)
                t1 = time.perf_counter()
                com = dense.commit(gens)
                proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=tape_seed)
                t2 = time.perf_counter()
                del dense
                ok = (hashlib.sha256(proof.bytes).hexdigest() == g["proof_sha256"]
                      and hashlib.sha256(com).hexdigest() == g["commitment_sha256"])
                if step >= args.warmup:
                    times[key].append(1e3 * (t2 - t0))
                    phases[key].append(1e3 * (t1 - t0))
                    golden_ok[key].append(ok)
                print("%s step %d %-22s %.2f ms (densify call %.2f ms) proof_sha256 == golden: %s" % (
                    name, step, key, 1e3 * (t2 - t0), 1e3 * (t1 - t0), ok), flush=True)
        res = {}
        for key in inputs:
            res[key] = {"median_ms": round(float(np.median(times[key])), 3), "min_ms": round(min(times[key]), 3),
                        "max_ms": round(max(times[key]), 3),
                        "median_densify_call_ms": round(float(np.median(phases[key])), 3),
                        "lookups_per_s": round((1 << log_s) / (float(np.median(times[key])) / 1e3)),
                        "proof_sha256_equals_golden_every_step": all(golden_ok[key]),
                        "steps_ms": [round(t, 2) for t in times[key]]}
        res["row_major_index_bytes"] = int(8 * idx.size)  # 8 B per index, read once by the extract
        doc["configs"][name] = res
        print(name, json.dumps(res), flush=True)
        del gens, inputs, row
        torch.cuda.empty_cache()
    ctx.close()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "densify_device_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    bad = [n for n, c in doc["configs"].items() for k, v in c.items() if isinstance(v, dict)
           and not v["proof_sha256_equals_golden_every_step"]]
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
