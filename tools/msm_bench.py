"""BASELINE config 5: the VariableBaseMSM-only sweep (bench.py --workload msm).

For n = 2^16 .. 2^max (step 2) and three scalar distributions — uniform full-width Fr, "Lasso-shaped" < 2^16 and
< 2^20 — ONE MSM on device-resident inputs (affine bases and Montgomery scalars already in HBM; everything else —
canonical scalars, internal base form, digits, sort, buckets — inside the timed region), CUDA events on the library's
stream, max over ranks.  N > 1 (torchrun): the terms are sharded over the GPUs by index, every GPU returns one partial
point, gather-then-add (SURVEY §8e).  CPU comparator on rank 0 up to 2^cpu_max: the restated msm_bigint_wnaf (one MSM
is serial in the reference, msm/mod.rs:125-147) with the max-bits shortcut (msm/mod.rs:95-106) and without it (= what
`--features ark-msm` selects).  Prints one JSON line: terms/s per case, mixed additions/s against the 7.2 G adds/s the
row-commitment kernel reaches (profiles/README.md), and the headline = full-width 2^22.
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

ADD_CEILING = 7.2e9  # mixed additions/s of msm_rows_direct_u32_kernel (84 % of the integer pipe), profiles/README.md


def main(args):
    import torch
    import torch.distributed as dist

    import lasso_b200 as lb
    import oracle_lib as ol
    from oracle_lib import P, sz

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = lb.Context(local_rank)
    if world > 1:
        ctx.init_comm(rank, world)
    max_log = int(getattr(args, "msm_max_log", 24))
    cpu_max = 18
    pool = np.ascontiguousarray(ol.generators(8194, persist=False)[:8192])
    rows = []
    for log_n in range(16, max_log + 1, 2):
        n = 1 << log_n
        n_loc = n // world
        for name, bits in (("full-253", 253), ("small-16", 16), ("small-20", 20)):
            rng = np.random.default_rng(1000 * log_n + bits)  # every rank draws the whole vector, keeps its block
            if bits <= 60:
                v = rng.integers(0, 1 << bits, size=n, dtype=np.uint64)
                sc = np.zeros((n, 4), dtype=np.uint64)
                ol.lib().orc_fr_from_u64_batch(P(v), sz(n), P(sc))
            else:
                raw = rng.integers(0, 2**63, size=(n, 4), dtype=np.uint64)
                raw[:, 3] &= (1 << 59) - 1
                sc = np.ascontiguousarray(raw)
            # rank g takes the terms [g * n_loc, (g+1) * n_loc): the tiled pool repeats every 8192 terms and n_loc is
            # a multiple of it, so every rank's term i uses base i % 8192
            mine = np.ascontiguousarray(sc[rank * n_loc:(rank + 1) * n_loc])
            job = lb.MsmJob(ctx, pool, mine)
            job.run(1)  # warm-up
            if world > 1:
                dist.barrier()
            iters = 5 if log_n <= 20 else 2
            pt, ms, info = job.run(iters)
            job.close()
            if world > 1:
                t = torch.tensor([ms], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t[0])
            row = {"log_n": log_n, "scalars": name, "ms": round(ms, 4), "terms_per_s": n / (ms * 1e-3),
                   "c": info["c"], "windows": info["windows"],
                   "mixed_adds_per_s": n * info["windows"] / (ms * 1e-3)}
            row["frac_of_add_ceiling"] = row["mixed_adds_per_s"] / (ADD_CEILING * world)
            if rank == 0 and log_n <= cpu_max:
                bases = np.ascontiguousarray(np.tile(pool, (n // 8192, 1)))
                for hack, key in ((1, "cpu_ms_maxbits_shortcut"), (0, "cpu_ms_ark_msm")):
                    ref = np.zeros(16, dtype=np.uint64)
                    t0 = time.perf_counter()
                    ol.lib().orc_msm(P(bases), P(sc), sz(n), hack, P(ref))
                    row[key] = round(1e3 * (time.perf_counter() - t0), 1)
                    row["same_point_as_cpu"] = bool(ol.lib().orc_point_eq(P(pt), P(ref)) == 1)
            rows.append(row)
    if rank == 0:
        head = next((r for r in rows if r["log_n"] == 22 and r["scalars"] == "full-253"), rows[-1])
        line = {"metric": "VariableBaseMSM terms/sec (2^22 full-width curve25519 scalars, device-resident)",
                "value": head["terms_per_s"], "unit": "terms/s", "n_gpus": world, "steps": 1, "warmup": 1,
                "ms_per_step": head["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u32 (8-limb 256-bit, Fq pseudo-Mersenne)", "data": "synthetic",
                "config": {"workload": "BASELINE configs[4]: VariableBaseMSM-only sweep 2^16..2^%d, bases = 8192 distinct subgroup "
                                       "points tiled, terms sharded over the GPUs by index (gather-then-add of partial points)" % max_log,
                           "cpu_comparator": "restated msm_bigint_wnaf, 1 thread (one MSM is serial in the reference)"},
                "roofline": {"kernel": "msm_accum_kernel", "bound": "integer-ALU (7 Fq mul per mixed addition)",
                             "achieved": head["mixed_adds_per_s"], "peak": ADD_CEILING * world, "unit": "mixed adds/s",
                             "frac": head["frac_of_add_ceiling"], "traffic": None},
                "sweep": rows}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
