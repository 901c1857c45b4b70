"""Run under torchrun with WORLD_SIZE ranks: ONE proof sharded over all ranks, every rank densifying from its own CUDA
tensor (lasso_densify_device: the same matrix on every rank's device, each rank extracts its own shard); rank 0 checks
that commitment, challenges and proof bytes equal the CPU oracle's, and an out-of-range index must be reported on every
rank.  One GPU per rank by default; with LASSO_SHARD_SAME_GPU=1 every rank uses GPU 0 (gloo for the plumbing), as in
tools/sharded_check.py.
usage: torchrun --nproc-per-node N tools/sharded_device_check.py"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.distributed as dist
import lasso_b200 as lb
import oracle_lib as ol

rank = int(os.environ.get("RANK", 0)); local = int(os.environ.get("LOCAL_RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
same_gpu = os.environ.get("LASSO_SHARD_SAME_GPU") == "1"
if same_gpu:
    local = 0
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
else:
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dev = torch.device("cuda", local)


def as_tensor(idx, dtype, layout):
    t = torch.from_numpy(idx.astype(np.int64)).to(dev, torch.int64 if dtype.endswith("64") else torch.int32)
    if layout == "col":
        t = t.t().contiguous().t()
    elif layout == "expand":
        t = t[:, :1].expand(idx.shape)
    return t.view(getattr(torch, dtype)) if dtype.startswith("u") else t


# kind, C, log_m, log_r, lookups, same, dtype, layout
cases = [(2, 4, 16, 0, 1 << 12, 1, "int64", "expand"), (3, 4, 4, 0, 128, 0, "int32", "row"),
         (0, 1, 16, 0, 1 << 10, 1, "uint64", "row"), (4, 3, 8, 40, 256, 0, "uint32", "col"),
         (3, 8, 8, 0, 512, 0, "int64", "col"), (1, 2, 8, 0, 700, 0, "int64", "row")]
ctx = lb.Context(local)
ctx.init_comm()
ok = True
for kind, C, log_m, log_r, n, same, dtype, layout in cases:
    rng = np.random.default_rng(kind * 7 + C)
    col = rng.integers(0, 1 << log_m, size=(n, 1), dtype=np.uint64)
    idx = np.ascontiguousarray(np.repeat(col, C, axis=1) if same else rng.integers(0, 1 << log_m, size=(n, C), dtype=np.uint64))
    s = 1 << (n - 1).bit_length()
    r = ol.rand_fr(rng, s.bit_length() - 1); seed = ol.rand_fr(rng, 1)[0]
    S = lb.Strategy(kind, C, log_m, log_r)
    need = lb.gens_points_needed(C, s, S.num_memories, log_m)
    stream = np.ascontiguousarray(ol.generators(max(need, 300))[:need])
    gens = lb.SparsePolyCommitmentGens.new(ctx, b"g", C, s, S.num_memories, log_m, stream=stream)
    t = as_tensor(idx, dtype, layout)
    t0 = time.time()
    dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, t, log_m)
    com = dense.commit(gens)
    proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=seed)
    dt = time.time() - t0
    if rank == 0:
        ref = ol.prove(kind, C, log_m, log_r, idx, r, stream, seed, flags=1)
        good = ref["rc"] == 0 and com == ref["commitment"] and proof.bytes == ref["proof"]
        print("case kind=%d C=%d log_m=%d n=%d %s/%s world=%d: %s (%.1f ms, commit_ok=%s)" % (
            kind, C, log_m, n, dtype, layout, world, "OK" if good else "MISMATCH", dt * 1e3, com == ref["commitment"]),
            flush=True)
        ok = ok and good
# an out-of-range index (densified.rs:46) near the end: every rank checks every element, so every rank reports it
n_bad = 1 << 12
bad = np.zeros((n_bad, 2), dtype=np.uint64)
bad[n_bad - 3, 1] = 1 << 8
try:
    lb.DensifiedRepresentation.from_lookup_indices(ctx, as_tensor(bad, "int64", "row"), 8)
    bad_ok = False
except lb.LassoError as e:
    bad_ok = e.code == 3
flags = [None] * world
dist.all_gather_object(flags, bad_ok)
if rank == 0:
    print("out-of-range index reported on every rank: %s" % ("OK" if all(flags) else "MISMATCH %s" % flags), flush=True)
    ok = ok and all(flags)
# the context is still usable after the rejected call
rng = np.random.default_rng(5)
idx = rng.integers(0, 1 << 8, size=(1 << 10, 2), dtype=np.uint64)
r = ol.rand_fr(rng, 10); seed = ol.rand_fr(rng, 1)[0]
S = lb.Strategy(lb.XOR, 2, 8)
need = lb.gens_points_needed(2, 1 << 10, 2, 8)
stream = np.ascontiguousarray(ol.generators(max(need, 300))[:need])
gens = lb.SparsePolyCommitmentGens.new(ctx, b"g", 2, 1 << 10, 2, 8, stream=stream)
dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, as_tensor(idx, "int64", "row"), 8)
com = dense.commit(gens)
proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=seed)
if rank == 0:
    ref = ol.prove(lb.XOR, 2, 8, 0, idx, r, stream, seed, flags=1)
    good = ref["rc"] == 0 and com == ref["commitment"] and proof.bytes == ref["proof"]
    print("proof after the rejected call: %s" % ("OK" if good else "MISMATCH"), flush=True)
    ok = ok and good
dist.barrier()
dist.destroy_process_group()
if rank == 0:
    print("SHARDED_DEVICE_CHECK", "PASS" if ok else "FAIL")
    sys.exit(0 if ok else 1)
