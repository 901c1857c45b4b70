"""DensifiedRepresentation.from_lookup_indices on a CUDA tensor (lasso_densify_device): the index matrix is read in
place on the device, in any of four integer types and any strides.  Every field, commitment and proof must equal what
the same indices give as a host array (and therefore the CPU oracle's bytes)."""
import ctypes
import hashlib
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
import workloads as wl
from test_gpu_prove import CASES, make_inputs

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DTYPES = ["int64", "uint64", "int32", "uint32"]
LAYOUTS = ["row", "col", "expand", "slice"]


@pytest.fixture(scope="module")
def ctx():
    import lasso_b200 as lb

    c = lb.Context(0)
    yield c
    c.close()


def to_cuda(idx, dtype="int64", layout="row"):
    """idx (n x C, uint64 numpy) as a CUDA tensor of `dtype` stored in `layout`:
    row: contiguous (n, C); col: a contiguous (C, n) tensor transposed; expand: column 0 broadcast to C columns
    (stride 0, so the caller must compare against np.repeat(idx[:, :1], C, 1)); slice: every other row of a (2n, C)."""
    import torch

    n, C_ = idx.shape
    signed = torch.int64 if dtype.endswith("64") else torch.int32
    src = torch.from_numpy(idx.astype(np.int64)).to("cuda", signed)
    if layout == "row":
        t = src
    elif layout == "col":
        t = src.t().contiguous().t()
    elif layout == "expand":
        t = src[:, :1].expand(n, C_)
    elif layout == "slice":
        big = torch.full((2 * n, C_), 12345, dtype=signed, device="cuda")
        big[::2] = src
        t = big[::2]
    else:
        raise ValueError(layout)
    if dtype.startswith("u"):
        t = t.view(getattr(torch, dtype))
    assert t.shape == (n, C_)
    if layout == "col" and C_ > 1:  # with one column both layouts are the same tensor
        assert t.stride() == (1, n)
    if layout == "expand":
        assert t.stride(1) == 0
    return t


def host_view(idx, layout):
    return np.ascontiguousarray(np.repeat(idx[:, :1], idx.shape[1], axis=1)) if layout == "expand" else idx


def fields(d):
    """dim_usize, dim, read, final and both merged polynomials (lasso_dense_read 0-5)"""
    nv_l = (2 * d.C * d.s - 1).bit_length()
    nv_m = (d.C - 1).bit_length() + d.log_m
    return [d.dim_usize, d.dim, d.read, d.final, d._read(4, 1 << nv_l, 4), d._read(5, 1 << nv_m, 4)]


def assert_same_fields(ctx, idx_host, t, log_m):
    import lasso_b200 as lb

    a = fields(lb.DensifiedRepresentation.from_lookup_indices(ctx, idx_host, log_m))
    b = fields(lb.DensifiedRepresentation.from_lookup_indices(ctx, t, log_m))
    for name, x, y in zip(["dim_usize", "dim", "read", "final", "l_variate", "log_m_variate"], a, b):
        assert x.shape == y.shape and (x == y).all(), name


def skewed(n, C_, log_m, seed):
    """test_gpu_prove.test_gpu_densify_matches_host_scan's addresses: one column of three addresses, a run of 300"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, 1 << log_m, size=(n, C_), dtype=np.uint64)
    idx[:, 1 % C_] = rng.integers(0, 3, size=n)
    idx[100:400, C_ - 1] = 17
    return idx


# ------------------------------------------------------------------ 1. fields equal the host path's
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_fields_match_host_path_every_dtype_and_layout(ctx, dtype, layout):
    idx = skewed(5000, 3, 8, 77)
    assert_same_fields(ctx, host_view(idx, layout), to_cuda(idx, dtype, layout), 8)


@pytest.mark.parametrize("C_,log_m,n", [(1, 4, 700), (1, 16, 1 << 12), (3, 8, 5000), (3, 16, 700), (4, 4, 1 << 10),
                                        (4, 16, 5000), (8, 8, 700), (8, 16, 1 << 11), (16, 4, 5000), (16, 8, 1 << 9),
                                        (16, 16, 700), (4, 16, 1 << 15)])
def test_fields_match_host_path_shapes(ctx, C_, log_m, n):
    rng = np.random.default_rng(C_ * 1000 + log_m * 10 + n)
    idx = rng.integers(0, 1 << log_m, size=(n, C_), dtype=np.uint64)
    assert_same_fields(ctx, idx, to_cuda(idx), log_m)
    assert_same_fields(ctx, idx, to_cuda(idx, "uint32", "col"), log_m)


def test_cpu_tensor_takes_the_host_path(ctx):
    import torch

    import lasso_b200 as lb

    idx = skewed(700, 4, 8, 5)
    before = ctx.launches
    a = fields(lb.DensifiedRepresentation.from_lookup_indices(ctx, torch.from_numpy(idx.astype(np.int64)), 8))
    b = fields(lb.DensifiedRepresentation.from_lookup_indices(ctx, idx, 8))
    assert ctx.launches > before
    for x, y in zip(a, b):
        assert (x == y).all()


def test_rejects_other_shapes_and_dtypes(ctx):
    import torch

    import lasso_b200 as lb

    for bad in (torch.zeros(16, dtype=torch.int64, device="cuda"), torch.zeros(4, 4, 2, dtype=torch.int64, device="cuda"),
                torch.zeros(16, 2, dtype=torch.float32, device="cuda"), torch.zeros(16, 2, dtype=torch.int16, device="cuda")):
        with pytest.raises(TypeError):
            lb.DensifiedRepresentation.from_lookup_indices(ctx, bad, 4)


# ------------------------------------------------------------------ 2. proof bytes equal the oracle's
PROVE = [("prove_4d_lt", "int64", "row"), ("prove_4d_and", "uint32", "expand"), ("prove_3d_range", "int32", "col"),
         ("xor_c4", "uint64", "expand"), ("or_c2_ragged", "int64", "slice"), ("lt_c8", "int32", "row"),
         ("xor_c16_m16", "int64", "col"), ("range_c4", "uint64", "slice")]


def prove_and_check(ctx, kind, C_, log_m, log_r, idx, r, seed, indices, mutate=None):
    import lasso_b200 as lb

    s = 1 << max(0, (idx.shape[0] - 1).bit_length())
    S = lb.Strategy(kind, C_, log_m, log_r)
    need = lb.gens_points_needed(C_, s, S.num_memories, log_m)
    stream = np.ascontiguousarray(ol.generators(max(need, 300))[:need])
    gens = lb.SparsePolyCommitmentGens.new(ctx, b"gens_sparse_poly", C_, s, S.num_memories, log_m, stream=stream)
    dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, indices, log_m)
    if mutate is not None:
        mutate()
    commitment = dense.commit(gens)
    proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=seed)
    ref = ol.prove(kind, C_, log_m, log_r, idx, r, stream, seed, flags=1)
    assert ref["rc"] == 0
    assert commitment == ref["commitment"]
    assert len(proof.challenges) == len(ref["challenges"]) and (proof.challenges == ref["challenges"]).all()
    assert proof.bytes == ref["proof"]


@pytest.mark.parametrize("name,dtype,layout", PROVE)
def test_prove_from_cuda_tensor_matches_oracle(ctx, name, dtype, layout):
    _, kind, C_, log_m, log_r, n, same = next(c for c in CASES if c[0] == name)
    if layout == "expand":
        assert same, "a broadcast column needs a case with the same index in every dimension"
    idx, r, seed, _ = make_inputs(C_, log_m, n, len(name), same)
    prove_and_check(ctx, kind, C_, log_m, log_r, idx, r, seed, to_cuda(idx, dtype, layout))


# ------------------------------------------------------------------ 3. at size: the golden hashes
@pytest.mark.parametrize("name", ["xor_c4_s20", "lt_c8_s22", "rc40_c4_s24"])
def test_big_config_from_cuda_tensor_matches_golden(ctx, name):
    import torch

    import lasso_b200 as lb

    g = json.load(open(os.path.join(HERE, "golden", "big_proofs.json")))["cases"][name]
    kind, C_, log_m, log_r, log_s, idx, r, tape_seed = wl.config_inputs(name)
    assert hashlib.sha256(idx.tobytes()).hexdigest() == g["indices_sha256"]
    S = lb.Strategy(kind, C_, log_m, log_r)
    s = 1 << log_s
    stream = np.ascontiguousarray(ol.generators(lb.gens_points_needed(C_, s, S.num_memories, log_m)))
    gens = lb.SparsePolyCommitmentGens.new(ctx, b"gens_sparse_poly", C_, s, S.num_memories, log_m, stream=stream)
    t = torch.from_numpy(idx.astype(np.int64)).cuda()
    dense = lb.DensifiedRepresentation.from_lookup_indices(ctx, t, log_m)
    del t
    com = dense.commit(gens)
    proof = lb.SparsePolynomialEvaluationProof.prove(ctx, S, dense, r, gens, tape_seed=tape_seed)
    assert hashlib.sha256(com).hexdigest() == g["commitment_sha256"]
    assert hashlib.sha256(proof.bytes).hexdigest() == g["proof_sha256"]


# ------------------------------------------------------------------ 4. out of range
@pytest.mark.parametrize("dtype", DTYPES)
def test_out_of_range_then_the_context_still_proves(ctx, dtype):
    import lasso_b200 as lb

    log_m = 8
    idx = skewed(1000, 3, log_m, 9)
    bad = idx.copy()
    bad[-1, 2] = 1 << log_m  # == m, in the last row
    with pytest.raises(lb.LassoError) as e:
        lb.DensifiedRepresentation.from_lookup_indices(ctx, to_cuda(bad, dtype), log_m)
    assert e.value.code == 3
    if dtype.startswith("int"):
        neg = to_cuda(idx, dtype)
        neg[-1, 1] = -1
        with pytest.raises(lb.LassoError) as e:
            lb.DensifiedRepresentation.from_lookup_indices(ctx, neg, log_m)
        assert e.value.code == 3
        neg = to_cuda(idx, dtype)
        neg[0, 0] = -(1 << 31)
        with pytest.raises(lb.LassoError) as e:
            lb.DensifiedRepresentation.from_lookup_indices(ctx, neg, log_m)
        assert e.value.code == 3
    idx, r, seed, _ = make_inputs(3, log_m, 1000, 31, False)
    prove_and_check(ctx, 2, 3, log_m, 0, idx, r, seed, to_cuda(idx, dtype))


def test_bad_shapes_strides_and_dtype_are_rejected(ctx):
    import torch

    import lasso_b200 as lb

    t = torch.zeros(64, 4, dtype=torch.int64, device="cuda")
    L = lb.lib()

    def call(dtype=lb.IDX_I64, n=64, C_=4, rs=4, cs=1, log_m=8):
        h = ctypes.c_void_p()
        rc = L.lasso_densify_device(ctx._h, ctypes.c_void_p(t.data_ptr()), dtype, ctypes.c_size_t(n), ctypes.c_size_t(C_),
                                    ctypes.c_int64(rs), ctypes.c_int64(cs), ctypes.c_size_t(log_m), None, ctypes.byref(h))
        if rc == 0:
            L.lasso_dense_destroy(h)
        return rc

    assert call() == 0
    for kw in (dict(dtype=4), dict(dtype=-1), dict(rs=-4), dict(cs=-1), dict(n=0), dict(C_=0), dict(C_=17),
               dict(log_m=0), dict(log_m=29)):
        assert call(**kw) == 4, kw


# ------------------------------------------------------------------ 5. ordered after the producer's stream
def test_waits_for_the_producer_stream(ctx):
    import torch

    import lasso_b200 as lb

    log_m = 8
    idx = skewed(5000, 4, log_m, 3)
    src = torch.from_numpy(idx.astype(np.int64)).cuda()
    x = torch.zeros_like(src)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # ~0.1 s of spinning before the indices are written
        x.copy_(src)
        d = lb.DensifiedRepresentation.from_lookup_indices(ctx, x, log_m)
    got = fields(d)
    want = fields(lb.DensifiedRepresentation.from_lookup_indices(ctx, idx, log_m))
    for a, b in zip(got, want):
        assert (a == b).all()


# ------------------------------------------------------------------ 6. the buffer is free on return
def test_buffer_is_free_on_return(ctx):
    name = "xor_c4_indep"
    _, kind, C_, log_m, log_r, n, same = next(c for c in CASES if c[0] == name)
    idx, r, seed, _ = make_inputs(C_, log_m, n, 17, same)
    t = to_cuda(idx)
    prove_and_check(ctx, kind, C_, log_m, log_r, idx, r, seed, t, mutate=lambda: t.fill_(0))


# ------------------------------------------------------------------ 7. host memory is refused before any work
def test_host_pointer_rejected_before_any_launch(ctx):
    import torch

    import lasso_b200 as lb

    idx = skewed(1000, 4, 8, 1)
    pinned = torch.from_numpy(idx.astype(np.int64)).pin_memory()
    L = lb.lib()
    for ptr in (idx.ctypes.data, pinned.data_ptr()):
        before = ctx.launches
        h = ctypes.c_void_p()
        rc = L.lasso_densify_device(ctx._h, ctypes.c_void_p(ptr), lb.IDX_U64, ctypes.c_size_t(1000), ctypes.c_size_t(4),
                                    ctypes.c_int64(4), ctypes.c_int64(1), ctypes.c_size_t(8), None, ctypes.byref(h))
        assert rc < 0
        assert "not device memory" in L.lasso_last_error().decode()
        assert ctx.launches == before and not h.value


# ------------------------------------------------------------------ 8. one proof sharded over several ranks
def _run_sharded(nproc, same_gpu, timeout=1500):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ)
    if same_gpu:
        env["LASSO_SHARD_SAME_GPU"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "sharded_device_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    assert "SHARDED_DEVICE_CHECK PASS" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


def test_sharded_two_ranks_one_gpu_from_cuda_tensors():
    _run_sharded(2, True)


def test_sharded_four_ranks_one_gpu_from_cuda_tensors():
    _run_sharded(4, True)


def test_sharded_two_gpus_from_cuda_tensors():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (the one-GPU variants above cover the same code on this box)")
    _run_sharded(2, False)
