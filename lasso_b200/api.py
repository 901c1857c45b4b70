"""ctypes binding of liblasso_b200.so (include/lasso_b200.h) + the reference-shaped Python surface.

Field elements are numpy uint64 arrays (..., 4): ark-ff Montgomery limbs.  Affine points (..., 8),
extended points (..., 16)."""
import ctypes as C
import os
import sys

import numpy as np

AND, OR, XOR, LT, RANGE_CHECK = 0, 1, 2, 3, 4
IDX_U64, IDX_I64, IDX_U32, IDX_I32 = 0, 1, 2, 3  # LASSO_IDX_*: element types of lasso_densify_device
_HERE = os.path.dirname(os.path.abspath(__file__))


class LassoError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("lasso_b200 error %d: %s" % (code, msg))
        self.code = code


def library_path():
    return os.path.join(_HERE, "liblasso_b200.so")


_lib = None


def lib():
    """Load the CUDA extension.  Fails loudly if it has not been built — there is no other code path."""
    global _lib
    if _lib is None:
        p = library_path()
        if not os.path.exists(p):
            raise RuntimeError("liblasso_b200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(nvcc, sm_100a).  lasso_b200 has no CPU fallback.")
        L = C.CDLL(p)
        L.lasso_last_error.restype = C.c_char_p
        L.lasso_gens_points_needed.restype = C.c_size_t
        L.lasso_gens_points_needed.argtypes = [C.c_size_t] * 4
        L.lasso_dense_s.restype = C.c_size_t
        L.lasso_dense_read.restype = C.c_size_t
        L.lasso_launch_count.restype = C.c_ulonglong
        L.lasso_spans.restype = C.c_size_t
        _lib = L
    return _lib


def _chk(rc):
    if rc != 0:
        raise LassoError(rc, lib().lasso_last_error().decode())


def _p(a):
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def _fr(a, shape_last=4):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    assert a.shape[-1] == shape_last
    return a


def _ptr_array(arrays):
    arr = (C.c_void_p * len(arrays))()
    for i, a in enumerate(arrays):
        arr[i] = a.ctypes.data
    return arr


class Strategy:
    """SubtableStrategy<F, C, M> (src/subtables/mod.rs:31-93) as runtime parameters."""

    def __init__(self, kind, C_, log_m, log_r=0):
        self.kind, self.C, self.log_m, self.log_r = int(kind), int(C_), int(log_m), int(log_r)

    @property
    def num_subtables(self):
        return {LT: 2, RANGE_CHECK: 3}.get(self.kind, 1)

    @property
    def num_memories(self):
        return 2 * self.C if self.kind == LT else self.C

    @property
    def sumcheck_poly_degree(self):
        return (self.C if self.kind == LT else 1) + 1


class Context:
    """One per GPU: device, stream, memory pool, scratch."""

    def __init__(self, device=0):
        h = C.c_void_p()
        _chk(lib().lasso_ctx_create(C.byref(h), int(device)))
        self._h = h
        self.device = int(device)
        self._scratch = {}

    def _buf(self, name, shape, dtype):
        """Output staging reused across calls (a fresh 4 MiB np.zeros per commit / prove is an mmap + page faults +
        munmap inside the caller's timed region); contents are overwritten by the library before they are read."""
        b = self._scratch.get(name)
        if b is None or b.shape != tuple(np.atleast_1d(shape)) or b.dtype != np.dtype(dtype):
            b = np.zeros(shape, dtype=dtype)
            self._scratch[name] = b
        return b

    def close(self):
        if self._h:
            lib().lasso_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def init_comm(self, rank=None, world=None):
        """Shard ONE proof over the ranks of a torch.distributed job (one process per GPU, world a power of two
        <= 8, one node).  The 128-byte job id (random bytes naming the job's shared host segments, or the NCCL
        unique id under LASSO_B200_XCHG=nccl) is created on rank 0 and broadcast through torch.distributed
        (any backend).  Collective: every rank must call it."""
        import torch.distributed as dist

        from . import parallel

        rank = dist.get_rank() if rank is None else rank
        world = dist.get_world_size() if world is None else world
        ident = np.zeros(128, dtype=np.uint8)
        if rank == 0:
            _chk(lib().lasso_comm_unique_id(_p(ident)))
        ident = np.frombuffer(parallel.broadcast_bytes(ident.tobytes(), src=0), dtype=np.uint8).copy()
        _chk(lib().lasso_ctx_init_comm(self._h, _p(ident), int(rank), int(world)))
        self.rank, self.world = rank, world

    def bind_host_threads(self):
        """One process per GPU: pin the CALLING thread (the one that proves and spins on the round messages) to a
        dedicated core of the GPU's NUMA node and give the library's helper threads the rest of the node; returns the
        node id or -1 when the topology is not exposed.  Threads created earlier keep their affinity."""
        return int(lib().lasso_ctx_bind_host_threads(self._h))

    @property
    def launches(self):
        return int(lib().lasso_launch_count(self._h))

    def last_timings_ms(self):
        t = (C.c_double * 3)()
        lib().lasso_last_timings(self._h, t)
        return dict(densify=t[0], commit=t[1], prove=t[2])

    def spans(self):
        buf = C.create_string_buffer(8192)
        lib().lasso_spans(self._h, buf, C.c_size_t(8192))
        return dict((kv.split("=")[0], float(kv.split("=")[1])) for kv in buf.value.decode().split(";") if kv)

    def bench_bind(self, length, npolys, iters):
        ms = C.c_double(0)
        _chk(lib().lasso_bench_bind(self._h, C.c_size_t(length), int(npolys), int(iters), C.byref(ms)))
        return ms.value


# ------------------------------------------------------------------ per-loop entry points
def bind_top(ctx, Z, r):
    Z = _fr(Z).copy()
    _chk(lib().lasso_bind_top(ctx._h, _p(Z), C.c_size_t(Z.shape[0]), _p(_fr(r))))
    return Z[: Z.shape[0] // 2]


def bind_bot(ctx, Z, r):
    Z = _fr(Z).copy()
    _chk(lib().lasso_bind_bot(ctx._h, _p(Z), C.c_size_t(Z.shape[0]), _p(_fr(r))))
    return Z[: Z.shape[0] // 2]


def eq_evals(ctx, r):
    r = _fr(r).reshape(-1, 4)
    out = np.zeros((1 << r.shape[0], 4), dtype=np.uint64)
    _chk(lib().lasso_eq_evals(ctx._h, _p(r), int(r.shape[0]), _p(out)))
    return out


def sumcheck_round_arbitrary(ctx, S, polys):
    polys = [_fr(p) for p in polys]
    out = np.zeros((S.sumcheck_poly_degree + 1, 4), dtype=np.uint64)
    _chk(lib().lasso_sumcheck_round_arbitrary(ctx._h, S.kind, S.C, S.log_m, S.log_r, _ptr_array(polys),
                                              C.c_size_t(polys[0].shape[0]), _p(out)))
    return out


def sumcheck_bind_round_arbitrary(ctx, S, polys, r):
    """Bind every polynomial's top variable to r, then evaluate the next round: (bound polys, evals)."""
    polys = [_fr(p).copy() for p in polys]
    out = np.zeros((S.sumcheck_poly_degree + 1, 4), dtype=np.uint64)
    n = polys[0].shape[0]
    _chk(lib().lasso_sumcheck_bind_round_arbitrary(ctx._h, S.kind, S.C, S.log_m, S.log_r, _ptr_array(polys),
                                                   C.c_size_t(n), _p(_fr(r)), _p(out)))
    return [p[: n // 2] for p in polys], out


def sumcheck_round_cubic(ctx, A, B, Ceq):
    A = [_fr(a) for a in A]
    B = [_fr(b) for b in B]
    Ceq = _fr(Ceq)
    out = np.zeros((len(A), 3, 4), dtype=np.uint64)
    _chk(lib().lasso_sumcheck_round_cubic(ctx._h, len(A), _ptr_array(A), _ptr_array(B), _p(Ceq),
                                          C.c_size_t(Ceq.shape[0]), _p(out)))
    return out


def materialize_subtables(ctx, S):
    tabs = [np.zeros((1 << S.log_m, 4), dtype=np.uint64) for _ in range(S.num_subtables)]
    _chk(lib().lasso_materialize_subtables(ctx._h, S.kind, S.C, S.log_m, S.log_r, _ptr_array(tabs)))
    return tabs


def gather_lookup_polys(ctx, S, nz):
    nz = [np.ascontiguousarray(d, dtype=np.uint64) for d in nz]
    s = nz[0].shape[0]
    E = [np.zeros((s, 4), dtype=np.uint64) for _ in range(S.num_memories)]
    _chk(lib().lasso_gather_lookup_polys(ctx._h, S.kind, S.C, S.log_m, S.log_r, _ptr_array(nz), C.c_size_t(s),
                                         _ptr_array(E)))
    return E


def msm(ctx, bases_affine, scalars):
    bases = _fr(bases_affine, 8)
    sc = _fr(scalars)
    if bases.shape[0] != sc.shape[0]:  # VariableBaseMSM::msm -> Err(min_len), msm/mod.rs:36-40
        raise LassoError(1, "msm: bases.len() != scalars.len() (min = %d)" % min(bases.shape[0], sc.shape[0]))
    out = np.zeros(16, dtype=np.uint64)
    _chk(lib().lasso_msm(ctx._h, _p(bases), _p(sc), C.c_size_t(sc.shape[0]), _p(out)))
    return out


class MsmJob:
    """One VariableBaseMSM (msm/mod.rs:36-40) on device-resident inputs: n terms, term i uses base i % len(bases)."""

    def __init__(self, ctx, bases_affine, scalars):
        bases = _fr(bases_affine, 8)
        sc = _fr(scalars)
        h = C.c_void_p()
        _chk(lib().lasso_msm_job_create(ctx._h, _p(bases), C.c_size_t(bases.shape[0]), _p(sc), C.c_size_t(sc.shape[0]),
                                        C.byref(h)))
        self.ctx, self._h, self.n = ctx, h, sc.shape[0]

    def run(self, iters=1):
        """-> (extended point (16 u64), average ms per MSM, info dict)"""
        out = np.zeros(16, dtype=np.uint64)
        ms = C.c_double(0)
        info = (C.c_int * 8)()
        _chk(lib().lasso_msm_job_run(self.ctx._h, self._h, int(iters), C.byref(ms), _p(out), info))
        return out, ms.value, dict(c=info[0], windows=info[1], scalar_bits=info[2], unit=info[3], L=info[4], T2=info[5],
                                   world=info[6])

    def naive(self):
        out = np.zeros(16, dtype=np.uint64)
        _chk(lib().lasso_msm_job_naive(self.ctx._h, self._h, _p(out)))
        return out

    def close(self):
        if self._h:
            lib().lasso_msm_job_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            if self.ctx._h:
                self.close()
        except Exception:
            pass


def commit_rows(ctx, gens_affine, Z, L_size, R_size):
    g = _fr(gens_affine, 8)
    Z = _fr(Z)
    assert g.shape[0] >= R_size and Z.shape[0] == L_size * R_size
    out = np.zeros((L_size, 16), dtype=np.uint64)
    _chk(lib().lasso_commit_rows(ctx._h, _p(g), _p(Z), C.c_size_t(L_size), C.c_size_t(R_size), _p(out)))
    return out


def gens_points_needed(c, s, num_memories, log_m):
    return int(lib().lasso_gens_points_needed(c, s, num_memories, log_m))


def sample_generators(label, count):
    out = np.zeros((count, 8), dtype=np.uint64)
    _chk(lib().lasso_sample_generators(label, C.c_size_t(count), _p(out)))
    return out


# ------------------------------------------------------------------ the reference-shaped surface
class SparsePolyCommitmentGens:
    """src/lasso/surge.rs:25-58"""

    def __init__(self, ctx, handle, stream):
        self.ctx, self._h, self.stream = ctx, handle, stream

    @classmethod
    def new(cls, ctx, label, c, s, num_memories, log_m, stream=None):
        need = gens_points_needed(c, s, num_memories, log_m)
        if stream is None:
            stream = sample_generators(label, need)
        stream = _fr(stream, 8)
        h = C.c_void_p()
        _chk(lib().lasso_gens_create(ctx._h, _p(stream), C.c_size_t(stream.shape[0]), C.c_size_t(c), C.c_size_t(s),
                                     C.c_size_t(num_memories), C.c_size_t(log_m), C.byref(h)))
        return cls(ctx, h, stream)

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().lasso_gens_destroy(self._h)
        except Exception:
            pass


def _is_cuda_tensor(x):
    torch = sys.modules.get("torch")  # a tensor implies torch is loaded; api.py never imports it itself
    return torch is not None and isinstance(x, torch.Tensor) and x.is_cuda


class DensifiedRepresentation:
    """src/lasso/densified.rs:8-96 (device resident)"""

    def __init__(self, ctx, handle, C_, log_m):
        self.ctx, self._h, self.C, self.log_m = ctx, handle, C_, log_m
        self.s = int(lib().lasso_dense_s(handle))
        self.m = 1 << log_m

    @classmethod
    def from_lookup_indices(cls, ctx, indices, log_m):
        """indices: n x C lookup indices.  A CUDA torch.Tensor (int64, uint64, int32 or uint32, any strides) on the
        context's device is read in place, after the work queued on the current stream of its device; anything else is
        converted to a host uint64 array."""
        if _is_cuda_tensor(indices):
            return cls._from_cuda_tensor(ctx, indices, log_m)
        idx = np.ascontiguousarray(indices, dtype=np.uint64)
        assert idx.ndim == 2
        h = C.c_void_p()
        _chk(lib().lasso_densify(ctx._h, _p(idx), C.c_size_t(idx.shape[0]), C.c_size_t(idx.shape[1]),
                                 C.c_size_t(log_m), C.byref(h)))
        return cls(ctx, h, idx.shape[1], log_m)

    @classmethod
    def _from_cuda_tensor(cls, ctx, t, log_m):
        import torch

        codes = {torch.int64: IDX_I64, torch.int32: IDX_I32}
        for name, code in (("uint64", IDX_U64), ("uint32", IDX_U32)):
            if hasattr(torch, name):
                codes[getattr(torch, name)] = code
        if t.dim() != 2:
            raise TypeError("lookup indices must be a 2-D (n, C) tensor, got shape %s" % (tuple(t.shape),))
        if t.dtype not in codes:
            raise TypeError("lookup indices must be int64, uint64, int32 or uint32, got %s" % t.dtype)
        if t.device.index != ctx.device:
            raise ValueError("lookup indices are on cuda:%d, the context on cuda:%d" % (t.device.index, ctx.device))
        stream = torch.cuda.current_stream(t.device).cuda_stream
        h = C.c_void_p()
        _chk(lib().lasso_densify_device(ctx._h, C.c_void_p(t.data_ptr()), codes[t.dtype], C.c_size_t(t.shape[0]),
                                        C.c_size_t(t.shape[1]), C.c_int64(t.stride(0)), C.c_int64(t.stride(1)),
                                        C.c_size_t(log_m), C.c_void_p(stream), C.byref(h)))
        return cls(ctx, h, t.shape[1], log_m)

    def _read(self, which, n, width):
        out = np.zeros((n, width) if width > 1 else (n,), dtype=np.uint64)
        got = lib().lasso_dense_read(self.ctx._h, self._h, which, _p(out), C.c_size_t(n))
        assert got == n, (got, n)
        return out

    @property
    def dim_usize(self):
        return self._read(0, self.C * self.s, 1).reshape(self.C, self.s)

    @property
    def dim(self):
        return self._read(1, self.C * self.s, 4).reshape(self.C, self.s, 4)

    @property
    def read(self):
        return self._read(2, self.C * self.s, 4).reshape(self.C, self.s, 4)

    @property
    def final(self):
        return self._read(3, self.C * self.m, 4).reshape(self.C, self.m, 4)

    def commit(self, gens):
        cap = 1 << 22
        out = self.ctx._buf("commitment", cap, np.uint8)
        n = C.c_size_t(0)
        _chk(lib().lasso_commit(self.ctx._h, self._h, gens._h, _p(out), C.c_size_t(cap), C.byref(n)))
        return bytes(out[: n.value])

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().lasso_dense_destroy(self._h)
        except Exception:
            pass


class SparsePolynomialEvaluationProof:
    """src/lasso/surge.rs:92-211.  `.bytes` is the ark-serialize (compressed) encoding of the proof."""

    def __init__(self, data, challenges):
        self.bytes, self.challenges = data, challenges

    @classmethod
    def prove(cls, ctx, strategy, dense, r, gens, transcript_label=b"example", tape_label=b"proof", tape_seed=None):
        r = _fr(r).reshape(-1, 4)
        seed = _fr(tape_seed if tape_seed is not None else np.zeros(4, dtype=np.uint64))
        cap = 1 << 22
        out = ctx._buf("proof", cap, np.uint8)
        chal = ctx._buf("challenges", (1 << 14, 4), np.uint64)
        n, nch = C.c_size_t(0), C.c_size_t(0)
        _chk(lib().lasso_prove(ctx._h, strategy.kind, strategy.log_r, dense._h, _p(r), C.c_size_t(r.shape[0]), gens._h,
                               transcript_label, tape_label, _p(seed), _p(out), C.c_size_t(cap), C.byref(n), _p(chal),
                               C.c_size_t(chal.shape[0]), C.byref(nch)))
        return cls(bytes(out[: n.value]), chal[: nch.value].copy())
