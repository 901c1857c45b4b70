"""ctypes loader for the CPU oracle (oracle/, test infrastructure only).

Field elements are numpy uint64 arrays of shape (..., 4): ark-ff Montgomery limbs.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_build", "liblasso_oracle.so")

L_FR = 2**252 + 27742317777372353535851937790883648493
Q_FQ = 2**255 - 19
R256 = 2**256

u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)


def build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            build()
        _lib = C.CDLL(SO)
        _lib.orc_num_memories.restype = C.c_size_t
        _lib.orc_num_subtables.restype = C.c_size_t
        _lib.orc_transcript_new.restype = C.c_void_p
        _lib.orc_spans.restype = C.c_size_t
    return _lib


def P(a):
    """pointer to a contiguous numpy array"""
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def sz(n):
    return C.c_size_t(int(n))


# ---- python big-int <-> limb helpers (independent of the oracle) ----
def int_to_limbs(x):
    return np.array([(x >> (64 * i)) & (2**64 - 1) for i in range(4)], dtype=np.uint64)


def limbs_to_int(a):
    a = np.asarray(a, dtype=np.uint64).reshape(-1)
    return sum(int(a[i]) << (64 * i) for i in range(4))


def to_mont(x, p=L_FR):
    return int_to_limbs((x % p) * R256 % p)


def from_mont(a, p=L_FR):
    return limbs_to_int(a) * pow(R256, -1, p) % p


def fr_array(ints):
    """list of python ints -> (n,4) uint64 Montgomery Fr array"""
    out = np.zeros((len(ints), 4), dtype=np.uint64)
    for i, x in enumerate(ints):
        out[i] = to_mont(x, L_FR)
    return out


def fr_ints(arr):
    arr = np.asarray(arr, dtype=np.uint64).reshape(-1, 4)
    return [from_mont(arr[i], L_FR) for i in range(arr.shape[0])]


def fq_array(ints):
    out = np.zeros((len(ints), 4), dtype=np.uint64)
    for i, x in enumerate(ints):
        out[i] = to_mont(x, Q_FQ)
    return out


def fq_ints(arr):
    arr = np.asarray(arr, dtype=np.uint64).reshape(-1, 4)
    return [from_mont(arr[i], Q_FQ) for i in range(arr.shape[0])]


def rand_fr(rng, n):
    """n uniform Fr elements (Montgomery limbs) from a numpy Generator"""
    return fr_array([int.from_bytes(rng.bytes(40), "little") % L_FR for _ in range(n)])


def f_op(which, op, a, b=None):
    out = np.zeros(4, dtype=np.uint64)
    lib().orc_f_op(which, op, P(np.ascontiguousarray(a)), P(np.ascontiguousarray(b)) if b is not None else None, P(out))
    return out


# ---- generators (cached on disk: sampling needs one sqrt + cofactor clearing per point) ----
_gens_cache = {}


def generators(count, label=b"gens_sparse_poly", persist=True):
    """The first `count` points of the oracle's generator stream; persist=False never writes the on-disk cache (for
    callers that must leave the source tree as they found it, such as bench.py)."""
    key = (label,)
    have = _gens_cache.get(key)
    if have is not None and have.shape[0] >= count:
        return have[:count]
    cache = os.path.join(ROOT, "oracle", "_build", "gens_%s_%d.npy" % (label.decode(), count))
    if os.path.exists(cache):
        g = np.load(cache)
    else:
        g = np.zeros((count, 8), dtype=np.uint64)
        lib().orc_sample_generators(sz(count), label, P(g))
        if persist:
            np.save(cache, g)
    _gens_cache[key] = g
    return g


STRATS = {"and": 0, "or": 1, "xor": 2, "lt": 3, "range": 4}


def prove(kind, Cdim, log_m, log_r, indices, r, gens, tape_seed, flags=1, nthreads=None):
    """Run Densify -> commit -> prove (-> verify) in the oracle.
    indices: (n, C) uint64.  Returns dict(rc, proof, commitment, challenges, timings_ms, spans)."""
    L = lib()
    if nthreads:
        L.orc_set_num_threads(int(nthreads))
    indices = np.ascontiguousarray(indices, dtype=np.uint64)
    n = indices.shape[0]
    cap = 1 << 24
    proof = np.zeros(cap, dtype=np.uint8)
    comm = np.zeros(cap, dtype=np.uint8)
    chal = np.zeros((1 << 16, 4), dtype=np.uint64)
    plen, clen, nch = C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
    tm = np.zeros(4, dtype=np.float64)
    r = np.ascontiguousarray(r, dtype=np.uint64)
    gens = np.ascontiguousarray(gens, dtype=np.uint64)
    tape_seed = np.ascontiguousarray(tape_seed, dtype=np.uint64)
    rc = L.orc_prove(int(kind), sz(Cdim), sz(log_m), sz(log_r), P(indices), sz(n), P(r), P(gens), sz(gens.shape[0]),
                     P(tape_seed), int(flags), P(proof), sz(cap), C.byref(plen), P(comm), sz(cap), C.byref(clen),
                     P(chal), sz(chal.shape[0]), C.byref(nch), P(tm))
    buf = C.create_string_buffer(4096)
    L.orc_spans(buf, sz(4096))
    spans = dict((kv.split("=")[0], float(kv.split("=")[1])) for kv in buf.value.decode().split(";") if kv)
    return dict(rc=rc, proof=bytes(proof[: plen.value]), commitment=bytes(comm[: clen.value]),
                challenges=chal[: nch.value].copy(), timings_ms=tm, spans=spans)
