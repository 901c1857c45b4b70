"""Pin the oracle's twisted-Edwards group + the restated reference MSM (msm/mod.rs) against an
independent Python implementation and against libsodium (its answers stored in tests/golden/libsodium_ed25519.json
by tests/golden/make_libsodium.py)."""
import json
import os
import sys

import numpy as np
import pytest

import oracle_lib as ol
import pyref
from oracle_lib import L_FR, Q_FQ, P, fq_ints, fr_array, lib, sz

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SODIUM = json.load(open(os.path.join(GOLDEN, "libsodium_ed25519.json")))
sys.path.insert(0, GOLDEN)
from make_libsodium import scalars  # noqa: E402


def sodium_base_noclamp(k):
    return bytes.fromhex(SODIUM["base_noclamp"][hex(k)])


def sodium_add(a, b):
    """libsodium's sum of a * B and b * B"""
    return bytes.fromhex(SODIUM["add"]["%s+%s" % (hex(a), hex(b))])


def affine_ints(a):
    x, y = fq_ints(np.asarray(a).reshape(2, 4))
    return (x, y)


def ext_to_affine(pt):
    out = np.zeros(8, dtype=np.uint64)
    lib().orc_point_to_affine(P(pt), P(out))
    return affine_ints(out)


def mk_affine(pt):
    return np.concatenate([ol.to_mont(pt[0], Q_FQ), ol.to_mont(pt[1], Q_FQ)])


def test_generator_matches_libsodium():
    g = np.zeros(8, dtype=np.uint64)
    lib().orc_generator(P(g))
    gx, gy = affine_ints(g)
    assert (gx, gy) == (pyref.BX, pyref.BY)
    assert pyref.rfc8032_encode((gx, gy)) == sodium_base_noclamp(1)
    assert lib().orc_on_curve(P(g)) == 1


def test_scalar_mul_add_vs_libsodium_and_python():
    g = np.zeros(8, dtype=np.uint64)
    lib().orc_generator(P(g))
    G = np.zeros(16, dtype=np.uint64)
    lib().orc_point_from_affine(P(g), P(G))
    prev = prev_k = None
    for k in scalars():
        out = np.zeros(16, dtype=np.uint64)
        lib().orc_point_mul(P(G), P(ol.to_mont(k)), P(out))
        aff = ext_to_affine(out)
        assert pyref.rfc8032_encode(aff) == sodium_base_noclamp(k)
        assert aff == pyref.te_mul((pyref.BX, pyref.BY), k)
        comp = np.zeros(32, dtype=np.uint8)
        lib().orc_point_compress(P(out), P(comp))
        assert bytes(comp) == pyref.ark_encode(aff)
        dec = np.zeros(8, dtype=np.uint64)
        assert lib().orc_decompress(P(comp), P(dec)) == 0
        assert affine_ints(dec) == aff
        if prev is not None:
            s = np.zeros(16, dtype=np.uint64)
            lib().orc_point_add(P(out), P(prev), P(s))
            assert pyref.rfc8032_encode(ext_to_affine(s)) == sodium_add(k, prev_k)
            d = np.zeros(16, dtype=np.uint64)
            lib().orc_point_dbl(P(out), P(d))
            assert ext_to_affine(d) == pyref.te_add(aff, aff)
        prev, prev_k = out, k


def test_sampled_generators_are_prime_order_points():
    g = ol.generators(66)
    assert len({bytes(x) for x in g}) == 66
    lm = ol.to_mont(0)  # l == 0 mod l: multiply by canonical l through python instead
    for i in range(0, 66, 13):
        assert lib().orc_on_curve(P(g[i])) == 1
        assert pyref.te_mul(affine_ints(g[i]), L_FR) == (0, 1)
    # deterministic
    g2 = np.zeros((4, 8), dtype=np.uint64)
    lib().orc_sample_generators(sz(4), b"gens_sparse_poly", P(g2))
    assert (g2 == g[:4]).all()


def test_make_digits_recompose():
    rng = np.random.default_rng(5)
    for w in (3, 5, 8, 10, 13):
        for nbits in (16, 20, 60, 253):
            k = int.from_bytes(rng.bytes(32), "little") % (1 << nbits) % L_FR
            out = np.zeros(128, dtype=np.int64)
            cnt = ol.C.c_size_t(0)
            lib().orc_make_digits(P(ol.int_to_limbs(k)), sz(w), sz(nbits), P(out), ol.C.byref(cnt))
            digs = out[: cnt.value].tolist()
            assert cnt.value == (nbits + w - 1) // w
            assert sum(d << (w * i) for i, d in enumerate(digs)) == k
            assert all(-(1 << (w - 1)) <= d for d in digs[:-1]) and all(d < (1 << (w - 1)) + 1 for d in digs[:-1])


@pytest.mark.parametrize("n,bits", [(1, 253), (5, 253), (31, 8), (33, 16), (100, 253), (257, 20), (64, 1)])
def test_msm_wnaf_equals_naive_equals_python(n, bits):
    rng = np.random.default_rng(100 + n)
    bases = ol.generators(300)[:n]
    ks = [int.from_bytes(rng.bytes(40), "little") % L_FR % (1 << bits) for _ in range(n)]
    ks[0] = 0
    S = fr_array(ks)
    outs = []
    for hack in (1, 0, 2):
        o = np.zeros(16, dtype=np.uint64)
        lib().orc_msm(P(np.ascontiguousarray(bases)), P(S), sz(n), hack, P(o))
        outs.append(ext_to_affine(o))
    assert outs[0] == outs[1] == outs[2]
    if n <= 33:
        assert outs[0] == pyref.te_msm([affine_ints(b) for b in bases], ks)
