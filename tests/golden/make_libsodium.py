"""Generate tests/golden/libsodium_ed25519.json: libsodium's answers (through PyNaCl) for the points
tests/test_oracle_curve.py checks the oracle's group law against, so that the comparison needs no PyNaCl at test time.

    base_noclamp[hex(k)]      crypto_scalarmult_ed25519_base_noclamp(k)  = RFC 8032 encoding of k * B
    add["hex(a)+hex(b)"]      crypto_core_ed25519_add(a * B, b * B)      for consecutive scalars of scalars()

Regenerate with:  python tests/golden/make_libsodium.py   (needs PyNaCl)
"""
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
L_FR = 2**252 + 27742317777372353535851937790883648493


def scalars():
    """the seeded scalars of test_scalar_mul_add_vs_libsodium_and_python"""
    rng = np.random.default_rng(11)
    return [int.from_bytes(rng.bytes(40), "little") % L_FR for _ in range(12)]


def main():
    import nacl
    import nacl.bindings as nb

    def mul(k):
        return nb.crypto_scalarmult_ed25519_base_noclamp(k.to_bytes(32, "little"))

    ks = scalars()
    out = {"source": "libsodium (bundled with PyNaCl %s)" % nacl.__version__,
           "base_noclamp": {hex(k): mul(k).hex() for k in [1] + ks},
           "add": {"%s+%s" % (hex(a), hex(b)): nb.crypto_core_ed25519_add(mul(a), mul(b)).hex()
                   for a, b in zip(ks[1:], ks[:-1])}}
    with open(os.path.join(HERE, "libsodium_ed25519.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", len(out["base_noclamp"]), "products and", len(out["add"]), "sums")


if __name__ == "__main__":
    main()
