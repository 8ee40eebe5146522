#!/usr/bin/env python3
"""Regenerates tests/golden/libsodium_ristretto255.json: ristretto255 products computed by libsodium, an implementation
independent of the oracle (SURVEY.md A.5), for the seeded scalars of tests/test_oracle_kats.py::test_libsodium_cross_check.

    python tests/golden/make_libsodium_vectors.py [path/to/libsodium.so]

Without an argument it uses the libsodium that the pyzmq wheel bundles in the running interpreter's site-packages.
"""
import ctypes
import glob
import json
import pathlib
import random
import sys
import sysconfig

L = 2**252 + 27742317777372353535851937790883648493
OUT = pathlib.Path(__file__).with_name("libsodium_ristretto255.json")


def sc(x):
    return (x % L).to_bytes(32, "little")


def main():
    libs = sys.argv[1:] or glob.glob(sysconfig.get_paths()["purelib"] + "/pyzmq.libs/libsodium*.so*")
    if not libs:
        raise SystemExit("no libsodium found: pass its path")
    sodium = ctypes.CDLL(libs[0])
    rnd = random.Random(4)
    vectors = []
    for _ in range(5):
        k = sc(rnd.randrange(1, L))
        kb = ctypes.create_string_buffer(32)
        assert sodium.crypto_scalarmult_ristretto255_base(kb, k) == 0
        k2 = sc(rnd.randrange(1, L))
        k2kb = ctypes.create_string_buffer(32)
        assert sodium.crypto_scalarmult_ristretto255(k2kb, k2, kb.raw) == 0
        vectors.append({"k": k.hex(), "k_base": kb.raw.hex(), "k2": k2.hex(), "k2_k_base": k2kb.raw.hex()})
    sodium.sodium_version_string.restype = ctypes.c_char_p
    doc = {"_source": "libsodium %s crypto_scalarmult_ristretto255_base / crypto_scalarmult_ristretto255, scalars from "
                      "random.Random(4)" % sodium.sodium_version_string().decode(),
           "vectors": vectors}
    OUT.write_text(json.dumps(doc, indent=1) + "\n")
    print("wrote", OUT, "with", len(vectors), "vectors")


if __name__ == "__main__":
    main()
