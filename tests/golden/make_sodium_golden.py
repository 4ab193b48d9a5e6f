"""libsodium's ristretto255 results on the inputs tests/test_oracle_group.py feeds the oracle: the hash-to-group map of sha512(b"pt%d"),
sums and differences of consecutive pairs, scalar multiples by numpy.random.default_rng(7) draws reduced mod q, the validity verdict on 300
sha256 strings, and a 16-term MSM over MultiCommitGens::new(16, b"sodium-msm").  Stored so that the differential test runs without libsodium.
Writes tests/golden/sodium_ristretto.json.
    python tests/golden/make_sodium_golden.py [path/to/libsodium.so]   (default: the copy bundled with pyzmq)"""
import ctypes as C
import glob
import hashlib
import json
import os
import site
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np
from oracle.spartan_ref import core as oc


def main():
    if len(sys.argv) > 1:
        path = sys.argv[1]
    else:
        path = [p for sp in site.getsitepackages() for p in glob.glob(sp + "/pyzmq.libs/libsodium*")][0]
    sod = C.CDLL(path)
    assert sod.sodium_init() >= 0
    o = C.create_string_buffer(32)
    rng = np.random.default_rng(7)
    out = {"from_hash": [], "add": [], "sub": [], "scalarmult": []}
    for i in range(40):
        sod.crypto_core_ristretto255_from_hash(o, C.c_char_p(hashlib.sha512(b"pt%d" % i).digest()))
        out["from_hash"].append(o.raw.hex())
    pts = [bytes.fromhex(h) for h in out["from_hash"]]
    for i in range(0, 40, 2):
        sod.crypto_core_ristretto255_add(o, C.c_char_p(pts[i]), C.c_char_p(pts[i + 1]))
        out["add"].append(o.raw.hex())
        sod.crypto_core_ristretto255_sub(o, C.c_char_p(pts[i]), C.c_char_p(pts[i + 1]))
        out["sub"].append(o.raw.hex())
        k = int.from_bytes(rng.bytes(32), "little") % oc.Q
        assert sod.crypto_scalarmult_ristretto255(o, C.c_char_p(k.to_bytes(32, "little")), C.c_char_p(pts[i])) == 0
        out["scalarmult"].append(o.raw.hex())
    out["valid"] = "".join("1" if sod.crypto_core_ristretto255_is_valid_point(C.c_char_p(hashlib.sha256(b"v%d" % i).digest())) else "0" for i in range(300))
    n = 16
    gens = oc.MultiCommitGens.new(n, b"sodium-msm")
    sc = oc.to_ints(oc.prg_scalars("s", n))
    acc = bytes(32)
    for i in range(n):
        sod.crypto_scalarmult_ristretto255(o, C.c_char_p(sc[i].to_bytes(32, "little")), C.c_char_p(gens.g(i).compress()))
        t = C.create_string_buffer(32)
        sod.crypto_core_ristretto255_add(t, C.c_char_p(acc), C.c_char_p(o.raw))
        acc = t.raw
    out["msm16"] = acc.hex()
    out["libsodium"] = os.path.basename(path)
    json.dump(out, open(os.path.join(ROOT, "tests", "golden", "sodium_ristretto.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
