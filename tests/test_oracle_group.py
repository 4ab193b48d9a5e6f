"""ristretto255 restatement (oracle/csrc/ristretto.c) pinned against RFC 9496 appendix A vectors and,
as an independent differential oracle, libsodium's results on the same inputs (tests/golden/sodium_ristretto.json, made by
tests/golden/make_sodium_golden.py) — SURVEY.md §8c item 3.
The reference holds no group-level known answers (its group is curve25519-dalek, a third-party crate)."""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle.spartan_ref import core as oc

SODIUM = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sodium_ristretto.json")))

# RFC 9496 A.1: multiples 0..4 of the generator
RFC_MULTIPLES = [
    "0000000000000000000000000000000000000000000000000000000000000000",
    "e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76",
    "6a493210f7499cd17fecb510ae0cea23a110e8d5b901f8acadd3095c73a3b919",
    "94741f5d5d52755ece4f23f044ee27d5d1ea1e2bd196b462166b16152a9d0259",
    "da80862773358b466ffadfe0b3293ab3d9fd53c5ea6c955358f568322daf6a57",
]


def test_rfc9496_basepoint_multiples():
    B = oc.Point.decompress(oc.BASEPOINT_COMPRESSED)
    acc = oc.Point.identity()
    for h in RFC_MULTIPLES:
        assert acc.compress().hex() == h
        acc = acc + B
    assert (B * 3).compress().hex() == RFC_MULTIPLES[3]


def test_decode_rejects_bad_encodings():
    # RFC 9496 A.2: non-canonical field encodings and negative field elements
    bad = [
        "00ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff",
        "ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        "f3ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        "edffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
        "0100000000000000000000000000000000000000000000000000000000000000",
        "01ffffffffffffffffffffffffffffffffffffffffffffffffffffffffffff7f",
    ]
    for h in bad:
        assert oc.Point.decompress(bytes.fromhex(h)) is None


def test_differential_vs_libsodium():
    rng = np.random.default_rng(7)
    pts = []
    for i in range(40):
        h = hashlib.sha512(b"pt%d" % i).digest()
        want = bytes.fromhex(SODIUM["from_hash"][i])
        mine = oc.Point.from_uniform_bytes(h)
        assert mine.compress() == want
        assert oc.Point.decompress(want).compress() == want
        pts.append(mine)
    for j, i in enumerate(range(0, 40, 2)):
        assert (pts[i] + pts[i + 1]).compress().hex() == SODIUM["add"][j]
        assert (pts[i] - pts[i + 1]).compress().hex() == SODIUM["sub"][j]
        k = int.from_bytes(rng.bytes(32), "little") % oc.Q
        assert (pts[i] * k).compress().hex() == SODIUM["scalarmult"][j]
    # validity of random byte strings agrees
    assert len(SODIUM["valid"]) == 300
    for i in range(300):
        b = hashlib.sha256(b"v%d" % i).digest()
        assert (oc.Point.decompress(b) is not None) == (SODIUM["valid"][i] == "1")


@pytest.mark.parametrize("n", [1, 2, 5, 33, 189, 190, 600, 1024])
def test_msm_matches_naive(n):
    """vartime_multiscalar_mul (group.rs:98-117): Straus / Pippenger paths against sum of scalar mults"""
    gens = oc.MultiCommitGens.new(n, b"test-msm")
    sc = oc.prg_scalars("msm%d" % n, n)
    if n >= 3:
        sc[0] = 0
        sc[1] = oc.to_arr([1])[0]
        sc[2] = oc.to_arr([oc.Q - 1])[0]
    got = oc.msm(sc, gens.G)
    ints = oc.to_ints(sc)
    if n <= 33:
        acc = oc.Point.identity()
        for i in range(n):
            acc = acc + gens.g(i) * ints[i]
        assert got.compress() == acc.compress()
    # linearity: MSM(2s) == 2*MSM(s)
    got2 = oc.msm([(2 * v) % oc.Q for v in ints], gens.G)
    assert got2.compress() == (got + got).compress()


def test_msm_vs_libsodium():
    """sum of libsodium's scalar multiples of the 16 generators (tests/golden/make_sodium_golden.py) against the oracle's MSM"""
    n = 16
    gens = oc.MultiCommitGens.new(n, b"sodium-msm")
    sc = oc.to_ints(oc.prg_scalars("s", n))
    assert oc.msm(sc, gens.G).compress().hex() == SODIUM["msm16"]


def test_gens_prefix_sharing():
    """r1csproof.rs:48-58: gens_3 / gens_4 built from the same label share the SHAKE prefix of gens_n"""
    g5 = oc.MultiCommitGens.new(5, b"gens_r1cs_sat")
    g3 = oc.MultiCommitGens.new(3, b"gens_r1cs_sat")
    assert np.array_equal(g3.G, g5.G[:3])
    assert g3.h.compress() == g5.g(3).compress()
    # generator derivation is exactly the RFC one-way map of consecutive 64-byte SHAKE blocks (commitments.rs:15-33)
    stream = hashlib.shake_256(b"gens_r1cs_sat" + oc.BASEPOINT_COMPRESSED).digest(64 * 6)
    assert oc.Point.from_uniform_bytes(stream[64:128]).compress() == g5.g(1).compress()
    assert g5.h.compress() == oc.Point.from_uniform_bytes(stream[320:384]).compress()
