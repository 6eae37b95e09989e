"""The product's host-side codecs (scroll-prover_b200/serde_bn254.hpp, SURVEY.md §8(f).3) on the reference's own files:
compressed G1 points and the `vk_*.vkey` layout (`SerdeFormat::Processed`).  The verifying keys shipped under
release-v0.13.1 must parse, every point must decompress to the coordinates chunk.protocol lists (where it lists them) and
re-serialise byte for byte.  CPU only (host build of csrc/ff.cuh)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_emul", "serde_host.cpp")
SO = os.path.join(HERE, "host_emul", "libserde_host.so")
HDRS = [os.path.join(HERE, "..", "scroll-prover_b200", p) for p in ("serde_bn254.hpp", os.path.join("csrc", "ff.cuh"))]
GOLD = json.load(open(os.path.join(HERE, "golden", "reference_fixtures.json")))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(p) for p in [SRC] + HDRS):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", SO, SRC])
    return C.CDLL(SO)


def read_vk(lib, raw: bytes):
    k, nf, npm = C.c_uint32(), C.c_uint32(), C.c_uint32()
    pts = np.zeros(((len(raw) - 8) // 32, 8), np.uint64)
    back = (C.c_uint8 * len(raw))()
    ok = lib.serde_host_read_vk(raw, C.c_uint64(len(raw)), C.byref(k), C.byref(nf), C.byref(npm), C.c_void_p(pts.ctypes.data), back)
    return ok, k.value, nf.value, npm.value, pts, bytes(back)


@pytest.mark.parametrize("name,k,n_fixed,n_perm", [("vk_chunk.vkey", 25, 4, 3), ("vk_batch.vkey", 26, 4, 5), ("vk_bundle.vkey", 26, 4, 3)])
def test_reference_vk_files_parse_and_round_trip(lib, name, k, n_fixed, n_perm):
    raw = bytes.fromhex(GOLD["files"][name]["hex"])
    ok, kk, nf, npm, pts, back = read_vk(lib, raw)
    assert ok == 1 and (kk, nf, npm) == (k, n_fixed, n_perm)
    assert back == raw  # decompress -> compress reproduces the file byte for byte
    assert pts.any(axis=1).all()  # no identity commitments in these keys


def test_vk_chunk_points_equal_the_protocols_preprocessed_points(lib):
    """chunk.protocol lists the same seven commitments as (x, y) Montgomery limbs: decompression must land on exactly those"""
    raw = bytes.fromhex(GOLD["files"]["vk_chunk.vkey"]["hex"])
    ok, _, _, _, pts, _ = read_vk(lib, raw)
    assert ok == 1
    pre = GOLD["chunk_protocol"]["preprocessed"]
    want = np.array([p["x"] + p["y"] for p in pre], dtype=np.uint64)
    assert np.array_equal(pts, want)


def test_identity_and_malformed_encodings(lib):
    out = np.zeros(8, np.uint64)
    ident = bytes(31) + b"\x80"
    assert lib.serde_host_decompress(ident, C.c_void_p(out.ctypes.data)) == 1 and not out.any()
    buf = (C.c_uint8 * 32)()
    lib.serde_host_compress(C.c_void_p(out.ctypes.data), buf)
    assert bytes(buf) == ident
    assert lib.serde_host_decompress(bytes(31) + b"\xc0", C.c_void_p(out.ctypes.data)) == 0        # identity with a sign bit
    assert lib.serde_host_decompress(b"\x01" + bytes(30) + b"\x80", C.c_void_p(out.ctypes.data)) == 0  # identity with x != 0
    q = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
    assert lib.serde_host_decompress(q.to_bytes(32, "little"), C.c_void_p(out.ctypes.data)) == 0    # x not reduced
    # x = 4: 4^3 + 3 = 67 is not a square mod q -> no point (checked against Euler's criterion)
    x = next(v for v in range(2, 50) if pow(v ** 3 + 3, (q - 1) // 2, q) != 1)
    assert lib.serde_host_decompress(x.to_bytes(32, "little"), C.c_void_p(out.ctypes.data)) == 0
    # truncated / inconsistent vk files
    raw = bytes.fromhex(GOLD["files"]["vk_chunk.vkey"]["hex"])
    assert read_vk(lib, raw[:-1])[0] == 0
    bad = bytearray(raw)
    bad[4:8] = (99).to_bytes(4, "big")  # more fixed commitments than points
    assert read_vk(lib, bytes(bad))[0] == 0


def test_generator_compresses_to_the_known_bytes(lib):
    # (1, 2): x = 1, y = 2 is even -> bit 254 clear
    one = (1 << 256) % 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
    two = 2 * one % 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
    limbs = lambda v: [(v >> (64 * i)) & (2**64 - 1) for i in range(4)]
    g = np.array(limbs(one) + limbs(two), dtype=np.uint64)
    buf = (C.c_uint8 * 32)()
    lib.serde_host_compress(C.c_void_p(g.ctypes.data), buf)
    assert bytes(buf) == (1).to_bytes(32, "little")
    out = np.zeros(8, np.uint64)
    assert lib.serde_host_decompress(bytes(buf), C.c_void_p(out.ctypes.data)) == 1 and np.array_equal(out, g)


def test_random_points_round_trip_and_agree_with_the_oracle(lib):
    """compress / decompress on 200 random curve points (both y parities): identity on the point, same bytes as the oracle's codec"""
    from oracle import oracle as O

    pts = O.fill_points(200, 0x5E4DE, 4)
    buf = (C.c_uint8 * 32)()
    out = np.zeros(8, np.uint64)
    parities = set()
    for p in pts:
        p = np.ascontiguousarray(p)
        lib.serde_host_compress(C.c_void_p(p.ctypes.data), buf)
        comp = bytes(buf)
        assert comp == O.g1_compress(p)
        parities.add(comp[31] >> 6 & 1)
        assert lib.serde_host_decompress(comp, C.c_void_p(out.ctypes.data)) == 1
        assert np.array_equal(out, p)
    assert parities == {0, 1}


def test_vk_bundle_points_are_the_constants_the_evm_verifier_hard_codes(lib):
    """Two artefacts of the reference tied together by OUR codec: the seven compressed commitments of release-v0.13.1/vk_bundle.vkey,
    decompressed (square root + sign bit) by the product's serde_bn254.hpp and by the oracle, are exactly the uncompressed (x, y)
    words the generated EVM verifier pushes (PUSH32) for its fixed / permutation commitments (evm_verifier.bin)."""
    from oracle import oracle as O
    from reference_data import REL

    raw = bytes.fromhex(GOLD["files"]["vk_bundle.vkey"]["hex"])
    code = open(os.path.join(REL, "evm_verifier.bin"), "rb").read()
    pushed = lambda v: b"\x7f" + v.to_bytes(32, "big") in code
    ok, _, _, _, pts, _ = read_vk(lib, raw)
    assert ok == 1 and len(pts) == 7
    for i, p in enumerate(pts):
        x, y = O.fq_to_int(p[:4]), O.fq_to_int(p[4:])
        assert pushed(x) and pushed(y), i
        assert np.array_equal(O.g1_decompress(raw[8 + 32 * i:40 + 32 * i]), p)
        assert not pushed(0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47 - y)  # the other square root is not in the program: the sign bit matters
