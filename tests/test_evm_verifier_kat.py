"""The reference's EVM verifier PROGRAM run on the reference's shipped proof (SURVEY.md §8(c) fixture 3, §8(f).4; the `verifier
bytecode check` of BASELINE configs[4]): the deployed artefact release-v0.13.1/evm_verifier.bin is run by a small stack machine
(tests/evm_bytecode.py), which executes its constructor, takes the 13 987-byte runtime it returns and calls it with calldata =
proof.data with pi.data spliced in after the 12 accumulator limbs (the layer-6 EVM proof).  It must accept, with the precompile
and Keccak call counts the program's Yul source (evm_verifier.yul) has on the same calldata, and must reject when a byte of the
proof or of the public input is flipped.  The artefacts and the Yul run's counts are stored under tests/golden.

The elliptic-curve precompiles (ecAdd 0x06, ecMul 0x07, ecPairing 0x08) are served twice: by the independent big-integer model
and by the PRODUCT's host-side code (csrc/ec.cuh group law + pairing_bn254.hpp, through tests/host_emul/libpairing_host.so) --
so the product's verifier-side arithmetic is held to a complete real proof of the reference, not only to its accumulator.
CPU only."""
import ctypes as C
import os
import subprocess

from pairing_model import Q, g1_add, g1_mul, pairing_check
from reference_data import GOLD, REL
from yul_verifier import keccak256

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def be(v):
    return int(v).to_bytes(32, "big")


# ---- precompiles on the big-integer model
def on_curve(p):
    return p == (0, 0) or (p[0] < Q and p[1] < Q and (p[1] * p[1] - p[0] ** 3 - 3) % Q == 0)


def m_add(p, q):
    if not on_curve(p) or not on_curve(q):
        raise ValueError
    r = g1_add(None if p == (0, 0) else p, None if q == (0, 0) else q)
    return be(0) + be(0) if r is None else be(r[0]) + be(r[1])


def m_mul(p, k):
    if not on_curve(p):
        raise ValueError
    r = None if p == (0, 0) else g1_mul(p, k)
    return be(0) + be(0) if r is None else be(r[0]) + be(r[1])


def m_pairing(data):
    pairs = []
    for i in range(0, len(data), 192):
        w = [int.from_bytes(data[i + 32 * j:i + 32 * j + 32], "big") for j in range(6)]
        p1 = None if (w[0], w[1]) == (0, 0) else (w[0], w[1])
        q2 = ((w[3], w[2]), (w[5], w[4]))  # EIP-197 order (x_c1, x_c0, y_c1, y_c0)
        if p1 is not None:
            pairs.append((p1, q2))
    return be(1 if pairing_check(pairs) else 0)


# ---- precompiles on the product's host code
def host_lib():
    src = os.path.join(ROOT, "tests", "host_emul", "pairing_host.cpp")
    so = os.path.join(ROOT, "tests", "host_emul", "libpairing_host.so")
    hdrs = [os.path.join(ROOT, "scroll-prover_b200", h) for h in ("pairing_bn254.hpp", "csrc/ec.cuh", "csrc/ff.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in [src] + hdrs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src])
    lib = C.CDLL(so)
    for f in (lib.ec_host_add, lib.ec_host_mul, lib.pairing_host_eip197):
        f.restype = C.c_int
    return lib


def h_add_mul(lib):
    def add(p, q):
        out = C.create_string_buffer(64)
        if lib.ec_host_add(be(p[0]) + be(p[1]) + be(q[0]) + be(q[1]), out) != 0:
            raise ValueError
        return out.raw

    def mul(p, k):
        out = C.create_string_buffer(64)
        if lib.ec_host_mul(be(p[0]) + be(p[1]) + be(k), out) != 0:
            raise ValueError
        return out.raw

    def pairing(data):
        rc = lib.pairing_host_eip197(data, len(data) // 192)
        if rc < 0:
            raise ValueError
        return be(rc)

    return add, mul, pairing


def load():
    pi, proof = open(os.path.join(REL, "pi.data"), "rb").read(), open(os.path.join(REL, "proof.data"), "rb").read()
    # the reference's own test assembles the calldata like this (integration/tests/unit_tests.rs:30-32,
    # `proof.splice(384..384, pi)`): the 12 accumulator limbs, the 13 public-input words, then the proof proper
    return proof[:384] + pi + proof[384:]


def test_keccak256_known_answers():
    assert keccak256(b"").hex() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"
    assert keccak256(b"abc").hex() == "4e03657aea45a94fc7d47ba826c8d667c0d1e6e33a64a036ec44f58fa12d6c45"
    assert keccak256(bytes(200)).hex() != keccak256(bytes(201)).hex()  # multi-block inputs absorb every block


# ---- the deployed bytecode (evm_verifier.bin)
def load_bin():
    return open(os.path.join(REL, "evm_verifier.bin"), "rb").read()


def test_reference_verifier_bytecode_deploys_and_accepts_the_shipped_proof():
    from evm_bytecode import call, deploy

    calldata = load()
    assert len(calldata) == 416 + 1632
    runtime = deploy(load_bin())
    assert len(runtime) == 0x36A3  # the size the constructor pushes before CODECOPY
    ok, m = call(runtime, calldata, m_add, m_mul, m_pairing)
    assert ok
    # same work as the Yul source does: one pairing, the same EC and hash call counts
    y = GOLD["evm_verifier_yul_run"]
    assert y["accepted"] and m.precompile_calls[8] == 1
    assert m.precompile_calls == {int(a): n for a, n in y["precompile_calls"].items()} and m.keccak_calls == y["keccak_calls"]


def test_reference_verifier_bytecode_on_the_products_host_curve_and_pairing_code():
    from evm_bytecode import call, deploy

    calldata = load()
    runtime = deploy(load_bin())
    add, mul, pairing = h_add_mul(host_lib())
    ok, m = call(runtime, calldata, add, mul, pairing)
    assert ok and m.precompile_calls[8] == 1
    # a flipped byte anywhere -- a public input, a commitment, an evaluation, the last opening point -- is rejected
    for pos in (40, 384 + 5, 800 + 5, 800 + 700, len(calldata) - 3):
        bad = bytearray(calldata)
        bad[pos] ^= 1
        ok2, _ = call(runtime, bytes(bad), add, mul, pairing)
        assert not ok2, pos
    # a truncated proof is rejected as well (CALLDATALOAD past the end reads zeros: not a curve point / wrong pairing)
    ok3, _ = call(runtime, calldata[:-32], add, mul, pairing)
    assert not ok3


# ---- the PRODUCT's EVMVerifier (scroll-prover_b200/evm_verifier_b200.hpp): the same bytecode on a C++ stack machine whose
# precompiles are the product's host curve / pairing code -- the reference's integration/src/verifier.rs without an EVM
EVM_SRC = os.path.join(ROOT, "tests", "cpp", "test_evm_verifier.cpp")
EVM_BIN = os.path.join(ROOT, "tests", "cpp", "test_evm_verifier")


def evm_binary():
    deps = [EVM_SRC] + [os.path.join(ROOT, "scroll-prover_b200", h) for h in ("evm_verifier_b200.hpp", "keccak256.hpp", "pairing_bn254.hpp", "csrc/ec.cuh", "csrc/ff.cuh")]
    if not os.path.exists(EVM_BIN) or any(os.path.getmtime(d) > os.path.getmtime(EVM_BIN) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", EVM_BIN, EVM_SRC])
    return EVM_BIN


def product_evm(*extra):
    out = subprocess.run([evm_binary(), os.path.join(REL, "evm_verifier.bin"), os.path.join(REL, "proof.data"), os.path.join(REL, "pi.data"), *map(str, extra)],
                         capture_output=True, text=True, timeout=120).stdout.split()
    return out[0], dict(kv.split("=") for kv in out[1:])


def test_the_products_evm_verifier_accepts_the_shipped_proof_like_the_python_machine():
    from evm_bytecode import call, deploy

    verdict, info = product_evm()
    calldata = load()
    ok, m = call(deploy(load_bin()), calldata, m_add, m_mul, m_pairing)
    assert verdict == "ACCEPT" and ok
    assert int(info["runtime_bytes"]) == 0x36A3 and int(info["steps"]) == m.steps  # instruction for instruction
    assert (int(info["keccak"]), int(info["modexp"]), int(info["ecadd"]), int(info["ecmul"]), int(info["pairing"])) == \
        (m.keccak_calls, m.precompile_calls[5], m.precompile_calls[6], m.precompile_calls[7], m.precompile_calls[8])
    for pos in (40, 384 + 5, 800 + 5, 800 + 700, len(calldata) - 3):
        assert product_evm(pos)[0] == "REJECT", pos
    assert product_evm(-32)[0] == "REJECT"  # truncated


def test_the_products_evm_word_arithmetic_matches_python_integers():
    import random

    rnd = random.Random(0xE7)
    top = (1 << 256) - 1
    R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
    cases = [(0, 0, 0), (top, top, top), (top, top, 1), (top, 1, 0), (5, 3, 7), (top, top, Q), (Q - 1, Q - 1, Q), (R_MOD - 1, R_MOD - 2, R_MOD),
             (1 << 255, 1 << 255, (1 << 255) + 1), (top, 255, top - 1), (1, 256, 0), (12345, 64, 1 << 200)]
    cases += [(rnd.getrandbits(256), rnd.getrandbits(rnd.choice((8, 64, 256))), rnd.getrandbits(rnd.choice((1, 64, 255, 256)))) for _ in range(40)]
    for a, b, m in cases:
        out = subprocess.run([evm_binary(), "--arith", "%064x" % a, "%064x" % b, "%064x" % m], capture_output=True, text=True, timeout=60).stdout.split()
        got = [int(x, 16) for x in out]
        want = [(a + b) % m if m else 0, a * b % m if m else 0, a % m if m else 0, pow(a, b, m) if m else 0, (a + b) & top, (a - b) & top,
                (a << b) & top if b < 256 else 0]
        assert got == want, (hex(a), hex(b), hex(m))
