"""The product-side reader of snark-verifier `*.protocol` files (scroll-prover_b200/protocol_json.hpp, SURVEY.md §8(f).3) against
Python's own reading of the same JSON: on a small synthetic protocol and on the reference's shipped
release-v0.13.1/chunk.protocol (stored under tests/golden): the domain equals the C++ mirror's EvaluationDomain::new_(5, 25),
the 7 preprocessed commitments equal the points of vk_chunk.vkey as serde_bn254.hpp decodes them, and the proof size implied by
the protocol (5 witness commitments + 4 quotient chunks + 17 evaluations + 2 SHPLONK points) is the 896 bytes of the reference's
chunk proofs (integration/tests/test_data/full_proof_1.json)."""
import json
import os
import subprocess

from reference_data import REL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_protocol_json.cpp")
BIN = os.path.join(ROOT, "tests", "cpp", "test_protocol_json")


def binary():
    deps = [SRC] + [os.path.join(ROOT, "scroll-prover_b200", h) for h in ("protocol_json.hpp", "serde_bn254.hpp", "halo2_b200.hpp")]
    if not os.path.exists(BIN) or any(os.path.getmtime(d) > os.path.getmtime(BIN) for d in deps):
        lib = os.path.join(ROOT, "scroll-prover_b200")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", BIN, SRC, "-L" + lib, "-lb200zk", "-Wl,-rpath," + lib])
    return BIN


def run(*paths):
    r = subprocess.run([binary(), *paths], capture_output=True, text=True, timeout=60)
    return r.returncode, json.loads(r.stdout)


def check_against_python(path, out):
    d = json.load(open(path))
    assert out["k"] == d["domain"]["k"] and out["n"] == d["domain"]["n"] and out["n_inv"] == d["domain"]["n_inv"] and out["gen"] == d["domain"]["gen"]
    assert out["n_preprocessed"] == len(d["preprocessed"]) and out["last_preprocessed_y"] == d["preprocessed"][-1]["y"]
    assert out["num_instance"] == d["num_instance"] and out["num_witness"] == d["num_witness"] and out["num_challenge"] == d["num_challenge"]
    assert out["n_evaluations"] == len(d["evaluations"]) and out["n_queries"] == len(d["queries"])
    assert out["quotient"] == [d["quotient"]["num_chunk"], d["quotient"]["chunk_degree"]]
    assert out["numerator_root"] == next(iter(d["quotient"]["numerator"]))
    rots = [q["rotation"] for q in d["queries"]]
    assert out["rotations"] == [min(0, min(rots)), max(0, max(rots))]
    assert out["has_initial_state"] == (d["transcript_initial_state"] is not None)
    if out["has_initial_state"]:
        assert out["transcript_initial_state"] == d["transcript_initial_state"]
    assert out["accumulator_limbs"] == (len(d["accumulator_indices"][0]) if d["accumulator_indices"] else 0)
    assert out["proof_bytes_shplonk"] == 32 * (sum(d["num_witness"]) + d["quotient"]["num_chunk"] + len(d["evaluations"]) + 2)


def test_synthetic_protocol(tmp_path):
    """a small protocol in the same schema: u64 limbs above 2^63, a negative rotation, null optional fields"""
    proto = {"domain": {"k": 6, "n": 64, "n_inv": [18446744073709551615, 1, 2, 3], "gen": [4, 5, 6, 7], "gen_inv": [8, 9, 10, 11]},
             "preprocessed": [{"x": [1, 2, 3, 4], "y": [5, 6, 7, 9223372036854775809]}],
             "num_instance": [2], "num_witness": [3, 1], "num_challenge": [1, 2],
             "evaluations": [{"poly": 2, "rotation": 0}, {"poly": 2, "rotation": -1}, {"poly": 0, "rotation": 0}],
             "queries": [{"poly": 2, "rotation": 0}, {"poly": 2, "rotation": -1}, {"poly": 0, "rotation": 0}, {"poly": 6, "rotation": 0}],
             "quotient": {"num_chunk": 3, "chunk_degree": 1, "numerator": {"Sum": [{"Polynomial": {"poly": 2, "rotation": 0}}, {"Constant": [1, 0, 0, 0]}]}},
             "transcript_initial_state": None, "instance_committing_key": None, "linearization": None, "accumulator_indices": []}
    path = tmp_path / "mini.protocol"
    path.write_text(json.dumps(proto))
    rc, out = run(str(path))
    assert rc == 0 and out["vk_match"] == -1 and out["instances_committed"] is False
    check_against_python(str(path), out)
    # malformed inputs are reported, not crashed on
    bad = dict(proto, domain=dict(proto["domain"], n=63))
    path.write_text(json.dumps(bad))
    rc, out = run(str(path))
    assert rc == 1 and "2^k" in out["error"]
    path.write_text(json.dumps(proto)[:-20])
    rc, out = run(str(path))
    assert rc == 1 and "error" in out
    bad = dict(proto, queries=proto["queries"] + [{"poly": 9, "rotation": 0}])
    path.write_text(json.dumps(bad))
    rc, out = run(str(path))
    assert rc == 1 and "unknown polynomial" in out["error"]


def test_reference_chunk_protocol_matches_the_mirror_and_the_shipped_vk():
    rc, out = run(os.path.join(REL, "chunk.protocol"), os.path.join(REL, "vk_chunk.vkey"))
    assert rc == 0
    check_against_python(os.path.join(REL, "chunk.protocol"), out)
    assert out["k"] == 25 and out["domain_matches_mirror"] is True and out["vk_match"] == 1 and out["n_preprocessed"] == 7
    assert out["num_witness"] == [1, 1, 3] and out["quotient"] == [4, 1] and out["accumulator_limbs"] == 12
    assert out["proof_bytes_shplonk"] == 896  # the size of the reference's chunk proofs
