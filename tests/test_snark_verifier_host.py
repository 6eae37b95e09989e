"""The product's host-side verifier for the reference's proof format (scroll-prover_b200/snark_verifier_b200.hpp: PlonkVerifier +
PoseidonTranscript + Bdfg21 + KZG decider, C++ mirror of snark-verifier @ 948671c as scroll-prover's ChunkVerifier / BatchVerifier use
it, integration/src/prove.rs:50-53,78-80 of the reference):

  * it ACCEPTS the reference's shipped chunk proofs (k = 25) and batch proofs (k = 26) from the protocol JSON, instances and proof
    bytes alone -- the same decisions as the independent big-integer model (tests/snark_verifier_model.py);
  * it rejects tampered proofs, wrong public inputs, a corrupted carried accumulator and another trusted setup;
  * it ACCEPTS the proofs our own create_proof makes with the Poseidon transcript (plonk_b200.hpp) under the exported protocol --
    i.e. prover and verifier of the product meet in the reference's format.
CPU only.  The reference's proofs are the sample stored in tests/golden/reference_proofs.json (tests/reference_data.py)."""
import base64
import json
import os
import subprocess

import pytest

from pairing_model import Q
from reference_data import GOLD, REL, proof_files_dir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_snark_verifier.cpp")
BIN = os.path.join(ROOT, "tests", "cpp", "test_snark_verifier")
DATA = proof_files_dir()
NEG_S_G2 = ((0x17944351223333f260ddc3b4af45191b856689eda9eab5cbcddbbe570ce860d2, 0x186282957db913abd99f91db59fe69922e95040603ef44c0bd7aa3adeef8f5ac),
            (0x06ecdb9f9567f59ed2eee36e1e1d58797fd13cc97fafc2910f5e8a12f202fa9a, 0x06d971ff4a7467c3ec596ed6efc674572e32fd6f52b721f97e35b0b3d3546753))
S_G2 = (NEG_S_G2[0], ((-NEG_S_G2[1][0]) % Q, (-NEG_S_G2[1][1]) % Q))


def binary():
    deps = [SRC] + [os.path.join(ROOT, "scroll-prover_b200", h) for h in ("snark_verifier_b200.hpp", "proof_files.hpp", "plonk_b200.hpp", "protocol_json.hpp", "pairing_bn254.hpp", "serde_bn254.hpp")]
    if not os.path.exists(BIN) or any(os.path.getmtime(d) > os.path.getmtime(BIN) for d in deps):
        lib = os.path.join(ROOT, "scroll-prover_b200")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", BIN, SRC, "-L" + lib, "-lb200zk", "-Wl,-rpath," + lib])
    return BIN


def g2_words(q):
    return ["%064x" % q[0][1], "%064x" % q[0][0], "%064x" % q[1][1], "%064x" % q[1][0]]


def verdict(tmp_path, proto, proof: bytes, instances, s_g2=S_G2):
    case = {"protocol": proto, "proof": proof.hex(), "instances": [["%064x" % v for v in col] for col in instances], "s_g2": g2_words(s_g2)}
    path = tmp_path / "case.json"
    path.write_text(json.dumps(case))
    return subprocess.run([binary(), str(path)], capture_output=True, text=True, timeout=120).stdout.strip()


def decode(entry):
    raw = base64.b64decode(entry["instances"])
    return json.loads(base64.b64decode(entry["protocol"])), base64.b64decode(entry["proof"]), [[int.from_bytes(raw[i:i + 32], "big") for i in range(0, len(raw), 32)]]


def test_reference_chunk_and_batch_proofs_are_accepted(tmp_path):
    from test_reference_proofs_kat import chunk_entries

    n = 0
    for name, i, e in chunk_entries():
        assert verdict(tmp_path, *decode(e)) == "ACCEPT", (name, i)
        n += 1
    for name in ("full_proof_batch_agg_1.json", "full_proof_batch_agg_2.json"):
        assert verdict(tmp_path, *decode(json.load(open(os.path.join(DATA, name))))) == "ACCEPT", name
        n += 1
    assert n == 10


def test_tampering_is_rejected(tmp_path):
    proto, proof, instances = decode(json.load(open(os.path.join(DATA, "full_proof_1.json")))["chunk_proofs"][0])
    for pos in (3, 200, 300, 500, 850, 895):
        bad = bytearray(proof)
        bad[pos] ^= 1
        assert verdict(tmp_path, proto, bytes(bad), instances).startswith("REJECT"), pos
    assert verdict(tmp_path, proto, proof[:-32], instances).startswith("REJECT")          # truncated
    assert verdict(tmp_path, proto, proof + bytes(32), instances).startswith("REJECT")  # trailing bytes
    wrong = [instances[0][:]]
    wrong[0][20] ^= 1   # a public input
    assert verdict(tmp_path, proto, proof, wrong).startswith("REJECT")
    wrong = [instances[0][:]]
    wrong[0][0] ^= 1    # a limb of the carried accumulator: the transcript changes AND the carried accumulator breaks
    assert verdict(tmp_path, proto, proof, wrong).startswith("REJECT")
    assert verdict(tmp_path, proto, proof, instances, s_g2=NEG_S_G2).startswith("REJECT")  # another (here: the negated) setup point
    assert verdict(tmp_path, proto, proof, instances) == "ACCEPT"


@pytest.mark.parametrize("k,seed,variant", [(6, 1, 1), (7, 4, 2), (7, 2, 3)])
def test_our_own_poseidon_proofs_are_accepted_under_the_exported_protocol(tmp_path, k, seed, variant):
    import test_plonk_session as TS

    _, out = TS.run("oracle", k, seed, variant)
    proofs, proto_text, instances, s_g2 = TS.parse_poseidon(out)
    proto, proof = json.loads(proto_text), proofs["oracle"]
    assert verdict(tmp_path, proto, proof, instances, s_g2=s_g2) == "ACCEPT"
    bad = bytearray(proof)
    bad[len(bad) // 3] ^= 1
    assert verdict(tmp_path, proto, bytes(bad), instances, s_g2=s_g2).startswith("REJECT")


def verify_file(path, s_g2=S_G2, tamper=False):
    r = subprocess.run([binary(), "--file", str(path)] + g2_words(s_g2) + (["--tamper"] if tamper else []), capture_output=True, text=True, timeout=600)
    lines = r.stdout.strip().splitlines()
    accepted, total = int(lines[-1].split()[1]), int(lines[-1].split()[3])
    return accepted, total, lines[:-1]


def test_every_proof_file_the_reference_ships_is_read_and_accepted():
    """scroll-prover_b200/proof_files.hpp reads the reference's proof files AS WRITTEN (serde_json objects with base64 fields, the
    chunk_proofs containers of batch tasks) and runs verify_chunk_proof / verify_batch_proof on every proof object in them: the 8
    stored chunk proofs (of the reference's 319) and both batch proofs are accepted -- the protocol they carry, the proof, the carried
    accumulator, and the vk bytes beside them matching the protocol's preprocessed commitments."""
    files = [os.path.join(DATA, name) for name in GOLD["files"]]
    chunk = batch = 0
    for f in files:
        accepted, total, lines = verify_file(f)
        assert accepted == total and total >= 1, (f, [l for l in lines if not l.startswith("ACCEPT")][:3])
        chunk += sum(1 for l in lines if l.startswith("ACCEPT chunk k=25 proof_bytes=896"))
        batch += sum(1 for l in lines if l.startswith("ACCEPT batch k=26"))
    assert (chunk, batch) == (8, 2)
    # and every one of those chunk proofs was made for the RELEASED circuit: the vk and the protocol it carries are byte-for-byte
    # release-v0.13.1/vk_chunk.vkey and chunk.protocol (four different git versions of the prover among them)
    rel_vk = open(os.path.join(REL, "vk_chunk.vkey"), "rb").read()
    rel_proto = json.load(open(os.path.join(REL, "chunk.protocol")))
    versions = set()
    for f in files:
        for cp in json.load(open(f)).get("chunk_proofs", []):
            assert base64.b64decode(cp["vk"]) == rel_vk and json.loads(base64.b64decode(cp["protocol"])) == rel_proto
            versions.add(cp["git_version"])
    assert len(versions) == 4


def test_proof_files_with_a_flipped_proof_byte_or_another_setup_are_rejected(tmp_path):
    f = os.path.join(DATA, "batch-task-with-blob-raw.json")
    assert verify_file(f)[:2] == (4, 4)
    assert verify_file(f, tamper=True)[:2] == (0, 4)
    assert verify_file(f, s_g2=NEG_S_G2)[:2] == (0, 4)
    # a vk that belongs to another circuit beside the proof: refused before any pairing
    j = json.load(open(os.path.join(DATA, "full_proof_1.json")))
    j["chunk_proofs"][0]["vk"] = json.load(open(os.path.join(DATA, "full_proof_batch_agg_1.json")))["vk"]
    p = tmp_path / "swapped_vk.json"
    p.write_text(json.dumps(j))
    accepted, total, lines = verify_file(p)
    assert (accepted, total) == (0, 1) and "vk" in lines[0]
    # malformed base64 is an error, not a crash
    j["chunk_proofs"][0]["vk"] = "@@@@"
    p.write_text(json.dumps(j))
    r = subprocess.run([binary(), "--file", str(p)] + g2_words(S_G2), capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and r.stdout.startswith("REJECT exception")


def test_keccak256_of_the_proof_file_reader_known_answers():
    from yul_verifier import keccak256

    for msg in (b"", b"abc", bytes(range(135)), bytes(range(136)), bytes(range(200)) * 3):
        out = subprocess.run([binary(), "--keccak", msg.hex()], capture_output=True, text=True, timeout=60).stdout.strip()
        assert out == keccak256(msg).hex()
    assert subprocess.run([binary(), "--keccak", ""], capture_output=True, text=True).stdout.strip() == "c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470"


def test_a_chunk_proof_is_bound_to_the_chunk_info_beside_it(tmp_path):
    """instances[12..44] = keccak256(chain_id || prev_state_root || post_state_root || withdraw_root || data_hash || keccak256(tx_bytes)):
    true for every shipped chunk proof (test_every_proof_file_... goes through the same check); any changed field is refused"""
    j = json.load(open(os.path.join(DATA, "full_proof_1.json")))
    p = tmp_path / "edited.json"
    for field, edit in (("chain_id", lambda v: v + 1), ("post_state_root", lambda v: v[:-1] + ("0" if v[-1] != "0" else "1")),
                        ("tx_bytes", lambda v: base64.b64encode(base64.b64decode(v) + b"\x00").decode())):
        k = json.loads(json.dumps(j))
        k["chunk_proofs"][0]["chunk_info"][field] = edit(k["chunk_proofs"][0]["chunk_info"][field])
        p.write_text(json.dumps(k))
        accepted, total, lines = verify_file(p)
        assert (accepted, total) == (0, 1) and "chunk_info" in lines[0], field
    p.write_text(json.dumps(j))
    assert verify_file(p)[:2] == (1, 1)


def test_a_batch_proof_carries_its_batch_hash_and_the_second_continues_the_first(tmp_path):
    b1, b2 = (json.load(open(os.path.join(DATA, f"full_proof_batch_agg_{i}.json"))) for i in (1, 2))
    w1, w2 = decode(b1)[2][0], decode(b2)[2][0]
    assert len(w1) == 23 and (w1[18] << 128) | w1[19] == int(b1["batch_hash"], 16) and (w2[18] << 128) | w2[19] == int(b2["batch_hash"], 16)
    assert w2[12:16] == w1[16:20] and w1[20] == w2[20]  # parent state root / batch hash of #2 = current of #1; same chain id
    p = tmp_path / "edited.json"
    b1["batch_hash"] = b1["batch_hash"][:-1] + ("0" if b1["batch_hash"][-1] != "0" else "1")
    p.write_text(json.dumps(b1))
    accepted, total, lines = verify_file(p)
    assert (accepted, total) == (0, 1) and "batch_hash" in lines[0]


def batch_task(path):
    out = subprocess.run([binary(), "--batch-task", str(path)], capture_output=True, text=True, timeout=120).stdout.strip()
    fields = dict(kv.split("=") for kv in out.split() if "=" in kv)
    return out.split()[0], fields, out


def test_batch_tasks_are_consistent_and_their_header_hashes_chain(tmp_path):
    """proof_files.hpp reads the reference's batch proving tasks (chunk_infos + chunk_proofs + batch_header): every chunk info is the
    one its proof carries, state roots chain, header.data_hash = keccak(chunk data hashes); BatchHeader::batch_hash (keccak of the
    193-byte encoding) is pinned by the reference's data twice: the headers of the ten consecutive tasks 293205..293214 chain through
    parent_batch_hash, and the header of full_proof_batch_prove_1.json hashes to the batch_hash of the batch proof made from it.
    Of those ten tasks only the headers are stored: a header without chunks is still hashed, and the task is refused."""
    p = tmp_path / "task.json"
    prev = None
    for index, header in sorted(GOLD["batch_headers"].items()):
        p.write_text(json.dumps({"chunk_infos": [], "chunk_proofs": [], "batch_header": header}))
        verdict, info, out = batch_task(p)
        assert verdict == "INCONSISTENT" and "one chunk info per chunk proof" in out and info["chunks"] == "0", out
        if prev is not None:
            assert info["parent"] == prev, index
        prev = info["batch_hash"]
    assert len(GOLD["batch_headers"]) == 10
    raw = os.path.join(DATA, "batch-task-with-blob-raw.json")
    verdict, info, out = batch_task(raw)
    assert verdict == "CONSISTENT" and info["chunks"] == "4", out
    # the batch proof full_proof_batch_agg_1.json was made from the task full_proof_batch_prove_1.json: same batch hash
    j = json.load(open(os.path.join(DATA, "full_proof_batch_prove_1.json")))
    j["chunk_infos"] = [cp["chunk_info"] for cp in j["chunk_proofs"]]
    p.write_text(json.dumps(j))
    verdict, info, out = batch_task(p)
    assert verdict == "CONSISTENT"
    # and all 11 public inputs of that batch proof are the ones the task determines (roots, hashes, chain id); not those of another task
    agg = os.path.join(DATA, "full_proof_batch_agg_1.json")
    out = subprocess.run([binary(), "--batch-task", str(p), agg], capture_output=True, text=True, timeout=120).stdout
    assert "proof_matches_task=1" in out
    out = subprocess.run([binary(), "--batch-task", raw, agg], capture_output=True, text=True, timeout=120).stdout
    assert "proof_matches_task=0" in out
    assert "0x" + info["batch_hash"] == json.load(open(os.path.join(DATA, "full_proof_batch_agg_1.json")))["batch_hash"], out
    # inconsistencies are named
    t = json.load(open(raw))
    t["chunk_infos"][3]["post_state_root"] = t["chunk_infos"][3]["post_state_root"][:-1] + ("0" if t["chunk_infos"][3]["post_state_root"][-1] != "0" else "1")
    p.write_text(json.dumps(t))
    assert batch_task(p)[0] == "INCONSISTENT"
    t = json.load(open(raw))
    t["chunk_infos"], t["chunk_proofs"] = t["chunk_infos"][:-1], t["chunk_proofs"][:-1]
    p.write_text(json.dumps(t))
    verdict, _, out = batch_task(p)
    assert verdict == "INCONSISTENT" and "data_hash" in out
