"""Stores the reference's proof files and release artefacts that the verifier tests read, sampled to stay small:
    python tests/golden/make_reference_proofs.py <scroll-prover checkout>

Writes
  release-v0.13.1/   chunk.protocol, vk_chunk.vkey, evm_verifier.bin, proof.data, pi.data, byte for byte;
  reference_proofs.json
    "files"          proof files of integration/tests/test_data in their own JSON layout.  Kept whole: full_proof_1,
                     full_proof_batch_prove_1, full_proof_batch_agg_{1,2} and the 4-chunk batch-task-with-blob-raw task (less its
                     blob_bytes).  Sampled: the chunk proof with the shortest tx_bytes of batch-task-with-blob.json and of
                     batch_tasks/batch_task_293209.json, stored as plain chunk-proof lists.  Together they hold 8 chunk proofs of all
                     4 prover versions the test data has, and both batch proofs.
    "shared"         the protocol strings every chunk proof (and both batch proofs) carry, stored once; a proof object's
                     "protocol" field names its entry here.
    "batch_headers"  the headers of the ten consecutive tasks batch_tasks/batch_task_2932{05..14}.json.
    "evm_verifier_yul_run"  what the Yul source of the EVM verifier (release-v0.13.1/evm_verifier.yul) does on
                     proof.data with pi.data spliced in: its verdict and its precompile / Keccak call counts.
tests/reference_data.py writes the proof files back out for the tests."""
import base64
import glob
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
RELEASE = ("chunk.protocol", "vk_chunk.vkey", "evm_verifier.bin", "proof.data", "pi.data")


def main(ref):
    data = os.path.join(ref, "integration", "tests", "test_data")
    rel_out = os.path.join(HERE, "release-v0.13.1")
    os.makedirs(rel_out, exist_ok=True)
    for name in RELEASE:
        shutil.copyfile(os.path.join(ref, "release-v0.13.1", name), os.path.join(rel_out, name))

    load = lambda name: json.load(open(os.path.join(data, name)))
    files = {name: load(name) for name in ("full_proof_1.json", "full_proof_batch_prove_1.json", "full_proof_batch_agg_1.json",
                                           "full_proof_batch_agg_2.json", "batch-task-with-blob-raw.json")}
    del files["batch-task-with-blob-raw.json"]["blob_bytes"]  # not read by a batch task's consistency check
    for name in ("batch-task-with-blob.json", "batch_tasks/batch_task_293209.json"):
        shortest = min(load(name)["chunk_proofs"], key=lambda cp: len(cp["chunk_info"]["tx_bytes"]))
        files[name] = {"chunk_proofs": [shortest]}

    shared = {}
    for f in files.values():
        for e in f.get("chunk_proofs", []) + ([f] if "protocol" in f else []):
            key = "chunk_protocol" if "chunk_info" in e else "batch_protocol"
            assert shared.setdefault(key, e["protocol"]) == e["protocol"], "one protocol string per proof kind"
            e["protocol"] = key
    headers = {os.path.basename(p)[len("batch_task_"):-len(".json")]: json.load(open(p))["batch_header"]
               for p in sorted(glob.glob(os.path.join(data, "batch_tasks", "*.json")))}

    sys.path.insert(0, os.path.dirname(HERE))
    from test_evm_verifier_kat import m_add, m_mul, m_pairing
    from yul_verifier import verify

    rel = lambda name: open(os.path.join(ref, "release-v0.13.1", name), "rb").read()
    proof = rel("proof.data")
    ok, m = verify(rel("evm_verifier.yul").decode(), proof[:384] + rel("pi.data") + proof[384:], m_add, m_mul, m_pairing)
    out = {"source": "scroll-tech/scroll-prover @ ecba83e", "shared": shared, "files": files, "batch_headers": headers,
           "evm_verifier_yul_run": {"accepted": ok, "precompile_calls": m.precompile_calls, "keccak_calls": m.keccak_calls}}
    path = os.path.join(HERE, "reference_proofs.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=0)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
