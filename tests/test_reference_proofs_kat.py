"""The reference's OWN proofs verified offline (SURVEY.md §8(c) fixture 4): the chunk proofs (layer 2, k = 25, 896 bytes) and the
batch proofs (layer 4, k = 26) shipped in the reference's integration/tests/test_data are read with the protocol JSON they carry,
their Poseidon transcript is replayed, the quotient identity is evaluated from the protocol's expression tree, the SHPLONK (Bdfg21)
opening is folded into a KZG accumulator and the accumulator is decided against the trusted setup's G2 constants
(release-v0.13.1/evm_verifier.yul:1230-1239) -- tests/snark_verifier_model.py, a big-integer model of snark-verifier's native
verifier.  Every proof must be accepted (with the pairing of the big-integer model AND with the product's host pairing code), the
accumulator each proof carries in its instances must be valid as well, and a flipped proof byte / instance must be rejected.

What this pins: the proof format the hot path's outputs end up in -- compressed commitments, evaluation order, rotation sets, the
powers of mu / gamma (= the `y` / `v` of halo2's ProverSHPLONK, ascending, which scroll-prover_b200/plonk_b200.hpp follows) --
against real proofs of the reference, not against our own reading of it.  CPU only; the proofs are the sample stored in
tests/golden/reference_proofs.json (tests/reference_data.py)."""
import base64
import ctypes as C
import json
import os

from pairing_model import G2_GEN, pairing_check
from reference_data import GOLD, REL, proof_files_dir
from snark_verifier_model import PoseidonSpec, verify_plonk

DATA = proof_files_dir()

# -[s]G2 of the degree-26 SRS as the EVM verifier holds it (evm_verifier.yul:1236-1239; EIP-197 word order x_c1, x_c0, y_c1, y_c0)
NEG_S_G2 = ((0x17944351223333f260ddc3b4af45191b856689eda9eab5cbcddbbe570ce860d2, 0x186282957db913abd99f91db59fe69922e95040603ef44c0bd7aa3adeef8f5ac),
            (0x06ecdb9f9567f59ed2eee36e1e1d58797fd13cc97fafc2910f5e8a12f202fa9a, 0x06d971ff4a7467c3ec596ed6efc674572e32fd6f52b721f97e35b0b3d3546753))
SPEC = PoseidonSpec()  # T = 5, RATE = 4, R_F = 8, R_P = 60


def decode(entry):
    proto = json.loads(base64.b64decode(entry["protocol"]))
    proof = base64.b64decode(entry["proof"])
    raw = base64.b64decode(entry["instances"])
    return proto, proof, [[int.from_bytes(raw[i:i + 32], "big") for i in range(0, len(raw), 32)]]


def carried_accumulator(instances):
    """the KZG accumulator a compression / aggregation proof exposes: 12 limbs of 88 bits = (lhs.x, lhs.y, rhs.x, rhs.y)"""
    l = instances[0][:12]
    c = [l[3 * i] + (l[3 * i + 1] << 88) + (l[3 * i + 2] << 176) for i in range(4)]
    return (c[0], c[1]), (c[2], c[3])


def decide(lhs, rhs):
    return pairing_check([(lhs, G2_GEN), (rhs, NEG_S_G2)])


def chunk_entries():
    """(file, index, proof object) of every stored chunk proof"""
    return [(name, i, e) for name in GOLD["files"] for i, e in enumerate(json.load(open(os.path.join(DATA, name))).get("chunk_proofs", []))]


def test_poseidon_constants_reproduce_the_published_t3_parameters():
    """the Grain generator is the Poseidon paper's: for (t = 3, R_F = 8, R_P = 57) it yields the widely deployed BN254 constants"""
    s3 = PoseidonSpec(3, 8, 57)
    assert s3.rc[0][0] == 0x0ee9a592ba9a9518d05986d656f40c2114c4993c11bb29938d21d47304cd8e6e
    assert s3.mds[0][0] == 0x109b7f411ba0e4c9b2b70caf5c36a7b194be7c11ad24378bfedb68592ba8118b
    assert len(SPEC.rc) == 68 and len(SPEC.mds) == 5


def test_reference_chunk_proofs_verify():
    entries = chunk_entries()
    assert len(entries) == 8
    release = json.load(open(os.path.join(REL, "chunk.protocol")))
    for name, i, e in entries:
        proto, proof, instances = decode(e)
        assert len(proof) == 896 and proto["domain"]["k"] == 25 and proto["quotient"]["num_chunk"] == 4 and len(instances[0]) == 44, (name, i)
        lhs, rhs, info = verify_plonk(proto, instances, proof, SPEC)
        assert info["n_sets"] == 3 and decide(lhs, rhs), (name, i)           # the proof itself
        assert decide(*carried_accumulator(instances)), (name, i)            # and the accumulator it carries forward
    assert decode(entries[0][2])[0] == release  # the released protocol is the one the test proofs were made under


def test_reference_batch_proofs_verify_under_their_own_protocol():
    for name in ("full_proof_batch_agg_1.json", "full_proof_batch_agg_2.json"):
        proto, proof, instances = decode(json.load(open(os.path.join(DATA, name))))
        assert proto["domain"]["k"] == 26
        lhs, rhs, _ = verify_plonk(proto, instances, proof, SPEC)
        assert decide(lhs, rhs) and decide(*carried_accumulator(instances)), name


def test_tampered_proofs_and_instances_are_rejected_and_the_product_pairing_agrees():
    proto, proof, instances = decode(json.load(open(os.path.join(DATA, "full_proof_1.json")))["chunk_proofs"][0])
    lhs, rhs, _ = verify_plonk(proto, instances, proof, SPEC)
    # the product's host pairing (pairing_bn254.hpp through tests/host_emul) takes the same decision
    from test_evm_verifier_kat import be, host_lib
    enc_g2 = lambda q: be(q[0][1]) + be(q[0][0]) + be(q[1][1]) + be(q[1][0])
    blob = be(lhs[0]) + be(lhs[1]) + enc_g2(G2_GEN) + be(rhs[0]) + be(rhs[1]) + enc_g2(NEG_S_G2)
    assert host_lib().pairing_host_eip197(blob, 2) == 1
    for pos in (3, 200, 300, 500, 850, 895):  # a witness commitment, a quotient chunk, evaluations, the two opening points
        bad = bytearray(proof)
        bad[pos] ^= 1
        try:
            l2, r2, _ = verify_plonk(proto, instances, bytes(bad), SPEC)
        except ValueError:
            continue  # not even a point / a canonical scalar any more
        assert not decide(l2, r2), pos
    wrong = [instances[0][:]]
    wrong[0][20] ^= 1  # a public-input byte
    l3, r3, _ = verify_plonk(proto, wrong, proof, SPEC)
    assert not decide(l3, r3)


def test_oracle_multiexp_redoes_the_msms_of_real_proofs_and_the_reference_srs_accepts_the_result():
    """A known-answer test of MSM OUTPUTS on the reference's real data: the two multi-scalar multiplications inside the verification
    of a shipped proof -- the quotient commitment sum_i z^(n i) h_i and the SHPLONK left-hand side over ALL of the proof's and the
    verifying key's commitments with the transcript-derived scalars (15 terms for the thin chunk proofs) -- are recomputed by the ORACLE's best_multiexp
    (oracle/halo2_arith.c, the restatement every CUDA result is compared with).  The result must be the model's point and, what no
    implementation can fake by agreeing with another, must be accepted by the pairing against the trusted setup's -[s]G2."""
    import numpy as np

    from oracle import oracle as O
    from pairing_model import g1_add, g1_mul

    def oracle_msm(pairs, threads):
        coeffs = np.stack([O.fr_from_int(s) for s, _ in pairs])
        bases = np.stack([np.concatenate([O.fq_from_int(p[0]), O.fq_from_int(p[1])]) for _, p in pairs])
        a = O.g1_to_affine(O.best_multiexp(coeffs, bases, threads=threads))
        return O.fq_to_int(a[:4]), O.fq_to_int(a[4:])

    picks = [decode(json.load(open(os.path.join(DATA, "full_proof_1.json")))["chunk_proofs"][0]),
             decode(json.load(open(os.path.join(DATA, "batch-task-with-blob-raw.json")))["chunk_proofs"][3]),
             decode(json.load(open(os.path.join(DATA, "full_proof_batch_agg_1.json"))))]
    for proto, proof, instances in picks:
        lhs, rhs, info = verify_plonk(proto, instances, proof, SPEC)
        terms = info["msm_terms"]
        assert len(terms) >= 12 and all(p is not None for _, p in terms)
        for threads in (1, 4):
            f = oracle_msm(terms, threads)
            assert f == info["f"]
            assert decide(g1_add(f, g1_mul(rhs, info["z_prime"])), rhs)
        q = oracle_msm(info["quotient_terms"], 1)
        assert q == terms[[i for i, (_, p) in enumerate(terms) if p == q][0]][1]  # the quotient commitment is one of the bases
        bad = list(terms)
        bad[7] = ((bad[7][0] + 1) % (1 << 253), bad[7][1])
        assert not decide(g1_add(oracle_msm(bad, 1), g1_mul(rhs, info["z_prime"])), rhs)
