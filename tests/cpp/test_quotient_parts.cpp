// The device-only prover session with the quotient built part by part (DeviceOps::quotient): the circuits of
// test_plonk_session.cpp (compiled into this driver, so both drivers prove the same circuits), proved at a size where the
// oracle would take minutes, accepted by the halo2-style verifier and by the snark-verifier mirror, plus the device bytes the
// quotient step held at its peak and the column count that bounds them.  First, the part forms of the host mirrors
// (EvaluationDomain::coeff_to_extended_part / extended_parts_to_coeff, GraphEvaluator::evaluate_part) against the full coset.
//   usage: test_quotient_parts <k> <seed> <variant>
#define main plonk_session_main
#include "test_plonk_session.cpp"
#undef main

int main(int argc, char** argv) {
    const uint32_t k = argc > 1 ? (uint32_t)std::atoi(argv[1]) : 18;
    const uint64_t seed = argc > 2 ? (uint64_t)std::atoll(argv[2]) : 1;
    const int variant = argc > 3 ? std::atoi(argv[3]) : 1;
    const uint64_t n = 1ull << k;
    try {
        {   // the host mirrors (halo2_b200.hpp): a column's parts are the strided slices of its coset, a program on a part is the
            // strided slice of its full-domain values, and the parts recombine to extended_to_coeff with and without the division
            EvaluationDomain d = EvaluationDomain::new_(5, 10);
            const uint64_t J = 1ull << (d.extended_k - d.k);
            Rng rng(7);
            Poly c(d.n);
            for (auto& x : c) x = rng.fr();
            const Poly ext = d.coeff_to_extended(c);
            GraphEvaluator ev;
            const uint32_t r1 = ev.add_rotation(1);
            ev.add(B200ZK_CALC_ADD, ev.add(B200ZK_CALC_MUL, ValueSource::Advice(0, r1), ValueSource::ExtendedX()), ValueSource::PreviousValue());
            const Fr zero = f_zero();
            DeviceColumn ext_col(ext), full_vals(Poly(ext.size(), zero));
            ev.evaluate(full_vals, d, {}, {&ext_col}, {}, {}, zero, zero, zero, zero);
            const Poly want = full_vals.to_host();
            Poly parts(ext.size()), divided(ext.size());
            for (uint32_t r = 0; r < J; ++r) {
                const Poly p = d.coeff_to_extended_part(c, r);
                DeviceColumn part_col(p), part_vals(Poly(d.n, zero));
                ev.evaluate_part(part_vals, d, r, {}, {&part_col}, {}, {}, zero, zero, zero, zero);
                const Poly got = part_vals.to_host();
                for (uint64_t i = 0; i < d.n; ++i) {
                    REQUIRE(p[i] == ext[r + J * i] && got[i] == want[r + J * i]);
                    parts[r * d.n + i] = p[i];
                }
            }
            Fr cur = f_pow(d.g_coset, d.n), wn = f_pow(d.extended_omega, d.n);
            std::vector<Fr> t_inv(J);
            for (auto& t : t_inv) { t = f_inv(f_sub(cur, f_one())); cur = f_mul(cur, wn); }
            for (size_t i = 0; i < ext.size(); ++i) divided[i] = f_mul(ext[i], t_inv[i % J]);
            REQUIRE(d.extended_parts_to_coeff(parts, false) == d.extended_to_coeff(ext));
            REQUIRE(d.extended_parts_to_coeff(parts, true) == d.extended_to_coeff(divided));
            std::printf("host mirrors: parts, part evaluation and recombination agree with the full coset (2^%u, J = %llu)\n", d.k,
                        (unsigned long long)J);
        }
        Circuit C = variant == 3 ? build_phased(k, seed, 0) : (variant == 2 ? build_wide(k, seed, 0) : build(k, seed, 0));
        EvaluationDomain dom = EvaluationDomain::new_(C.cs.degree(), k);
        const Fr tau = f_from_bytes_wide((const uint8_t*)"b200zk test srs: tau is NOT secret -- a toxic-waste-free toy..!!");
        ParamsKZG params;
        ParamsKZG::setup(params, k, tau);
        VerifierParams vp;
        vp.g2 = pairing::g2_generator();
        uint8_t repr[32];
        f_to_repr(tau, repr);
        uint64_t limbs[4];
        std::memcpy(limbs, repr, 32);
        vp.s_g2 = pairing::g2_mul(vp.g2, limbs);
        DeviceOps dops(params, dom);
        ProvingKey pk = keygen(dops, dom, C.cs, C.fixed, *C.assembly);
        ProofArtifacts pr = C.synth ? create_proof(dops, dom, pk, C.synth, C.instances, 0xB200 + seed, TranscriptKind::Poseidon)
                                    : create_proof(dops, dom, pk, C.advice, C.instances, 0xB200 + seed, TranscriptKind::Poseidon);
        std::string why;
        REQUIRE(verify_proof(dom, pk.vk, vp, C.instances, pr.proof, &why, TranscriptKind::Poseidon));
        protocol::PlonkProtocol P = protocol::parse_protocol(export_protocol_json(dom, pk.vk));
        const uint64_t u = n - C.cs.blinding_factors() - 1;
        std::vector<std::vector<Fr>> inst;
        for (auto& col : C.instances) inst.emplace_back(col.begin(), col.begin() + u);
        REQUIRE(snark::verify(P, inst, pr.proof, vp.g2, vp.s_g2, &why));
        std::vector<uint8_t> bad = pr.proof;
        bad[bad.size() / 2] ^= 1;
        REQUIRE(!snark::verify(P, inst, bad, vp.g2, vp.s_g2, &why));
        // the columns the quotient reads: fixed | l0 l_last l_active | sigma, advice | z sets | (m, phi) per lookup, instance
        const size_t columns = pk.fixed_polys.size() + 3 + pk.sigma_polys.size() + C.cs.num_advice + aux_layout(C.cs).n_sets +
                               2 * C.cs.lookups.size() + C.cs.num_instance;
        std::printf("quotient_peak_bytes %zu columns %zu parts %u n %llu\n", dops.quotient_peak_bytes(), columns,
                    1u << (dom.extended_k - dom.k), (unsigned long long)n);
        std::printf("device proof of 2^%u rows: %zu bytes, accepted by both verifiers\nOK\n", k, pr.proof.size());
        return 0;
    } catch (const std::exception& e) {
        std::printf("EXCEPTION: %s\n", e.what());
        return 1;
    }
}
