// plonk_b200.hpp — a create_proof / verify_proof SESSION over the hot path (SURVEY.md §8 rows a9, f4).
//
// C++ host-side mirror (the reference is Rust; no toolchain here) of the control flow of
//   halo2_proofs::plonk::{keygen_vk, keygen_pk, create_proof, verify_proof}            (src/plonk/{keygen,prover,verifier}.rs)
//   plonk::{permutation, mv_lookup, vanishing} prover / verifier arguments               (src/plonk/*/{prover,verifier}.rs)
//   poly::kzg::multiopen::{ProverSHPLONK, VerifierSHPLONK}                                (src/poly/kzg/multiopen/shplonk/*)
//   transcript::{Blake2bWrite, Blake2bRead, Challenge255}                                 (src/transcript.rs)
//   dev::MockProver (constraint check without proving)                                   (src/dev.rs)
// of scroll-tech/halo2 @ e5ddf67 (pin /root/reference/Cargo.lock:1886-1888), the function the reference enters at
// /root/reference/integration/src/prove.rs:37-39 (gen_halo2_chunk_proof) and checks at :50-53 (verify_chunk_proof).
//
// Every field-vector / group operation of the prover goes through the `Ops` interface below -- exactly the operations
// libb200zk replaces (commit_lagrange, commit, lagrange_to_coeff, coeff_to_extended, extended_to_coeff, GraphEvaluator,
// permutation product, log-derivative sum, eval_polynomial, kate_division, linear combinations).  `DeviceOps` implements it
// over the C ABI (include/b200zk.h); the tests implement the same interface over the CPU oracle and require IDENTICAL PROOF
// BYTES from both.  The host keeps what upstream keeps on the host: the transcript, challenge arithmetic, blinding rows,
// multiplicity counting, rotation-set bookkeeping.  The verifier is host-only (pairing_bn254.hpp), as in the reference.
//
// Fidelity: the phase loop (advice columns and challenges per phase, ConstraintSystem::{advice_column_phase, challenge_phase}),
// argument order, constraint order, y-folding, evaluation order and the SHPLONK construction follow upstream;
// `VerifyingKey::transcript_repr` is our own pinning (upstream hashes the Debug rendering of its Rust structs) and no
// reference proof of a known circuit + SRS exists offline, so byte-compatibility WITH UPSTREAM PROOFS is not claimed
// ("parity unpinned" at that level); what is tested is: proofs verify under an independent pairing check, device and
// oracle runs give identical bytes, and any tampering is rejected.
#pragma once
#include <array>
#include <functional>
#include <map>
#include <memory>
#include <set>

#include "csrc/ec.cuh"
#include "halo2_b200.hpp"
#include "pairing_bn254.hpp"
#include "serde_bn254.hpp"

namespace halo2_b200 {
namespace plonk {

using detail::DFr;
using detail::from_dev;
using detail::to_dev;

// ------------------------------------------------------------------------------------------------ small field helpers (host)
inline Fr f_zero() { return from_dev(DFr::zero()); }
inline Fr f_one() { return from_dev(DFr::one()); }
inline Fr f_u64(uint64_t v) { return from_dev(detail::from_u64(v)); }
inline Fr f_add(const Fr& a, const Fr& b) { return from_dev(to_dev(a) + to_dev(b)); }
inline Fr f_sub(const Fr& a, const Fr& b) { return from_dev(to_dev(a) - to_dev(b)); }
inline Fr f_mul(const Fr& a, const Fr& b) { return from_dev(to_dev(a) * to_dev(b)); }
inline Fr f_neg(const Fr& a) { return from_dev(to_dev(a).neg()); }
inline Fr f_inv(const Fr& a) { return from_dev(to_dev(a).inv()); }
inline bool f_is_zero(const Fr& a) { return (a.l[0] | a.l[1] | a.l[2] | a.l[3]) == 0; }
inline Fr f_pow(const Fr& a, uint64_t e) { return from_dev(to_dev(a).pow_u64(e)); }
inline void f_to_repr(const Fr& a, uint8_t out[32]) {  // canonical little-endian bytes (Fr::to_repr)
    DFr c = to_dev(a).from_mont();
    std::memcpy(out, c.l.v, 32);
}
inline bool f_from_repr(const uint8_t in[32], Fr* out) {
    DFr c;
    std::memcpy(c.l.v, in, 32);
    uint32_t m[8], d[8];
    DFr::modulus(m);
    if (!b200zk::leaf::sub8(d, c.l.v, m)) return false;  // no borrow: the value is >= r
    *out = from_dev(c.to_mont());
    return true;
}
// Fr::from_uniform_bytes / from_bytes_wide: 512-bit little-endian integer mod r
inline Fr f_from_bytes_wide(const uint8_t in[64]) {
    DFr lo, hi;
    std::memcpy(lo.l.v, in, 32);
    std::memcpy(hi.l.v, in + 32, 32);
    // lo, hi < 2^256 are not reduced: x.to_mont() = x * R2 * R^-1 = x R is a valid Montgomery product for any x < 2^256
    DFr two256 = DFr::one();  // Montgomery form of 1 is R = 2^256 mod r: as a field element it IS 2^256
    return from_dev(lo.to_mont() + hi.to_mont() * two256.to_mont());
}
inline Fr f_delta() {  // halo2curves Fr::DELTA = GENERATOR^(2^S): generator of the t-order multiplicative subgroup
    return f_pow(f_pow(f_u64(7), 1ull << 14), 1ull << 14);  // 7^(2^28)
}

// ------------------------------------------------------------------------------------------------ Blake2b transcript
// RFC 7693 BLAKE2b-512 with the 16-byte personalisation "Halo2-Transcript" (transcript.rs: Blake2bParams::new()
// .hash_length(64).personal(b"Halo2-Transcript")); checked against Python's hashlib in tests/test_plonk_session.py.
class Blake2b {
  public:
    explicit Blake2b(const char personal[16]) {
        static const uint64_t IV[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                                       0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
        for (int i = 0; i < 8; ++i) h_[i] = IV[i];
        h_[0] ^= 0x01010000ull ^ 64ull;  // depth 1, fanout 1, no key, 64-byte digest
        uint64_t p0, p1;
        std::memcpy(&p0, personal, 8);
        std::memcpy(&p1, personal + 8, 8);
        h_[6] ^= p0;
        h_[7] ^= p1;
    }
    void update(const uint8_t* data, size_t len) {
        while (len) {
            if (fill_ == 128) {
                t_ += 128;
                compress(false);
                fill_ = 0;
            }
            size_t take = std::min(len, (size_t)128 - fill_);
            std::memcpy(buf_ + fill_, data, take);
            fill_ += take;
            data += take;
            len -= take;
        }
    }
    std::array<uint8_t, 64> finalize() const {  // on a copy: the running state stays usable (hasher.clone().finalize())
        Blake2b c = *this;
        c.t_ += c.fill_;
        std::memset(c.buf_ + c.fill_, 0, 128 - c.fill_);
        c.compress(true);
        std::array<uint8_t, 64> out;
        std::memcpy(out.data(), c.h_, 64);
        return out;
    }

  private:
    static uint64_t rotr(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }
    void compress(bool last) {
        static const uint8_t S[12][16] = {{0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
                                          {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
                                          {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
                                          {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
                                          {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0},
                                          {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3}};
        static const uint64_t IV[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                                       0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
        uint64_t m[16], v[16];
        std::memcpy(m, buf_, 128);
        for (int i = 0; i < 8; ++i) v[i] = h_[i], v[i + 8] = IV[i];
        v[12] ^= t_;
        if (last) v[14] = ~v[14];
        auto G = [&](int r, int i, int a, int b, int c, int d) {
            v[a] = v[a] + v[b] + m[S[r][2 * i]];
            v[d] = rotr(v[d] ^ v[a], 32);
            v[c] = v[c] + v[d];
            v[b] = rotr(v[b] ^ v[c], 24);
            v[a] = v[a] + v[b] + m[S[r][2 * i + 1]];
            v[d] = rotr(v[d] ^ v[a], 16);
            v[c] = v[c] + v[d];
            v[b] = rotr(v[b] ^ v[c], 63);
        };
        for (int r = 0; r < 12; ++r) {
            G(r, 0, 0, 4, 8, 12); G(r, 1, 1, 5, 9, 13); G(r, 2, 2, 6, 10, 14); G(r, 3, 3, 7, 11, 15);
            G(r, 4, 0, 5, 10, 15); G(r, 5, 1, 6, 11, 12); G(r, 6, 2, 7, 8, 13); G(r, 7, 3, 4, 9, 14);
        }
        for (int i = 0; i < 8; ++i) h_[i] ^= v[i] ^ v[i + 8];
    }
    uint64_t h_[8], t_ = 0;
    uint8_t buf_[128] = {0};
    size_t fill_ = 0;
};

inline serde::G1Point to_affine_point(const G1& j) {  // normalised Jacobian (x, y, 1) or identity (z = 0) -> affine
    serde::G1Point p;
    if (j.is_identity()) {
        p.x = b200zk::Fq::zero();
        p.y = b200zk::Fq::zero();
        return p;
    }
    std::memcpy(p.x.l.v, j.x.l, 32);
    std::memcpy(p.y.l.v, j.y.l, 32);
    return p;
}

// ------------------------------------------------------------------------------------------------ Poseidon (snark-verifier's transcript hash)
// snark-verifier's native transcript for the chunk / batch proofs (`PoseidonTranscript`, system/halo2/transcript/halo2.rs) hashes with
// the Poseidon sponge of util/hash/poseidon.rs at T = 5, RATE = 4, R_F = 8, R_P = 60; the round constants and the Cauchy MDS matrix
// come from the Grain LFSR of the Poseidon paper.  tests/test_reference_proofs_kat.py pins these parameters and conventions on the
// reference's shipped proofs (through the Python model tests/snark_verifier_model.py); this C++ sponge is checked against that model.
class PoseidonSpec {
  public:
    static constexpr int T = 5, RATE = 4, R_F = 8, R_P = 60;
    std::vector<std::array<DFr, T>> rc;
    std::array<std::array<DFr, T>, T> mds;
    static const PoseidonSpec& get() {
        static const PoseidonSpec s;
        return s;
    }
    void permute(std::array<DFr, T>& st) const {
        auto pow5 = [](const DFr& x) { DFr x2 = x.sqr(); return x2.sqr() * x; };
        auto mix = [&](std::array<DFr, T>& s) {
            std::array<DFr, T> o;
            for (int i = 0; i < T; ++i) {
                DFr acc = DFr::zero();
                for (int j = 0; j < T; ++j) acc = acc + mds[i][j] * s[j];
                o[i] = acc;
            }
            s = o;
        };
        size_t r = 0;
        for (int k = 0; k < R_F / 2; ++k, ++r) {
            for (int i = 0; i < T; ++i) st[i] = pow5(st[i] + rc[r][i]);
            mix(st);
        }
        for (int k = 0; k < R_P; ++k, ++r) {
            for (int i = 0; i < T; ++i) st[i] = st[i] + rc[r][i];
            st[0] = pow5(st[0]);
            mix(st);
        }
        for (int k = 0; k < R_F / 2; ++k, ++r) {
            for (int i = 0; i < T; ++i) st[i] = pow5(st[i] + rc[r][i]);
            mix(st);
        }
    }

  private:
    struct Grain {  // generate_parameters_grain: 80-bit LFSR, taps 62 51 38 23 13 0, self-shrinking output
        std::vector<uint8_t> s;
        Grain(uint32_t t, uint32_t r_f, uint32_t r_p) {
            auto put = [&](uint32_t v, int width) { for (int i = width - 1; i >= 0; --i) s.push_back((v >> i) & 1); };
            put(1, 2); put(0, 4); put(254, 12); put(t, 12); put(r_f, 10); put(r_p, 10); put((1u << 30) - 1, 30);
            for (int i = 0; i < 160; ++i) update();
        }
        uint8_t update() {
            uint8_t b = s[62] ^ s[51] ^ s[38] ^ s[23] ^ s[13] ^ s[0];
            s.erase(s.begin());
            s.push_back(b);
            return b;
        }
        uint8_t bit() {
            for (;;) {
                uint8_t first = update(), second = update();
                if (first) return second;
            }
        }
        void bits254_le(uint8_t out[64]) {  // 254 output bits, most significant first, as a little-endian 64-byte integer
            std::memset(out, 0, 64);
            for (int i = 253; i >= 0; --i)
                if (bit()) out[i / 8] |= (uint8_t)(1u << (i % 8));
        }
        Fr element(bool reject) {
            for (;;) {
                uint8_t b[64];
                bits254_le(b);
                Fr v;
                if (!reject) return f_from_bytes_wide(b);
                if (f_from_repr(b, &v)) return v;
            }
        }
    };
    PoseidonSpec() {
        Grain g(T, R_F, R_P);
        rc.resize(R_F + R_P);
        for (auto& row : rc)
            for (auto& c : row) c = to_dev(g.element(true));
        for (;;) {
            Fr v[2 * T];
            for (auto& e : v) e = g.element(false);
            bool distinct = true;
            for (int i = 0; i < 2 * T; ++i)
                for (int j = i + 1; j < 2 * T; ++j) distinct &= !(v[i] == v[j]);
            if (!distinct) continue;
            for (int i = 0; i < T; ++i)
                for (int j = 0; j < T; ++j) mds[i][j] = (to_dev(v[i]) + to_dev(v[T + j])).inv();
            break;
        }
    }
};

// util/hash/poseidon.rs: state [2^64, 0, ..]; update() buffers; squeeze() absorbs the buffer in RATE chunks -- a partial (or empty)
// last chunk is followed by a one -- and returns state[1]; the state carries over from one squeeze to the next
class PoseidonSponge {
  public:
    PoseidonSponge() {
        for (auto& x : st_) x = DFr::zero();
        st_[0] = to_dev(f_pow(f_u64(2), 64));
    }
    void update(const Fr& v) { buf_.push_back(to_dev(v)); }
    Fr squeeze() {
        std::vector<DFr> buf;
        buf.swap(buf_);
        const bool exact = buf.size() % PoseidonSpec::RATE == 0;
        for (size_t i = 0; i < buf.size(); i += PoseidonSpec::RATE) permutation(buf.data() + i, std::min(buf.size() - i, (size_t)PoseidonSpec::RATE));
        if (exact) permutation(nullptr, 0);
        return from_dev(st_[1]);
    }

  private:
    void permutation(const DFr* chunk, size_t len) {
        for (size_t i = 0; i < len; ++i) st_[i + 1] = st_[i + 1] + chunk[i];
        if (len + 1 < (size_t)PoseidonSpec::T) st_[len + 1] = st_[len + 1] + DFr::one();
        PoseidonSpec::get().permute(st_);
    }
    std::array<DFr, PoseidonSpec::T> st_;
    std::vector<DFr> buf_;
};

// transcript::{Blake2bWrite, Blake2bRead}<_, G1Affine, Challenge255<_>> (halo2's default), or snark-verifier's PoseidonTranscript
// (the one the reference's chunk / batch proofs are made with): same proof bytes layout, different challenge derivation
enum class TranscriptKind { Blake2b, Poseidon };
class Transcript {
  public:
    static constexpr uint8_t PREFIX_CHALLENGE = 0, PREFIX_POINT = 1, PREFIX_SCALAR = 2;
    explicit Transcript(TranscriptKind kind = TranscriptKind::Blake2b) : kind_(kind), state_("Halo2-Transcript") {}
    explicit Transcript(const std::vector<uint8_t>& proof, TranscriptKind kind = TranscriptKind::Blake2b)
        : kind_(kind), state_("Halo2-Transcript"), proof_(proof) {}

    void common_scalar(const Fr& s) {
        if (kind_ == TranscriptKind::Poseidon) {
            sponge_.update(s);
            return;
        }
        uint8_t b[33];
        b[0] = PREFIX_SCALAR;
        f_to_repr(s, b + 1);
        state_.update(b, 33);
    }
    void common_point(const serde::G1Point& p) {  // coordinates, little-endian canonical (x then y)
        if (p.x.is_zero() && p.y.is_zero()) throw Panic("cannot write points at infinity to the transcript");
        if (kind_ == TranscriptKind::Poseidon) {  // fe_to_fe::<Fq, Fr>: the coordinates reduced into the scalar field
            uint8_t w[64] = {0};
            serde::fq_to_le32(p.x, w);
            sponge_.update(f_from_bytes_wide(w));
            serde::fq_to_le32(p.y, w);
            sponge_.update(f_from_bytes_wide(w));
            return;
        }
        uint8_t b[65];
        b[0] = PREFIX_POINT;
        serde::fq_to_le32(p.x, b + 1);
        serde::fq_to_le32(p.y, b + 33);
        state_.update(b, 65);
    }
    void write_point(const G1& commitment) {
        serde::G1Point p = to_affine_point(commitment);
        common_point(p);
        uint8_t c[32];
        serde::g1_to_compressed(p, c);
        proof_.insert(proof_.end(), c, c + 32);
    }
    void write_scalar(const Fr& s) {
        common_scalar(s);
        uint8_t b[32];
        f_to_repr(s, b);
        proof_.insert(proof_.end(), b, b + 32);
    }
    serde::G1Point read_point() {
        if (pos_ + 32 > proof_.size()) throw Panic("proof too short (point)");
        serde::G1Point p;
        if (!serde::g1_from_compressed(proof_.data() + pos_, &p)) throw Panic("invalid point encoding in proof");
        pos_ += 32;
        common_point(p);
        return p;
    }
    Fr read_scalar() {
        if (pos_ + 32 > proof_.size()) throw Panic("proof too short (scalar)");
        Fr s;
        if (!f_from_repr(proof_.data() + pos_, &s)) throw Panic("invalid field element encoding in proof");
        pos_ += 32;
        common_scalar(s);
        return s;
    }
    Fr squeeze_challenge() {
        if (kind_ == TranscriptKind::Poseidon) return sponge_.squeeze();
        state_.update(&PREFIX_CHALLENGE, 1);
        auto h = state_.finalize();
        return f_from_bytes_wide(h.data());
    }
    std::vector<uint8_t> finalize() const { return proof_; }
    bool exhausted() const { return pos_ == proof_.size(); }

  private:
    TranscriptKind kind_;
    Blake2b state_;
    PoseidonSponge sponge_;
    std::vector<uint8_t> proof_;
    size_t pos_ = 0;
};

// ------------------------------------------------------------------------------------------------ plonk::Expression
struct Expr;
using ExprP = std::shared_ptr<const Expr>;
struct Expr {
    enum Kind { Constant, Fixed, Advice, Instance, Negated, Sum, Product, Scaled, Challenge } kind;
    Fr c{};          // Constant, Scaled
    uint32_t col = 0;  // column index (Challenge: index of the challenge)
    int32_t rot = 0;   // Rotation
    ExprP a, b;
    static ExprP constant(const Fr& v) { auto e = std::make_shared<Expr>(); e->kind = Constant; e->c = v; return e; }
    static ExprP fixed(uint32_t col, int32_t rot = 0) { auto e = std::make_shared<Expr>(); e->kind = Fixed; e->col = col; e->rot = rot; return e; }
    static ExprP advice(uint32_t col, int32_t rot = 0) { auto e = std::make_shared<Expr>(); e->kind = Advice; e->col = col; e->rot = rot; return e; }
    static ExprP instance(uint32_t col, int32_t rot = 0) { auto e = std::make_shared<Expr>(); e->kind = Instance; e->col = col; e->rot = rot; return e; }
    static ExprP challenge(uint32_t index) { auto e = std::make_shared<Expr>(); e->kind = Challenge; e->col = index; return e; }  // Expression::Challenge
    static ExprP neg(ExprP x) { auto e = std::make_shared<Expr>(); e->kind = Negated; e->a = x; return e; }
    static ExprP sum(ExprP x, ExprP y) { auto e = std::make_shared<Expr>(); e->kind = Sum; e->a = x; e->b = y; return e; }
    static ExprP sub(ExprP x, ExprP y) { return sum(x, neg(y)); }
    static ExprP mul(ExprP x, ExprP y) { auto e = std::make_shared<Expr>(); e->kind = Product; e->a = x; e->b = y; return e; }
    static ExprP scaled(ExprP x, const Fr& s) { auto e = std::make_shared<Expr>(); e->kind = Scaled; e->a = x; e->c = s; return e; }

    uint32_t degree() const {
        switch (kind) {
            case Constant: case Challenge: return 0;
            case Fixed: case Advice: case Instance: return 1;
            case Negated: case Scaled: return a->degree();
            case Sum: return std::max(a->degree(), b->degree());
            default: return a->degree() + b->degree();
        }
    }
    // Expression::evaluate with one closure per leaf kind
    template <typename T>
    T evaluate(const std::function<T(const Fr&)>& constant, const std::function<T(int, uint32_t, int32_t)>& query,
               const std::function<T(const T&)>& negated, const std::function<T(const T&, const T&)>& sum,
               const std::function<T(const T&, const T&)>& product, const std::function<T(const T&, const Fr&)>& scaled) const {
        switch (kind) {
            case Constant: return constant(c);
            case Fixed: case Advice: case Instance: return query((int)kind, col, rot);
            case Challenge: return query((int)kind, col, 0);  // the leaf closure resolves challenges by index
            case Negated: return negated(a->evaluate<T>(constant, query, negated, sum, product, scaled));
            case Sum: return sum(a->evaluate<T>(constant, query, negated, sum, product, scaled), b->evaluate<T>(constant, query, negated, sum, product, scaled));
            case Product: return product(a->evaluate<T>(constant, query, negated, sum, product, scaled), b->evaluate<T>(constant, query, negated, sum, product, scaled));
            default: return scaled(a->evaluate<T>(constant, query, negated, sum, product, scaled), c);
        }
    }
    void collect_queries(std::set<std::pair<uint32_t, int32_t>>& fx, std::set<std::pair<uint32_t, int32_t>>& ad,
                         std::set<std::pair<uint32_t, int32_t>>& in) const {
        if (kind == Fixed) fx.insert({col, rot});
        if (kind == Advice) ad.insert({col, rot});
        if (kind == Instance) in.insert({col, rot});
        if (a) a->collect_queries(fx, ad, in);
        if (b) b->collect_queries(fx, ad, in);
    }
    // field value of the expression from already-known query values (the verifier, and the host-side lookup compression)
    Fr eval_with(const std::function<Fr(int, uint32_t, int32_t)>& q) const {
        return evaluate<Fr>([](const Fr& v) { return v; }, q, [](const Fr& v) { return f_neg(v); },
                            [](const Fr& x, const Fr& y) { return f_add(x, y); }, [](const Fr& x, const Fr& y) { return f_mul(x, y); },
                            [](const Fr& x, const Fr& s) { return f_mul(x, s); });
    }
};

// GraphEvaluator::add_expression (evaluation.rs): lowers an Expression into calculations of `ev`
inline ValueSource add_expression(GraphEvaluator& ev, const Expr& e) {
    switch (e.kind) {
        case Expr::Constant: return ev.add_constant(e.c);
        case Expr::Fixed: return ValueSource::Fixed(e.col, ev.add_rotation(e.rot));
        case Expr::Advice: return ValueSource::Advice(e.col, ev.add_rotation(e.rot));
        case Expr::Instance: return ValueSource::Instance(e.col, ev.add_rotation(e.rot));
        case Expr::Challenge: return ValueSource::Challenge(e.col);
        case Expr::Negated: return ev.add(B200ZK_CALC_NEGATE, add_expression(ev, *e.a));
        case Expr::Sum: {
            if (e.b->kind == Expr::Negated) return ev.add(B200ZK_CALC_SUB, add_expression(ev, *e.a), add_expression(ev, *e.b->a));  // a + (-b) = a - b, as upstream
            return ev.add(B200ZK_CALC_ADD, add_expression(ev, *e.a), add_expression(ev, *e.b));
        }
        case Expr::Product: return ev.add(B200ZK_CALC_MUL, add_expression(ev, *e.a), add_expression(ev, *e.b));
        default: return ev.add(B200ZK_CALC_MUL, add_expression(ev, *e.a), ev.add_constant(e.c));
    }
}

// ------------------------------------------------------------------------------------------------ ConstraintSystem
struct Column {
    int kind;  // Expr::Fixed / Advice / Instance
    uint32_t index;
    bool operator<(const Column& o) const { return kind != o.kind ? kind < o.kind : index < o.index; }
    bool operator==(const Column& o) const { return kind == o.kind && index == o.index; }
};
struct Lookup {  // mv_lookup::Argument: input expressions (one set) and table expressions, compressed with theta
    std::vector<ExprP> inputs, table;
};
struct ConstraintSystem {
    uint32_t num_fixed = 0, num_advice = 0, num_instance = 0;
    std::vector<ExprP> gates;             // every polynomial identity (selector already multiplied in), in gate order
    std::vector<Lookup> lookups;
    std::vector<Column> permutation;      // columns under equality constraints, in enable_equality order
    // multi-phase proving (ConstraintSystem::advice_column_phase / challenge_phase): advice column c is assigned in phase
    // advice_phase[c] (empty = every column in the first phase); challenge i becomes available after the commitments of phase
    // challenge_phase[i] and may be used by the witness of later phases and by any expression (Expr::challenge(i))
    std::vector<uint8_t> advice_phase, challenge_phase;
    uint32_t phase_of_advice(uint32_t col) const { return advice_phase.empty() ? 0 : advice_phase[col]; }
    uint32_t num_phases() const {
        uint32_t p = 0;
        for (auto v : advice_phase) p = std::max<uint32_t>(p, v);
        for (auto v : challenge_phase) p = std::max<uint32_t>(p, v);
        return p + 1;
    }
    std::vector<std::pair<uint32_t, int32_t>> fixed_queries, advice_queries, instance_queries;  // in first-use order

    void finalize() {  // collects the queries the way ConstraintSystem::query_*_index registers them
        std::set<std::pair<uint32_t, int32_t>> fx, ad, in;
        auto take = [&](const ExprP& e) {
            std::set<std::pair<uint32_t, int32_t>> f2, a2, i2;
            e->collect_queries(f2, a2, i2);
            for (auto& q : f2) if (fx.insert(q).second) fixed_queries.push_back(q);
            for (auto& q : a2) if (ad.insert(q).second) advice_queries.push_back(q);
            for (auto& q : i2) if (in.insert(q).second) instance_queries.push_back(q);
        };
        for (auto& g : gates) take(g);
        for (auto& l : lookups) {
            for (auto& e : l.inputs) take(e);
            for (auto& e : l.table) take(e);
        }
        for (auto& c : permutation) {  // enable_equality queries the column at the current rotation
            std::pair<uint32_t, int32_t> q{c.index, 0};
            if (c.kind == Expr::Fixed && fx.insert(q).second) fixed_queries.push_back(q);
            if (c.kind == Expr::Advice && ad.insert(q).second) advice_queries.push_back(q);
            if (c.kind == Expr::Instance && in.insert(q).second) instance_queries.push_back(q);
        }
    }
    uint32_t degree() const {  // ConstraintSystem::degree: max over the arguments' required degrees
        uint32_t d = permutation.empty() ? 1 : 3;  // permutation::Argument::required_degree
        for (auto& l : lookups) {  // mv_lookup required_degree: l_active * (table + beta) * prod(inputs + beta) * phi
            uint32_t in_deg = 1, t_deg = 1;
            for (auto& e : l.inputs) in_deg = std::max(in_deg, e->degree());
            for (auto& e : l.table) t_deg = std::max(t_deg, e->degree());
            d = std::max(d, 2 + in_deg + t_deg);
        }
        for (auto& g : gates) d = std::max(d, g->degree());
        return std::max(d, 3u);
    }
    uint32_t blinding_factors() const {  // ConstraintSystem::blinding_factors
        std::map<uint32_t, uint32_t> per_col;
        for (auto& q : advice_queries) per_col[q.first]++;
        uint32_t factors = 1;
        for (auto& kv : per_col) factors = std::max(factors, kv.second);
        factors = std::max(3u, factors);  // the permutation argument opens z at x, omega x, omega^last x
        return factors + 2;               // + 1 for the multiopen argument, + 1 for h(x)
    }
    uint32_t permutation_chunk_len() const { return degree() - 2; }
};

// ------------------------------------------------------------------------------------------------ the hot-path operations
struct Program {  // a GraphEvaluator program in the ABI's (= upstream's) form
    std::vector<b200zk_calculation> calcs;
    std::vector<b200zk_value_source> parts;
    std::vector<Fr> constants;
    std::vector<int32_t> rotations;
};
using Poly = std::vector<Fr>;
struct ProvingKey;

struct Ops {
    virtual ~Ops() = default;
    virtual G1 commit_lagrange(const Poly& values) = 0;                      // Params::commit_lagrange
    virtual G1 commit(const Poly& coeffs) = 0;                               // ParamsProver::commit (first len bases of g)
    virtual Poly lagrange_to_coeff(Poly values) = 0;                         // EvaluationDomain::lagrange_to_coeff
    virtual Poly coeff_to_extended(const Poly& coeffs) = 0;                  // EvaluationDomain::coeff_to_extended
    virtual Poly extended_to_coeff(Poly ext) = 0;                            // EvaluationDomain::extended_to_coeff (n * (j-1) coefficients)
    virtual Fr eval_polynomial(const Poly& coeffs, const Fr& x) = 0;         // arithmetic::eval_polynomial
    virtual Poly kate_division(const Poly& coeffs, const Fr& b) = 0;         // arithmetic::kate_division
    virtual Poly poly_mul(const Poly& a, const Poly& b) = 0;                 // pointwise product
    virtual Poly poly_lincomb(const std::vector<const Poly*>& polys, const std::vector<Fr>& scalars) = 0;  // sum_j s_j p_j
    // GraphEvaluator::evaluate over the extended domain; values in = PreviousValue, out = result
    virtual void graph_evaluate(const Program& p, const std::vector<const Poly*>& fixed, const std::vector<const Poly*>& advice,
                                const std::vector<const Poly*>& instance, const std::vector<Fr>& challenges, const Fr& beta,
                                const Fr& gamma, const Fr& theta, const Fr& y, Poly& values) = 0;
    // permutation::Argument::commit, one column set (all 2^k rows; the caller applies blinding)
    virtual Poly permutation_product(const std::vector<const Poly*>& values, const std::vector<const Poly*>& sigma, const Fr& beta,
                                     const Fr& gamma, const Fr& delta_omega_start, const Fr& delta, const Fr& z_init) = 0;
    // mv_lookup phi(X) running sum
    virtual Poly logup_running_sum(const std::vector<const Poly*>& inputs, const Poly& table, const Poly& m, const Fr& beta,
                                   const Fr& phi_init) = 0;
    // evaluate_h (gates, permutation, lookups folded with y) + divide_by_vanishing_poly + extended_to_coeff: the
    // n * quotient_poly_degree coefficients of h.  Columns in coefficient form, in the programs' table order:
    // advice = [cs advice..., z sets..., (m, phi) per lookup].  The default works on full extended cosets (defined below).
    virtual Poly quotient(const ProvingKey& pk, const EvaluationDomain& dom, const std::vector<const Poly*>& advice,
                          const std::vector<const Poly*>& instance, const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma,
                          const Fr& theta, const Fr& y);
};

// The product: every operation through the C ABI.  Host vectors in and out (the ABI stages them); the quotient-construction
// group takes device-resident columns, which DeviceColumn provides.
class DeviceOps : public Ops {
  public:
    DeviceOps(ParamsKZG& params, const EvaluationDomain& dom) : params_(params), dom_(dom) {}
    G1 commit_lagrange(const Poly& v) override { return params_.commit_lagrange(v); }
    G1 commit(const Poly& c) override { return params_.commit(c); }
    Poly lagrange_to_coeff(Poly v) override { return dom_.lagrange_to_coeff(std::move(v)); }
    Poly coeff_to_extended(const Poly& c) override { return dom_.coeff_to_extended(c); }
    Poly extended_to_coeff(Poly e) override { return dom_.extended_to_coeff(std::move(e)); }
    Fr eval_polynomial(const Poly& c, const Fr& x) override { return arithmetic::eval_polynomial(c, x); }
    Poly kate_division(const Poly& c, const Fr& b) override { return arithmetic::kate_division(c, b); }
    Poly poly_mul(const Poly& a, const Poly& b) override {
        if (a.size() != b.size()) throw Panic("poly_mul: length mismatch");
        Poly r(a.size());
        auto& be = Backend::get();
        be.check(b200zk_poly_mul(be.ctx(), r.data(), a.data(), b.data(), a.size()), "poly_mul");
        return r;
    }
    Poly poly_lincomb(const std::vector<const Poly*>& polys, const std::vector<Fr>& scalars) override {
        size_t n = 0;
        for (auto* p : polys) n = std::max(n, p->size());
        std::vector<DeviceColumn> cols;
        std::vector<const void*> ptrs;
        for (auto* p : polys) {
            Poly padded = *p;
            padded.resize(n, f_zero());
            cols.emplace_back(padded);
            ptrs.push_back(cols.back().ptr());
        }
        DeviceColumn out(n);
        auto& be = Backend::get();
        be.check(b200zk_poly_lincomb(be.ctx(), out.ptr(), ptrs.data(), scalars.data(), (uint32_t)ptrs.size(), n), "poly_lincomb");
        return out.to_host();
    }
    void graph_evaluate(const Program& p, const std::vector<const Poly*>& fixed, const std::vector<const Poly*>& advice,
                        const std::vector<const Poly*>& instance, const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma,
                        const Fr& theta, const Fr& y, Poly& values) override {
        auto& be = Backend::get();
        b200zk_graph* g = nullptr;
        be.check(b200zk_graph_create(be.ctx(), p.calcs.data(), (uint32_t)p.calcs.size(), p.parts.data(), (uint32_t)p.parts.size(),
                                     p.constants.data(), (uint32_t)p.constants.size(), p.rotations.data(), (uint32_t)p.rotations.size(), &g),
                 "graph_create");
        std::vector<DeviceColumn> keep;
        auto up = [&](const std::vector<const Poly*>& v) {
            std::vector<const void*> t;
            for (auto* c : v) {
                keep.emplace_back(*c);
                t.push_back(keep.back().ptr());
            }
            return t;
        };
        keep.reserve(fixed.size() + advice.size() + instance.size() + 1);
        auto tf = up(fixed), ta = up(advice), ti = up(instance);
        DeviceColumn vals(values);
        int32_t rc = b200zk_graph_evaluate(be.ctx(), g, tf.data(), (uint32_t)tf.size(), ta.data(), (uint32_t)ta.size(), ti.data(),
                                           (uint32_t)ti.size(), challenges.data(), (uint32_t)challenges.size(), &beta, &gamma, &theta, &y,
                                           &dom_.extended_omega, vals.ptr(), dom_.extended_k, 1 << (dom_.extended_k - dom_.k));
        b200zk_graph_destroy(be.ctx(), g);
        be.check(rc, "graph_evaluate");
        values = vals.to_host();
    }
    Poly permutation_product(const std::vector<const Poly*>& values, const std::vector<const Poly*>& sigma, const Fr& beta, const Fr& gamma,
                             const Fr& delta_omega_start, const Fr& delta, const Fr& z_init) override {
        std::vector<DeviceColumn> keep;
        keep.reserve(values.size() + sigma.size());
        std::vector<const DeviceColumn*> dv, ds;
        for (auto* c : values) { keep.emplace_back(*c); dv.push_back(&keep.back()); }
        for (auto* c : sigma) { keep.emplace_back(*c); ds.push_back(&keep.back()); }
        DeviceColumn z((size_t)dom_.n);
        plonk::permutation_product(dv, ds, beta, gamma, delta_omega_start, delta, dom_, z_init, z);
        return z.to_host();
    }
    Poly logup_running_sum(const std::vector<const Poly*>& inputs, const Poly& table, const Poly& m, const Fr& beta, const Fr& phi_init) override {
        std::vector<DeviceColumn> keep;
        keep.reserve(inputs.size());
        std::vector<const DeviceColumn*> di;
        for (auto* c : inputs) { keep.emplace_back(*c); di.push_back(&keep.back()); }
        DeviceColumn t(table), mm(m), phi((size_t)dom_.n);
        plonk::logup_running_sum(di, t, mm, beta, dom_, phi_init, phi);
        return phi.to_host();
    }

    // Part by part (DESIGN.md "Quotient construction"): every coefficient-form column is uploaded once; for each of the J
    // parts of the extended coset, all columns are transformed into one reused set of n-row scratch columns and the programs
    // chain into slot r of one 2^extended_k buffer; one b200zk_extended_parts_to_coeff divides by X^n - 1 and recombines.
    // No column is ever held at extended size.  Domains with more parts than the kernels support take the full-coset path.
    Poly quotient(const ProvingKey& pk, const EvaluationDomain& dom, const std::vector<const Poly*>& advice,
                  const std::vector<const Poly*>& instance, const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma,
                  const Fr& theta, const Fr& y) override;
    // device bytes the last quotient() held at its peak (columns, scratch and the part buffer)
    size_t quotient_peak_bytes() const { return quotient_peak_; }

  private:
    ParamsKZG& params_;
    const EvaluationDomain& dom_;
    size_t quotient_peak_ = 0;
};

// ------------------------------------------------------------------------------------------------ keys
struct Assembly {  // permutation::keygen::Assembly: the cell mapping built from copy constraints
    std::vector<std::vector<std::pair<uint32_t, uint32_t>>> mapping;  // mapping[col][row] = (col', row') next cell of the cycle
    Assembly(size_t n_cols, size_t n) : mapping(n_cols, std::vector<std::pair<uint32_t, uint32_t>>(n)) {
        for (size_t c = 0; c < n_cols; ++c)
            for (size_t r = 0; r < n; ++r) mapping[c][r] = {(uint32_t)c, (uint32_t)r};
    }
    // copy(left, right): merges the two cycles (swapping successors joins two disjoint cycles)
    void copy(uint32_t lc, uint32_t lr, uint32_t rc, uint32_t rr) {
        // walk left's cycle: if right is already in it, nothing to do
        auto cur = mapping[lc][lr];
        while (!(cur.first == lc && cur.second == lr)) {
            if (cur.first == rc && cur.second == rr) return;
            cur = mapping[cur.first][cur.second];
        }
        if (lc == rc && lr == rr) return;
        std::swap(mapping[lc][lr], mapping[rc][rr]);
    }
};

struct VerifyingKey {
    uint32_t k = 0;
    ConstraintSystem cs;
    std::vector<serde::G1Point> fixed_commitments, permutation_commitments;
    Fr transcript_repr{};
};
struct ProvingKey {
    VerifyingKey vk;
    Poly l0, l_last, l_active_row;                       // extended cosets
    Poly l0_poly, l_last_poly, l_active_row_poly;        // the same in coefficient form
    std::vector<Poly> fixed_values, fixed_polys, fixed_cosets;
    std::vector<Poly> sigma_values, sigma_polys, sigma_cosets;
    Program gates;                                        // custom gates folded with y
    Program permutation;                                  // evaluate_h "Permutations" section
    std::vector<Program> lookups;                         // one program per lookup
};

inline Program take_program(const GraphEvaluator& ev) { return Program{ev.calculations(), ev.horner_parts(), ev.constants(), ev.rotations()}; }

inline Fr vk_transcript_repr(const VerifyingKey& vk) {
    Blake2b h("Halo2-Verify-Key");
    auto u32 = [&](uint32_t v) { h.update((const uint8_t*)&v, 4); };
    u32(vk.k); u32(vk.cs.num_fixed); u32(vk.cs.num_advice); u32(vk.cs.num_instance); u32((uint32_t)vk.cs.gates.size());
    u32((uint32_t)vk.cs.lookups.size()); u32((uint32_t)vk.cs.permutation.size()); u32(vk.cs.degree());
    for (auto& q : vk.cs.advice_queries) { u32(q.first); u32((uint32_t)q.second); }
    for (auto& q : vk.cs.fixed_queries) { u32(q.first); u32((uint32_t)q.second); }
    if (!vk.cs.advice_phase.empty() || !vk.cs.challenge_phase.empty()) {  // single-phase keys hash as before
        u32((uint32_t)vk.cs.advice_phase.size());
        for (auto v : vk.cs.advice_phase) u32(v);
        u32((uint32_t)vk.cs.challenge_phase.size());
        for (auto v : vk.cs.challenge_phase) u32(v);
    }
    uint8_t c[32];
    for (auto& p : vk.fixed_commitments) { serde::g1_to_compressed(p, c); h.update(c, 32); }
    for (auto& p : vk.permutation_commitments) { serde::g1_to_compressed(p, c); h.update(c, 32); }
    return f_from_bytes_wide(h.finalize().data());
}

// column indices inside the GraphEvaluator's tables: fixed = [cs fixed..., l0, l_last, l_active, sigma...],
// advice = [cs advice..., z sets..., lookup m / phi / ...] -- the auxiliary polynomials are addressed like columns so that
// the permutation and lookup identities run through the same kernel as the gates (halo2_b200.hpp)
struct AuxLayout {
    uint32_t l0, l_last, l_active, sigma0;  // fixed-table indices
    uint32_t z0;                            // advice-table index of the first permutation product
    uint32_t n_sets;
};
inline AuxLayout aux_layout(const ConstraintSystem& cs) {
    AuxLayout a;
    a.l0 = cs.num_fixed;
    a.l_last = cs.num_fixed + 1;
    a.l_active = cs.num_fixed + 2;
    a.sigma0 = cs.num_fixed + 3;
    a.z0 = cs.num_advice;
    uint32_t chunk = cs.permutation_chunk_len();
    a.n_sets = cs.permutation.empty() ? 0 : (uint32_t)((cs.permutation.size() + chunk - 1) / chunk);
    return a;
}

// evaluate_h on full extended cosets: every column's coset, the programs over the whole extended domain, the 1/(X^n - 1) column
inline Poly Ops::quotient(const ProvingKey& pk, const EvaluationDomain& dom, const std::vector<const Poly*>& advice,
                          const std::vector<const Poly*>& instance, const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma,
                          const Fr& theta, const Fr& y) {
    const ConstraintSystem& cs = pk.vk.cs;
    const uint64_t n = dom.n;
    std::vector<Poly> advice_cosets, instance_cosets;
    for (auto* c : advice) advice_cosets.push_back(coeff_to_extended(*c));
    for (auto* c : instance) instance_cosets.push_back(coeff_to_extended(*c));
    const size_t ext_n = (size_t)1 << dom.extended_k;
    Poly h_ext(ext_n, f_zero());
    std::vector<const Poly*> fixed_tab, advice_tab, instance_tab;
    for (auto& c : pk.fixed_cosets) fixed_tab.push_back(&c);
    fixed_tab.push_back(&pk.l0);
    fixed_tab.push_back(&pk.l_last);
    fixed_tab.push_back(&pk.l_active_row);
    for (auto& c : pk.sigma_cosets) fixed_tab.push_back(&c);
    for (auto& c : advice_cosets) advice_tab.push_back(&c);
    for (auto& c : instance_cosets) instance_tab.push_back(&c);
    if (!pk.gates.calcs.empty()) graph_evaluate(pk.gates, fixed_tab, advice_tab, instance_tab, challenges, beta, gamma, theta, y, h_ext);
    if (!cs.permutation.empty()) graph_evaluate(pk.permutation, fixed_tab, advice_tab, instance_tab, challenges, beta, gamma, theta, y, h_ext);
    for (auto& prog : pk.lookups) graph_evaluate(prog, fixed_tab, advice_tab, instance_tab, challenges, beta, gamma, theta, y, h_ext);
    {   // EvaluationDomain::divide_by_vanishing_poly: (zeta * w_ext^i)^n - 1 takes 2^(extended_k - k) distinct values
        const size_t period = (size_t)1 << (dom.extended_k - dom.k);
        std::vector<Fr> t_inv(period);
        Fr zn = f_pow(dom.g_coset, n), wn = f_pow(dom.extended_omega, n), cur = zn;
        for (size_t i = 0; i < period; ++i) { t_inv[i] = f_inv(f_sub(cur, f_one())); cur = f_mul(cur, wn); }
        Poly t_col(ext_n);
        for (size_t i = 0; i < ext_n; ++i) t_col[i] = t_inv[i % period];
        h_ext = poly_mul(h_ext, t_col);
    }
    return extended_to_coeff(std::move(h_ext));  // n * quotient_poly_degree coefficients
}

inline Poly DeviceOps::quotient(const ProvingKey& pk, const EvaluationDomain& dom, const std::vector<const Poly*>& advice,
                                const std::vector<const Poly*>& instance, const std::vector<Fr>& challenges, const Fr& beta,
                                const Fr& gamma, const Fr& theta, const Fr& y) {
    const uint32_t k = dom.k, ek = dom.extended_k;
    if (ek - k > 4) return Ops::quotient(pk, dom, advice, instance, challenges, beta, gamma, theta, y);  // J > 16 parts
    const uint32_t J = 1u << (ek - k);
    const uint64_t n = dom.n;
    auto& be = Backend::get();
    size_t held = 0;
    quotient_peak_ = 0;
    auto hold = [&](uint64_t elems) { held += 32 * (size_t)elems; quotient_peak_ = std::max(quotient_peak_, held); };
    // the columns in the programs' table order (fixed | advice | instance), coefficient form, each uploaded once
    std::vector<const Poly*> cols;
    for (auto& c : pk.fixed_polys) cols.push_back(&c);
    cols.push_back(&pk.l0_poly);
    cols.push_back(&pk.l_last_poly);
    cols.push_back(&pk.l_active_row_poly);
    for (auto& c : pk.sigma_polys) cols.push_back(&c);
    const uint32_t n_fixed = (uint32_t)cols.size();
    cols.insert(cols.end(), advice.begin(), advice.end());
    cols.insert(cols.end(), instance.begin(), instance.end());
    const uint32_t n_advice = (uint32_t)advice.size(), n_instance = (uint32_t)instance.size();
    std::vector<DeviceColumn> coeff, part_cols;
    coeff.reserve(cols.size());
    part_cols.reserve(cols.size());
    std::vector<const void*> coeff_ptrs;
    std::vector<void*> part_ptrs;
    for (auto* c : cols) {
        coeff.emplace_back(*c);
        hold(n);
        coeff_ptrs.push_back(coeff.back().ptr());
    }
    for (size_t i = 0; i < cols.size(); ++i) {
        part_cols.emplace_back((size_t)n);
        hold(n);
        part_ptrs.push_back(part_cols.back().ptr());
    }
    DeviceColumn parts((size_t)J * n);
    hold((uint64_t)J * n);
    struct Graphs {  // the evaluate_h programs, released on every exit
        std::vector<b200zk_graph*> g;
        ~Graphs() { for (auto* h : g) b200zk_graph_destroy(Backend::get().ctx(), h); }
    } graphs;
    auto compile = [&](const Program& p) {
        b200zk_graph* g = nullptr;
        be.check(b200zk_graph_create(be.ctx(), p.calcs.data(), (uint32_t)p.calcs.size(), p.parts.data(), (uint32_t)p.parts.size(),
                                     p.constants.data(), (uint32_t)p.constants.size(), p.rotations.data(), (uint32_t)p.rotations.size(), &g),
                 "graph_create");
        graphs.g.push_back(g);
    };
    if (!pk.gates.calcs.empty()) compile(pk.gates);
    if (!pk.vk.cs.permutation.empty()) compile(pk.permutation);
    for (auto& prog : pk.lookups) compile(prog);
    const Poly zeros(n, f_zero());
    const void* const* tf = (const void* const*)part_ptrs.data();
    for (uint32_t r = 0; r < J; ++r) {
        be.check(b200zk_coeff_to_extended_parts(be.ctx(), coeff_ptrs.data(), (uint32_t)cols.size(), k, ek, r, part_ptrs.data()),
                 "coeff_to_extended_parts");
        void* slot = (char*)parts.ptr() + 32 * (size_t)r * n;
        be.check(b200zk_buf_upload(be.ctx(), slot, zeros.data(), 32 * n), "quotient: clear part");
        for (auto* g : graphs.g)
            be.check(b200zk_graph_evaluate_part(be.ctx(), g, tf, n_fixed, tf + n_fixed, n_advice, tf + n_fixed + n_advice, n_instance,
                                                challenges.data(), (uint32_t)challenges.size(), &beta, &gamma, &theta, &y, k, ek, r, slot),
                     "graph_evaluate_part");
    }
    const uint64_t pieces = dom.quotient_poly_degree;
    be.check(b200zk_extended_parts_to_coeff(be.ctx(), parts.ptr(), k, ek, (uint32_t)pieces, 1, parts.ptr()), "extended_parts_to_coeff");
    Poly h(pieces * n);
    be.check(b200zk_buf_download(be.ctx(), h.data(), parts.ptr(), 32 * pieces * n), "quotient: download");
    return h;
}

// keygen_vk + keygen_pk: fixed columns (Lagrange values), the permutation assembly; polynomials and cosets through `ops`
inline ProvingKey keygen(Ops& ops, const EvaluationDomain& dom, ConstraintSystem cs, const std::vector<Poly>& fixed, const Assembly& assembly) {
    if (cs.advice_queries.empty() && cs.fixed_queries.empty()) cs.finalize();
    const uint64_t n = dom.n;
    if (fixed.size() != cs.num_fixed) throw Panic("keygen: wrong number of fixed columns");
    if (!cs.advice_phase.empty() && cs.advice_phase.size() != cs.num_advice) throw Panic("keygen: one phase per advice column");
    {   // every Expression::Challenge names a declared challenge
        std::function<void(const Expr&)> check = [&](const Expr& e) {
            if (e.kind == Expr::Challenge && e.col >= cs.challenge_phase.size()) throw Panic("keygen: expression uses an undeclared challenge");
            if (e.a) check(*e.a);
            if (e.b) check(*e.b);
        };
        for (auto& g : cs.gates) check(*g);
        for (auto& l : cs.lookups) {
            for (auto& e : l.inputs) check(*e);
            for (auto& e : l.table) check(*e);
        }
    }
    if (cs.degree() - 1 > dom.quotient_poly_degree) throw Panic("keygen: the domain's quotient degree is too small for this constraint system");
    ProvingKey pk;
    pk.vk.k = dom.k;
    pk.vk.cs = cs;
    for (auto& col : fixed) {
        if (col.size() != n) throw Panic("keygen: fixed column length");
        pk.fixed_values.push_back(col);
        pk.vk.fixed_commitments.push_back(to_affine_point(ops.commit_lagrange(col)));
        pk.fixed_polys.push_back(ops.lagrange_to_coeff(col));
        pk.fixed_cosets.push_back(ops.coeff_to_extended(pk.fixed_polys.back()));
    }
    // permutation::keygen::Assembly::build_{vk,pk}: sigma_i(omega^j) = delta^{i'} omega^{j'} for mapping[i][j] = (i', j')
    const Fr delta = f_delta();
    std::vector<Fr> omega_pow(n), delta_pow(cs.permutation.size());
    Fr cur = f_one();
    for (uint64_t j = 0; j < n; ++j) { omega_pow[j] = cur; cur = f_mul(cur, dom.omega); }
    cur = f_one();
    for (auto& d : delta_pow) { d = cur; cur = f_mul(cur, delta); }
    for (size_t i = 0; i < cs.permutation.size(); ++i) {
        Poly s(n);
        for (uint64_t j = 0; j < n; ++j) {
            auto m = assembly.mapping[i][j];
            s[j] = f_mul(delta_pow[m.first], omega_pow[m.second]);
        }
        pk.sigma_values.push_back(s);
        pk.vk.permutation_commitments.push_back(to_affine_point(ops.commit_lagrange(s)));
        pk.sigma_polys.push_back(ops.lagrange_to_coeff(s));
        pk.sigma_cosets.push_back(ops.coeff_to_extended(pk.sigma_polys.back()));
    }
    // l0, l_last, l_active_row (keygen_pk): l_blind covers the last blinding_factors rows, l_last the row before them
    const uint32_t bf = cs.blinding_factors();
    if (n < (uint64_t)bf + 3) throw Panic("keygen: not enough rows");
    Poly l0(n, f_zero()), l_blind(n, f_zero()), l_last(n, f_zero());
    l0[0] = f_one();
    for (uint64_t r = n - bf; r < n; ++r) l_blind[r] = f_one();
    l_last[n - bf - 1] = f_one();
    pk.l0_poly = ops.lagrange_to_coeff(l0);
    pk.l0 = ops.coeff_to_extended(pk.l0_poly);
    Poly lb_poly = ops.lagrange_to_coeff(l_blind);
    Poly lb = ops.coeff_to_extended(lb_poly);
    pk.l_last_poly = ops.lagrange_to_coeff(l_last);
    pk.l_last = ops.coeff_to_extended(pk.l_last_poly);
    pk.l_active_row.resize(pk.l0.size());
    for (size_t i = 0; i < pk.l0.size(); ++i) pk.l_active_row[i] = f_sub(f_sub(f_one(), pk.l_last[i]), lb[i]);
    // 1 - l_last - l_blind in coefficient form (the constant 1 is coefficient 0): its coset is l_active_row exactly
    pk.l_active_row_poly.resize(n);
    for (uint64_t i = 0; i < n; ++i) pk.l_active_row_poly[i] = f_sub(f_sub(i == 0 ? f_one() : f_zero(), pk.l_last_poly[i]), lb_poly[i]);
    pk.vk.transcript_repr = vk_transcript_repr(pk.vk);

    // ---- Evaluator::new: the programs of evaluate_h
    const AuxLayout aux = aux_layout(cs);
    {
        GraphEvaluator ev;  // custom gates: value = value * y + gate_i  (one Horner over all gate polynomials)
        std::vector<ValueSource> parts;
        for (auto& g : cs.gates) parts.push_back(add_expression(ev, *g));
        if (!parts.empty()) ev.add_horner(ValueSource::PreviousValue(), parts, ValueSource::Y());
        pk.gates = take_program(ev);
    }
    if (!cs.permutation.empty()) {
        GraphEvaluator ev;
        const uint32_t r0 = ev.add_rotation(0);
        std::vector<ValueSource> z, vals, sig;
        for (uint32_t s = 0; s < aux.n_sets; ++s) z.push_back(ValueSource::Advice(aux.z0 + s, r0));
        for (size_t i = 0; i < cs.permutation.size(); ++i) {
            const Column& c = cs.permutation[i];
            vals.push_back(c.kind == Expr::Advice ? ValueSource::Advice(c.index, r0)
                                                  : (c.kind == Expr::Fixed ? ValueSource::Fixed(c.index, r0) : ValueSource::Instance(c.index, r0)));
            sig.push_back(ValueSource::Fixed(aux.sigma0 + (uint32_t)i, r0));
        }
        permutation_constraints(ev, z, cs.permutation_chunk_len(), vals, sig, ValueSource::Fixed(aux.l0, r0), ValueSource::Fixed(aux.l_last, r0),
                                ValueSource::Fixed(aux.l_active, r0), -(int32_t)(bf + 1), delta);
        pk.permutation = take_program(ev);
    }
    for (size_t li = 0; li < cs.lookups.size(); ++li) {
        // evaluate_h's lookup section: the input / table expressions are compressed with theta ON the extended coset
        // (Horner(0, parts, Theta), evaluation.rs `evaluate_lc`) -- as products of column cosets, not as interpolants of their
        // row values; m and phi are supplied as advice-like columns after the z sets: base + 0 = m, base + 1 = phi
        GraphEvaluator ev;
        const uint32_t r0 = ev.add_rotation(0);
        const uint32_t base = aux.z0 + aux.n_sets + 2 * (uint32_t)li;
        const ValueSource zero = ev.add_constant(f_zero());
        auto compress = [&](const std::vector<ExprP>& exprs) {
            std::vector<ValueSource> parts;
            for (auto& e : exprs) parts.push_back(add_expression(ev, *e));
            return ev.add_horner(zero, parts, ValueSource::Theta());
        };
        const ValueSource input = compress(cs.lookups[li].inputs), table = compress(cs.lookups[li].table);
        lookup_constraints(ev, {input}, table, ValueSource::Advice(base, r0), ValueSource::Advice(base + 1, r0), ValueSource::Fixed(aux.l0, r0),
                           ValueSource::Fixed(aux.l_last, r0), ValueSource::Fixed(aux.l_active, r0));
        pk.lookups.push_back(take_program(ev));
    }
    return pk;
}

// ------------------------------------------------------------------------------------------------ helpers shared by prover and verifier
struct Rng {  // deterministic blinding (fixed-seed xorshift64*; upstream takes an RngCore)
    uint64_t s;
    explicit Rng(uint64_t seed) : s(seed ? seed : 0x9E3779B97F4A7C15ull) {}
    uint64_t next() {
        s ^= s >> 12; s ^= s << 25; s ^= s >> 27;
        return s * 0x2545F4914F6CDD1Dull;
    }
    Fr fr() {
        uint8_t b[64];
        for (int i = 0; i < 8; ++i) { uint64_t v = next(); std::memcpy(b + 8 * i, &v, 8); }
        return f_from_bytes_wide(b);
    }
};

inline Fr rotate_omega(const EvaluationDomain& dom, const Fr& x, int32_t rot) {  // EvaluationDomain::rotate_omega
    Fr w = rot >= 0 ? f_pow(dom.omega, (uint64_t)rot) : f_pow(dom.omega_inv, (uint64_t)(-(int64_t)rot));
    return f_mul(x, w);
}

// lagrange_interpolate(points, evals) -> coefficients (arithmetic.rs); the point sets of a proof have <= 3 points
inline Poly lagrange_interpolate(const std::vector<Fr>& pts, const std::vector<Fr>& evals) {
    size_t m = pts.size();
    Poly out(m, f_zero());
    for (size_t j = 0; j < m; ++j) {
        Poly num{f_one()};  // prod_{k != j} (X - x_k)
        Fr den = f_one();
        for (size_t k = 0; k < m; ++k) {
            if (k == j) continue;
            Poly nx(num.size() + 1, f_zero());
            for (size_t i = 0; i < num.size(); ++i) {
                nx[i + 1] = f_add(nx[i + 1], num[i]);
                nx[i] = f_sub(nx[i], f_mul(num[i], pts[k]));
            }
            num = nx;
            den = f_mul(den, f_sub(pts[j], pts[k]));
        }
        Fr s = f_mul(evals[j], f_inv(den));
        for (size_t i = 0; i < num.size(); ++i) out[i] = f_add(out[i], f_mul(num[i], s));
    }
    return out;
}
inline Fr eval_small(const Poly& p, const Fr& x) {
    Fr acc = f_zero();
    for (size_t i = p.size(); i-- > 0;) acc = f_add(f_mul(acc, x), p[i]);
    return acc;
}

// one opening claim: polynomial (prover) / commitment (verifier), point, evaluation
struct Query {
    size_t poly_id;  // identity of the polynomial / commitment (queries of the same id share a rotation set)
    Fr point, eval;
};
struct RotationSets {  // shplonk::construct_intermediate_sets
    struct Set {
        std::vector<Fr> points;
        std::vector<size_t> polys;                 // poly ids, in first-appearance order
        std::vector<std::vector<Fr>> evals;        // evals[poly][point]
    };
    std::vector<Set> sets;
    std::vector<Fr> super_points;
};
inline RotationSets build_rotation_sets(const std::vector<Query>& queries) {
    auto same = [](const Fr& a, const Fr& b) { return a == b; };
    std::vector<size_t> order;                       // distinct poly ids in first-appearance order
    std::map<size_t, std::vector<std::pair<Fr, Fr>>> per_poly;
    RotationSets rs;
    for (auto& q : queries) {
        if (!per_poly.count(q.poly_id)) order.push_back(q.poly_id);
        auto& v = per_poly[q.poly_id];
        bool dup = false;
        for (auto& pe : v) dup |= same(pe.first, q.point);
        if (!dup) v.push_back({q.point, q.eval});
        bool seen = false;
        for (auto& p : rs.super_points) seen |= same(p, q.point);
        if (!seen) rs.super_points.push_back(q.point);
    }
    for (size_t id : order) {
        auto& v = per_poly[id];
        RotationSets::Set* target = nullptr;
        for (auto& s : rs.sets) {  // same point SET (order-insensitive)
            if (s.points.size() != v.size()) continue;
            bool all = true;
            for (auto& pe : v) {
                bool in = false;
                for (auto& p : s.points) in |= same(p, pe.first);
                all &= in;
            }
            if (all) { target = &s; break; }
        }
        if (!target) {
            rs.sets.emplace_back();
            target = &rs.sets.back();
            for (auto& pe : v) target->points.push_back(pe.first);
        }
        std::vector<Fr> ev;
        for (auto& p : target->points)
            for (auto& pe : v)
                if (same(pe.first, p)) ev.push_back(pe.second);
        target->polys.push_back(id);
        target->evals.push_back(ev);
    }
    return rs;
}

// ------------------------------------------------------------------------------------------------ create_proof
struct ProofArtifacts {  // what a caller may want beside the bytes (tests)
    std::vector<uint8_t> proof;
    size_t n_commitments = 0, n_evals = 0;
};

// The caller's witness generation (upstream: Circuit::synthesize run once per phase through WitnessCollection): called for
// phase 0, 1, ... with the challenges squeezed so far (entries of later phases are zero) and the advice table; it fills the usable
// rows of the columns of THAT phase (columns of earlier phases hold what was committed, writes to them are discarded).
using WitnessFn = std::function<void(uint32_t phase, const std::vector<Fr>& challenges, std::vector<Poly>& advice)>;

// plonk::create_proof for one circuit instance.  Per phase: witness, blinding rows, commit_lagrange of that phase's advice columns,
// then the phase's challenges from the transcript (prover.rs `for current_phase in pk.vk.cs.phases()`); instances: Lagrange values
// of the instance columns.
inline ProofArtifacts create_proof(Ops& ops, const EvaluationDomain& dom, const ProvingKey& pk, const WitnessFn& synthesize,
                                   const std::vector<Poly>& instances, uint64_t rng_seed,
                                   TranscriptKind transcript_kind = TranscriptKind::Blake2b) {
    const ConstraintSystem& cs = pk.vk.cs;
    const uint64_t n = dom.n;
    const uint32_t bf = cs.blinding_factors();
    const uint64_t u = n - bf - 1;  // last usable row index (the l_last row); rows > u are blinding rows
    const AuxLayout aux = aux_layout(cs);
    if (instances.size() != cs.num_instance) throw Panic("create_proof: wrong number of columns");
    if (!cs.advice_phase.empty() && cs.advice_phase.size() != cs.num_advice) throw Panic("create_proof: one phase per advice column");
    Rng rng(rng_seed);
    Transcript tr(transcript_kind);
    ProofArtifacts art;
    auto write_point = [&](const G1& c) { tr.write_point(c); art.n_commitments++; };

    // 0. vk and instances into the transcript (vk.hash_into; instance values as common scalars -- KZG: query_instance = false)
    tr.common_scalar(pk.vk.transcript_repr);
    std::vector<Poly> instance_polys;
    for (auto& inst : instances) {
        if (inst.size() != n) throw Panic("create_proof: instance column length");
        for (uint64_t r = u; r < n; ++r)
            if (!f_is_zero(inst[r])) throw Panic("create_proof: instance values beyond the usable rows");
        instance_polys.push_back(ops.lagrange_to_coeff(inst));
    }
    for (auto& inst : instances)
        for (uint64_t r = 0; r < u; ++r) tr.common_scalar(inst[r]);

    // 1. advice, phase by phase: witness, blinding rows, commitments (commit_lagrange), the phase's challenges; then the
    //    coefficient form of every column
    std::vector<Poly> advice(cs.num_advice, Poly(n, f_zero())), advice_polys;
    std::vector<Fr> challenges(cs.challenge_phase.size(), f_zero());
    for (uint32_t phase = 0; phase < cs.num_phases(); ++phase) {
        std::vector<Poly> work = advice;
        synthesize(phase, challenges, work);
        if (work.size() != cs.num_advice) throw Panic("create_proof: wrong number of columns");
        for (uint32_t c = 0; c < cs.num_advice; ++c) {
            if (cs.phase_of_advice(c) != phase) continue;
            if (work[c].size() != n) throw Panic("create_proof: advice column length");
            advice[c] = std::move(work[c]);
            for (uint64_t r = u; r < n; ++r) advice[c][r] = rng.fr();  // unusable_rows_start = n - (blinding_factors + 1)
        }
        for (uint32_t c = 0; c < cs.num_advice; ++c)
            if (cs.phase_of_advice(c) == phase) write_point(ops.commit_lagrange(advice[c]));
        for (size_t i = 0; i < challenges.size(); ++i)
            if (cs.challenge_phase[i] == phase) challenges[i] = tr.squeeze_challenge();
    }
    for (auto& col : advice) advice_polys.push_back(ops.lagrange_to_coeff(col));
    const Fr theta = tr.squeeze_challenge();

    // 2. lookups, first half (mv_lookup::Argument::prepare): compress with theta, count multiplicities, commit m
    auto lagrange_query = [&](uint64_t row) {
        return [&, row](int kind, uint32_t col, int32_t rot) -> Fr {
            uint64_t r = (uint64_t)(((int64_t)row + rot) % (int64_t)n + (int64_t)n) % n;
            if (kind == Expr::Challenge) return challenges[col];
            if (kind == Expr::Fixed) return pk.fixed_values[col][r];
            if (kind == Expr::Advice) return advice[col][r];
            return instances[col][r];
        };
    };
    auto compress = [&](const std::vector<ExprP>& exprs) {  // fold(acc * theta + expr) over the rows of the domain
        Poly out(n);
        for (uint64_t r = 0; r < n; ++r) {
            Fr acc = f_zero();
            auto q = lagrange_query(r);
            for (auto& e : exprs) acc = f_add(f_mul(acc, theta), e->eval_with(q));
            out[r] = acc;
        }
        return out;
    };
    struct LookupState { Poly input, table, m, phi, m_poly, phi_poly; };
    std::vector<LookupState> lk(cs.lookups.size());
    for (size_t li = 0; li < cs.lookups.size(); ++li) {
        lk[li].input = compress(cs.lookups[li].inputs);
        lk[li].table = compress(cs.lookups[li].table);
        lk[li].m.assign(n, f_zero());
        std::map<std::array<uint64_t, 4>, uint64_t> index;  // table value -> first row holding it (usable rows only)
        for (uint64_t r = 0; r < u; ++r) {
            std::array<uint64_t, 4> key{lk[li].table[r].l[0], lk[li].table[r].l[1], lk[li].table[r].l[2], lk[li].table[r].l[3]};
            index.emplace(key, r);
        }
        std::vector<uint64_t> counts(n, 0);
        for (uint64_t r = 0; r < u; ++r) {
            std::array<uint64_t, 4> key{lk[li].input[r].l[0], lk[li].input[r].l[1], lk[li].input[r].l[2], lk[li].input[r].l[3]};
            auto it = index.find(key);
            if (it == index.end()) throw Panic("lookup input is not in the table (the witness does not satisfy the lookup)");
            counts[it->second]++;
        }
        for (uint64_t r = 0; r < n; ++r) lk[li].m[r] = f_u64(counts[r]);
        write_point(ops.commit_lagrange(lk[li].m));
    }
    const Fr beta = tr.squeeze_challenge();
    const Fr gamma = tr.squeeze_challenge();

    // 3. permutation::Argument::commit: one grand product per column set, chained through z[u]
    const Fr delta = f_delta();
    std::vector<Poly> z_values, z_polys;
    if (!cs.permutation.empty()) {
        const uint32_t chunk = cs.permutation_chunk_len();
        Fr z_init = f_one(), delta_omega = f_one();
        for (uint32_t s = 0; s < aux.n_sets; ++s) {
            std::vector<const Poly*> vals, sig;
            for (size_t i = (size_t)s * chunk; i < std::min(cs.permutation.size(), (size_t)(s + 1) * chunk); ++i) {
                const Column& c = cs.permutation[i];
                vals.push_back(c.kind == Expr::Advice ? &advice[c.index] : (c.kind == Expr::Fixed ? &pk.fixed_values[c.index] : &instances[c.index]));
                sig.push_back(&pk.sigma_values[i]);
            }
            Poly z = ops.permutation_product(vals, sig, beta, gamma, delta_omega, delta, z_init);
            z_init = z[u];
            for (uint64_t r = u + 1; r < n; ++r) z[r] = rng.fr();
            for (size_t i = 0; i < vals.size(); ++i) delta_omega = f_mul(delta_omega, delta);
            z_values.push_back(z);
        }
        if (!(z_init == f_one())) throw Panic("permutation product does not close: the witness violates a copy constraint");
        for (auto& z : z_values) write_point(ops.commit_lagrange(z));
        for (auto& z : z_values) z_polys.push_back(ops.lagrange_to_coeff(z));
    }
    // 4. lookups, second half (commit_grand_sum): phi running sum, blinded, committed
    for (auto& l : lk) {
        l.phi = ops.logup_running_sum({&l.input}, l.table, l.m, beta, f_zero());
        if (!f_is_zero(l.phi[u])) throw Panic("lookup running sum does not close");
        for (uint64_t r = u + 1; r < n; ++r) l.phi[r] = rng.fr();
        write_point(ops.commit_lagrange(l.phi));
    }
    // 5. vanishing::Argument::commit: a random polynomial of degree n - 1
    Poly random_poly(n);
    for (auto& c : random_poly) c = rng.fr();
    write_point(ops.commit(random_poly));
    const Fr y = tr.squeeze_challenge();

    // 6. evaluate_h: gates, permutation, lookups folded with y; divided by X^n - 1; back to coefficients
    std::vector<const Poly*> advice_tab, instance_tab;
    for (auto& c : advice_polys) advice_tab.push_back(&c);
    for (auto& c : z_polys) advice_tab.push_back(&c);
    for (auto& l : lk) {
        l.m_poly = ops.lagrange_to_coeff(l.m);
        l.phi_poly = ops.lagrange_to_coeff(l.phi);
        advice_tab.push_back(&l.m_poly);
        advice_tab.push_back(&l.phi_poly);
    }
    for (auto& c : instance_polys) instance_tab.push_back(&c);
    Poly h_coeffs = ops.quotient(pk, dom, advice_tab, instance_tab, challenges, beta, gamma, theta, y);  // n * quotient_poly_degree
    // vanishing::Committed::construct: pieces of n coefficients, each committed
    std::vector<Poly> h_pieces;
    for (size_t i = 0; i < dom.quotient_poly_degree; ++i) h_pieces.emplace_back(h_coeffs.begin() + i * n, h_coeffs.begin() + (i + 1) * n);
    for (auto& p : h_pieces) write_point(ops.commit(p));
    const Fr x = tr.squeeze_challenge();
    const Fr xn = f_pow(x, n);

    // 7. evaluations, in upstream's order; every evaluated polynomial also becomes an opening query
    std::vector<const Poly*> open_polys;  // poly id -> coefficients
    std::vector<Query> queries;
    auto poly_id = [&](const Poly* p) {
        for (size_t i = 0; i < open_polys.size(); ++i)
            if (open_polys[i] == p) return i;
        open_polys.push_back(p);
        return open_polys.size() - 1;
    };
    auto eval_and_write = [&](const Poly& p, const Fr& at, bool write) {
        Fr v = ops.eval_polynomial(p, at);
        if (write) { tr.write_scalar(v); art.n_evals++; }
        return v;
    };
    std::vector<Query> q_advice, q_fixed, q_perm_common, q_perm, q_lookup, q_vanishing;
    for (auto& q : cs.advice_queries) {
        Fr at = rotate_omega(dom, x, q.second);
        q_advice.push_back({poly_id(&advice_polys[q.first]), at, eval_and_write(advice_polys[q.first], at, true)});
    }
    for (auto& q : cs.fixed_queries) {
        Fr at = rotate_omega(dom, x, q.second);
        q_fixed.push_back({poly_id(&pk.fixed_polys[q.first]), at, eval_and_write(pk.fixed_polys[q.first], at, true)});
    }
    // vanishing::Constructed::evaluate: h(X) = sum_i x^(n i) h_i(X) folded, and the random polynomial's evaluation
    Poly h_poly;
    {
        std::vector<const Poly*> ps;
        std::vector<Fr> sc;
        Fr p = f_one();
        for (auto& piece : h_pieces) { ps.push_back(&piece); sc.push_back(p); p = f_mul(p, xn); }
        h_poly = ops.poly_lincomb(ps, sc);
    }
    const Fr random_eval = eval_and_write(random_poly, x, true);
    for (auto& s : pk.sigma_polys) q_perm_common.push_back({poly_id(&s), x, eval_and_write(s, x, true)});  // permutation::ProvingKey::evaluate
    const Fr x_next = rotate_omega(dom, x, 1), x_last = rotate_omega(dom, x, -(int32_t)(bf + 1));
    for (size_t s = 0; s < z_polys.size(); ++s) {  // permutation::Constructed::evaluate
        q_perm.push_back({poly_id(&z_polys[s]), x, eval_and_write(z_polys[s], x, true)});
        q_perm.push_back({poly_id(&z_polys[s]), x_next, eval_and_write(z_polys[s], x_next, true)});
        if (s + 1 < z_polys.size()) q_perm.push_back({poly_id(&z_polys[s]), x_last, eval_and_write(z_polys[s], x_last, true)});
    }
    for (auto& l : lk) {  // mv_lookup::Committed::evaluate: phi(x), phi(omega x), m(x)
        q_lookup.push_back({poly_id(&l.phi_poly), x, eval_and_write(l.phi_poly, x, true)});
        q_lookup.push_back({poly_id(&l.phi_poly), x_next, eval_and_write(l.phi_poly, x_next, true)});
        q_lookup.push_back({poly_id(&l.m_poly), x, eval_and_write(l.m_poly, x, true)});
    }
    q_vanishing.push_back({poly_id(&h_poly), x, eval_and_write(h_poly, x, false)});
    q_vanishing.push_back({poly_id(&random_poly), x, random_eval});
    // the query order of create_proof: advice, permutation, lookups, fixed, permutation common, vanishing
    for (auto* v : {&q_advice, &q_perm, &q_lookup, &q_fixed, &q_perm_common, &q_vanishing})
        queries.insert(queries.end(), v->begin(), v->end());

    // 8. ProverSHPLONK::create_proof
    const Fr sy = tr.squeeze_challenge();  // y of the multiopen argument
    const Fr sv = tr.squeeze_challenge();  // v
    RotationSets rs = build_rotation_sets(queries);
    std::vector<Poly> set_numerators;      // per set: sum_j y^j (p_j(X) - r_j(X)), ascending powers in query order
    std::vector<std::vector<Poly>> set_r;  // r_j(X) per set and polynomial
    Poly h_open;                           // sum_i v^i quotient_set_i, ascending powers in set order
    {
        std::vector<Poly> quotients;
        for (auto& set : rs.sets) {
            std::vector<Poly> diffs, rpolys;
            for (size_t j = 0; j < set.polys.size(); ++j) {
                Poly r = lagrange_interpolate(set.points, set.evals[j]);
                Poly d = *open_polys[set.polys[j]];
                for (size_t i = 0; i < r.size(); ++i) d[i] = f_sub(d[i], r[i]);
                diffs.push_back(std::move(d));
                rpolys.push_back(std::move(r));
            }
            std::vector<const Poly*> ps;
            std::vector<Fr> sc(diffs.size());
            Fr p = f_one();
            for (size_t j = 0; j < diffs.size(); ++j) { sc[j] = p; p = f_mul(p, sy); }  // numerators.zip(powers(y)): ascending powers, as upstream
            for (auto& d : diffs) ps.push_back(&d);
            Poly num = ops.poly_lincomb(ps, sc);
            Poly q = num;
            for (auto& pt : set.points) q = ops.kate_division(q, pt);  // div_by_vanishing: one root at a time
            quotients.push_back(std::move(q));
            set_numerators.push_back(std::move(num));
            set_r.push_back(std::move(rpolys));
        }
        std::vector<const Poly*> ps;
        std::vector<Fr> sc(quotients.size());
        Fr p = f_one();
        for (size_t i = 0; i < quotients.size(); ++i) { sc[i] = p; p = f_mul(p, sv); }  // .zip(powers(v))
        for (auto& q : quotients) ps.push_back(&q);
        h_open = ops.poly_lincomb(ps, sc);
    }
    write_point(ops.commit(h_open));
    const Fr su = tr.squeeze_challenge();  // u
    {
        // L(X) = sum_i v^(..) z_diff_i (N_i(X) - N_i's remainder at u) - Z_T(u) h(X), normalised by 1 / z_diff_0; L(u) = 0
        Fr zt = f_one();
        for (auto& p : rs.super_points) zt = f_mul(zt, f_sub(su, p));
        std::vector<Fr> z_diff(rs.sets.size());
        for (size_t i = 0; i < rs.sets.size(); ++i) {
            Fr zs = f_one();
            for (auto& p : rs.sets[i].points) zs = f_mul(zs, f_sub(su, p));
            z_diff[i] = f_mul(zt, f_inv(zs));
        }
        const Fr z0_inv = f_inv(z_diff[0]);
        std::vector<const Poly*> ps;
        std::vector<Fr> sc;
        Fr constant = f_zero();  // the r_ij(u) part, subtracted from the constant coefficient
        Fr vp = f_one();
        std::vector<Fr> vpow(rs.sets.size());
        for (size_t i = 0; i < rs.sets.size(); ++i) { vpow[i] = vp; vp = f_mul(vp, sv); }
        for (size_t i = 0; i < rs.sets.size(); ++i) {
            const Fr w = f_mul(f_mul(vpow[i], z_diff[i]), z0_inv);
            // N_i(X) + sum_j y^(..) r_ij(X)  is  sum_j y^(..) p_ij(X); we need  sum_j y^(..) (p_ij(X) - r_ij(u))
            Fr yp = f_one(), ru = f_zero();
            std::vector<Fr> ypow(set_r[i].size());
            for (size_t j = 0; j < set_r[i].size(); ++j) { ypow[j] = yp; yp = f_mul(yp, sy); }
            for (size_t j = 0; j < set_r[i].size(); ++j) {
                ps.push_back(open_polys[rs.sets[i].polys[j]]);
                sc.push_back(f_mul(w, ypow[j]));
                ru = f_add(ru, f_mul(ypow[j], eval_small(set_r[i][j], su)));
            }
            constant = f_add(constant, f_mul(w, ru));
        }
        ps.push_back(&h_open);
        sc.push_back(f_neg(f_mul(zt, z0_inv)));
        Poly L = ops.poly_lincomb(ps, sc);
        L[0] = f_sub(L[0], constant);
        if (!f_is_zero(ops.eval_polynomial(L, su))) throw Panic("SHPLONK: the linearisation polynomial does not vanish at u");
        write_point(ops.commit(ops.kate_division(L, su)));
    }
    art.proof = tr.finalize();
    return art;
}

// the witness known up front (single-phase circuits, or a caller that already holds every phase's columns)
inline ProofArtifacts create_proof(Ops& ops, const EvaluationDomain& dom, const ProvingKey& pk, std::vector<Poly> advice,
                                   const std::vector<Poly>& instances, uint64_t rng_seed,
                                   TranscriptKind transcript_kind = TranscriptKind::Blake2b) {
    if (advice.size() != pk.vk.cs.num_advice) throw Panic("create_proof: wrong number of columns");
    const ConstraintSystem& cs = pk.vk.cs;
    WitnessFn fill = [&](uint32_t phase, const std::vector<Fr>&, std::vector<Poly>& table) {
        for (uint32_t c = 0; c < cs.num_advice; ++c)
            if (cs.phase_of_advice(c) == phase) table[c] = advice[c];
    };
    return create_proof(ops, dom, pk, fill, instances, rng_seed, transcript_kind);
}

// ------------------------------------------------------------------------------------------------ MockProver (host only)
// dev::MockProver::run + verify, the check the reference's `make mock` performs before any proving
// (/root/reference/integration/src/mock.rs:11-30 -> MockProver::verify_par): the witness is synthesised phase by phase (challenges
// from `seed` instead of a transcript), the rows beyond the usable ones are filled with random values as create_proof would blind
// them, and every constraint is evaluated with plain field arithmetic -- no polynomial, no commitment, no device:
//   gates on EVERY row of the domain (what the quotient identity demands; a selector that is live on a row whose rotations reach
//   into the blinding rows shows up here), lookup inputs against the table on the usable rows, copy constraints cell by cell.
struct MockFailure {
    enum Kind { Gate, Lookup, Permutation } kind;
    size_t index;  // gate index, lookup index, or index of the column in cs.permutation
    uint64_t row;
    bool operator==(const MockFailure& o) const { return kind == o.kind && index == o.index && row == o.row; }
};
inline std::vector<MockFailure> mock_prove(const EvaluationDomain& dom, ConstraintSystem cs, const std::vector<Poly>& fixed, const Assembly& assembly,
                                           const WitnessFn& synthesize, const std::vector<Poly>& instances, uint64_t seed = 1) {
    if (cs.advice_queries.empty() && cs.fixed_queries.empty()) cs.finalize();
    const uint64_t n = dom.n, u = n - cs.blinding_factors() - 1;
    if (fixed.size() != cs.num_fixed || instances.size() != cs.num_instance) throw Panic("mock_prove: wrong number of columns");
    Rng rng(seed);
    std::vector<Poly> advice(cs.num_advice, Poly(n, f_zero()));
    std::vector<Fr> challenges(cs.challenge_phase.size(), f_zero());
    for (uint32_t phase = 0; phase < cs.num_phases(); ++phase) {
        std::vector<Poly> work = advice;
        synthesize(phase, challenges, work);
        for (uint32_t c = 0; c < cs.num_advice; ++c) {
            if (cs.phase_of_advice(c) != phase) continue;
            if (work[c].size() != n) throw Panic("mock_prove: advice column length");
            advice[c] = std::move(work[c]);
            for (uint64_t r = u; r < n; ++r) advice[c][r] = rng.fr();
        }
        for (size_t i = 0; i < challenges.size(); ++i)
            if (cs.challenge_phase[i] == phase) challenges[i] = rng.fr();
    }
    const Fr theta = rng.fr();
    auto cell = [&](uint64_t row) {
        return [&, row](int kind, uint32_t col, int32_t rot) -> Fr {
            if (kind == Expr::Challenge) return challenges[col];
            const uint64_t r = (uint64_t)((((int64_t)row + rot) % (int64_t)n + (int64_t)n) % (int64_t)n);
            return kind == Expr::Fixed ? fixed[col][r] : (kind == Expr::Advice ? advice[col][r] : instances[col][r]);
        };
    };
    std::vector<MockFailure> failures;
    for (size_t g = 0; g < cs.gates.size(); ++g)
        for (uint64_t r = 0; r < n; ++r)
            if (!f_is_zero(cs.gates[g]->eval_with(cell(r)))) failures.push_back({MockFailure::Gate, g, r});
    for (size_t li = 0; li < cs.lookups.size(); ++li) {
        auto compress = [&](const std::vector<ExprP>& es, uint64_t r) {
            Fr acc = f_zero();
            auto q = cell(r);
            for (auto& e : es) acc = f_add(f_mul(acc, theta), e->eval_with(q));
            return std::array<uint64_t, 4>{acc.l[0], acc.l[1], acc.l[2], acc.l[3]};
        };
        std::set<std::array<uint64_t, 4>> table;
        for (uint64_t r = 0; r < u; ++r) table.insert(compress(cs.lookups[li].table, r));
        for (uint64_t r = 0; r < u; ++r)
            if (!table.count(compress(cs.lookups[li].inputs, r))) failures.push_back({MockFailure::Lookup, li, r});
    }
    auto value = [&](size_t pcol, uint64_t r) {
        const Column& c = cs.permutation[pcol];
        return c.kind == Expr::Fixed ? fixed[c.index][r] : (c.kind == Expr::Advice ? advice[c.index][r] : instances[c.index][r]);
    };
    for (size_t c = 0; c < cs.permutation.size(); ++c)
        for (uint64_t r = 0; r < n; ++r) {
            const auto next = assembly.mapping[c][r];
            if (!(value(c, r) == value(next.first, next.second))) failures.push_back({MockFailure::Permutation, c, r});
        }
    return failures;
}

// ------------------------------------------------------------------------------------------------ snark-verifier protocol export
// What snark-verifier's `compile(params, vk, config)` (system/halo2.rs) produces for a halo2 verifying key, written for OUR key in the
// serde_json schema of the reference's `*.protocol` files (protocol_json.hpp reads it back): polynomial indices = preprocessed (fixed,
// then permutation commitments) | instance columns | witnesses in commitment order (advice, lookup m, permutation z, lookup phi,
// random) | quotient; the evaluations in the order create_proof writes them; the opening queries in the order the SHPLONK prover
// takes them; the quotient numerator as an expression tree folded with the last challenge.  A proof made by create_proof with
// TranscriptKind::Poseidon verifies under a verifier that is driven by this JSON alone -- tests/snark_verifier_model.py, the model
// that accepts the reference's shipped chunk and batch proofs.
inline std::string export_protocol_json(const EvaluationDomain& dom, const VerifyingKey& vk) {
    const ConstraintSystem& cs = vk.cs;
    const uint32_t bf = cs.blinding_factors();
    const uint64_t u = dom.n - bf - 1;
    const AuxLayout aux = aux_layout(cs);
    const size_t n_pre = vk.fixed_commitments.size() + vk.permutation_commitments.size(), n_inst = cs.num_instance;
    const size_t A = cs.num_advice, L = cs.lookups.size(), S = aux.n_sets;
    const size_t w0 = n_pre + n_inst, p_m = w0 + A, p_z = p_m + L, p_phi = p_z + S, p_random = p_phi + L, p_quotient = p_random + 1;
    // snark-verifier orders witnesses and challenges by phase (Polynomials::new `remapping`): the index of advice column c among
    // the witnesses is its position in phase-major order -- which is the order create_proof commits them in
    const uint32_t P = cs.num_phases();
    std::vector<size_t> advice_index(A), challenge_index(cs.challenge_phase.size()), advice_per_phase(P, 0), challenge_per_phase(P, 0);
    {
        size_t next = 0;
        for (uint32_t ph = 0; ph < P; ++ph)
            for (uint32_t c = 0; c < A; ++c)
                if (cs.phase_of_advice(c) == ph) { advice_index[c] = next++; advice_per_phase[ph]++; }
        next = 0;
        for (uint32_t ph = 0; ph < P; ++ph)
            for (size_t i = 0; i < challenge_index.size(); ++i)
                if (cs.challenge_phase[i] == ph) { challenge_index[i] = next++; challenge_per_phase[ph]++; }
    }
    const int C = (int)challenge_index.size();  // theta, beta, gamma, y follow the circuit's own challenges
    auto limbs = [](const uint64_t l[4]) {
        return "[" + std::to_string(l[0]) + ", " + std::to_string(l[1]) + ", " + std::to_string(l[2]) + ", " + std::to_string(l[3]) + "]";
    };
    auto fr = [&](const Fr& v) { return limbs(v.l); };
    auto fq = [&](const b200zk::Fq& v) {
        uint64_t l[4];
        std::memcpy(l, v.l.v, 32);
        return limbs(l);
    };
    auto poly = [](size_t idx, int32_t rot) { return "{\"Polynomial\": {\"poly\": " + std::to_string(idx) + ", \"rotation\": " + std::to_string(rot) + "}}"; };
    auto constant = [&](const Fr& v) { return "{\"Constant\": " + fr(v) + "}"; };
    auto challenge = [](int i) { return "{\"Challenge\": " + std::to_string(i) + "}"; };
    auto lagrange = [](int64_t i) { return "{\"CommonPolynomial\": {\"Lagrange\": " + std::to_string(i) + "}}"; };
    const std::string identity = "{\"CommonPolynomial\": \"Identity\"}";
    auto neg = [](const std::string& a) { return "{\"Negated\": " + a + "}"; };
    auto sum = [](const std::string& a, const std::string& b) { return "{\"Sum\": [" + a + ", " + b + "]}"; };
    auto sub = [&](const std::string& a, const std::string& b) { return sum(a, neg(b)); };
    auto mul = [](const std::string& a, const std::string& b) { return "{\"Product\": [" + a + ", " + b + "]}"; };
    const std::string theta = challenge(C), beta = challenge(C + 1), gamma = challenge(C + 2), one = constant(f_one());
    std::function<std::string(const Expr&)> expr = [&](const Expr& e) -> std::string {
        switch (e.kind) {
            case Expr::Constant: return constant(e.c);
            case Expr::Fixed: return poly(e.col, e.rot);
            case Expr::Advice: return poly(w0 + advice_index[e.col], e.rot);
            case Expr::Instance: return poly(n_pre + e.col, e.rot);
            case Expr::Challenge: return challenge((int)challenge_index[e.col]);
            case Expr::Negated: return neg(expr(*e.a));
            case Expr::Sum: return sum(expr(*e.a), expr(*e.b));
            case Expr::Product: return mul(expr(*e.a), expr(*e.b));
            default: return "{\"Scaled\": [" + expr(*e.a) + ", " + fr(e.c) + "]}";
        }
    };
    auto column = [&](const Column& c) { return c.kind == Expr::Advice ? poly(w0 + advice_index[c.index], 0) : (c.kind == Expr::Fixed ? poly(c.index, 0) : poly(n_pre + c.index, 0)); };
    const int32_t last = -(int32_t)(bf + 1);
    std::string l_blind = lagrange(-1);
    for (uint32_t i = 2; i <= bf; ++i) l_blind = sum(l_blind, lagrange(-(int64_t)i));
    const std::string l_0 = lagrange(0), l_last = lagrange(last), l_active = sub(one, sum(l_last, l_blind));
    std::vector<std::string> terms;
    for (auto& g : cs.gates) terms.push_back(expr(*g));
    if (!cs.permutation.empty()) {
        const uint32_t chunk = cs.permutation_chunk_len();
        terms.push_back(mul(l_0, sub(one, poly(p_z, 0))));
        terms.push_back(mul(l_last, sub(mul(poly(p_z + S - 1, 0), poly(p_z + S - 1, 0)), poly(p_z + S - 1, 0))));
        for (size_t sidx = 1; sidx < S; ++sidx) terms.push_back(mul(l_0, sub(poly(p_z + sidx, 0), poly(p_z + sidx - 1, last))));
        Fr dpow = f_one();
        const Fr delta = f_delta();
        for (size_t sidx = 0; sidx < S; ++sidx) {
            std::string left = poly(p_z + sidx, 1), right = poly(p_z + sidx, 0);
            for (size_t i = sidx * chunk; i < std::min(cs.permutation.size(), (sidx + 1) * (size_t)chunk); ++i) {
                const std::string v = column(cs.permutation[i]);
                left = mul(left, sum(sum(v, mul(beta, poly(vk.fixed_commitments.size() + i, 0))), gamma));
                right = mul(right, sum(sum(v, mul(mul(beta, identity), constant(dpow))), gamma));
                dpow = f_mul(dpow, delta);
            }
            terms.push_back(mul(sub(left, right), l_active));
        }
    }
    for (size_t li = 0; li < L; ++li) {
        auto compress = [&](const std::vector<ExprP>& es) {
            std::string acc = constant(f_zero());
            for (auto& e : es) acc = sum(mul(acc, theta), expr(*e));
            return acc;
        };
        const std::string fi = sum(compress(cs.lookups[li].inputs), beta), tau = sum(compress(cs.lookups[li].table), beta);
        const std::string phi = poly(p_phi + li, 0), phi_next = poly(p_phi + li, 1), m = poly(p_m + li, 0);
        terms.push_back(mul(l_0, phi));
        terms.push_back(mul(l_last, phi));
        terms.push_back(mul(sub(mul(mul(tau, fi), sub(phi_next, phi)), sub(tau, mul(m, fi))), l_active));
    }
    // evaluations (write order of create_proof) and queries (order of its SHPLONK opening claims)
    std::vector<std::pair<size_t, int32_t>> evals, queries, q_fixed, q_sigma;
    for (auto& q : cs.advice_queries) evals.push_back({w0 + advice_index[q.first], q.second});
    for (auto& q : cs.fixed_queries) { evals.push_back({q.first, q.second}); q_fixed.push_back({q.first, q.second}); }
    evals.push_back({p_random, 0});
    for (size_t i = 0; i < vk.permutation_commitments.size(); ++i) { evals.push_back({vk.fixed_commitments.size() + i, 0}); q_sigma.push_back({vk.fixed_commitments.size() + i, 0}); }
    for (auto& q : cs.advice_queries) queries.push_back({w0 + advice_index[q.first], q.second});
    for (size_t sidx = 0; sidx < S; ++sidx)
        for (int32_t rot : {0, 1, last}) {
            if (rot == last && sidx + 1 == S) continue;
            evals.push_back({p_z + sidx, rot});
            queries.push_back({p_z + sidx, rot});
        }
    for (size_t li = 0; li < L; ++li)
        for (auto pr : {std::pair<size_t, int32_t>{p_phi + li, 0}, {p_phi + li, 1}, {p_m + li, 0}}) {
            evals.push_back(pr);
            queries.push_back(pr);
        }
    queries.insert(queries.end(), q_fixed.begin(), q_fixed.end());
    queries.insert(queries.end(), q_sigma.begin(), q_sigma.end());
    queries.push_back({p_quotient, 0});
    queries.push_back({p_random, 0});
    auto list = [](const std::vector<std::pair<size_t, int32_t>>& v) {
        std::string o = "[";
        for (size_t i = 0; i < v.size(); ++i) o += std::string(i ? ", " : "") + "{\"poly\": " + std::to_string(v[i].first) + ", \"rotation\": " + std::to_string(v[i].second) + "}";
        return o + "]";
    };
    std::string numerator = "{\"DistributePowers\": [[";
    for (size_t i = 0; i < terms.size(); ++i) numerator += (i ? ", " : "") + terms[i];
    numerator += "], " + challenge(C + 3) + "]}";
    std::string pre = "[";
    size_t cnt = 0;
    for (auto* v : {&vk.fixed_commitments, &vk.permutation_commitments})
        for (auto& pt : *v) pre += std::string(cnt++ ? ", " : "") + "{\"x\": " + fq(pt.x) + ", \"y\": " + fq(pt.y) + "}";
    pre += "]";
    std::string num_witness, num_challenge;  // per phase, then [lookup m] [z, phi, random]; theta joins the last phase's challenges
    for (uint32_t ph = 0; ph < P; ++ph) {
        num_witness += std::to_string(advice_per_phase[ph]) + ", ";
        num_challenge += std::to_string(challenge_per_phase[ph] + (ph + 1 == P ? 1 : 0)) + ", ";
    }
    num_witness += std::to_string(L) + ", " + std::to_string(S + L + 1);
    num_challenge += "2, 1";
    std::string inst = "[";
    for (size_t i = 0; i < n_inst; ++i) inst += std::string(i ? ", " : "") + std::to_string(u);
    inst += "]";
    return "{\"domain\": {\"k\": " + std::to_string(dom.k) + ", \"n\": " + std::to_string(dom.n) + ", \"n_inv\": " + fr(dom.ifft_divisor) + ", \"gen\": " +
           fr(dom.omega) + ", \"gen_inv\": " + fr(dom.omega_inv) + "}, \"preprocessed\": " + pre + ", \"num_instance\": " + inst +
           ", \"num_witness\": [" + num_witness + "], \"num_challenge\": [" + num_challenge + "], \"evaluations\": " +
           list(evals) + ", \"queries\": " + list(queries) + ", \"quotient\": {\"num_chunk\": " + std::to_string(dom.quotient_poly_degree) +
           ", \"chunk_degree\": 1, \"numerator\": " + numerator + "}, \"transcript_initial_state\": " + fr(vk.transcript_repr) +
           ", \"instance_committing_key\": null, \"linearization\": null, \"accumulator_indices\": []}";
}

// ------------------------------------------------------------------------------------------------ verify_proof (host only)
struct VerifierParams {  // ParamsVerifierKZG: g2 and s_g2 (and G1's generator)
    pairing::G2Point g2, s_g2;
};

namespace hostg1 {
using b200zk::Affine;
using b200zk::XYZZ;
inline XYZZ from_point(const serde::G1Point& p) {
    Affine a;
    a.x = p.x;
    a.y = p.y;
    return b200zk::xyzz_from_affine(a);
}
inline XYZZ mul(const serde::G1Point& p, const Fr& s) {
    DFr c = to_dev(s).from_mont();
    XYZZ acc = XYZZ::identity();
    if (p.x.is_zero() && p.y.is_zero()) return acc;
    for (int limb = 7; limb >= 0; --limb)
        for (int b = 31; b >= 0; --b) {
            acc = b200zk::xyzz_dbl(acc);
            if ((c.l.v[limb] >> b) & 1) b200zk::xyzz_madd(acc, p.x, p.y);
        }
    return acc;
}
inline pairing::G1Point to_pairing_point(const XYZZ& p) {
    Affine a = b200zk::xyzz_to_affine(p);
    return {a.x, a.y};
}
}  // namespace hostg1

// plonk::verify_proof + VerifierSHPLONK + the final pairing (the "decide" of snark-verifier's KzgAs)
inline bool verify_proof(const EvaluationDomain& dom, const VerifyingKey& vk, const VerifierParams& vp, const std::vector<Poly>& instances,
                         const std::vector<uint8_t>& proof, std::string* why = nullptr,
                         TranscriptKind transcript_kind = TranscriptKind::Blake2b) {
    auto fail = [&](const char* m) { if (why) *why = m; return false; };
    try {
        const ConstraintSystem& cs = vk.cs;
        const uint64_t n = dom.n;
        const uint32_t bf = cs.blinding_factors();
        const uint64_t u = n - bf - 1;
        const AuxLayout aux = aux_layout(cs);
        Transcript tr(proof, transcript_kind);
        tr.common_scalar(vk.transcript_repr);
        if (instances.size() != cs.num_instance) return fail("wrong number of instance columns");
        for (auto& inst : instances)
            for (uint64_t r = 0; r < u; ++r) tr.common_scalar(inst[r]);
        std::vector<serde::G1Point> advice_c(cs.num_advice), m_c, z_c, phi_c, h_c;
        std::vector<Fr> challenges(cs.challenge_phase.size(), f_zero());
        for (uint32_t phase = 0; phase < cs.num_phases(); ++phase) {  // per phase: its advice commitments, then its challenges
            for (uint32_t c = 0; c < cs.num_advice; ++c)
                if (cs.phase_of_advice(c) == phase) advice_c[c] = tr.read_point();
            for (size_t i = 0; i < challenges.size(); ++i)
                if (cs.challenge_phase[i] == phase) challenges[i] = tr.squeeze_challenge();
        }
        const Fr theta = tr.squeeze_challenge();
        for (size_t i = 0; i < cs.lookups.size(); ++i) m_c.push_back(tr.read_point());
        const Fr beta = tr.squeeze_challenge(), gamma = tr.squeeze_challenge();
        for (uint32_t s = 0; s < aux.n_sets; ++s) z_c.push_back(tr.read_point());
        for (size_t i = 0; i < cs.lookups.size(); ++i) phi_c.push_back(tr.read_point());
        const serde::G1Point random_c = tr.read_point();
        const Fr y = tr.squeeze_challenge();
        for (size_t i = 0; i < dom.quotient_poly_degree; ++i) h_c.push_back(tr.read_point());
        const Fr x = tr.squeeze_challenge();
        const Fr xn = f_pow(x, n);
        std::vector<Fr> advice_e, fixed_e, sigma_e;
        for (size_t i = 0; i < cs.advice_queries.size(); ++i) advice_e.push_back(tr.read_scalar());
        for (size_t i = 0; i < cs.fixed_queries.size(); ++i) fixed_e.push_back(tr.read_scalar());
        const Fr random_eval = tr.read_scalar();
        for (size_t i = 0; i < cs.permutation.size(); ++i) sigma_e.push_back(tr.read_scalar());
        struct ZE { Fr cur, next, last; };
        std::vector<ZE> z_e(aux.n_sets);
        for (uint32_t s = 0; s < aux.n_sets; ++s) {
            z_e[s].cur = tr.read_scalar();
            z_e[s].next = tr.read_scalar();
            z_e[s].last = (s + 1 < aux.n_sets) ? tr.read_scalar() : f_zero();
        }
        struct LE { Fr phi, phi_next, m; };
        std::vector<LE> l_e(cs.lookups.size());
        for (auto& l : l_e) { l.phi = tr.read_scalar(); l.phi_next = tr.read_scalar(); l.m = tr.read_scalar(); }

        // Lagrange basis evaluations at x: l_i(x) = (omega^i / n) (x^n - 1) / (x - omega^i)
        auto lagrange_at = [&](int64_t i) {
            Fr w = i >= 0 ? f_pow(dom.omega, (uint64_t)i) : f_pow(dom.omega_inv, (uint64_t)(-i));
            return f_mul(f_mul(f_mul(w, dom.ifft_divisor), f_sub(xn, f_one())), f_inv(f_sub(x, w)));
        };
        const Fr l_0 = lagrange_at(0), l_last = lagrange_at(-(int64_t)(bf + 1));
        Fr l_blind = f_zero();
        for (uint32_t i = 1; i <= bf; ++i) l_blind = f_add(l_blind, lagrange_at(-(int64_t)i));
        const Fr l_active = f_sub(f_sub(f_one(), l_last), l_blind);
        // instance evaluations by interpolation (query_instance = false): sum_r inst[r] l_{r + rot}(x)... computed per query
        auto instance_eval = [&](uint32_t col, int32_t rot) {
            Fr acc = f_zero();
            for (uint64_t r = 0; r < u; ++r)
                if (!f_is_zero(instances[col][r])) acc = f_add(acc, f_mul(instances[col][r], lagrange_at((int64_t)r - rot)));
            return acc;
        };
        auto query = [&](int kind, uint32_t col, int32_t rot) -> Fr {
            if (kind == Expr::Challenge) return challenges[col];
            if (kind == Expr::Instance) return instance_eval(col, rot);
            auto& qs = kind == Expr::Fixed ? cs.fixed_queries : cs.advice_queries;
            auto& ev = kind == Expr::Fixed ? fixed_e : advice_e;
            for (size_t i = 0; i < qs.size(); ++i)
                if (qs[i].first == col && qs[i].second == rot) return ev[i];
            throw Panic("verifier: expression queries a cell that was not opened");
        };
        // expected h(x): gates, permutation, lookups folded with y, divided by x^n - 1
        Fr acc = f_zero();
        auto fold = [&](const Fr& v) { acc = f_add(f_mul(acc, y), v); };
        for (auto& g : cs.gates) fold(g->eval_with(query));
        if (!cs.permutation.empty()) {
            const uint32_t chunk = cs.permutation_chunk_len();
            const Fr delta = f_delta();
            fold(f_mul(l_0, f_sub(f_one(), z_e.front().cur)));
            fold(f_mul(l_last, f_sub(f_mul(z_e.back().cur, z_e.back().cur), z_e.back().cur)));
            for (uint32_t s = 1; s < aux.n_sets; ++s) fold(f_mul(l_0, f_sub(z_e[s].cur, z_e[s - 1].last)));
            Fr dpow = f_one();
            for (uint32_t s = 0; s < aux.n_sets; ++s) {
                Fr left = z_e[s].next, right = z_e[s].cur;
                size_t c0 = (size_t)s * chunk, c1 = std::min(cs.permutation.size(), c0 + chunk);
                for (size_t i = c0; i < c1; ++i) {
                    Fr v = query(cs.permutation[i].kind, cs.permutation[i].index, 0);
                    left = f_mul(left, f_add(f_add(v, f_mul(beta, sigma_e[i])), gamma));
                    right = f_mul(right, f_add(f_add(v, f_mul(f_mul(beta, x), dpow)), gamma));
                    dpow = f_mul(dpow, delta);
                }
                fold(f_mul(f_sub(left, right), l_active));
            }
        }
        for (size_t li = 0; li < cs.lookups.size(); ++li) {
            Fr in = f_zero(), tb = f_zero();
            for (auto& e : cs.lookups[li].inputs) in = f_add(f_mul(in, theta), e->eval_with(query));
            for (auto& e : cs.lookups[li].table) tb = f_add(f_mul(tb, theta), e->eval_with(query));
            const Fr fi = f_add(in, beta), tau = f_add(tb, beta);
            fold(f_mul(l_0, l_e[li].phi));
            fold(f_mul(l_last, l_e[li].phi));
            // tau * prod(f_i + beta) * (phi(omega x) - phi(x)) - (tau * sum_i prod_{j != i} - m * prod)   with one input set
            Fr lhs = f_mul(f_mul(tau, fi), f_sub(l_e[li].phi_next, l_e[li].phi));
            Fr rhs = f_sub(tau, f_mul(l_e[li].m, fi));
            fold(f_mul(f_sub(lhs, rhs), l_active));
        }
        const Fr expected_h = f_mul(acc, f_inv(f_sub(xn, f_one())));

        // the opening claims, in the prover's order; commitments by id
        std::vector<hostg1::XYZZ> commitments;
        std::vector<Query> queries;
        auto cid = [&](const hostg1::XYZZ& c) { commitments.push_back(c); return commitments.size() - 1; };
        std::vector<size_t> advice_id, fixed_id, sigma_id, z_id, phi_id, m_id;
        for (auto& c : advice_c) advice_id.push_back(cid(hostg1::from_point(c)));
        for (auto& c : z_c) z_id.push_back(cid(hostg1::from_point(c)));
        for (size_t i = 0; i < phi_c.size(); ++i) { phi_id.push_back(cid(hostg1::from_point(phi_c[i]))); m_id.push_back(cid(hostg1::from_point(m_c[i]))); }
        for (auto& c : vk.fixed_commitments) fixed_id.push_back(cid(hostg1::from_point(c)));
        for (auto& c : vk.permutation_commitments) sigma_id.push_back(cid(hostg1::from_point(c)));
        hostg1::XYZZ h_comm = hostg1::XYZZ::identity();  // sum_i x^(n i) [h_i]
        for (size_t i = h_c.size(); i-- > 0;) {
            hostg1::XYZZ t = hostg1::XYZZ::identity();
            if (!h_comm.is_identity()) t = hostg1::mul(serde::G1Point{hostg1::to_pairing_point(h_comm).x, hostg1::to_pairing_point(h_comm).y}, xn);
            b200zk::xyzz_madd(t, h_c[i].x, h_c[i].y);
            h_comm = t;
        }
        const size_t h_id = cid(h_comm), random_id = cid(hostg1::from_point(random_c));
        const Fr x_next = rotate_omega(dom, x, 1), x_last = rotate_omega(dom, x, -(int32_t)(bf + 1));
        for (size_t i = 0; i < cs.advice_queries.size(); ++i)
            queries.push_back({advice_id[cs.advice_queries[i].first], rotate_omega(dom, x, cs.advice_queries[i].second), advice_e[i]});
        for (uint32_t s = 0; s < aux.n_sets; ++s) {
            queries.push_back({z_id[s], x, z_e[s].cur});
            queries.push_back({z_id[s], x_next, z_e[s].next});
            if (s + 1 < aux.n_sets) queries.push_back({z_id[s], x_last, z_e[s].last});
        }
        for (size_t i = 0; i < l_e.size(); ++i) {
            queries.push_back({phi_id[i], x, l_e[i].phi});
            queries.push_back({phi_id[i], x_next, l_e[i].phi_next});
            queries.push_back({m_id[i], x, l_e[i].m});
        }
        for (size_t i = 0; i < cs.fixed_queries.size(); ++i)
            queries.push_back({fixed_id[cs.fixed_queries[i].first], rotate_omega(dom, x, cs.fixed_queries[i].second), fixed_e[i]});
        for (size_t i = 0; i < sigma_id.size(); ++i) queries.push_back({sigma_id[i], x, sigma_e[i]});
        queries.push_back({h_id, x, expected_h});
        queries.push_back({random_id, x, random_eval});

        // VerifierSHPLONK::verify_proof
        const Fr sy = tr.squeeze_challenge(), sv = tr.squeeze_challenge();
        const serde::G1Point h1 = tr.read_point();
        const Fr su = tr.squeeze_challenge();
        const serde::G1Point h2 = tr.read_point();
        if (!tr.exhausted()) return fail("trailing bytes after the proof");
        RotationSets rs = build_rotation_sets(queries);
        Fr zt = f_one();
        for (auto& p : rs.super_points) zt = f_mul(zt, f_sub(su, p));
        std::vector<Fr> z_diff(rs.sets.size());
        for (size_t i = 0; i < rs.sets.size(); ++i) {
            Fr zs = f_one();
            for (auto& p : rs.sets[i].points) zs = f_mul(zs, f_sub(su, p));
            z_diff[i] = f_mul(zt, f_inv(zs));
        }
        const Fr z0_inv = f_inv(z_diff[0]);
        std::vector<Fr> vpow(rs.sets.size());
        Fr vacc = f_one();
        for (size_t i = 0; i < rs.sets.size(); ++i) { vpow[i] = vacc; vacc = f_mul(vacc, sv); }  // gamma.powers(sets.len()) of snark-verifier's Bdfg21
        hostg1::XYZZ E = hostg1::XYZZ::identity();
        Fr r_total = f_zero();
        for (size_t i = 0; i < rs.sets.size(); ++i) {
            const Fr w = f_mul(f_mul(vpow[i], z_diff[i]), z0_inv);
            std::vector<Fr> ypow(rs.sets[i].polys.size());
            Fr yp = f_one();
            for (size_t j = 0; j < ypow.size(); ++j) { ypow[j] = yp; yp = f_mul(yp, sy); }  // mu.powers(..)
            for (size_t j = 0; j < rs.sets[i].polys.size(); ++j) {
                Poly r = lagrange_interpolate(rs.sets[i].points, rs.sets[i].evals[j]);
                const Fr s = f_mul(w, ypow[j]);
                pairing::G1Point cp = hostg1::to_pairing_point(commitments[rs.sets[i].polys[j]]);
                hostg1::XYZZ t = hostg1::mul(serde::G1Point{cp.x, cp.y}, s);
                b200zk::xyzz_add(E, t);
                r_total = f_add(r_total, f_mul(s, eval_small(r, su)));
            }
        }
        // E = sum s_ij [P_ij] - r_total G - (Z_T(u) / z_diff_0) [h1] + u [h2];   check e(E, g2) = e(h2, s_g2)
        serde::G1Point gen;
        gen.x = b200zk::Fq::one();
        gen.y = b200zk::Fq::one().dbl();
        hostg1::XYZZ t = hostg1::mul(gen, f_neg(r_total));
        b200zk::xyzz_add(E, t);
        t = hostg1::mul(h1, f_neg(f_mul(zt, z0_inv)));
        b200zk::xyzz_add(E, t);
        t = hostg1::mul(h2, su);
        b200zk::xyzz_add(E, t);
        pairing::G1Point lhs = hostg1::to_pairing_point(E);
        pairing::G1Point neg_h2{h2.x, h2.y.neg()};
        if (!pairing::pairing_check({{lhs, vp.g2}, {neg_h2, vp.s_g2}})) return fail("pairing check failed");
        return true;
    } catch (const Panic& e) {
        if (why) *why = e.what();
        return false;
    }
}

}  // namespace plonk
}  // namespace halo2_b200
