// halo2_b200.hpp — C++ host-side mirror of the halo2_proofs functions that libb200zk replaces.
//
// The reference's host language is Rust (no toolchain in this image), so the host layer above the C ABI
// (include/b200zk.h) is provided in C++ with the SAME names, argument meaning and failure behaviour as
// halo2_proofs 1.1.0 (scroll-tech/halo2 @ e5ddf67, pin /root/reference/Cargo.lock:1886-1888):
//
//   halo2_b200::arithmetic::best_multiexp / best_fft / eval_polynomial / kate_division   (src/arithmetic.rs)
//   halo2_b200::EvaluationDomain::{new_, lagrange_to_coeff, coeff_to_extended, extended_to_coeff}  (src/poly/domain.rs),
//     plus coeff_to_extended_part / extended_parts_to_coeff: the extended coset as J parts of n points
//   halo2_b200::ParamsKZG::{setup, read_custom, write_custom, commit, commit_lagrange, downsize-less accessors}
//                                                                                    (src/poly/kzg/commitment.rs)
// A Rust panic (assert_eq!, unwrap) is mirrored by throwing halo2_b200::Panic.  Types are layout-identical to
// halo2curves::bn256::{Fr, G1Affine, G1} (raw Montgomery limbs).  Header-only; link with -lb200zk.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../include/b200zk.h"
#include "csrc/ff.cuh"  // host emulation of the field layer for the (tiny) domain-constant computations

namespace halo2_b200 {

struct Panic : std::runtime_error {
    using std::runtime_error::runtime_error;
};

struct Fr {
    uint64_t l[4];
    bool operator==(const Fr& o) const { return std::memcmp(l, o.l, 32) == 0; }
};
struct Fq {
    uint64_t l[4];
};
struct G1Affine {
    Fq x, y;  // identity = (0, 0)
};
struct G1 {
    Fq x, y, z;  // Jacobian, identity z = 0
    bool is_identity() const { return (z.l[0] | z.l[1] | z.l[2] | z.l[3]) == 0; }
};
static_assert(sizeof(Fr) == 32 && sizeof(G1Affine) == 64 && sizeof(G1) == 96, "ABI layout");

namespace detail {
using DFr = b200zk::Fr;
inline DFr to_dev(const Fr& a) {
    DFr r;
    std::memcpy(r.l.v, a.l, 32);
    return r;
}
inline Fr from_dev(const DFr& a) {
    Fr r;
    std::memcpy(r.l, a.l.v, 32);
    return r;
}
inline DFr from_u64(uint64_t v) {
    DFr t = DFr::zero();
    t.l.v[0] = (uint32_t)v;
    t.l.v[1] = (uint32_t)(v >> 32);
    return t.to_mont();
}
inline DFr root_of_unity() {  // halo2curves Fr::ROOT_OF_UNITY (Montgomery limbs)
    DFr r;
    const uint32_t v[8] = {0xb639feb8u, 0x9632c7c5u, 0x0d0ff299u, 0x985ce340u, 0x01b0ecd8u, 0xb2dd8800u, 0x6d98ce29u, 0x1d69070du};
    for (int i = 0; i < 8; ++i) r.l.v[i] = v[i];
    return r;
}
inline DFr zeta() {  // halo2curves Fr::ZETA
    DFr z;
    const uint32_t v[8] = {0x55fcd653u, 0x0363f299u, 0x5fc1e200u, 0x73e7950bu, 0x576d9d24u, 0xc5fce83eu, 0xa1c3a4d4u, 0x059c805du};
    for (int i = 0; i < 8; ++i) z.l.v[i] = v[i];
    return z;
}
}  // namespace detail

// One context per process per GPU (B200ZK_DEVICE selects the ordinal); created on first use.
class Backend {
  public:
    static Backend& get() {
        static Backend b;
        return b;
    }
    b200zk_ctx* ctx() const { return ctx_; }
    void check(int32_t rc, const char* what) const {
        if (rc != B200ZK_OK) throw Panic(std::string(what) + ": b200zk error " + std::to_string(rc) + ": " + b200zk_last_error(ctx_));
    }

  private:
    Backend() {
        int dev = 0;
        if (const char* e = std::getenv("B200ZK_DEVICE")) dev = std::atoi(e);
        if (b200zk_ctx_create(&dev, 1, &ctx_) != B200ZK_OK)
            throw Panic("b200zk_ctx_create failed: no CUDA device (there is no CPU fallback)");
    }
    ~Backend() {
        if (ctx_) b200zk_ctx_destroy(ctx_);
    }
    b200zk_ctx* ctx_ = nullptr;
};

namespace arithmetic {
// pub fn best_multiexp<C: CurveAffine>(coeffs: &[C::Scalar], bases: &[C]) -> C::Curve
inline G1 best_multiexp(const std::vector<Fr>& coeffs, const std::vector<G1Affine>& bases) {
    if (coeffs.size() != bases.size()) throw Panic("assertion failed: `(left == right)` coeffs.len() == bases.len()");
    G1 out;
    auto& b = Backend::get();
    b.check(b200zk_msm_g1_bases(b.ctx(), bases.data(), coeffs.data(), coeffs.size(), &out), "best_multiexp");
    return out;
}
// pub fn best_fft<Scalar, G>(a: &mut [G], omega: Scalar, log_n: u32)      (G = Fr)
inline void best_fft(std::vector<Fr>& a, const Fr& omega, uint32_t log_n) {
    if (a.size() != (size_t(1) << log_n)) throw Panic("assertion failed: `(left == right)` a.len() == 1 << log_n");
    auto& b = Backend::get();
    b.check(b200zk_ntt_fr(b.ctx(), a.data(), log_n, &omega, 0, B200ZK_COSET_NONE), "best_fft");
}
inline Fr eval_polynomial(const std::vector<Fr>& poly, const Fr& point) {
    Fr out;
    auto& b = Backend::get();
    b.check(b200zk_eval_poly(b.ctx(), poly.data(), poly.size(), &point, &out), "eval_polynomial");
    return out;
}
inline std::vector<Fr> kate_division(const std::vector<Fr>& a, const Fr& bpt) {
    if (a.empty()) throw Panic("attempt to subtract with overflow (a.len() - 1)");
    std::vector<Fr> q(a.size() - 1);
    auto& b = Backend::get();
    b.check(b200zk_kate_division(b.ctx(), q.data(), a.data(), a.size(), &bpt), "kate_division");
    return q;
}
}  // namespace arithmetic

// halo2_proofs::poly::EvaluationDomain<Fr>
class EvaluationDomain {
  public:
    uint32_t k, extended_k;
    uint64_t n, quotient_poly_degree;
    Fr omega, omega_inv, extended_omega, extended_omega_inv, g_coset, g_coset_inv, ifft_divisor, extended_ifft_divisor;

    // EvaluationDomain::new(j, k)
    static EvaluationDomain new_(uint32_t j, uint32_t k) {
        using detail::DFr;
        EvaluationDomain d;
        d.quotient_poly_degree = (uint64_t)j - 1;
        d.n = 1ull << k;
        d.k = k;
        uint32_t ek = k;
        while ((1ull << ek) < d.n * d.quotient_poly_degree) ek++;
        if (ek > 28) throw Panic("assertion failed: extended_k <= Fr::S");
        d.extended_k = ek;
        DFr eo = detail::root_of_unity();
        for (uint32_t i = ek; i < 28; ++i) eo = eo.sqr();
        DFr om = eo;
        for (uint32_t i = k; i < ek; ++i) om = om.sqr();
        d.extended_omega = detail::from_dev(eo);
        d.omega = detail::from_dev(om);
        d.extended_omega_inv = detail::from_dev(eo.inv());
        d.omega_inv = detail::from_dev(om.inv());
        d.g_coset = detail::from_dev(detail::zeta());
        d.g_coset_inv = detail::from_dev(detail::zeta().sqr());
        d.ifft_divisor = detail::from_dev(detail::from_u64(1ull << k).inv());
        d.extended_ifft_divisor = detail::from_dev(detail::from_u64(1ull << ek).inv());
        return d;
    }
    // consumes and returns the polynomial like the Rust methods (moved in, moved out)
    std::vector<Fr> lagrange_to_coeff(std::vector<Fr> a) const {
        if (a.size() != n) throw Panic("assertion failed: a.values.len() == 1 << self.k");
        auto& b = Backend::get();
        b.check(b200zk_ntt_fr(b.ctx(), a.data(), k, &omega_inv, 1, B200ZK_COSET_NONE), "lagrange_to_coeff");
        return a;
    }
    std::vector<Fr> coeff_to_extended(const std::vector<Fr>& a) const {
        if (a.size() != n) throw Panic("assertion failed: a.values.len() == 1 << self.k");
        std::vector<Fr> out(size_t(1) << extended_k);
        auto& b = Backend::get();
        b.check(b200zk_ntt_fr_ext(b.ctx(), a.data(), k, out.data(), extended_k, &extended_omega, 0, B200ZK_COSET_PRE), "coeff_to_extended");
        return out;
    }
    std::vector<Fr> extended_to_coeff(std::vector<Fr> a) const {
        if (a.size() != (size_t(1) << extended_k)) throw Panic("assertion failed: a.values.len() == self.extended_len()");
        auto& b = Backend::get();
        b.check(b200zk_ntt_fr(b.ctx(), a.data(), extended_k, &extended_omega_inv, 1, B200ZK_COSET_POST), "extended_to_coeff");
        a.resize((size_t)(n * quotient_poly_degree));  // truncate to the quotient degree
        return a;
    }
    // The extended coset as J = 2^(extended_k - k) parts of n points, part r = zeta * extended_omega^r * <omega>:
    // coeff_to_extended(a)[part + J*i] for i < n
    std::vector<Fr> coeff_to_extended_part(const std::vector<Fr>& a, uint32_t part) const {
        if (a.size() != n) throw Panic("assertion failed: a.values.len() == 1 << self.k");
        std::vector<Fr> out(n);
        auto& b = Backend::get();
        void* dev = nullptr;
        b.check(b200zk_buf_alloc(b.ctx(), 32 * n, &dev), "coeff_to_extended_part");
        const void* in = a.data();
        int32_t rc = b200zk_coeff_to_extended_parts(b.ctx(), &in, 1, k, extended_k, part, &dev);
        if (rc == B200ZK_OK) rc = b200zk_buf_download(b.ctx(), out.data(), dev, 32 * n);
        b200zk_buf_free(b.ctx(), dev);
        b.check(rc, "coeff_to_extended_part");
        return out;
    }
    // extended_to_coeff (after divide_by_vanishing_poly when asked) of the extended coset given part-major: parts[r * n + i] is
    // row r + J*i.  Returns the n * quotient_poly_degree coefficients, as extended_to_coeff does.
    std::vector<Fr> extended_parts_to_coeff(const std::vector<Fr>& parts, bool divide_by_vanishing) const {
        if (parts.size() != (size_t(1) << extended_k)) throw Panic("assertion failed: a.values.len() == self.extended_len()");
        std::vector<Fr> out((size_t)(n * quotient_poly_degree));
        auto& b = Backend::get();
        void* dev = nullptr;
        b.check(b200zk_buf_alloc(b.ctx(), 32 * parts.size(), &dev), "extended_parts_to_coeff");
        int32_t rc = b200zk_buf_upload(b.ctx(), dev, parts.data(), 32 * parts.size());
        if (rc == B200ZK_OK)
            rc = b200zk_extended_parts_to_coeff(b.ctx(), dev, k, extended_k, (uint32_t)quotient_poly_degree, divide_by_vanishing ? 1 : 0, dev);
        if (rc == B200ZK_OK) rc = b200zk_buf_download(b.ctx(), out.data(), dev, 32 * out.size());
        b200zk_buf_free(b.ctx(), dev);
        b.check(rc, "extended_parts_to_coeff");
        return out;
    }
};

// halo2_proofs::poly::kzg::commitment::ParamsKZG<Bn256>
class ParamsKZG {
  public:
    uint32_t k = 0;
    uint64_t n = 0;
    std::vector<G1Affine> g, g_lagrange;
    uint8_t g2[128] = {0}, s_g2[128] = {0};  // G2Affine RawBytes, carried opaquely (verification stays on the host)

    ParamsKZG() = default;
    ParamsKZG(const ParamsKZG&) = delete;
    ParamsKZG& operator=(const ParamsKZG&) = delete;
    ~ParamsKZG() { release(); }

    // ParamsKZG::setup(k, rng) with a caller-provided s ("unsafe" test SRS): g[i] = s^i G; g_lagrange[i] = L_i(s) G
    static void setup(ParamsKZG& p, uint32_t k, const Fr& s) {
        using detail::DFr;
        p.release();
        p.k = k;
        p.n = 1ull << k;
        std::vector<Fr> sc(p.n);
        DFr ds = detail::to_dev(s), cur = DFr::one();
        for (uint64_t i = 0; i < p.n; ++i) {
            sc[i] = detail::from_dev(cur);
            cur = cur * ds;
        }
        auto& b = Backend::get();
        p.g.resize(p.n);
        b.check(b200zk_g1_generator_mul_batch(b.ctx(), sc.data(), p.n, p.g.data()), "setup(g)");
        DFr root = detail::root_of_unity();
        for (uint32_t i = k; i < 28; ++i) root = root.sqr();
        DFr mult = (cur - DFr::one()) * detail::from_u64(p.n).inv();  // (s^n - 1) / n
        DFr rp = DFr::one();
        for (uint64_t i = 0; i < p.n; ++i) {
            sc[i] = detail::from_dev(mult * rp * (ds - rp).inv());
            rp = rp * root;
        }
        p.g_lagrange.resize(p.n);
        b.check(b200zk_g1_generator_mul_batch(b.ctx(), sc.data(), p.n, p.g_lagrange.data()), "setup(g_lagrange)");
    }

    // SerdeFormat::RawBytes: k u32 LE | n x G1 (64 B) g | n x G1 g_lagrange | G2 g2 (128 B) | G2 s_g2 (128 B)
    void write_custom(const std::string& path) const {
        FILE* f = std::fopen(path.c_str(), "wb");
        if (!f) throw Panic("write_custom: cannot open " + path);
        bool ok = std::fwrite(&k, 4, 1, f) == 1 && std::fwrite(g.data(), 64, n, f) == n && std::fwrite(g_lagrange.data(), 64, n, f) == n &&
                  std::fwrite(g2, 128, 1, f) == 1 && std::fwrite(s_g2, 128, 1, f) == 1;
        std::fclose(f);
        if (!ok) throw Panic("write_custom: short write");
    }
    static void read_custom(ParamsKZG& p, const std::string& path) {
        p.release();
        FILE* f = std::fopen(path.c_str(), "rb");
        if (!f) throw Panic("read_custom: cannot open " + path);
        uint32_t k = 0;
        bool ok = std::fread(&k, 4, 1, f) == 1 && k <= 28;
        if (ok) {
            p.k = k;
            p.n = 1ull << k;
            p.g.resize(p.n);
            p.g_lagrange.resize(p.n);
            ok = std::fread(p.g.data(), 64, p.n, f) == p.n && std::fread(p.g_lagrange.data(), 64, p.n, f) == p.n &&
                 std::fread(p.g2, 128, 1, f) == 1 && std::fread(p.s_g2, 128, 1, f) == 1;
        }
        std::fclose(f);
        if (!ok) throw Panic("read_custom: malformed params file " + path);
    }

    // ParamsProver::commit(poly, Blind): best_multiexp(poly, g[..poly.len()])   (blind ignored for KZG)
    G1 commit(const std::vector<Fr>& poly) { return msm(dev_g_, g, B200ZK_SRS_G, poly); }
    // Params::commit_lagrange(poly, Blind)
    G1 commit_lagrange(const std::vector<Fr>& poly) { return msm(dev_gl_, g_lagrange, B200ZK_SRS_G_LAGRANGE, poly); }

    // Params::downsize(k): truncate g and rebuild g_lagrange with the G1 FFT on the device
    // (reference call site /root/reference/integration/tests/integration.rs:17-18)
    void downsize(uint32_t new_k) {
        if (new_k > k) throw Panic("assertion failed: k <= self.k");
        release();
        k = new_k;
        n = 1ull << new_k;
        g.resize(n);
        g_lagrange.resize(n);
        auto& b = Backend::get();
        b.check(b200zk_g_to_lagrange(b.ctx(), g.data(), new_k, g_lagrange.data()), "downsize");
    }

    // device handles (registered lazily): for b200zk_commit_columns and other batched entry points
    b200zk_srs* lagrange_handle() { return handle(dev_gl_, g_lagrange, B200ZK_SRS_G_LAGRANGE); }
    b200zk_srs* monomial_handle() { return handle(dev_g_, g, B200ZK_SRS_G); }

    void release() {
        auto* c = Backend::get().ctx();
        if (dev_g_) b200zk_srs_release(c, dev_g_);
        if (dev_gl_) b200zk_srs_release(c, dev_gl_);
        dev_g_ = dev_gl_ = nullptr;
    }

  private:
    b200zk_srs *dev_g_ = nullptr, *dev_gl_ = nullptr;
    b200zk_srs* handle(b200zk_srs*& h, const std::vector<G1Affine>& bases, uint32_t tag) {
        auto& b = Backend::get();
        if (!h) b.check(b200zk_srs_register(b.ctx(), bases.data(), bases.size(), tag, &h), "srs_register");  // once, lazily
        return h;
    }
    G1 msm(b200zk_srs*& h, const std::vector<G1Affine>& bases, uint32_t tag, const std::vector<Fr>& poly) {
        if (poly.size() > bases.size()) throw Panic("assertion failed: `(left == right)` coeffs.len() == bases.len()");
        auto& b = Backend::get();
        handle(h, bases, tag);
        G1 out;
        b.check(b200zk_msm_g1(b.ctx(), h, poly.data(), poly.size(), &out), "commit");
        return out;
    }
};

// The per-column work of one create_proof phase for a batch of Lagrange-form columns held on the host:
// commitments[j] = commit_lagrange(cols[j]); with mode >= 1 the coefficient form (and with mode 2 the extended coset
// evaluations) are produced on the device into coeff_dev[j] / ext_dev[j] (b200zk_buf_alloc handles; may be null).
inline std::vector<G1> commit_columns(ParamsKZG& params, const EvaluationDomain& dom, const std::vector<const Fr*>& cols, int mode,
                                      void* const* coeff_dev = nullptr, void* const* ext_dev = nullptr) {
    std::vector<G1> out(cols.size());
    auto& b = Backend::get();
    std::vector<const void*> ptrs(cols.begin(), cols.end());
    b.check(b200zk_commit_columns(b.ctx(), params.lagrange_handle(), ptrs.data(), (uint32_t)ptrs.size(), dom.k, &dom.omega_inv,
                                  &dom.extended_omega, dom.extended_k, out.data(), coeff_dev, ext_dev, mode),
            "commit_columns");
    return out;
}

// A column (Polynomial<Fr, _>) resident on the device between calls: b200zk_buf_alloc / upload / download.
class DeviceColumn {
  public:
    DeviceColumn() = default;
    explicit DeviceColumn(size_t len) : len_(len) {
        auto& b = Backend::get();
        b.check(b200zk_buf_alloc(b.ctx(), 32 * (uint64_t)len, &dev_), "DeviceColumn::alloc");
    }
    explicit DeviceColumn(const std::vector<Fr>& host) : DeviceColumn(host.size()) { upload(host); }
    DeviceColumn(const DeviceColumn&) = delete;
    DeviceColumn& operator=(const DeviceColumn&) = delete;
    DeviceColumn(DeviceColumn&& o) noexcept : dev_(o.dev_), len_(o.len_) { o.dev_ = nullptr; }
    ~DeviceColumn() {
        if (dev_) b200zk_buf_free(Backend::get().ctx(), dev_);
    }
    void upload(const std::vector<Fr>& host) {
        if (host.size() != len_) throw Panic("DeviceColumn::upload: length mismatch");
        auto& b = Backend::get();
        b.check(b200zk_buf_upload(b.ctx(), dev_, host.data(), 32 * (uint64_t)len_), "DeviceColumn::upload");
    }
    std::vector<Fr> to_host() const {
        std::vector<Fr> out(len_);
        auto& b = Backend::get();
        b.check(b200zk_buf_download(b.ctx(), out.data(), dev_, 32 * (uint64_t)len_), "DeviceColumn::download");
        return out;
    }
    void* ptr() const { return dev_; }
    size_t len() const { return len_; }

  private:
    void* dev_ = nullptr;
    size_t len_ = 0;
};

// halo2_proofs::plonk -- the prover steps between the transforms, on device-resident columns (SURVEY.md §8(f).2)
namespace plonk {

// plonk::evaluation::ValueSource / Calculation / GraphEvaluator (evaluation.rs): same construction interface --
// add_constant / add_rotation / add_calculation return the index a later ValueSource names.
struct ValueSource {
    uint32_t kind, index, rotation;
    static ValueSource Constant(uint32_t i) { return {B200ZK_SRC_CONSTANT, i, 0}; }
    static ValueSource Intermediate(uint32_t i) { return {B200ZK_SRC_INTERMEDIATE, i, 0}; }
    static ValueSource Fixed(uint32_t col, uint32_t rot) { return {B200ZK_SRC_FIXED, col, rot}; }
    static ValueSource Advice(uint32_t col, uint32_t rot) { return {B200ZK_SRC_ADVICE, col, rot}; }
    static ValueSource Instance(uint32_t col, uint32_t rot) { return {B200ZK_SRC_INSTANCE, col, rot}; }
    static ValueSource Challenge(uint32_t i) { return {B200ZK_SRC_CHALLENGE, i, 0}; }
    static ValueSource Beta() { return {B200ZK_SRC_BETA, 0, 0}; }
    static ValueSource Gamma() { return {B200ZK_SRC_GAMMA, 0, 0}; }
    static ValueSource Theta() { return {B200ZK_SRC_THETA, 0, 0}; }
    static ValueSource Y() { return {B200ZK_SRC_Y, 0, 0}; }
    static ValueSource PreviousValue() { return {B200ZK_SRC_PREVIOUS_VALUE, 0, 0}; }
    static ValueSource ExtendedX() { return {B200ZK_SRC_EXTENDED_X, 0, 0}; }  // not upstream: the coset point of the row
};

class GraphEvaluator {
  public:
    GraphEvaluator() {  // upstream seeds the constants with 0, 1, 2
        add_constant(detail::from_dev(detail::DFr::zero()));
        add_constant(detail::from_dev(detail::DFr::one()));
        add_constant(detail::from_dev(detail::DFr::one() + detail::DFr::one()));
    }
    GraphEvaluator(const GraphEvaluator&) = delete;
    GraphEvaluator& operator=(const GraphEvaluator&) = delete;
    ~GraphEvaluator() { release(); }

    uint32_t add_rotation(int32_t rotation) {
        for (size_t i = 0; i < rotations_.size(); ++i)
            if (rotations_[i] == rotation) return (uint32_t)i;
        rotations_.push_back(rotation);
        dirty();
        return (uint32_t)rotations_.size() - 1;
    }
    ValueSource add_constant(const Fr& c) {
        for (size_t i = 0; i < constants_.size(); ++i)
            if (constants_[i] == c) return ValueSource::Constant((uint32_t)i);
        constants_.push_back(c);
        dirty();
        return ValueSource::Constant((uint32_t)constants_.size() - 1);
    }
    ValueSource add(uint32_t op, ValueSource a, ValueSource b = ValueSource::Constant(0)) {
        calcs_.push_back(b200zk_calculation{op, {a.kind, a.index, a.rotation}, {b.kind, b.index, b.rotation}, 0, 0});
        dirty();
        return ValueSource::Intermediate((uint32_t)calcs_.size() - 1);
    }
    // Calculation::Horner(start_value, parts, factor)
    ValueSource add_horner(ValueSource start, const std::vector<ValueSource>& parts, ValueSource factor) {
        b200zk_calculation c{B200ZK_CALC_HORNER, {start.kind, start.index, start.rotation}, {factor.kind, factor.index, factor.rotation},
                             (uint32_t)parts_.size(), (uint32_t)parts.size()};
        for (const auto& p : parts) parts_.push_back(b200zk_value_source{p.kind, p.index, p.rotation});
        calcs_.push_back(c);
        dirty();
        return ValueSource::Intermediate((uint32_t)calcs_.size() - 1);
    }
    size_t num_calculations() const { return calcs_.size(); }
    // the program in the ABI's form (what b200zk_graph_create takes): for callers that run it through another backend
    const std::vector<b200zk_calculation>& calculations() const { return calcs_; }
    const std::vector<b200zk_value_source>& horner_parts() const { return parts_; }
    const std::vector<Fr>& constants() const { return constants_; }
    const std::vector<int32_t>& rotations() const { return rotations_; }
    // validation + lowering without a device (b200zk_graph_check): {instructions, on-chip slots}; throws Panic with the reason
    std::pair<uint32_t, uint32_t> check() const {
        uint32_t ni = 0, ns = 0;
        char msg[256];
        int32_t rc = b200zk_graph_check(calcs_.data(), (uint32_t)calcs_.size(), parts_.data(), (uint32_t)parts_.size(),
                                        (uint32_t)constants_.size(), (uint32_t)rotations_.size(), &ni, &ns, msg, sizeof msg);
        if (rc != B200ZK_OK) throw Panic(std::string("GraphEvaluator::check: ") + msg);
        return {ni, ns};
    }

    // GraphEvaluator::evaluate for every row of the extended domain: values[row] = f(previous = values[row], row)
    void evaluate(DeviceColumn& values, const EvaluationDomain& dom, const std::vector<const DeviceColumn*>& fixed,
                  const std::vector<const DeviceColumn*>& advice, const std::vector<const DeviceColumn*>& instance,
                  const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma, const Fr& theta, const Fr& y) {
        auto& b = Backend::get();
        if (values.len() != (size_t(1) << dom.extended_k)) throw Panic("GraphEvaluator::evaluate: values must cover the extended domain");
        if (!graph_)
            b.check(b200zk_graph_create(b.ctx(), calcs_.data(), (uint32_t)calcs_.size(), parts_.data(), (uint32_t)parts_.size(),
                                        constants_.data(), (uint32_t)constants_.size(), rotations_.data(), (uint32_t)rotations_.size(),
                                        &graph_),
                    "GraphEvaluator::compile");
        auto table = [](const std::vector<const DeviceColumn*>& v) {
            std::vector<const void*> t;
            for (auto* c : v) t.push_back(c->ptr());
            return t;
        };
        auto tf = table(fixed), ta = table(advice), ti = table(instance);
        const int32_t rot_scale = 1 << (dom.extended_k - dom.k);
        b.check(b200zk_graph_evaluate(b.ctx(), graph_, tf.data(), (uint32_t)tf.size(), ta.data(), (uint32_t)ta.size(), ti.data(),
                                      (uint32_t)ti.size(), challenges.data(), (uint32_t)challenges.size(), &beta, &gamma, &theta, &y,
                                      &dom.extended_omega, values.ptr(), dom.extended_k, rot_scale),
                "GraphEvaluator::evaluate");
    }
    // the same on the n rows of one part of the extended coset (columns hold that part's values, rotations wrap within it)
    void evaluate_part(DeviceColumn& values, const EvaluationDomain& dom, uint32_t part, const std::vector<const DeviceColumn*>& fixed,
                       const std::vector<const DeviceColumn*>& advice, const std::vector<const DeviceColumn*>& instance,
                       const std::vector<Fr>& challenges, const Fr& beta, const Fr& gamma, const Fr& theta, const Fr& y) {
        auto& b = Backend::get();
        if (values.len() != dom.n) throw Panic("GraphEvaluator::evaluate_part: values must cover one part (n rows)");
        if (!graph_)
            b.check(b200zk_graph_create(b.ctx(), calcs_.data(), (uint32_t)calcs_.size(), parts_.data(), (uint32_t)parts_.size(),
                                        constants_.data(), (uint32_t)constants_.size(), rotations_.data(), (uint32_t)rotations_.size(),
                                        &graph_),
                    "GraphEvaluator::compile");
        auto table = [](const std::vector<const DeviceColumn*>& v) {
            std::vector<const void*> t;
            for (auto* c : v) t.push_back(c->ptr());
            return t;
        };
        auto tf = table(fixed), ta = table(advice), ti = table(instance);
        b.check(b200zk_graph_evaluate_part(b.ctx(), graph_, tf.data(), (uint32_t)tf.size(), ta.data(), (uint32_t)ta.size(), ti.data(),
                                           (uint32_t)ti.size(), challenges.data(), (uint32_t)challenges.size(), &beta, &gamma, &theta, &y,
                                           dom.k, dom.extended_k, part, values.ptr()),
                "GraphEvaluator::evaluate_part");
    }
    void release() {
        if (graph_) b200zk_graph_destroy(Backend::get().ctx(), graph_);
        graph_ = nullptr;
    }

  private:
    void dirty() { release(); }
    std::vector<b200zk_calculation> calcs_;
    std::vector<b200zk_value_source> parts_;
    std::vector<Fr> constants_;
    std::vector<int32_t> rotations_;
    b200zk_graph* graph_ = nullptr;
};

// evaluate_h's `// Permutations` section as a program appended to `ev` (upstream spells it out as a Rust loop; here the
// same kernel serves gates, permutation and lookups).  z[s]: the permutation product cosets (advice-like sources at
// rotation index 0 are re-issued at the next / last rotations); values[j] / sigma[j]: the permuted columns and their
// sigma cosets; l0, l_last, l_active_row: the Lagrange cosets.  Folds into PreviousValue with y in upstream's order.
inline ValueSource permutation_constraints(GraphEvaluator& ev, const std::vector<ValueSource>& z, uint32_t chunk_len,
                                           const std::vector<ValueSource>& values, const std::vector<ValueSource>& sigma,
                                           ValueSource l0, ValueSource l_last, ValueSource l_active_row, int32_t last_rotation,
                                           const Fr& delta) {
    if (z.empty() || values.size() != sigma.size()) throw Panic("permutation_constraints: bad shape");
    const uint32_t r_next = ev.add_rotation(1), r_last = ev.add_rotation(last_rotation);
    auto at = [](ValueSource s, uint32_t rot) { s.rotation = rot; return s; };
    const ValueSource one = ev.add_constant(detail::from_dev(detail::DFr::one()));
    std::vector<ValueSource> terms;
    terms.push_back(ev.add(B200ZK_CALC_MUL, ev.add(B200ZK_CALC_SUB, one, z.front()), l0));
    ValueSource zl2 = ev.add(B200ZK_CALC_SQUARE, z.back());
    terms.push_back(ev.add(B200ZK_CALC_MUL, ev.add(B200ZK_CALC_SUB, zl2, z.back()), l_last));
    for (size_t s = 1; s < z.size(); ++s)
        terms.push_back(ev.add(B200ZK_CALC_MUL, ev.add(B200ZK_CALC_SUB, z[s], at(z[s - 1], r_last)), l0));
    const ValueSource bx = ev.add(B200ZK_CALC_MUL, ValueSource::Beta(), ValueSource::ExtendedX());  // beta * zeta * w_ext^idx
    detail::DFr dpow = detail::DFr::one();
    for (size_t s = 0; s < z.size(); ++s) {
        size_t c0 = s * chunk_len, c1 = std::min(values.size(), c0 + chunk_len);
        ValueSource left = at(z[s], r_next), right = z[s];
        for (size_t j = c0; j < c1; ++j) {
            ValueSource u = ev.add(B200ZK_CALC_MUL, ValueSource::Beta(), sigma[j]);
            u = ev.add(B200ZK_CALC_ADD, u, values[j]);
            u = ev.add(B200ZK_CALC_ADD, u, ValueSource::Gamma());
            left = ev.add(B200ZK_CALC_MUL, left, u);
        }
        for (size_t j = c0; j < c1; ++j) {
            ValueSource d = (j == 0) ? bx : ev.add(B200ZK_CALC_MUL, bx, ev.add_constant(detail::from_dev(dpow)));
            ValueSource u = ev.add(B200ZK_CALC_ADD, values[j], d);
            u = ev.add(B200ZK_CALC_ADD, u, ValueSource::Gamma());
            right = ev.add(B200ZK_CALC_MUL, right, u);
            dpow = dpow * detail::to_dev(delta);
        }
        terms.push_back(ev.add(B200ZK_CALC_MUL, ev.add(B200ZK_CALC_SUB, left, right), l_active_row));
    }
    return ev.add_horner(ValueSource::PreviousValue(), terms, ValueSource::Y());
}

// evaluate_h's section for one log-derivative lookup: inputs[i] = compressed input expressions, table, m, phi on the coset.
// rhs uses the polynomial form tau * sum_i prod_{j != i} (f_j + beta) - m * prod (no per-row inversion).
inline ValueSource lookup_constraints(GraphEvaluator& ev, const std::vector<ValueSource>& inputs, ValueSource table, ValueSource m,
                                      ValueSource phi, ValueSource l0, ValueSource l_last, ValueSource l_active_row) {
    const uint32_t r_next = ev.add_rotation(1);
    const ValueSource one = ev.add_constant(detail::from_dev(detail::DFr::one()));
    const ValueSource zero = ev.add_constant(detail::from_dev(detail::DFr::zero()));
    const size_t n = inputs.size();
    std::vector<ValueSource> ph(n), pre(n, one), suf(n, one);
    for (size_t i = 0; i < n; ++i) ph[i] = ev.add(B200ZK_CALC_ADD, inputs[i], ValueSource::Beta());
    ValueSource prod = one;
    for (size_t i = 0; i < n; ++i) {
        pre[i] = prod;
        prod = (i == 0) ? ph[0] : ev.add(B200ZK_CALC_MUL, prod, ph[i]);
    }
    ValueSource acc = one;
    for (size_t i = n; i-- > 0;) {
        suf[i] = acc;
        acc = (i + 1 == n) ? ph[i] : ev.add(B200ZK_CALC_MUL, acc, ph[i]);
    }
    ValueSource ssum = zero;
    for (size_t i = 0; i < n; ++i) {
        ValueSource term = (i == 0) ? suf[i] : (i + 1 == n) ? pre[i] : ev.add(B200ZK_CALC_MUL, pre[i], suf[i]);
        ssum = (i == 0) ? term : ev.add(B200ZK_CALC_ADD, ssum, term);
    }
    ValueSource phi_next = phi;
    phi_next.rotation = r_next;
    ValueSource tau = ev.add(B200ZK_CALC_ADD, table, ValueSource::Beta());
    ValueSource lhs = ev.add(B200ZK_CALC_MUL, ev.add(B200ZK_CALC_MUL, tau, prod), ev.add(B200ZK_CALC_SUB, phi_next, phi));
    ValueSource rhs = ev.add(B200ZK_CALC_SUB, ev.add(B200ZK_CALC_MUL, tau, ssum), ev.add(B200ZK_CALC_MUL, m, prod));
    ValueSource q = ev.add(B200ZK_CALC_MUL, ev.add(B200ZK_CALC_SUB, lhs, rhs), l_active_row);
    return ev.add_horner(ValueSource::PreviousValue(), {ev.add(B200ZK_CALC_MUL, l0, phi), ev.add(B200ZK_CALC_MUL, l_last, phi), q},
                         ValueSource::Y());
}

// permutation::Argument::commit, one column set: z in Lagrange form (the caller applies the blinding rows and chains
// z[n - (blinding_factors + 1)] into the next set as z_init, as upstream does)
inline void permutation_product(const std::vector<const DeviceColumn*>& values, const std::vector<const DeviceColumn*>& sigma,
                                const Fr& beta, const Fr& gamma, const Fr& delta_omega_start, const Fr& delta,
                                const EvaluationDomain& dom, const Fr& z_init, DeviceColumn& z_out) {
    if (values.size() != sigma.size()) throw Panic("permutation_product: columns.len() != permutations.len()");
    std::vector<const void*> tv, ts;
    for (auto* c : values) tv.push_back(c->ptr());
    for (auto* c : sigma) ts.push_back(c->ptr());
    auto& b = Backend::get();
    b.check(b200zk_permutation_product(b.ctx(), tv.data(), ts.data(), (uint32_t)tv.size(), &beta, &gamma, &delta_omega_start, &delta,
                                       &dom.omega, dom.k, &z_init, z_out.ptr()),
            "permutation_product");
}

// mv_lookup prover: the phi(X) running sum
inline void logup_running_sum(const std::vector<const DeviceColumn*>& inputs, const DeviceColumn& table, const DeviceColumn& m,
                              const Fr& beta, const EvaluationDomain& dom, const Fr& phi_init, DeviceColumn& phi_out) {
    std::vector<const void*> ti;
    for (auto* c : inputs) ti.push_back(c->ptr());
    auto& b = Backend::get();
    b.check(b200zk_logup_running_sum(b.ctx(), ti.data(), (uint32_t)ti.size(), table.ptr(), m.ptr(), &beta, dom.k, &phi_init, phi_out.ptr()),
            "logup_running_sum");
}

}  // namespace plonk

}  // namespace halo2_b200
