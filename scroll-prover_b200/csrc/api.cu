// extern "C" boundary of libb200zk (include/b200zk.h): argument checking, host<->device staging,
// error codes.  No exceptions cross this file; every failure path sets b200zk_last_error.
#include <stdlib.h>

#include <new>

#include "common.cuh"
#include "ec.cuh"

namespace b200zk {
int32_t msm_run(b200zk_ctx* ctx, const Affine* bases, const Fr* scalars, uint64_t n, Jacobian* out_dev, uint32_t pre_c,
                uint64_t pre_stride);
int32_t msm_run_batch(b200zk_ctx* ctx, const Affine* bases, const Fr* const* cols, uint32_t batch, uint64_t n, Jacobian* out_dev,
                      uint32_t pre_c, uint64_t pre_stride);
uint32_t msm_max_batch(uint64_t n, uint32_t pre_c);
uint32_t msm_pick_window_precomputed(uint64_t n);
int32_t srs_precompute_run(b200zk_ctx* ctx, Affine* tables, uint64_t n, uint32_t c, uint32_t W);
int32_t g1_sum_run(b200zk_ctx* ctx, const Jacobian* pts, uint64_t count, Jacobian* out_dev);
int32_t g1_generator_mul_run(b200zk_ctx* ctx, const Fr* scalars, uint64_t n, Affine* out);
int32_t poly_ew(b200zk_ctx* ctx, int op, Fr* r, const Fr* a, const Fr* b, const Fr& s, uint64_t n);
int32_t eval_poly(b200zk_ctx* ctx, const Fr* poly, uint64_t n, const Fr& x, Fr* out_dev);
int32_t batch_invert(b200zk_ctx* ctx, Fr* data, uint64_t n);
int32_t inner_product(b200zk_ctx* ctx, const Fr* a, const Fr* b, uint64_t n, Fr* out_dev);
int32_t kate_division(b200zk_ctx* ctx, Fr* q, const Fr* a, uint64_t n, const Fr& b);
int32_t g1_fft_run(b200zk_ctx* ctx, const void* in, bool from_jac, void* out, bool to_jac, uint32_t log_n, const Fr& omega,
                   const Fr* scale);
int32_t field_op(b200zk_ctx* ctx, int field, int op, void* r, const void* a, const void* b, uint64_t n);
}  // namespace b200zk

using namespace b200zk;

#define CHECK_CTX(ctx) \
    if (!(ctx)) return B200ZK_E_INVALID

extern "C" {

int32_t b200zk_ctx_create(const int* devices, int n_devices, b200zk_ctx** out) {
    if (!out) return B200ZK_E_INVALID;
    *out = nullptr;
    if (n_devices != 1 && !(n_devices == 0 && devices == nullptr)) return B200ZK_E_UNSUPPORTED;
    int dev = (devices && n_devices == 1) ? devices[0] : 0;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        (void)cudaGetLastError();
        return B200ZK_E_CUDA;  // no CPU fallback by design
    }
    if (dev < 0 || dev >= count) return B200ZK_E_INVALID;
    if (cudaSetDevice(dev) != cudaSuccess) return B200ZK_E_CUDA;
    b200zk_ctx* ctx = new (std::nothrow) b200zk_ctx();
    if (!ctx) return B200ZK_E_OOM;
    ctx->device = dev;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return B200ZK_E_CUDA;
    }
    ctx->own_stream = true;
    if (const char* e = getenv("B200ZK_OVERLAP")) ctx->overlap = atoi(e);
    if (const char* e = getenv("B200ZK_ACC_L")) ctx->msm_acc_l = (uint32_t)atoi(e);
    if (const char* e = getenv("B200ZK_SCATTER_SWEEPS")) ctx->msm_scatter_sweeps = (uint32_t)atoi(e);  // experiment knob
    if (cudaMalloc(&ctx->msm_adds_dev, 8) == cudaSuccess) cudaMemset(ctx->msm_adds_dev, 0, 8);
    else ctx->msm_adds_dev = nullptr;
    *out = ctx;
    return B200ZK_OK;
}

int32_t b200zk_ctx_destroy(b200zk_ctx* ctx) {
    CHECK_CTX(ctx);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    comm_destroy(ctx);
    for (Scratch* s : {&ctx->ntt_work, &ctx->stage_in, &ctx->stage_out, &ctx->msm_work, &ctx->misc})
        if (s->p) cudaFree(s->p);
    for (auto& t : ctx->tables) cudaFree(t.dev);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->msm_adds_dev) cudaFree(ctx->msm_adds_dev);
    for (Scratch* s : {&ctx->colstage[0], &ctx->colstage[1], &ctx->col_coeff, &ctx->col_ext, &ctx->col_commits})
        if (s->p) cudaFree(s->p);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
        if (ctx->ev_used[i]) cudaEventDestroy(ctx->ev_used[i]);
        if (ctx->ev_used_aux[i]) cudaEventDestroy(ctx->ev_used_aux[i]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return B200ZK_OK;
}

const char* b200zk_last_error(const b200zk_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int32_t b200zk_ctx_set_stream(b200zk_ctx* ctx, void* cuda_stream) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (cuda_stream == nullptr) {
        if (!ctx->own_stream) {
            B2_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
            ctx->own_stream = true;
        }
        return B200ZK_OK;
    }
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return B200ZK_OK;
}

int32_t b200zk_ctx_synchronize(b200zk_ctx* ctx) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_ctx_launch_count(const b200zk_ctx* ctx, uint64_t* out) {
    if (!ctx || !out) return B200ZK_E_INVALID;
    *out = ctx->launches;
    return B200ZK_OK;
}

// ---- buffers ---------------------------------------------------------------------------------
int32_t b200zk_buf_alloc(b200zk_ctx* ctx, uint64_t bytes, void** out_dev) {
    CHECK_CTX(ctx);
    if (!out_dev) return fail(ctx, B200ZK_E_INVALID, "buf_alloc: null out");
    Guard g(ctx);
    *out_dev = nullptr;
    cudaError_t e = cudaMalloc(out_dev, bytes ? bytes : 1);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(ctx, B200ZK_E_OOM, "buf_alloc(%llu) failed: %s", (unsigned long long)bytes, cudaGetErrorString(e));
    }
    return B200ZK_OK;
}
int32_t b200zk_buf_free(b200zk_ctx* ctx, void* dev) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    if (!dev) return B200ZK_OK;
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B2_CUDA(ctx, cudaFree(dev));
    return B200ZK_OK;
}
int32_t b200zk_buf_upload(b200zk_ctx* ctx, void* dev, const void* host, uint64_t bytes) {
    CHECK_CTX(ctx);
    if (bytes && (!dev || !host)) return fail(ctx, B200ZK_E_INVALID, "buf_upload: null pointer");
    Guard g(ctx);
    B2_TRY(h2d(ctx, dev, host, bytes));
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // caller may reuse / free the host buffer
    return B200ZK_OK;
}
int32_t b200zk_buf_download(b200zk_ctx* ctx, void* host, const void* dev, uint64_t bytes) {
    CHECK_CTX(ctx);
    if (bytes && (!dev || !host)) return fail(ctx, B200ZK_E_INVALID, "buf_download: null pointer");
    Guard g(ctx);
    return d2h(ctx, host, dev, bytes);
}

// ---- SRS ---------------------------------------------------------------------------------------
int32_t b200zk_srs_register(b200zk_ctx* ctx, const void* g1_affine, uint64_t n, uint32_t tag, b200zk_srs** out) {
    CHECK_CTX(ctx);
    if (!out || (n && !g1_affine)) return fail(ctx, B200ZK_E_INVALID, "srs_register: null pointer");
    if (n >= (1ull << 31)) return fail(ctx, B200ZK_E_UNSUPPORTED, "srs_register: n >= 2^31");
    Guard g(ctx);
    b200zk_srs* s = new (std::nothrow) b200zk_srs();
    if (!s) return fail(ctx, B200ZK_E_OOM, "srs_register: host OOM");
    s->ctx = ctx;
    s->n = n;
    s->tag = tag;
    s->dev_bases = nullptr;
    s->pre_c = 0;
    s->pre_W = 1;
    size_t bytes = sizeof(Affine) * (n ? n : 1);
    if (ctx->srs_precompute && n >= (1ull << 16)) {
        // keep 2^(c*w) * P_i for every window w: all windows then share ONE bucket set (no per-window reduction, no
        // Horner doublings) and a wider window pays off.  Costs W x the base storage; skipped when memory is short.
        uint32_t c = msm_pick_window_precomputed(n), W = 254 / c + 1;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && (double)bytes * W < 0.35 * (double)free_b) {
            s->pre_c = c;
            s->pre_W = W;
            bytes *= W;
        }
    }
    cudaError_t e = cudaMalloc(&s->dev_bases, bytes);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        delete s;
        return fail(ctx, B200ZK_E_OOM, "srs_register: cudaMalloc(%zu) failed", bytes);
    }
    cudaMemcpyKind kind = is_device_ptr(g1_affine) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    e = n ? cudaMemcpyAsync(s->dev_bases, g1_affine, sizeof(Affine) * n, kind, ctx->stream) : cudaSuccess;
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        cudaFree(s->dev_bases);
        delete s;
        return fail(ctx, B200ZK_E_CUDA, "srs_register: upload failed: %s", cudaGetErrorString(e));
    }
    if (s->pre_c) {
        int32_t rc = srs_precompute_run(ctx, (Affine*)s->dev_bases, n, s->pre_c, s->pre_W);
        if (rc == B200ZK_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = B200ZK_E_CUDA;
        if (rc != B200ZK_OK) {
            cudaFree(s->dev_bases);
            delete s;
            return fail(ctx, rc, "srs_register: precomputation failed");
        }
    }
    *out = s;
    return B200ZK_OK;
}
int32_t b200zk_srs_release(b200zk_ctx* ctx, b200zk_srs* srs) {
    CHECK_CTX(ctx);
    if (!srs) return B200ZK_OK;
    Guard g(ctx);
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (srs->dev_bases) cudaFree(srs->dev_bases);
    delete srs;
    return B200ZK_OK;
}
int32_t b200zk_srs_len(const b200zk_srs* srs, uint64_t* out) {
    if (!srs || !out) return B200ZK_E_INVALID;
    *out = srs->n;
    return B200ZK_OK;
}

// ---- MSM ---------------------------------------------------------------------------------------
static int32_t msm_common(b200zk_ctx* ctx, const Affine* bases_dev, const void* scalars, uint64_t n, void* out96,
                          uint32_t pre_c = 0, uint64_t pre_stride = 0) {
    const void* sc_dev = nullptr;
    if (n) B2_TRY(stage_in(ctx, ctx->stage_in, scalars, sizeof(Fr) * n, &sc_dev));
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, 256));
    Jacobian* res = (Jacobian*)ctx->stage_out.p;
    B2_TRY(msm_run(ctx, bases_dev, (const Fr*)sc_dev, n, res, pre_c, pre_stride));
    return deliver(ctx, out96, res, sizeof(Jacobian));
}

int32_t b200zk_msm_g1(b200zk_ctx* ctx, const b200zk_srs* srs, const void* scalars, uint64_t n, void* out_jacobian96) {
    CHECK_CTX(ctx);
    if (!srs || !out_jacobian96 || (n && !scalars)) return fail(ctx, B200ZK_E_INVALID, "msm_g1: null pointer");
    if (srs->ctx != ctx) return fail(ctx, B200ZK_E_INVALID, "msm_g1: SRS belongs to another context");
    if (n > srs->n)
        return fail(ctx, B200ZK_E_INVALID, "msm_g1: %llu scalars but only %llu bases (assert_eq!(coeffs.len(), bases.len()))",
                    (unsigned long long)n, (unsigned long long)srs->n);
    Guard g(ctx);
    // a commit over a short prefix of a large precomputed SRS is cheaper with the plain bases (table 0) and a window
    // sized for n than with the handle's wide window (2^(c-1) buckets to reduce)
    uint32_t pre_c = (srs->pre_c && n * 16 >= srs->n) ? srs->pre_c : 0;
    return msm_common(ctx, (const Affine*)srs->dev_bases, scalars, n, out_jacobian96, pre_c, srs->n);
}

int32_t b200zk_msm_g1_batch(b200zk_ctx* ctx, const b200zk_srs* srs, const void* const* scalars, uint32_t count, uint64_t n,
                            void* out_jacobian96) {
    CHECK_CTX(ctx);
    if (!srs || (count && (!scalars || !out_jacobian96))) return fail(ctx, B200ZK_E_INVALID, "msm_g1_batch: null pointer");
    if (srs->ctx != ctx) return fail(ctx, B200ZK_E_INVALID, "msm_g1_batch: SRS belongs to another context");
    if (n > srs->n)
        return fail(ctx, B200ZK_E_INVALID, "msm_g1_batch: %llu scalars but only %llu bases (assert_eq!(coeffs.len(), bases.len()))",
                    (unsigned long long)n, (unsigned long long)srs->n);
    for (uint32_t j = 0; j < count; ++j)
        if (n && !scalars[j]) return fail(ctx, B200ZK_E_INVALID, "msm_g1_batch: scalars[%u] is null", j);
    Guard g(ctx);
    if (!count) return B200ZK_OK;
    try {
    const uint32_t pre_c = (srs->pre_c && n * 16 >= srs->n) ? srs->pre_c : 0;
    const uint32_t bmax = msm_max_batch(n, pre_c);
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, sizeof(Jacobian) * count));
    Jacobian* res = (Jacobian*)ctx->stage_out.p;
    size_t host_bytes = 0;  // staging for the host-resident columns of one batch
    for (uint32_t j0 = 0; j0 < count; j0 += bmax) {
        size_t b = 0;
        for (uint32_t j = j0; j < count && j < j0 + bmax; ++j)
            if (!is_device_ptr(scalars[j])) b += sizeof(Fr) * n;
        if (b > host_bytes) host_bytes = b;
    }
    if (host_bytes) B2_TRY(scratch_reserve(ctx, ctx->stage_in, host_bytes));
    std::vector<const Fr*> cols(bmax);
    for (uint32_t j0 = 0; j0 < count; j0 += bmax) {
        uint32_t len = count - j0 < bmax ? count - j0 : bmax;
        size_t off = 0;
        for (uint32_t q = 0; q < len; ++q) {
            const void* p = scalars[j0 + q];
            if (n && !is_device_ptr(p)) {
                B2_TRY(h2d(ctx, (char*)ctx->stage_in.p + off, p, sizeof(Fr) * n));
                p = (char*)ctx->stage_in.p + off;
                off += sizeof(Fr) * n;
            }
            cols[q] = (const Fr*)p;
        }
        B2_TRY(msm_run_batch(ctx, (const Affine*)srs->dev_bases, cols.data(), len, n, res + j0, pre_c, srs->n));
        // the staging buffer is reused by the next batch, and the caller's host columns must not be read after we return
        if (host_bytes && (j0 + bmax < count || is_device_ptr(out_jacobian96))) B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return deliver(ctx, out_jacobian96, res, sizeof(Jacobian) * count);
    } catch (const std::bad_alloc&) {  // nothing may unwind across the C boundary
        return fail(ctx, B200ZK_E_OOM, "msm_g1_batch: host allocation failed");
    }
}

int32_t b200zk_msm_g1_bases(b200zk_ctx* ctx, const void* g1_affine, const void* scalars, uint64_t n, void* out_jacobian96) {
    CHECK_CTX(ctx);
    if (!out_jacobian96 || (n && (!scalars || !g1_affine))) return fail(ctx, B200ZK_E_INVALID, "msm_g1_bases: null pointer");
    Guard g(ctx);
    const void* b_dev = nullptr;
    if (n) B2_TRY(stage_in(ctx, ctx->misc, g1_affine, sizeof(Affine) * n, &b_dev));
    // NB: ctx->misc is not used by msm_run
    return msm_common(ctx, (const Affine*)b_dev, scalars, n, out_jacobian96);
}

int32_t b200zk_g1_sum(b200zk_ctx* ctx, const void* jacobian_points, uint64_t count, void* out_jacobian96) {
    CHECK_CTX(ctx);
    if (!out_jacobian96 || (count && !jacobian_points)) return fail(ctx, B200ZK_E_INVALID, "g1_sum: null pointer");
    Guard g(ctx);
    const void* p_dev = nullptr;
    if (count) B2_TRY(stage_in(ctx, ctx->stage_in, jacobian_points, sizeof(Jacobian) * count, &p_dev));
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, 256));
    Jacobian* res = (Jacobian*)ctx->stage_out.p;
    B2_TRY(g1_sum_run(ctx, (const Jacobian*)p_dev, count, res));
    return deliver(ctx, out_jacobian96, res, sizeof(Jacobian));
}

int32_t b200zk_g1_generator_mul_batch(b200zk_ctx* ctx, const void* scalars, uint64_t n, void* out_affine) {
    CHECK_CTX(ctx);
    if (n && (!scalars || !out_affine)) return fail(ctx, B200ZK_E_INVALID, "g1_generator_mul_batch: null pointer");
    Guard g(ctx);
    if (!n) return B200ZK_OK;
    const void* sc_dev = nullptr;
    B2_TRY(stage_in(ctx, ctx->stage_in, scalars, sizeof(Fr) * n, &sc_dev));
    bool out_dev = is_device_ptr(out_affine);
    Affine* res = (Affine*)out_affine;
    if (!out_dev) {
        B2_TRY(scratch_reserve(ctx, ctx->stage_out, sizeof(Affine) * n));
        res = (Affine*)ctx->stage_out.p;
    }
    B2_TRY(g1_generator_mul_run(ctx, (const Fr*)sc_dev, n, res));
    if (!out_dev) return d2h(ctx, out_affine, res, sizeof(Affine) * n);
    return B200ZK_OK;
}

// ---- FFT over G1 (SRS tooling) -------------------------------------------------------------------
static int32_t g1_fft_common(b200zk_ctx* ctx, const void* in, bool from_jac, void* out, bool to_jac, uint32_t log_n,
                             const Fr& omega, const Fr* scale) {
    uint64_t n = 1ull << log_n;
    size_t in_bytes = (from_jac ? sizeof(Jacobian) : sizeof(Affine)) * n, out_bytes = (to_jac ? sizeof(Jacobian) : sizeof(Affine)) * n;
    const void* in_dev = nullptr;
    B2_TRY(stage_in(ctx, ctx->stage_in, in, in_bytes, &in_dev));
    bool out_is_dev = is_device_ptr(out);
    void* out_dev = out;
    if (!out_is_dev) {
        B2_TRY(scratch_reserve(ctx, ctx->stage_out, out_bytes));
        out_dev = ctx->stage_out.p;
    }
    B2_TRY(g1_fft_run(ctx, in_dev, from_jac, out_dev, to_jac, log_n, omega, scale));
    if (!out_is_dev) return d2h(ctx, out, out_dev, out_bytes);
    return B200ZK_OK;
}

int32_t b200zk_fft_g1(b200zk_ctx* ctx, void* jacobian_points, uint32_t log_n, const void* omega32) {
    CHECK_CTX(ctx);
    if (!jacobian_points || !omega32 || log_n > 28) return fail(ctx, B200ZK_E_INVALID, "fft_g1: bad arguments");
    Guard g(ctx);
    Fr omega;
    B2_TRY(read_fr(ctx, omega32, &omega));
    return g1_fft_common(ctx, jacobian_points, true, jacobian_points, true, log_n, omega, nullptr);
}

int32_t b200zk_g_to_lagrange(b200zk_ctx* ctx, const void* g_affine, uint32_t k, void* out_affine) {
    CHECK_CTX(ctx);
    if (!g_affine || !out_affine || k > 28) return fail(ctx, B200ZK_E_INVALID, "g_to_lagrange: bad arguments");
    Guard g(ctx);
    // omega_inv = ROOT_OF_UNITY_INV^(2^(S-k)), n_inv = TWO_INV^k   (g_to_lagrange in poly/kzg/commitment.rs)
    Fr root;
    const uint32_t rv[8] = {0xb639feb8u, 0x9632c7c5u, 0x0d0ff299u, 0x985ce340u, 0x01b0ecd8u, 0xb2dd8800u, 0x6d98ce29u, 0x1d69070du};
    for (int i = 0; i < 8; ++i) root.l.v[i] = rv[i];
    for (uint32_t i = k; i < 28; ++i) root = root.sqr();
    Fr omega_inv = root.inv();
    Fr nf = Fr::zero();
    nf.l.v[0] = (uint32_t)(1ull << k);
    nf.l.v[1] = (uint32_t)((1ull << k) >> 32);
    Fr n_inv = nf.to_mont().inv();
    return g1_fft_common(ctx, g_affine, false, out_affine, false, k, omega_inv, &n_inv);
}

// ---- NTT ---------------------------------------------------------------------------------------
int32_t b200zk_ntt_fr_ext(b200zk_ctx* ctx, const void* in, uint32_t log_in, void* out, uint32_t log_n, const void* omega32,
                          int inverse_scale, int coset_mode) {
    CHECK_CTX(ctx);
    if (!in || !out || !omega32) return fail(ctx, B200ZK_E_INVALID, "ntt: null pointer");
    if (log_n > 28 || log_in > log_n) return fail(ctx, B200ZK_E_INVALID, "ntt: bad sizes log_in=%u log_n=%u", log_in, log_n);
    Guard g(ctx);
    Fr omega;
    B2_TRY(read_fr(ctx, omega32, &omega));
    size_t in_bytes = sizeof(Fr) << log_in, out_bytes = sizeof(Fr) << log_n;
    bool out_is_dev = is_device_ptr(out);
    Fr* out_dev = (Fr*)out;
    if (!out_is_dev) {
        B2_TRY(scratch_reserve(ctx, ctx->stage_out, out_bytes));
        out_dev = (Fr*)ctx->stage_out.p;
    }
    const void* in_dev = nullptr;
    if (!is_device_ptr(in) && !out_is_dev && log_in == log_n) {
        // host in / host out of equal size: upload straight into the output staging buffer and run in place
        B2_TRY(h2d(ctx, out_dev, in, in_bytes));
        in_dev = out_dev;
    } else {
        B2_TRY(stage_in(ctx, ctx->stage_in, in, in_bytes, &in_dev));
    }
    B2_TRY(ntt_run(ctx, (const Fr*)in_dev, log_in, out_dev, log_n, omega, inverse_scale, coset_mode));
    if (!out_is_dev) return d2h(ctx, out, out_dev, out_bytes);
    return B200ZK_OK;
}

int32_t b200zk_ntt_fr(b200zk_ctx* ctx, void* data, uint32_t log_n, const void* omega32, int inverse_scale, int coset_mode) {
    return b200zk_ntt_fr_ext(ctx, data, log_n, data, log_n, omega32, inverse_scale, coset_mode);
}

// ---- the extended coset by parts (DESIGN.md "Quotient construction") ----------------------------
int32_t b200zk_coeff_to_extended_parts(b200zk_ctx* ctx, const void* const* coeffs, uint32_t count, uint32_t k, uint32_t extended_k,
                                       uint32_t part, void* const* out_dev) {
    CHECK_CTX(ctx);
    B2_TRY(check_part_args(ctx, "coeff_to_extended_parts", k, extended_k, part));
    if (count && (!coeffs || !out_dev)) return fail(ctx, B200ZK_E_INVALID, "coeff_to_extended_parts: null pointer table");
    Guard g(ctx);
    for (uint32_t j = 0; j < count; ++j) {
        if (!coeffs[j]) return fail(ctx, B200ZK_E_INVALID, "coeff_to_extended_parts: coeffs[%u] is null", j);
        if (!out_dev[j] || !is_device_ptr(out_dev[j]))
            return fail(ctx, B200ZK_E_INVALID, "coeff_to_extended_parts: out[%u] must be a device pointer", j);
    }
    const size_t bytes = sizeof(Fr) << k;
    for (uint32_t j = 0; j < count; ++j) {
        const void* in_dev = nullptr;
        B2_TRY(stage_in(ctx, ctx->stage_in, coeffs[j], bytes, &in_dev));  // stream order keeps the staging buffer's reuse safe
        B2_TRY(ntt_part_run(ctx, (const Fr*)in_dev, (Fr*)out_dev[j], k, extended_k, part, false, Fr::one()));
    }
    return B200ZK_OK;
}

int32_t b200zk_extended_parts_to_coeff(b200zk_ctx* ctx, void* parts_dev, uint32_t k, uint32_t extended_k, uint32_t n_pieces,
                                       int divide_by_vanishing, void* out_dev) {
    CHECK_CTX(ctx);
    B2_TRY(check_part_args(ctx, "extended_parts_to_coeff", k, extended_k, 0));
    const uint32_t log_j = extended_k - k, J = 1u << log_j;
    if (n_pieces < 1 || n_pieces > J)
        return fail(ctx, B200ZK_E_INVALID, "extended_parts_to_coeff: n_pieces = %u must lie in [1, J = %u]", n_pieces, J);
    Guard g(ctx);
    if (!parts_dev || !is_device_ptr(parts_dev)) return fail(ctx, B200ZK_E_INVALID, "extended_parts_to_coeff: parts must be a device pointer");
    if (!out_dev || !is_device_ptr(out_dev)) return fail(ctx, B200ZK_E_INVALID, "extended_parts_to_coeff: out must be a device pointer");
    const uint64_t n = 1ull << k;
    // part r: g_r^n = zeta^n w_J^r, w_J = w_ext^n the primitive J-th root; divide_by_vanishing_poly is 1 / (g_r^n - 1) on the part
    Fr zeta_n = Fr::one(), zeta = host_zeta();
    for (uint64_t i = 0; i < n % 3; ++i) zeta_n = zeta_n * zeta;  // zeta^3 = 1
    const Fr w_j = host_root_of_unity(log_j);
    Fr g_n = zeta_n;
    for (uint32_t r = 0; r < J; ++r, g_n = g_n * w_j) {
        Fr scale = divide_by_vanishing ? (g_n - Fr::one()).inv() : Fr::one();
        Fr* p = (Fr*)parts_dev + (uint64_t)r * n;
        B2_TRY(ntt_part_run(ctx, p, p, k, extended_k, r, true, scale));
    }
    Fr jf = Fr::zero();
    jf.l.v[0] = J;
    const Fr j_inv = jf.to_mont().inv();
    return parts_recombine_run(ctx, (const Fr*)parts_dev, k, log_j, n_pieces, zeta_n.inv(), w_j.inv(), j_inv, (Fr*)out_dev);
}

// ---- device-resident column pipeline (SURVEY.md §8(f).1) -------------------------------------------
static int32_t pipeline_init(b200zk_ctx* ctx) {
    if (ctx->copy_stream) return B200ZK_OK;
    B2_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    B2_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_used[i], cudaEventDisableTiming));
        B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_used_aux[i], cudaEventDisableTiming));
    }
    B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    B2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    return B200ZK_OK;
}

// One call = a list of independent per-column jobs of plonk::create_proof whose inputs are in HOST memory (pinned for
// overlap) or already on the device.  Jobs are taken in GROUPS: a group is uploaded (copy stream) while the previous one
// computes, and the commitments of a group's consecutive jobs over the same SRS go through ONE batched MSM pipeline
// (msm_run_batch) -- for 2^20-row columns that is up to 16 columns per pipeline, a 2^24+ column is a group of its own.
// No host synchronisation inside the loop.
static int32_t run_column_jobs_impl(b200zk_ctx* ctx, const b200zk_column_job* jobs, uint32_t count, uint32_t k, const void* omega_inv32,
                                    const void* extended_omega32, const void* extended_omega_inv32, uint32_t extended_k,
                                    void* commits_out);
int32_t b200zk_run_column_jobs(b200zk_ctx* ctx, const b200zk_column_job* jobs, uint32_t count, uint32_t k, const void* omega_inv32,
                               const void* extended_omega32, const void* extended_omega_inv32, uint32_t extended_k,
                               void* commits_out) {
    CHECK_CTX(ctx);
    try {  // the job bookkeeping allocates host memory: nothing may unwind across the C boundary
        return run_column_jobs_impl(ctx, jobs, count, k, omega_inv32, extended_omega32, extended_omega_inv32, extended_k, commits_out);
    } catch (const std::bad_alloc&) {
        return fail(ctx, B200ZK_E_OOM, "run_column_jobs: host allocation failed");
    } catch (...) {
        return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: unexpected host-side failure");
    }
}
static int32_t run_column_jobs_impl(b200zk_ctx* ctx, const b200zk_column_job* jobs, uint32_t count, uint32_t k, const void* omega_inv32,
                                    const void* extended_omega32, const void* extended_omega_inv32, uint32_t extended_k,
                                    void* commits_out) {
    if (k > 28 || (count && !jobs)) return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: bad arguments");
    const uint64_t n = 1ull << k;
    bool any_commit = false, any_coeff = false, any_ext = false, any_quot = false;
    for (uint32_t j = 0; j < count; ++j) {
        const b200zk_column_job& jb = jobs[j];
        if (!jb.host_values || jb.mode < 0 || jb.mode > 5) return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: job %u malformed", j);
        if (jb.mode <= 2) {
            if (!jb.srs || jb.srs->ctx != ctx || n > jb.srs->n)
                return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: job %u needs an SRS of this context with >= 2^k bases", j);
            any_commit = true;
        }
        any_coeff |= (jb.mode >= 1 && jb.mode <= 3);
        any_ext |= (jb.mode == 2 || jb.mode == 3 || jb.mode == 5);
        any_quot |= (jb.mode == 4);
    }
    if (any_commit && !commits_out) return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: commits_out is null");
    if (any_coeff && !omega_inv32) return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: omega_inv required");
    if ((any_ext && !extended_omega32) || (any_quot && !extended_omega_inv32) || ((any_ext || any_quot) && (extended_k < k || extended_k > 28)))
        return fail(ctx, B200ZK_E_INVALID, "run_column_jobs: bad extended domain");
    Guard g(ctx);
    if (!count) return B200ZK_OK;
    B2_TRY(pipeline_init(ctx));
    Fr omega_inv = Fr::one(), ext_omega = Fr::one(), ext_omega_inv = Fr::one();
    if (any_coeff) B2_TRY(read_fr(ctx, omega_inv32, &omega_inv));
    if (any_ext) B2_TRY(read_fr(ctx, extended_omega32, &ext_omega));
    if (any_quot) B2_TRY(read_fr(ctx, extended_omega_inv32, &ext_omega_inv));
    const size_t col_bytes = sizeof(Fr) * n, ext_bytes = sizeof(Fr) << extended_k;

    // ---- groups: [first, first + len); a mode-4 job (2^extended_k input values) is always a group of its own
    auto pre_of = [&](const b200zk_srs* s) -> uint32_t { return (n * 16 >= s->n) ? s->pre_c : 0; };
    uint32_t gmax = 1;
    for (uint32_t j = 0; j < count; ++j)
        if (jobs[j].mode <= 2) {
            gmax = msm_max_batch(n, pre_of(jobs[j].srs));
            break;
        }
    if (gmax > 16) gmax = 16;
    struct Group { uint32_t first, len; };
    std::vector<Group> groups;
    std::vector<uint8_t> is_dev(count);
    for (uint32_t j = 0; j < count; ++j) is_dev[j] = is_device_ptr(jobs[j].host_values) ? 1 : 0;
    for (uint32_t j = 0; j < count;) {
        if (jobs[j].mode == 4) {
            groups.push_back({j, 1});
            ++j;
            continue;
        }
        uint32_t len = 0;
        while (j + len < count && len < gmax && jobs[j + len].mode != 4) ++len;
        groups.push_back({j, len});
        j += len;
    }
    size_t stage_bytes = 0;  // host inputs of the largest group
    for (const Group& gr : groups) {
        size_t b = 0;
        for (uint32_t j = gr.first; j < gr.first + gr.len; ++j)
            if (!is_dev[j]) b += (jobs[j].mode == 4) ? ext_bytes : col_bytes;
        if (b > stage_bytes) stage_bytes = b;
    }
    for (int i = 0; i < 2; ++i)
        if (stage_bytes) B2_TRY(scratch_reserve(ctx, ctx->colstage[i], stage_bytes));
    B2_TRY(scratch_reserve(ctx, ctx->col_commits, sizeof(Jacobian) * count));
    if (any_coeff) B2_TRY(scratch_reserve(ctx, ctx->col_coeff, col_bytes));
    if (any_ext || any_quot) B2_TRY(scratch_reserve(ctx, ctx->col_ext, ext_bytes));
    Jacobian* commits = (Jacobian*)ctx->col_commits.p;
    if (any_commit) B2_CUDA(ctx, cudaMemsetAsync(commits, 0, sizeof(Jacobian) * count, ctx->stream));

    // Two compute streams: the commitments (MSM) run on the context stream, the transforms of the same column on
    // aux_stream.  Only msm_accumulate and the NTT passes are bound by the INT32 pipe; the MSM's sort / reduction phases
    // are latency- or memory-bound and overlap with the other stream's butterflies.
    const bool overlap = ctx->overlap && (any_coeff || any_quot || any_ext) && any_commit;
    cudaStream_t main_stream = ctx->stream, ntt_stream = overlap ? ctx->aux_stream : ctx->stream;
    struct StreamSwap {  // ntt_run / msm_run launch on ctx->stream
        b200zk_ctx* c;
        cudaStream_t saved;
        StreamSwap(b200zk_ctx* c_, cudaStream_t s) : c(c_), saved(c_->stream) { c->stream = s; }
        ~StreamSwap() { c->stream = saved; }
    };
    if (any_coeff) {  // twiddle tables are built once, on the context stream, before the streams fork
        const Fr* t = nullptr;
        B2_TRY(ntt_get_table(ctx, omega_inv, k, &t));
    }
    if (any_ext && extended_k >= 1) {
        const Fr* t = nullptr;
        B2_TRY(ntt_get_table(ctx, ext_omega, extended_k, &t));
    }
    if (any_quot && extended_k >= 1) {
        const Fr* t = nullptr;
        B2_TRY(ntt_get_table(ctx, ext_omega_inv, extended_k, &t));
    }
    // neither the copy stream nor the aux stream may overtake work already queued on the context stream
    B2_CUDA(ctx, cudaEventRecord(ctx->ev_fork, main_stream));
    B2_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_fork, 0));
    if (overlap) B2_CUDA(ctx, cudaStreamWaitEvent(ntt_stream, ctx->ev_fork, 0));

    bool used_main[2] = {false, false}, used_aux[2] = {false, false};
    std::vector<const Fr*> src(count);  // device address of every job's input
    bool any_host_copy = false;
    auto upload = [&](uint32_t gi) -> int32_t {  // returns with ev_copied[gi & 1] recorded when the group has host inputs
        const Group& gr = groups[gi];
        const int b = gi & 1;
        size_t off = 0;
        bool first_copy = true;
        for (uint32_t j = gr.first; j < gr.first + gr.len; ++j) {
            if (is_dev[j]) {
                src[j] = (const Fr*)jobs[j].host_values;  // already resident: used in place
                continue;
            }
            if (first_copy) {
                if (used_main[b]) B2_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_used[b], 0));
                if (used_aux[b]) B2_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_used_aux[b], 0));
                first_copy = false;
            }
            size_t bytes = (jobs[j].mode == 4) ? ext_bytes : col_bytes;
            char* dst = (char*)ctx->colstage[b].p + off;
            B2_CUDA(ctx, cudaMemcpyAsync(dst, jobs[j].host_values, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
            src[j] = (const Fr*)dst;
            off += bytes;
        }
        if (!first_copy) {
            B2_CUDA(ctx, cudaEventRecord(ctx->ev_copied[b], ctx->copy_stream));
            any_host_copy = true;
        }
        return B200ZK_OK;
    };
    B2_TRY(upload(0));
    for (uint32_t gi = 0; gi < groups.size(); ++gi) {
        const Group& gr = groups[gi];
        const int b = gi & 1;
        if (gi + 1 < groups.size()) B2_TRY(upload(gi + 1));
        bool host_in = false, grp_msm = false, grp_ntt = false;
        for (uint32_t j = gr.first; j < gr.first + gr.len; ++j) {
            host_in |= !is_dev[j];
            grp_msm |= jobs[j].mode <= 2;
            grp_ntt |= jobs[j].mode >= 1;
        }
        if (grp_msm) {
            if (host_in) B2_CUDA(ctx, cudaStreamWaitEvent(main_stream, ctx->ev_copied[b], 0));
            for (uint32_t j = gr.first; j < gr.first + gr.len;) {  // runs of consecutive commitments over the same SRS
                if (jobs[j].mode > 2) {
                    ++j;
                    continue;
                }
                const b200zk_srs* srs = jobs[j].srs;
                const uint32_t pre_c = pre_of(srs), bmax = msm_max_batch(n, pre_c);
                uint32_t len = 1;
                while (j + len < gr.first + gr.len && len < bmax && jobs[j + len].mode <= 2 && jobs[j + len].srs == srs) ++len;
                B2_TRY(msm_run_batch(ctx, (const Affine*)srs->dev_bases, &src[j], len, n, commits + j, pre_c, srs->n));
                j += len;
            }
            if (host_in) {
                B2_CUDA(ctx, cudaEventRecord(ctx->ev_used[b], main_stream));
                used_main[b] = true;
            }
        }
        if (grp_ntt) {
            StreamSwap sw(ctx, ntt_stream);
            if (host_in) B2_CUDA(ctx, cudaStreamWaitEvent(ntt_stream, ctx->ev_copied[b], 0));
            for (uint32_t j = gr.first; j < gr.first + gr.len; ++j) {
                const b200zk_column_job& jb = jobs[j];
                if (jb.mode < 1) continue;
                if (jb.mode <= 3) {
                    Fr* coeff = jb.coeff_out_dev ? (Fr*)jb.coeff_out_dev : (Fr*)ctx->col_coeff.p;
                    B2_TRY(ntt_run(ctx, src[j], k, coeff, k, omega_inv, 1, B200ZK_COSET_NONE));
                    if (jb.mode >= 2) {
                        Fr* ext = jb.ext_out_dev ? (Fr*)jb.ext_out_dev : (Fr*)ctx->col_ext.p;
                        B2_TRY(ntt_run(ctx, coeff, k, ext, extended_k, ext_omega, 0, B200ZK_COSET_PRE));
                    }
                } else if (jb.mode == 4) {
                    Fr* out = jb.coeff_out_dev ? (Fr*)jb.coeff_out_dev : (Fr*)ctx->col_ext.p;
                    B2_TRY(ntt_run(ctx, src[j], extended_k, out, extended_k, ext_omega_inv, 1, B200ZK_COSET_POST));
                } else {  // mode 5: coefficients -> extended coset
                    Fr* ext = jb.ext_out_dev ? (Fr*)jb.ext_out_dev : (Fr*)ctx->col_ext.p;
                    B2_TRY(ntt_run(ctx, src[j], k, ext, extended_k, ext_omega, 0, B200ZK_COSET_PRE));
                }
            }
            if (host_in) {
                B2_CUDA(ctx, cudaEventRecord(overlap ? ctx->ev_used_aux[b] : ctx->ev_used[b], ntt_stream));
                (overlap ? used_aux : used_main)[b] = true;
            }
        }
    }
    if (overlap) {  // join: everything issued on the aux stream is ordered before later work on the context stream
        B2_CUDA(ctx, cudaEventRecord(ctx->ev_join, ntt_stream));
        B2_CUDA(ctx, cudaStreamWaitEvent(main_stream, ctx->ev_join, 0));
    }
    if (!any_commit) {
        // no result to read back: still make sure every H2D copy has left the caller's host buffers before returning
        if (any_host_copy) B2_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
        return B200ZK_OK;
    }
    return deliver(ctx, commits_out, commits, sizeof(Jacobian) * count);
}

// Homogeneous convenience form: the same mode and SRS for every column.
int32_t b200zk_commit_columns(b200zk_ctx* ctx, const b200zk_srs* srs, const void* const* host_cols, uint32_t count, uint32_t k,
                              const void* omega_inv32, const void* extended_omega32, uint32_t extended_k, void* commits_out,
                              void* const* coeff_out_dev, void* const* ext_out_dev, int mode) {
    CHECK_CTX(ctx);
    if (mode < 0 || mode > 3) return fail(ctx, B200ZK_E_INVALID, "commit_columns: mode must be 0 (commit), 1 (+coeff), 2 (+coeff+extended), 3 (coeff+extended only)");
    if (count && !host_cols) return fail(ctx, B200ZK_E_INVALID, "commit_columns: null host_cols");
    std::vector<b200zk_column_job> jobs;
    try {
        jobs.resize(count);
    } catch (const std::bad_alloc&) {
        return fail(ctx, B200ZK_E_OOM, "commit_columns: host allocation failed");
    }
    for (uint32_t j = 0; j < count; ++j) {
        jobs[j].host_values = host_cols[j];
        jobs[j].srs = srs;
        jobs[j].mode = mode;
        jobs[j].coeff_out_dev = coeff_out_dev ? coeff_out_dev[j] : nullptr;
        jobs[j].ext_out_dev = ext_out_dev ? ext_out_dev[j] : nullptr;
    }
    return b200zk_run_column_jobs(ctx, jobs.data(), count, k, omega_inv32, extended_omega32, nullptr, extended_k, commits_out);
}

// ---- poly ops ------------------------------------------------------------------------------------
static int32_t ew_common(b200zk_ctx* ctx, int op, void* r, const void* a, const void* b, const void* s32, uint64_t n) {
    CHECK_CTX(ctx);
    bool need_b = (op == 0 || op == 1 || op == 2 || op == 4), need_s = (op == 3 || op == 4);
    if (n && (!r || !a || (need_b && !b) || (need_s && !s32))) return fail(ctx, B200ZK_E_INVALID, "poly op: null pointer");
    Guard g(ctx);
    if (!n) return B200ZK_OK;
    Fr s = Fr::zero();
    if (need_s) B2_TRY(read_fr(ctx, s32, &s));
    size_t bytes = sizeof(Fr) * n;
    const void *a_dev = nullptr, *b_dev = nullptr;
    B2_TRY(stage_in(ctx, ctx->stage_in, a, bytes, &a_dev));
    if (need_b) B2_TRY(stage_in(ctx, ctx->ntt_work, b, bytes, &b_dev));
    bool r_is_dev = is_device_ptr(r);
    Fr* r_dev = (Fr*)r;
    if (!r_is_dev) {
        B2_TRY(scratch_reserve(ctx, ctx->stage_out, bytes));
        r_dev = (Fr*)ctx->stage_out.p;
    }
    B2_TRY(poly_ew(ctx, op, r_dev, (const Fr*)a_dev, (const Fr*)b_dev, s, n));
    if (!r_is_dev) return d2h(ctx, r, r_dev, bytes);
    return B200ZK_OK;
}
int32_t b200zk_poly_add(b200zk_ctx* ctx, void* r, const void* a, const void* b, uint64_t n) { return ew_common(ctx, 0, r, a, b, nullptr, n); }
int32_t b200zk_poly_sub(b200zk_ctx* ctx, void* r, const void* a, const void* b, uint64_t n) { return ew_common(ctx, 1, r, a, b, nullptr, n); }
int32_t b200zk_poly_mul(b200zk_ctx* ctx, void* r, const void* a, const void* b, uint64_t n) { return ew_common(ctx, 2, r, a, b, nullptr, n); }
int32_t b200zk_poly_scale(b200zk_ctx* ctx, void* r, const void* a, const void* s32, uint64_t n) { return ew_common(ctx, 3, r, a, nullptr, s32, n); }
int32_t b200zk_poly_axpy(b200zk_ctx* ctx, void* r, const void* a, const void* s32, const void* b, uint64_t n) {
    return ew_common(ctx, 4, r, a, b, s32, n);
}

int32_t b200zk_eval_poly(b200zk_ctx* ctx, const void* poly, uint64_t n, const void* point32, void* out32) {
    CHECK_CTX(ctx);
    if (!out32 || !point32 || (n && !poly)) return fail(ctx, B200ZK_E_INVALID, "eval_poly: null pointer");
    Guard g(ctx);
    Fr x;
    B2_TRY(read_fr(ctx, point32, &x));
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, 256));
    Fr* res = (Fr*)ctx->stage_out.p;
    if (!n) {
        B2_CUDA(ctx, cudaMemsetAsync(res, 0, sizeof(Fr), ctx->stream));
    } else {
        const void* p_dev = nullptr;
        B2_TRY(stage_in(ctx, ctx->stage_in, poly, sizeof(Fr) * n, &p_dev));
        B2_TRY(eval_poly(ctx, (const Fr*)p_dev, n, x, res));
    }
    return deliver(ctx, out32, res, sizeof(Fr));
}

int32_t b200zk_inner_product(b200zk_ctx* ctx, const void* a, const void* b, uint64_t n, void* out32) {
    CHECK_CTX(ctx);
    if (!out32 || (n && (!a || !b))) return fail(ctx, B200ZK_E_INVALID, "inner_product: null pointer");
    Guard g(ctx);
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, 256));
    Fr* res = (Fr*)ctx->stage_out.p;
    if (!n) {
        B2_CUDA(ctx, cudaMemsetAsync(res, 0, sizeof(Fr), ctx->stream));
    } else {
        const void *a_dev = nullptr, *b_dev = nullptr;
        B2_TRY(stage_in(ctx, ctx->stage_in, a, sizeof(Fr) * n, &a_dev));
        B2_TRY(stage_in(ctx, ctx->ntt_work, b, sizeof(Fr) * n, &b_dev));
        B2_TRY(inner_product(ctx, (const Fr*)a_dev, (const Fr*)b_dev, n, res));
    }
    return deliver(ctx, out32, res, sizeof(Fr));
}

int32_t b200zk_batch_invert(b200zk_ctx* ctx, void* data, uint64_t n) {
    CHECK_CTX(ctx);
    if (n && !data) return fail(ctx, B200ZK_E_INVALID, "batch_invert: null pointer");
    Guard g(ctx);
    if (!n) return B200ZK_OK;
    if (is_device_ptr(data)) return batch_invert(ctx, (Fr*)data, n);
    size_t bytes = sizeof(Fr) * n;
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, bytes));
    B2_TRY(h2d(ctx, ctx->stage_out.p, data, bytes));
    B2_TRY(batch_invert(ctx, (Fr*)ctx->stage_out.p, n));
    return d2h(ctx, data, ctx->stage_out.p, bytes);
}

int32_t b200zk_kate_division(b200zk_ctx* ctx, void* q, const void* a, uint64_t n, const void* b32) {
    CHECK_CTX(ctx);
    if (n < 1 || !a || !b32 || (n > 1 && !q)) return fail(ctx, B200ZK_E_INVALID, "kate_division: bad arguments");
    Guard g(ctx);
    if (n == 1) return B200ZK_OK;
    Fr b;
    B2_TRY(read_fr(ctx, b32, &b));
    const void* a_dev = nullptr;
    B2_TRY(stage_in(ctx, ctx->stage_in, a, sizeof(Fr) * n, &a_dev));
    bool q_is_dev = is_device_ptr(q);
    Fr* q_dev = (Fr*)q;
    size_t qbytes = sizeof(Fr) * (n - 1);
    if (!q_is_dev) {
        B2_TRY(scratch_reserve(ctx, ctx->stage_out, qbytes));
        q_dev = (Fr*)ctx->stage_out.p;
    }
    B2_TRY(kate_division(ctx, q_dev, (const Fr*)a_dev, n, b));
    if (!q_is_dev) return d2h(ctx, q, q_dev, qbytes);
    return B200ZK_OK;
}

// ---- diagnostics -----------------------------------------------------------------------------------
int32_t b200zk_debug_field_op(b200zk_ctx* ctx, int field, int op, void* r, const void* a, const void* b, uint64_t n) {
    CHECK_CTX(ctx);
    if (n && (!r || !a || !b)) return fail(ctx, B200ZK_E_INVALID, "debug_field_op: null pointer");
    Guard g(ctx);
    if (!n) return B200ZK_OK;
    size_t bytes = 32 * n;
    const void *a_dev = nullptr, *b_dev = nullptr;
    B2_TRY(stage_in(ctx, ctx->stage_in, a, bytes, &a_dev));
    B2_TRY(stage_in(ctx, ctx->ntt_work, b, bytes, &b_dev));
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, bytes));
    B2_TRY(field_op(ctx, field, op, ctx->stage_out.p, a_dev, b_dev, n));
    return deliver(ctx, r, ctx->stage_out.p, bytes);
}

int32_t b200zk_profile_enable(b200zk_ctx* ctx, int on) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    ctx->profiling = on != 0;
    return B200ZK_OK;
}
int32_t b200zk_profile_reset(b200zk_ctx* ctx) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    prof_resolve(ctx);
    for (int i = 0; i < PROF_NKEYS; ++i) {
        ctx->prof_ms[i] = 0;
        ctx->prof_cnt[i] = 0;
    }
    return B200ZK_OK;
}
int32_t b200zk_profile_read(b200zk_ctx* ctx, const char* name, double* total_ms, uint64_t* count) {
    CHECK_CTX(ctx);
    if (!name) return fail(ctx, B200ZK_E_INVALID, "profile_read: null name");
    Guard g(ctx);
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    prof_resolve(ctx);
    for (int i = 0; i < PROF_NKEYS; ++i)
        if (strcmp(name, PROF_NAMES[i]) == 0) {
            if (total_ms) *total_ms = ctx->prof_ms[i];
            if (count) *count = ctx->prof_cnt[i];
            return B200ZK_OK;
        }
    return fail(ctx, B200ZK_E_INVALID, "profile_read: unknown kernel class '%s'", name);
}

int32_t b200zk_ctx_set_overlap(b200zk_ctx* ctx, int on) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    ctx->overlap = on != 0;
    return B200ZK_OK;
}
int32_t b200zk_srs_set_precompute(b200zk_ctx* ctx, int mode) {
    CHECK_CTX(ctx);
    if (mode != 0 && mode != 1) return fail(ctx, B200ZK_E_INVALID, "srs_set_precompute: mode must be 0 or 1");
    ctx->srs_precompute = mode;
    return B200ZK_OK;
}
int32_t b200zk_msm_set_window(b200zk_ctx* ctx, uint32_t c) {
    CHECK_CTX(ctx);
    if (c != 0 && (c < 2 || c > 24)) return fail(ctx, B200ZK_E_INVALID, "msm window %u out of range", c);
    ctx->msm_window = c;
    return B200ZK_OK;
}
int32_t b200zk_msm_total_adds(b200zk_ctx* ctx, uint64_t* actual_adds, int reset) {
    CHECK_CTX(ctx);
    Guard g(ctx);
    unsigned long long v = 0;
    if (ctx->msm_adds_dev) {
        B2_CUDA(ctx, cudaMemcpyAsync(&v, ctx->msm_adds_dev, 8, cudaMemcpyDeviceToHost, ctx->stream));
        B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (reset) B2_CUDA(ctx, cudaMemsetAsync(ctx->msm_adds_dev, 0, 8, ctx->stream));
    }
    if (actual_adds) *actual_adds = v;
    return B200ZK_OK;
}
int32_t b200zk_msm_last_stats(const b200zk_ctx* ctx, uint32_t* window_bits, uint32_t* n_windows, uint64_t* n_bucket_adds) {
    if (!ctx) return B200ZK_E_INVALID;
    if (window_bits) *window_bits = ctx->last_c;
    if (n_windows) *n_windows = ctx->last_windows;
    if (n_bucket_adds) *n_bucket_adds = ctx->last_adds;
    return B200ZK_OK;
}

}  // extern "C"
