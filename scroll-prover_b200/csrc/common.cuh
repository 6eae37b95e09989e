// Shared host-side plumbing of libb200zk: context, error reporting, scratch memory, staging.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200zk.h"
#include "ff.cuh"

namespace b200zk {

struct TwiddleTable {  // universal per-stage twiddles for one root: tab[2^(u-1) + j] = w_{2^u}^j
    Fr omega;          // the 2^log_n-th root the table was built for
    uint32_t log_n;
    Fr* dev;
};

// per-kernel-class device timing (CUDA events on the context stream), read by bench.py for the roofline
enum ProfKey { PROF_NTT_PASS = 0, PROF_NTT_TABLE, PROF_MSM_COUNT, PROF_MSM_SCAN, PROF_MSM_SCATTER, PROF_MSM_ACCUM,
               PROF_MSM_COMBINE, PROF_MSM_REDUCE, PROF_MSM_FINISH, PROF_POLY, PROF_NKEYS };
static const char* const PROF_NAMES[PROF_NKEYS] = {"ntt_pass", "ntt_table", "msm_count", "msm_scan", "msm_scatter",
                                                   "msm_accumulate", "msm_combine", "msm_reduce", "msm_finish", "poly"};
struct ProfSpan {
    int key;
    cudaEvent_t e0, e1;
};

struct Scratch {  // grow-only device allocation
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace b200zk

struct b200zk_srs {
    b200zk_ctx* ctx;
    void* dev_bases;  // n x 64 B affine (x,y Montgomery Fq); W tables back to back when precomputed
    uint64_t n;
    uint32_t tag;
    uint32_t pre_c;   // 0: plain bases; else window bits the 2^(c*w) tables were built for
    uint32_t pre_W;
};

struct b200zk_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    std::recursive_mutex mu;
    std::string err;
    uint64_t launches = 0;
    int sm_count = 148;
    // scratch pools
    b200zk::Scratch ntt_work, stage_in, stage_out, msm_work, misc;
    void* pinned = nullptr;
    size_t pinned_cap = 0;
    std::vector<b200zk::TwiddleTable> tables;
    // column pipeline (b200zk_commit_columns): copy stream + double-buffered staging
    cudaStream_t copy_stream = nullptr;
    cudaStream_t aux_stream = nullptr;     // transforms of a column run here, concurrently with its MSM on `stream`
    cudaEvent_t ev_used_aux[2] = {nullptr, nullptr}, ev_fork = nullptr, ev_join = nullptr;
    int overlap = 1;                       // B200ZK_OVERLAP=0 serialises MSM and transforms on one stream
    b200zk::Scratch colstage[2], col_coeff, col_ext, col_commits;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_used[2] = {nullptr, nullptr};
    // profiling
    bool profiling = false;
    std::vector<b200zk::ProfSpan> prof_open;
    std::vector<cudaEvent_t> prof_pool;
    double prof_ms[b200zk::PROF_NKEYS] = {0};
    uint64_t prof_cnt[b200zk::PROF_NKEYS] = {0};
    // msm knobs / stats
    uint32_t msm_window = 0;
    uint32_t msm_scatter_sweeps = 0;
    uint32_t msm_acc_l = 0;
    int srs_precompute = 1;  // 1 auto: SRS handles of >= 2^16 points keep 2^(c*w) multiples when memory allows
    unsigned long long* msm_adds_dev = nullptr;  // running count of bucket additions actually performed
    uint32_t last_c = 0, last_windows = 0;
    uint64_t last_adds = 0;
    // cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a per-DEVICE opt-in: the "already done" flags live in the
    // context (one device per context), not in process-wide statics
    uint32_t smem_optin = 0;
    // multi-GPU (comm.cu): the context owns its NCCL communicator
    void* nccl_comm = nullptr;   // ncclComm_t
    void* comm_buf = nullptr;    // (world + 1) x 96 B: gathered partial points + this rank's own
    int comm_rank = 0, comm_world = 1;  // bit i: kernel family i has its opt-in on this context's device
};

namespace b200zk {

inline int32_t fail(b200zk_ctx* ctx, int32_t code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

#define B2_CUDA(ctx, call)                                                                                   \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess)                                                                              \
            return ::b200zk::fail(ctx, e__ == cudaErrorMemoryAllocation ? B200ZK_E_OOM : B200ZK_E_CUDA,      \
                                  "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

#define B2_TRY(expr)                    \
    do {                                \
        int32_t rc__ = (expr);          \
        if (rc__ != B200ZK_OK) return rc__; \
    } while (0)

#define B2_LAUNCH_CHECK(ctx)                 \
    do {                                     \
        (ctx)->launches++;                   \
        B2_CUDA(ctx, cudaGetLastError());    \
    } while (0)

inline cudaEvent_t prof_event(b200zk_ctx* ctx) {
    if (!ctx->prof_pool.empty()) {
        cudaEvent_t e = ctx->prof_pool.back();
        ctx->prof_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
// usage: ProfScope ps(ctx, PROF_X); ...launches...   (records on the context stream when profiling is on)
struct ProfScope {
    b200zk_ctx* ctx;
    ProfSpan sp;
    bool on;
    ProfScope(b200zk_ctx* c, int key) : ctx(c), on(c->profiling) {
        if (!on) return;
        sp.key = key;
        sp.e0 = prof_event(c);
        sp.e1 = prof_event(c);
        cudaEventRecord(sp.e0, c->stream);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(sp.e1, ctx->stream);
        ctx->prof_open.push_back(sp);
    }
};
inline void prof_resolve(b200zk_ctx* ctx) {
    for (auto& sp : ctx->prof_open) {
        float ms = 0;
        if (cudaEventSynchronize(sp.e1) == cudaSuccess && cudaEventElapsedTime(&ms, sp.e0, sp.e1) == cudaSuccess) {
            ctx->prof_ms[sp.key] += ms;
            ctx->prof_cnt[sp.key] += 1;
        }
        ctx->prof_pool.push_back(sp.e0);
        ctx->prof_pool.push_back(sp.e1);
    }
    ctx->prof_open.clear();
}

inline int32_t scratch_reserve(b200zk_ctx* ctx, Scratch& s, size_t bytes) {
    if (bytes <= s.cap) return B200ZK_OK;
    if (s.p) {
        B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        B2_CUDA(ctx, cudaFree(s.p));
        s.p = nullptr;
        s.cap = 0;
    }
    size_t want = bytes + (bytes >> 3);
    cudaError_t e = cudaMalloc(&s.p, want);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        want = bytes;
        e = cudaMalloc(&s.p, want);
    }
    if (e != cudaSuccess) return fail(ctx, B200ZK_E_OOM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    s.cap = want;
    return B200ZK_OK;
}

inline bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Copy host->device (pageable or pinned) on the context stream.
inline int32_t h2d(b200zk_ctx* ctx, void* dev, const void* host, size_t bytes) {
    if (!bytes) return B200ZK_OK;
    B2_CUDA(ctx, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return B200ZK_OK;
}
inline int32_t d2h(b200zk_ctx* ctx, void* host, const void* dev, size_t bytes) {
    if (!bytes) return B200ZK_OK;
    B2_CUDA(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

inline bool is_pinned_host_ptr(const void* p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// Input staging: returns a device pointer holding `bytes` of `p` (p itself if already on device).
// The caller's HOST buffer is no longer read once this returns: a copy from pageable memory has left the buffer when
// cudaMemcpyAsync returns (the runtime stages it), a copy from PINNED memory is truly asynchronous, so it is waited for here --
// an entry point whose result stays on the device would otherwise return while the DMA still reads the caller's memory.
inline int32_t stage_in(b200zk_ctx* ctx, Scratch& s, const void* p, size_t bytes, const void** out) {
    if (is_device_ptr(p)) {
        *out = p;
        return B200ZK_OK;
    }
    B2_TRY(scratch_reserve(ctx, s, bytes));
    B2_TRY(h2d(ctx, s.p, p, bytes));
    if (bytes && is_pinned_host_ptr(p)) B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out = s.p;
    return B200ZK_OK;
}

struct Guard {
    std::lock_guard<std::recursive_mutex> lk;
    explicit Guard(b200zk_ctx* c) : lk(c->mu) { cudaSetDevice(c->device); }
};

// a 32 B field element argument (host or device pointer) -> host value; rejects unreduced limbs
inline int32_t read_fr(b200zk_ctx* ctx, const void* p, Fr* out) {
    if (!p) return fail(ctx, B200ZK_E_INVALID, "null field element pointer");
    if (is_device_ptr(p)) {
        B2_CUDA(ctx, cudaMemcpyAsync(out, p, sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
        B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    } else {
        memcpy(out, p, sizeof(Fr));
    }
    uint32_t m[8], d[8];
    Fr::modulus(m);
    if (!leaf::sub8(d, out->l.v, m)) return fail(ctx, B200ZK_E_INVALID, "field element is not reduced (>= modulus)");
    return B200ZK_OK;
}

// result delivery: dev -> (host | device) pointer
inline int32_t deliver(b200zk_ctx* ctx, void* dst, const void* dev_src, size_t bytes) {
    if (is_device_ptr(dst)) {
        if (dst != dev_src) B2_CUDA(ctx, cudaMemcpyAsync(dst, dev_src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
        return B200ZK_OK;
    }
    return d2h(ctx, dst, dev_src, bytes);
}

// implemented in ntt.cu / msm.cu / poly.cu
int32_t ntt_get_table(b200zk_ctx* ctx, const Fr& omega, uint32_t log_n, const Fr** out);
Fr host_zeta();
int32_t comm_destroy(b200zk_ctx* ctx);  // comm.cu
int32_t ntt_run(b200zk_ctx* ctx, const Fr* in, uint32_t log_in, Fr* out, uint32_t log_n, const Fr& omega,
                int inverse_scale, int coset_mode);
Fr host_root_of_unity(uint32_t log_n);  // EvaluationDomain's primitive 2^log_n-th root
int32_t ntt_part_run(b200zk_ctx* ctx, const Fr* in, Fr* out, uint32_t k, uint32_t ext_k, uint32_t part, bool inverse,
                     const Fr& scale);
int32_t parts_recombine_run(b200zk_ctx* ctx, const Fr* parts, uint32_t k, uint32_t log_j, uint32_t n_pieces, const Fr& zeta_n_inv,
                            const Fr& w_j_inv, const Fr& j_inv, Fr* out);  // quotient.cu

// the extended domain of 2^extended_k points split into J = 2^(extended_k - k) parts of 2^k points (the coset-part entries)
constexpr uint32_t MAX_PART_LOG = 4;  // J <= 16
inline int32_t check_part_args(b200zk_ctx* ctx, const char* what, uint32_t k, uint32_t extended_k, uint32_t part) {
    if (k < 1) return fail(ctx, B200ZK_E_INVALID, "%s: k = %u, must be at least 1", what, k);
    if (extended_k < k || extended_k > 28)
        return fail(ctx, B200ZK_E_INVALID, "%s: extended_k = %u must lie in [k, 28] (k = %u)", what, extended_k, k);
    if (extended_k - k > MAX_PART_LOG)
        return fail(ctx, B200ZK_E_INVALID, "%s: J = 2^%u parts exceeds the supported maximum of %u", what, extended_k - k,
                    1u << MAX_PART_LOG);
    if (part >= (1u << (extended_k - k)))
        return fail(ctx, B200ZK_E_INVALID, "%s: part %u >= J = %u", what, part, 1u << (extended_k - k));
    return B200ZK_OK;
}

}  // namespace b200zk
