// Quotient construction on the device: the prover work BETWEEN the transforms of plonk::create_proof (SURVEY.md §8(f).2).
//
//   graph_eval_kernel     plonk::evaluation::GraphEvaluator::evaluate over the extended domain      (evaluation.rs)
//   scan_*                the z(X) running product of permutation::Argument::commit and the phi(X) running sum of
//                         the log-derivative lookup                                  (permutation/prover.rs, mv_lookup/prover.rs)
//   perm_* / logup_*      the per-row numerators / denominators those loops fold
// of halo2_proofs 1.1.0 @ scroll-tech/halo2 e5ddf67 (pin /root/reference/Cargo.lock:1886-1888).
//
// All of it is HBM-streaming work with ~1-2 field multiplications per 32 B moved: columns are read once with 128-bit
// accesses by consecutive threads, intermediates of a row never leave the SM (shared-memory slots assigned by the
// host-side lowering in graph.hpp), and the scans are three streaming phases whose middle one is a single block.
#include <new>

#include "common.cuh"
#include "graph_exec.cuh"

struct b200zk_graph {
    b200zk::GraphProgram prog;
    b200zk::GInstr* dev_instrs = nullptr;
    b200zk::Fr* dev_consts = nullptr;  // [program constants | beta gamma theta y | challenges] -- tail rewritten per call
    uint32_t consts_cap = 0;           // elements
    uint32_t* dev_rot = nullptr;       // per call: (rotation * rot_scale) mod size
    const void** dev_cols = nullptr;   // per call: column pointer tables, fixed | advice | instance
    uint32_t cols_cap = 0;
    std::vector<int32_t> rotations;    // row offsets depend on rot_scale and the domain size of each evaluate call
};

namespace b200zk {

int32_t batch_invert(b200zk_ctx* ctx, Fr* data, uint64_t n);

__device__ __forceinline__ Fr q_ld(const Fr* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1];
    Fr r;
    r.l.v[0] = a.x; r.l.v[1] = a.y; r.l.v[2] = a.z; r.l.v[3] = a.w;
    r.l.v[4] = b.x; r.l.v[5] = b.y; r.l.v[6] = b.z; r.l.v[7] = b.w;
    return r;
}
__device__ __forceinline__ void q_st(Fr* p, const Fr& r) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(r.l.v[0], r.l.v[1], r.l.v[2], r.l.v[3]);
    q[1] = make_uint4(r.l.v[4], r.l.v[5], r.l.v[6], r.l.v[7]);
}

// ------------------------------------------------------------------------------------------------ graph evaluator
struct GraphLaunch {
    const GInstr* instrs;
    uint32_t n_instr;
    const Fr* consts;
    const Fr* const* cols;     // device table of column pointers: fixed | advice | instance (only those the program reads)
    const uint32_t* rot_off;
    uint32_t log_size;
    Fr* values;
    uint32_t out_slot;
    uint32_t uses_x, uses_prev;
    const Fr* xtab;  // omega_ext^j, j < size/2   (the level-log_size run of the twiddle table)
    Fr zeta;
    uint64_t row_first, row_count;  // the rows this launch evaluates (a rank's slice of the extended domain)
};

// slot s of the row owned by thread `tid`: limb l at word (s * 8 + l) * T + tid  -- a warp reads 32 consecutive words
struct SmemSlots {
    uint32_t* base;  // + tid
    uint32_t T;
    __device__ __forceinline__ Fr load(uint32_t s) const {
        Fr r;
        const uint32_t* p = base + (size_t)s * 8 * T;
#pragma unroll
        for (int l = 0; l < 8; ++l) r.l.v[l] = p[l * T];
        return r;
    }
    __device__ __forceinline__ void store(uint32_t s, const Fr& v) {
        uint32_t* p = base + (size_t)s * 8 * T;
#pragma unroll
        for (int l = 0; l < 8; ++l) p[l * T] = v.l.v[l];
    }
};
struct HbmCols {
    const Fr* const* cols;
    const uint32_t* rot_off;
    uint64_t row, mask;
    __device__ __forceinline__ Fr load(uint32_t col, uint32_t rot) const {
        const Fr* p = cols[col];
        return q_ld(p + ((row + rot_off[rot]) & mask));
    }
};
struct DevConsts {
    const Fr* c;
    __device__ __forceinline__ Fr load(uint32_t i) const { return q_ld(c + i); }
};

__global__ void graph_eval_kernel(GraphLaunch L) {
    extern __shared__ uint32_t gsm[];
    const uint32_t T = blockDim.x;
    const uint64_t size = 1ull << L.log_size;
    const uint64_t idx = (uint64_t)blockIdx.x * T + threadIdx.x;
    if (idx >= L.row_count) return;  // slots are private to a thread: no block-wide barrier below
    const uint64_t row = L.row_first + idx;
    SmemSlots S{gsm + threadIdx.x, T};
    if (L.uses_prev) S.store(G_SLOT_PREV, q_ld(L.values + row));
    if (L.uses_x) {
        Fr x = L.zeta;
        if (L.log_size) {
            const uint64_t half = size >> 1;
            Fr w = q_ld(L.xtab + (row & (half - 1)));
            if (row >= half) w = Fr::zero() - w;  // omega^(j + size/2) = -omega^j
            x = x * w;
        }
        S.store(G_SLOT_X, x);
    }
    HbmCols Cc{L.cols, L.rot_off, row, size - 1};
    DevConsts K{L.consts};
    graph_exec_row(L.instrs, L.n_instr, S, Cc, K);
    Fr out = (L.out_slot == G_NO_RESULT) ? Fr::zero() : S.load(L.out_slot);
    q_st(L.values + row, out);
}

// rows per block: the widest block whose slots still let several blocks share an SM
static uint32_t graph_block_rows(uint32_t n_slots, size_t* smem_bytes) {
    const size_t budget = 220 * 1024;
    uint32_t best_t = 32;
    size_t best_rows = 0;
    for (uint32_t t = 128; t >= 32; t >>= 1) {
        size_t per_block = (size_t)n_slots * 32 * t;
        if (per_block > budget) continue;
        size_t blocks = budget / (per_block + 1024);  // + the per-block shared-memory reservation of the driver
        if (blocks > 32) blocks = 32;                 // resident-block limit of an SM
        size_t rows = blocks * t;
        if (rows > 1280) rows = 1280;                 // ~52 registers per thread: 64 K registers hold ~1260 rows
        if (rows > best_rows) {                       // ties go to the wider block (fewer blocks to schedule)
            best_rows = rows;
            best_t = t;
        }
    }
    *smem_bytes = (size_t)n_slots * 32 * best_t;
    return best_t;
}

int32_t graph_evaluate_run(b200zk_ctx* ctx, const b200zk_graph* g, GraphLaunch L) {
    size_t smem = 0;
    uint32_t T = graph_block_rows(g->prog.n_slots, &smem);
    if (!(ctx->smem_optin & (1u << 8))) {
        B2_CUDA(ctx, cudaFuncSetAttribute(graph_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(224 * 1024)));
        ctx->smem_optin |= 1u << 8;
    }
    uint32_t blocks = (uint32_t)((L.row_count + T - 1) / T);
    if (!blocks) return B200ZK_OK;
    ProfScope ps_(ctx, PROF_POLY);
    graph_eval_kernel<<<blocks, T, smem, ctx->stream>>>(L);
    B2_LAUNCH_CHECK(ctx);
    return B200ZK_OK;
}

// ------------------------------------------------------------------------------------------------ exclusive scans
// out[0] = init, out[i] = out[i-1] (op) in[i-1].  Thread-sequential chunks (one multiplication per element and phase,
// the arithmetic minimum), chunk totals scanned recursively; the top level is one block.
constexpr uint32_t SCAN_CHUNK = 64, SCAN_TOP = 4096;

template <int OP>
__device__ __forceinline__ Fr scan_op(const Fr& a, const Fr& b) {
    return OP == B200ZK_SCAN_PRODUCT ? a * b : a + b;
}
template <int OP>
__device__ __forceinline__ Fr scan_unit() {
    return OP == B200ZK_SCAN_PRODUCT ? Fr::one() : Fr::zero();
}

template <int OP>
__global__ void __launch_bounds__(128) scan_totals_kernel(const Fr* in, uint64_t n, uint32_t nchunks, Fr* totals) {
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchunks) return;
    uint64_t s = (uint64_t)c * SCAN_CHUNK, e = s + SCAN_CHUNK;
    if (e > n) e = n;
    Fr acc = scan_unit<OP>();
    for (uint64_t i = s; i < e; ++i) acc = scan_op<OP>(acc, q_ld(in + i));
    q_st(totals + c, acc);
}

template <int OP>
__global__ void __launch_bounds__(128) scan_apply_kernel(const Fr* in, uint64_t n, uint32_t nchunks, const Fr* carry, Fr* out) {
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchunks) return;
    uint64_t s = (uint64_t)c * SCAN_CHUNK, e = s + SCAN_CHUNK;
    if (e > n) e = n;
    Fr acc = q_ld(carry + c);
    for (uint64_t i = s; i < e; ++i) {
        Fr v = q_ld(in + i);  // read before the write: in == out is allowed
        q_st(out + i, acc);
        acc = scan_op<OP>(acc, v);
    }
}

// one block, n <= SCAN_TOP: per-thread runs of 16, Hillis-Steele over the 256 run totals in shared memory
template <int OP>
__global__ void __launch_bounds__(256) scan_top_kernel(const Fr* in, uint32_t n, Fr init, Fr* out) {
    __shared__ Fr sh[256];
    const uint32_t t = threadIdx.x, per = (n + 255) / 256;
    uint32_t s = t * per, e = s + per;
    if (s > n) s = n;
    if (e > n) e = n;
    Fr acc = scan_unit<OP>();
    for (uint32_t i = s; i < e; ++i) acc = scan_op<OP>(acc, q_ld(in + i));
    sh[t] = acc;
    __syncthreads();
    for (uint32_t d = 1; d < 256; d <<= 1) {
        Fr v = sh[t];
        if (t >= d) v = scan_op<OP>(sh[t - d], v);
        __syncthreads();
        sh[t] = v;
        __syncthreads();
    }
    Fr carry = t ? scan_op<OP>(init, sh[t - 1]) : init;
    for (uint32_t i = s; i < e; ++i) {
        Fr v = q_ld(in + i);
        q_st(out + i, carry);
        carry = scan_op<OP>(carry, v);
    }
}

template <int OP>
static int32_t scan_level(b200zk_ctx* ctx, const Fr* in, uint64_t n, const Fr& init, Fr* out, Fr* scratch) {
    if (n <= SCAN_TOP) {
        scan_top_kernel<OP><<<1, 256, 0, ctx->stream>>>(in, (uint32_t)n, init, out);
        B2_LAUNCH_CHECK(ctx);
        return B200ZK_OK;
    }
    uint32_t nchunks = (uint32_t)((n + SCAN_CHUNK - 1) / SCAN_CHUNK);
    Fr* totals = scratch;  // nchunks entries, scanned in place into the chunk carries
    uint32_t blocks = (nchunks + 127) / 128;
    scan_totals_kernel<OP><<<blocks, 128, 0, ctx->stream>>>(in, n, nchunks, totals);
    B2_LAUNCH_CHECK(ctx);
    B2_TRY(scan_level<OP>(ctx, totals, nchunks, init, totals, scratch + nchunks));
    scan_apply_kernel<OP><<<blocks, 128, 0, ctx->stream>>>(in, n, nchunks, totals, out);
    B2_LAUNCH_CHECK(ctx);
    return B200ZK_OK;
}

static size_t scan_scratch_elems(uint64_t n) {
    size_t tot = 0;
    while (n > SCAN_TOP) {
        n = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
        tot += n;
    }
    return tot + 1;
}

// scratch: caller-provided device memory of scan_scratch_elems(n) elements
int32_t prefix_scan_run(b200zk_ctx* ctx, int op, const Fr* in, uint64_t n, const Fr& init, Fr* out, Fr* scratch) {
    if (n == 0) return B200ZK_OK;
    ProfScope ps_(ctx, PROF_POLY);
    if (op == B200ZK_SCAN_PRODUCT) return scan_level<B200ZK_SCAN_PRODUCT>(ctx, in, n, init, out, scratch);
    return scan_level<B200ZK_SCAN_SUM>(ctx, in, n, init, out, scratch);
}

// ------------------------------------------------------------------------------------------------ permutation argument
// mv[i] = prod_j (beta * sigma_j[i] + gamma + v_j[i])
__global__ void __launch_bounds__(256) perm_denominator_kernel(const Fr* const* values, const Fr* const* sigma, uint32_t n_cols,
                                                               Fr beta, Fr gamma, uint64_t n, Fr* mv) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        Fr acc = Fr::one();
        for (uint32_t j = 0; j < n_cols; ++j) acc = acc * (beta * q_ld(sigma[j] + i) + gamma + q_ld(values[j] + i));
        q_st(mv + i, acc);
    }
}
// mv[i] *= prod_j (delta_omega_j * omega^i * beta + gamma + v_j[i]);  dbeta[j] = delta_omega_start * delta^j * beta
__global__ void __launch_bounds__(256) perm_numerator_kernel(const Fr* const* values, const Fr* dbeta, uint32_t n_cols, Fr gamma,
                                                             const Fr* wtab, uint64_t n, Fr* mv) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t half = n >> 1;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        Fr w = Fr::one();
        if (half) {
            w = q_ld(wtab + (i & (half - 1)));
            if (i >= half) w = Fr::zero() - w;
        }
        Fr acc = q_ld(mv + i);
        for (uint32_t j = 0; j < n_cols; ++j) acc = acc * (q_ld(dbeta + j) * w + gamma + q_ld(values[j] + i));
        q_st(mv + i, acc);
    }
}

// ------------------------------------------------------------------------------------------------ log-derivative lookup
// den[j * n + i] = inputs_j[i] + beta  (j < n_inputs);  den[n_inputs * n + i] = table[i] + beta
__global__ void __launch_bounds__(256) logup_denominator_kernel(const Fr* const* inputs, uint32_t n_inputs, const Fr* table, Fr beta,
                                                                uint64_t n, Fr* den) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        for (uint32_t j = 0; j < n_inputs; ++j) q_st(den + (uint64_t)j * n + i, q_ld(inputs[j] + i) + beta);
        q_st(den + (uint64_t)n_inputs * n + i, q_ld(table + i) + beta);
    }
}
// d[i] = sum_j inv[j * n + i] - m[i] * inv[n_inputs * n + i]
__global__ void __launch_bounds__(256) logup_combine_kernel(const Fr* inv, uint32_t n_inputs, const Fr* m, uint64_t n, Fr* d) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        Fr acc = Fr::zero();
        for (uint32_t j = 0; j < n_inputs; ++j) acc = acc + q_ld(inv + (uint64_t)j * n + i);
        acc = acc - q_ld(m + i) * q_ld(inv + (uint64_t)n_inputs * n + i);
        q_st(d + i, acc);
    }
}

static uint32_t stream_blocks(b200zk_ctx* ctx, uint64_t n) {
    uint64_t want = (n + 255) / 256, cap = (uint64_t)ctx->sm_count * 16;
    if (want > cap) want = cap;
    return (uint32_t)(want ? want : 1);
}

// uploads `count` host pointers into a device table carved from ctx->misc at byte offset `off`
static int32_t upload_ptrs(b200zk_ctx* ctx, const void* const* host, uint32_t count, char* dev_base, size_t off, const Fr* const** out) {
    *out = (const Fr* const*)(dev_base + off);
    if (count) B2_CUDA(ctx, cudaMemcpyAsync(dev_base + off, host, sizeof(void*) * count, cudaMemcpyHostToDevice, ctx->stream));
    return B200ZK_OK;
}

int32_t permutation_product_run(b200zk_ctx* ctx, const void* const* values, const void* const* sigma, uint32_t n_cols, const Fr& beta,
                                const Fr& gamma, const Fr& delta_omega_start, const Fr& delta, const Fr& omega, uint32_t k,
                                const Fr& z_init, Fr* z_out) {
    const uint64_t n = 1ull << k;
    const Fr* wtab = nullptr;
    if (k) {
        B2_TRY(ntt_get_table(ctx, omega, k, &wtab));
        wtab += n >> 1;
    }
    // scratch in ctx->stage_out: mv | scan scratch | pointer tables | dbeta      (ctx->misc is batch_invert's)
    size_t o_mv = 0, o_scan = o_mv + sizeof(Fr) * n, o_pv = o_scan + sizeof(Fr) * scan_scratch_elems(n);
    size_t o_ps = o_pv + sizeof(void*) * (n_cols + 1), o_db = (o_ps + sizeof(void*) * (n_cols + 1) + 31) / 32 * 32;
    size_t total = o_db + sizeof(Fr) * (n_cols + 1);
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, total));
    char* base = (char*)ctx->stage_out.p;
    Fr* mv = (Fr*)(base + o_mv);
    const Fr *const *dv, *const *ds;
    B2_TRY(upload_ptrs(ctx, values, n_cols, base, o_pv, &dv));
    B2_TRY(upload_ptrs(ctx, sigma, n_cols, base, o_ps, &ds));
    std::vector<Fr> dbeta(n_cols + 1);
    Fr dw = delta_omega_start;
    for (uint32_t j = 0; j < n_cols; ++j) {
        dbeta[j] = dw * beta;
        dw = dw * delta;
    }
    // the host vector dies with this frame: pageable cudaMemcpyAsync returns after staging, so that is safe
    if (n_cols) B2_CUDA(ctx, cudaMemcpyAsync(base + o_db, dbeta.data(), sizeof(Fr) * n_cols, cudaMemcpyHostToDevice, ctx->stream));
    uint32_t blocks = stream_blocks(ctx, n);
    {
        ProfScope ps_(ctx, PROF_POLY);
        perm_denominator_kernel<<<blocks, 256, 0, ctx->stream>>>(dv, ds, n_cols, beta, gamma, n, mv);
        B2_LAUNCH_CHECK(ctx);
    }
    B2_TRY(batch_invert(ctx, mv, n));
    {
        ProfScope ps_(ctx, PROF_POLY);
        perm_numerator_kernel<<<blocks, 256, 0, ctx->stream>>>(dv, (const Fr*)(base + o_db), n_cols, gamma, wtab, n, mv);
        B2_LAUNCH_CHECK(ctx);
    }
    return prefix_scan_run(ctx, B200ZK_SCAN_PRODUCT, mv, n, z_init, z_out, (Fr*)(base + o_scan));
}

int32_t logup_running_sum_run(b200zk_ctx* ctx, const void* const* inputs, uint32_t n_inputs, const Fr* table, const Fr* m,
                              const Fr& beta, uint32_t k, const Fr& phi_init, Fr* phi_out) {
    const uint64_t n = 1ull << k;
    size_t o_den = 0, o_d = o_den + sizeof(Fr) * n * ((size_t)n_inputs + 1), o_scan = o_d + sizeof(Fr) * n;
    size_t o_pi = o_scan + sizeof(Fr) * scan_scratch_elems(n);
    size_t total = o_pi + sizeof(void*) * (n_inputs + 1);
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, total));
    char* base = (char*)ctx->stage_out.p;
    Fr* den = (Fr*)(base + o_den);
    Fr* d = (Fr*)(base + o_d);
    const Fr* const* di;
    B2_TRY(upload_ptrs(ctx, inputs, n_inputs, base, o_pi, &di));
    uint32_t blocks = stream_blocks(ctx, n);
    {
        ProfScope ps_(ctx, PROF_POLY);
        logup_denominator_kernel<<<blocks, 256, 0, ctx->stream>>>(di, n_inputs, table, beta, n, den);
        B2_LAUNCH_CHECK(ctx);
    }
    B2_TRY(batch_invert(ctx, den, n * ((uint64_t)n_inputs + 1)));
    {
        ProfScope ps_(ctx, PROF_POLY);
        logup_combine_kernel<<<blocks, 256, 0, ctx->stream>>>(den, n_inputs, m, n, d);
        B2_LAUNCH_CHECK(ctx);
    }
    return prefix_scan_run(ctx, B200ZK_SCAN_SUM, d, n, phi_init, phi_out, (Fr*)(base + o_scan));
}

// ------------------------------------------------------------------------------------------------ linear combination
// out[i] = sum_j s_j * p_j[i]: every input is read once and the output written once (a chain of axpy calls would move
// 3x the bytes).  The SHPLONK prover's  sum_i v^i p_i(X)  per rotation set, and the final L(X) combination.
__global__ void __launch_bounds__(256) lincomb_kernel(const Fr* const* polys, const Fr* scalars, uint32_t count, uint64_t n, Fr* out) {
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        Fr acc = Fr::zero();
        for (uint32_t j = 0; j < count; ++j) acc = acc + q_ld(scalars + j) * q_ld(polys[j] + i);
        q_st(out + i, acc);
    }
}

int32_t lincomb_run(b200zk_ctx* ctx, const void* const* polys, const Fr* scalars_host, uint32_t count, uint64_t n, Fr* out) {
    size_t o_sc = 0, o_pt = sizeof(Fr) * ((size_t)count + 1);
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, o_pt + sizeof(void*) * ((size_t)count + 1)));
    char* base = (char*)ctx->stage_out.p;
    const Fr* const* dp;
    B2_TRY(upload_ptrs(ctx, polys, count, base, o_pt, &dp));
    if (count) B2_CUDA(ctx, cudaMemcpyAsync(base + o_sc, scalars_host, sizeof(Fr) * count, cudaMemcpyHostToDevice, ctx->stream));
    ProfScope ps_(ctx, PROF_POLY);
    lincomb_kernel<<<stream_blocks(ctx, n), 256, 0, ctx->stream>>>(dp, (const Fr*)(base + o_sc), count, n, out);
    B2_LAUNCH_CHECK(ctx);
    return B200ZK_OK;
}

// ------------------------------------------------------------------------------------------------ quotient from coset parts
// e_r[m] (r < J parts of n coefficients, part-major) -> h_j[m] = zeta^(-n j) J^-1 sum_r w_J^(-r j) e_r[m], j < n_pieces:
// a J-point inverse DFT per coefficient index, held in registers (radix-2 DIT, bit-reversed loads).  HBM-bound:
// (J + n_pieces) * 32 B per index.  out may equal parts (every index is read in full before its pieces are written).
struct PartsDft {
    Fr tw[8];   // w_J^-k, k < J/2
    Fr sc[16];  // zeta^(-n j) / J
};

template <int J>
__global__ void __launch_bounds__(128) parts_recombine_kernel(const Fr* parts, uint64_t n, uint32_t n_pieces, PartsDft D, Fr* out) {
    constexpr int LOGJ = J == 1 ? 0 : J == 2 ? 1 : J == 4 ? 2 : J == 8 ? 3 : 4;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; m < n; m += stride) {
        Fr a[J];
#pragma unroll
        for (int r = 0; r < J; ++r) {
            int br = 0;
#pragma unroll
            for (int b = 0; b < LOGJ; ++b) br |= ((r >> b) & 1) << (LOGJ - 1 - b);
            a[br] = q_ld(parts + (uint64_t)r * n + m);
        }
#pragma unroll
        for (int len = 2; len <= J; len <<= 1) {
#pragma unroll
            for (int s0 = 0; s0 < J; s0 += len) {
#pragma unroll
                for (int q = 0; q < len / 2; ++q) {
                    Fr u = a[s0 + q], v = a[s0 + q + len / 2];
                    if (q) v = v * D.tw[q * (J / len)];
                    a[s0 + q] = u + v;
                    a[s0 + q + len / 2] = u - v;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < J; ++j)
            if ((uint32_t)j < n_pieces) q_st(out + (uint64_t)j * n + m, a[j] * D.sc[j]);
    }
}

int32_t parts_recombine_run(b200zk_ctx* ctx, const Fr* parts, uint32_t k, uint32_t log_j, uint32_t n_pieces, const Fr& zeta_n_inv,
                            const Fr& w_j_inv, const Fr& j_inv, Fr* out) {
    const uint64_t n = 1ull << k;
    const uint32_t J = 1u << log_j;
    PartsDft D;
    Fr w = Fr::one();
    for (uint32_t i = 0; i < 8; ++i) {
        D.tw[i] = w;
        w = w * w_j_inv;
    }
    Fr sc = j_inv;
    for (uint32_t j = 0; j < 16; ++j) {
        D.sc[j] = sc;
        sc = sc * zeta_n_inv;
    }
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((n + 127) / 128, (uint64_t)ctx->sm_count * 16);
    ProfScope ps_(ctx, PROF_POLY);
    switch (J) {
        case 1: parts_recombine_kernel<1><<<blocks, 128, 0, ctx->stream>>>(parts, n, n_pieces, D, out); break;
        case 2: parts_recombine_kernel<2><<<blocks, 128, 0, ctx->stream>>>(parts, n, n_pieces, D, out); break;
        case 4: parts_recombine_kernel<4><<<blocks, 128, 0, ctx->stream>>>(parts, n, n_pieces, D, out); break;
        case 8: parts_recombine_kernel<8><<<blocks, 128, 0, ctx->stream>>>(parts, n, n_pieces, D, out); break;
        case 16: parts_recombine_kernel<16><<<blocks, 128, 0, ctx->stream>>>(parts, n, n_pieces, D, out); break;
        default: return fail(ctx, B200ZK_E_UNSUPPORTED, "extended_parts_to_coeff: J = %u is not supported", J);
    }
    B2_LAUNCH_CHECK(ctx);
    return B200ZK_OK;
}

}  // namespace b200zk

using namespace b200zk;

#define CHECK_CTX(ctx) \
    if (!(ctx)) return B200ZK_E_INVALID

static int32_t require_device(b200zk_ctx* ctx, const void* p, const char* what) {
    if (!p || !is_device_ptr(p)) return fail(ctx, B200ZK_E_INVALID, "%s must be a device pointer", what);
    return B200ZK_OK;
}
static int32_t require_device_cols(b200zk_ctx* ctx, const void* const* cols, uint32_t count, const char* what) {
    if (count && !cols) return fail(ctx, B200ZK_E_INVALID, "%s: null pointer table", what);
    for (uint32_t i = 0; i < count; ++i)
        if (!cols[i] || !is_device_ptr(cols[i])) return fail(ctx, B200ZK_E_INVALID, "%s[%u] must be a device pointer", what, i);
    return B200ZK_OK;
}

extern "C" {

int32_t b200zk_poly_lincomb(b200zk_ctx* ctx, void* out_dev, const void* const* polys_dev, const void* scalars32, uint32_t count, uint64_t n) {
    CHECK_CTX(ctx);
    if (count && !scalars32) return fail(ctx, B200ZK_E_INVALID, "poly_lincomb: null scalars");
    Guard g(ctx);
    if (!n) return B200ZK_OK;
    B2_TRY(require_device(ctx, out_dev, "poly_lincomb: out"));
    B2_TRY(require_device_cols(ctx, polys_dev, count, "poly_lincomb: polys"));
    std::vector<Fr> sc(count + 1);
    for (uint32_t j = 0; j < count; ++j) B2_TRY(read_fr(ctx, (const char*)scalars32 + 32 * (size_t)j, &sc[j]));
    return lincomb_run(ctx, polys_dev, sc.data(), count, n, (Fr*)out_dev);
}

int32_t b200zk_prefix_scan(b200zk_ctx* ctx, int op, const void* in_dev, uint64_t n, const void* init32, void* out_dev) {
    CHECK_CTX(ctx);
    if (op != B200ZK_SCAN_PRODUCT && op != B200ZK_SCAN_SUM) return fail(ctx, B200ZK_E_INVALID, "prefix_scan: unknown op %d", op);
    Guard g(ctx);
    Fr init;
    B2_TRY(read_fr(ctx, init32, &init));
    if (!n) return B200ZK_OK;
    B2_TRY(require_device(ctx, in_dev, "prefix_scan: in"));
    B2_TRY(require_device(ctx, out_dev, "prefix_scan: out"));
    B2_TRY(scratch_reserve(ctx, ctx->stage_out, sizeof(Fr) * scan_scratch_elems(n)));
    return prefix_scan_run(ctx, op, (const Fr*)in_dev, n, init, (Fr*)out_dev, (Fr*)ctx->stage_out.p);
}

int32_t b200zk_permutation_product(b200zk_ctx* ctx, const void* const* values_dev, const void* const* sigma_dev, uint32_t n_cols,
                                   const void* beta32, const void* gamma32, const void* delta_omega_start32, const void* delta32,
                                   const void* omega32, uint32_t k, const void* z_init32, void* z_out_dev) {
    CHECK_CTX(ctx);
    if (k > 28) return fail(ctx, B200ZK_E_INVALID, "permutation_product: k = %u > 28", k);
    Guard g(ctx);
    Fr beta, gamma, dws, delta, omega, z0;
    B2_TRY(read_fr(ctx, beta32, &beta));
    B2_TRY(read_fr(ctx, gamma32, &gamma));
    B2_TRY(read_fr(ctx, delta_omega_start32, &dws));
    B2_TRY(read_fr(ctx, delta32, &delta));
    B2_TRY(read_fr(ctx, omega32, &omega));
    B2_TRY(read_fr(ctx, z_init32, &z0));
    B2_TRY(require_device_cols(ctx, values_dev, n_cols, "permutation_product: values"));
    B2_TRY(require_device_cols(ctx, sigma_dev, n_cols, "permutation_product: sigma"));
    B2_TRY(require_device(ctx, z_out_dev, "permutation_product: z_out"));
    return permutation_product_run(ctx, values_dev, sigma_dev, n_cols, beta, gamma, dws, delta, omega, k, z0, (Fr*)z_out_dev);
}

int32_t b200zk_logup_running_sum(b200zk_ctx* ctx, const void* const* inputs_dev, uint32_t n_inputs, const void* table_dev,
                                 const void* m_dev, const void* beta32, uint32_t k, const void* phi_init32, void* phi_out_dev) {
    CHECK_CTX(ctx);
    if (k > 28) return fail(ctx, B200ZK_E_INVALID, "logup_running_sum: k = %u > 28", k);
    Guard g(ctx);
    Fr beta, phi0;
    B2_TRY(read_fr(ctx, beta32, &beta));
    B2_TRY(read_fr(ctx, phi_init32, &phi0));
    B2_TRY(require_device_cols(ctx, inputs_dev, n_inputs, "logup_running_sum: inputs"));
    B2_TRY(require_device(ctx, table_dev, "logup_running_sum: table"));
    B2_TRY(require_device(ctx, m_dev, "logup_running_sum: m"));
    B2_TRY(require_device(ctx, phi_out_dev, "logup_running_sum: phi_out"));
    return logup_running_sum_run(ctx, inputs_dev, n_inputs, (const Fr*)table_dev, (const Fr*)m_dev, beta, k, phi0, (Fr*)phi_out_dev);
}

int32_t b200zk_graph_create(b200zk_ctx* ctx, const b200zk_calculation* calculations, uint32_t n_calculations,
                            const b200zk_value_source* horner_parts, uint32_t n_parts, const void* constants32, uint32_t n_constants,
                            const int32_t* rotations, uint32_t n_rotations, b200zk_graph** out) {
    CHECK_CTX(ctx);
    if (!out) return fail(ctx, B200ZK_E_INVALID, "graph_create: null out");
    *out = nullptr;
    if ((n_calculations && !calculations) || (n_parts && !horner_parts) || (n_constants && !constants32) ||
        (n_rotations && !rotations))
        return fail(ctx, B200ZK_E_INVALID, "graph_create: null pointer");
    Guard g(ctx);
    b200zk_graph* gr = new (std::nothrow) b200zk_graph();
    if (!gr) return fail(ctx, B200ZK_E_OOM, "graph_create: out of host memory");
    std::string err = graph_compile(calculations, n_calculations, horner_parts, n_parts, n_constants, n_rotations, &gr->prog);
    if (!err.empty()) {
        delete gr;
        return fail(ctx, err.find("too many intermediates") != std::string::npos ? B200ZK_E_UNSUPPORTED : B200ZK_E_INVALID,
                    "graph_create: %s", err.c_str());
    }
    std::vector<Fr> consts(n_constants);
    uint32_t mod[8], dif[8];
    Fr::modulus(mod);
    for (uint32_t i = 0; i < n_constants; ++i) {
        memcpy(&consts[i], (const char*)constants32 + 32 * (size_t)i, 32);
        if (!leaf::sub8(dif, consts[i].l.v, mod)) {
            delete gr;
            return fail(ctx, B200ZK_E_INVALID, "graph_create: constant %u is not reduced", i);
        }
    }
    gr->rotations.assign(rotations, rotations + n_rotations);
    auto cleanup = [&]() {
        if (gr->dev_instrs) cudaFree(gr->dev_instrs);
        if (gr->dev_consts) cudaFree(gr->dev_consts);
        if (gr->dev_rot) cudaFree(gr->dev_rot);
        if (gr->dev_cols) cudaFree(gr->dev_cols);
        delete gr;
    };
    gr->consts_cap = n_constants + 4 + gr->prog.need_challenges;
    gr->cols_cap = gr->prog.need_cols[0] + gr->prog.need_cols[1] + gr->prog.need_cols[2];
    if (cudaMalloc(&gr->dev_instrs, sizeof(GInstr) * (gr->prog.instrs.size() + 1)) != cudaSuccess ||
        cudaMalloc(&gr->dev_consts, sizeof(Fr) * (gr->consts_cap + 1)) != cudaSuccess ||
        cudaMalloc(&gr->dev_rot, sizeof(uint32_t) * (n_rotations + 1)) != cudaSuccess ||
        cudaMalloc(&gr->dev_cols, sizeof(void*) * (gr->cols_cap + 1)) != cudaSuccess) {
        (void)cudaGetLastError();
        cleanup();
        return fail(ctx, B200ZK_E_OOM, "graph_create: device allocation failed");
    }
    cudaError_t e = cudaSuccess;
    if (!gr->prog.instrs.empty())
        e = cudaMemcpyAsync(gr->dev_instrs, gr->prog.instrs.data(), sizeof(GInstr) * gr->prog.instrs.size(), cudaMemcpyHostToDevice,
                            ctx->stream);
    if (e == cudaSuccess && n_constants)
        e = cudaMemcpyAsync(gr->dev_consts, consts.data(), sizeof(Fr) * n_constants, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        cleanup();
        return fail(ctx, B200ZK_E_CUDA, "graph_create: upload failed: %s", cudaGetErrorString(e));
    }
    *out = gr;
    return B200ZK_OK;
}

int32_t b200zk_graph_destroy(b200zk_ctx* ctx, b200zk_graph* graph) {
    CHECK_CTX(ctx);
    if (!graph) return B200ZK_OK;
    Guard g(ctx);
    cudaStreamSynchronize(ctx->stream);
    if (graph->dev_instrs) cudaFree(graph->dev_instrs);
    if (graph->dev_consts) cudaFree(graph->dev_consts);
    if (graph->dev_rot) cudaFree(graph->dev_rot);
    if (graph->dev_cols) cudaFree(graph->dev_cols);
    delete graph;
    return B200ZK_OK;
}

int32_t b200zk_graph_info(const b200zk_graph* graph, uint32_t* n_instructions, uint32_t* n_slots) {
    if (!graph) return B200ZK_E_INVALID;
    if (n_instructions) *n_instructions = (uint32_t)graph->prog.instrs.size();
    if (n_slots) *n_slots = graph->prog.n_slots;
    return B200ZK_OK;
}

int32_t b200zk_graph_check(const b200zk_calculation* calculations, uint32_t n_calculations, const b200zk_value_source* horner_parts,
                           uint32_t n_parts, uint32_t n_constants, uint32_t n_rotations, uint32_t* n_instructions, uint32_t* n_slots,
                           char* message, uint64_t message_cap) {
    if (message && message_cap) message[0] = 0;
    if ((n_calculations && !calculations) || (n_parts && !horner_parts)) return B200ZK_E_INVALID;
    GraphProgram prog;
    std::string err = graph_compile(calculations, n_calculations, horner_parts, n_parts, n_constants, n_rotations, &prog);
    if (!err.empty()) {
        if (message && message_cap) snprintf(message, (size_t)message_cap, "%s", err.c_str());
        return err.find("too many intermediates") != std::string::npos ? B200ZK_E_UNSUPPORTED : B200ZK_E_INVALID;
    }
    if (n_instructions) *n_instructions = (uint32_t)prog.instrs.size();
    if (n_slots) *n_slots = prog.n_slots;
    return B200ZK_OK;
}

int32_t b200zk_graph_evaluate(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev, uint32_t n_fixed,
                              const void* const* advice_dev, uint32_t n_advice, const void* const* instance_dev, uint32_t n_instance,
                              const void* challenges32, uint32_t n_challenges, const void* beta32, const void* gamma32,
                              const void* theta32, const void* y32, const void* extended_omega32, void* values_dev, uint32_t log_size,
                              int32_t rot_scale) {
    return b200zk_graph_evaluate_rows(ctx, graph, fixed_dev, n_fixed, advice_dev, n_advice, instance_dev, n_instance, challenges32,
                                      n_challenges, beta32, gamma32, theta32, y32, extended_omega32, values_dev, log_size, rot_scale, 0,
                                      log_size <= 30 ? (1ull << log_size) : 0);
}

}  // extern "C"

// rows [row_first, +row_count) of a domain of 2^log_size points x_zeta * w^row (w read from x_omega32 when the program uses x)
static int32_t graph_evaluate_impl(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev, uint32_t n_fixed,
                                   const void* const* advice_dev, uint32_t n_advice, const void* const* instance_dev, uint32_t n_instance,
                                   const void* challenges32, uint32_t n_challenges, const void* beta32, const void* gamma32,
                                   const void* theta32, const void* y32, const void* x_omega32, void* values_dev, uint32_t log_size,
                                   int32_t rot_scale, uint64_t row_first, uint64_t row_count, const Fr& x_zeta) {
    if (!graph) return fail(ctx, B200ZK_E_INVALID, "graph_evaluate: null graph");
    if (log_size > 30) return fail(ctx, B200ZK_E_INVALID, "graph_evaluate: log_size = %u > 30", log_size);
    if (row_first > (1ull << log_size) || row_count > (1ull << log_size) - row_first)
        return fail(ctx, B200ZK_E_INVALID, "graph_evaluate: rows [%llu, +%llu) exceed the domain of 2^%u", (unsigned long long)row_first,
                    (unsigned long long)row_count, log_size);
    const GraphProgram& P = graph->prog;
    if (P.need_cols[0] > n_fixed || P.need_cols[1] > n_advice || P.need_cols[2] > n_instance)
        return fail(ctx, B200ZK_E_INVALID, "graph_evaluate: the program reads fixed/advice/instance columns up to %u/%u/%u, got %u/%u/%u",
                    P.need_cols[0], P.need_cols[1], P.need_cols[2], n_fixed, n_advice, n_instance);
    if (P.need_challenges > n_challenges) return fail(ctx, B200ZK_E_INVALID, "graph_evaluate: the program reads %u challenges, got %u", P.need_challenges, n_challenges);
    if (n_challenges && !challenges32) return fail(ctx, B200ZK_E_INVALID, "graph_evaluate: null challenges");
    Guard g(ctx);
    B2_TRY(require_device(ctx, values_dev, "graph_evaluate: values"));
    B2_TRY(require_device_cols(ctx, fixed_dev, P.need_cols[0], "graph_evaluate: fixed"));
    B2_TRY(require_device_cols(ctx, advice_dev, P.need_cols[1], "graph_evaluate: advice"));
    B2_TRY(require_device_cols(ctx, instance_dev, P.need_cols[2], "graph_evaluate: instance"));
    // per-call constants: beta gamma theta y | challenges
    std::vector<Fr> tail(4 + P.need_challenges);
    B2_TRY(read_fr(ctx, beta32, &tail[0]));
    B2_TRY(read_fr(ctx, gamma32, &tail[1]));
    B2_TRY(read_fr(ctx, theta32, &tail[2]));
    B2_TRY(read_fr(ctx, y32, &tail[3]));
    for (uint32_t i = 0; i < P.need_challenges; ++i) B2_TRY(read_fr(ctx, (const char*)challenges32 + 32 * (size_t)i, &tail[4 + i]));
    const uint64_t size = 1ull << log_size;
    const int32_t* rotations = graph->rotations.data();
    std::vector<uint32_t> rot_off(P.n_rotations + 1);
    for (uint32_t r = 0; r < P.n_rotations; ++r) {
        int64_t v = ((int64_t)rotations[r] * rot_scale) % (int64_t)size;  // rem_euclid, as get_rotation_idx
        if (v < 0) v += (int64_t)size;
        rot_off[r] = (uint32_t)v;
    }
    std::vector<const void*> cols(graph->cols_cap + 1);
    uint32_t off1 = P.need_cols[0], off2 = off1 + P.need_cols[1];
    for (uint32_t i = 0; i < P.need_cols[0]; ++i) cols[i] = fixed_dev[i];
    for (uint32_t i = 0; i < P.need_cols[1]; ++i) cols[off1 + i] = advice_dev[i];
    for (uint32_t i = 0; i < P.need_cols[2]; ++i) cols[off2 + i] = instance_dev[i];
    GraphLaunch L;
    L.instrs = graph->dev_instrs;
    L.n_instr = (uint32_t)P.instrs.size();
    L.consts = graph->dev_consts;
    L.cols = (const Fr* const*)graph->dev_cols;
    L.rot_off = graph->dev_rot;
    L.log_size = log_size;
    L.values = (Fr*)values_dev;
    L.out_slot = P.out_slot;
    L.uses_x = P.uses_x;
    L.uses_prev = P.uses_prev;
    L.xtab = nullptr;
    L.zeta = x_zeta;
    L.row_first = row_first;
    L.row_count = row_count;
    if (P.uses_x && log_size) {
        Fr w;
        B2_TRY(read_fr(ctx, x_omega32, &w));
        const Fr* tab = nullptr;
        B2_TRY(ntt_get_table(ctx, w, log_size, &tab));
        L.xtab = tab + (size >> 1);
    }
    // the small per-call tables ride on the context stream ahead of the kernel; a previous evaluate of this graph on
    // the same stream has finished reading them by then (stream order)
    B2_CUDA(ctx, cudaMemcpyAsync(graph->dev_consts + P.n_constants, tail.data(), sizeof(Fr) * tail.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (P.n_rotations) B2_CUDA(ctx, cudaMemcpyAsync(graph->dev_rot, rot_off.data(), sizeof(uint32_t) * P.n_rotations, cudaMemcpyHostToDevice, ctx->stream));
    if (graph->cols_cap) B2_CUDA(ctx, cudaMemcpyAsync(graph->dev_cols, cols.data(), sizeof(void*) * graph->cols_cap, cudaMemcpyHostToDevice, ctx->stream));
    return graph_evaluate_run(ctx, graph, L);
}

extern "C" {

int32_t b200zk_graph_evaluate_rows(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev, uint32_t n_fixed,
                                   const void* const* advice_dev, uint32_t n_advice, const void* const* instance_dev, uint32_t n_instance,
                                   const void* challenges32, uint32_t n_challenges, const void* beta32, const void* gamma32,
                                   const void* theta32, const void* y32, const void* extended_omega32, void* values_dev, uint32_t log_size,
                                   int32_t rot_scale, uint64_t row_first, uint64_t row_count) {
    CHECK_CTX(ctx);
    return graph_evaluate_impl(ctx, graph, fixed_dev, n_fixed, advice_dev, n_advice, instance_dev, n_instance, challenges32, n_challenges,
                               beta32, gamma32, theta32, y32, extended_omega32, values_dev, log_size, rot_scale, row_first, row_count,
                               host_zeta());
}

int32_t b200zk_graph_evaluate_part(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev, uint32_t n_fixed,
                                   const void* const* advice_dev, uint32_t n_advice, const void* const* instance_dev, uint32_t n_instance,
                                   const void* challenges32, uint32_t n_challenges, const void* beta32, const void* gamma32,
                                   const void* theta32, const void* y32, uint32_t k, uint32_t extended_k, uint32_t part, void* values_dev) {
    CHECK_CTX(ctx);
    B2_TRY(check_part_args(ctx, "graph_evaluate_part", k, extended_k, part));
    // part r is the coset g_r * <w> of the n-th roots, g_r = zeta * w_ext^r: rotations move within the part (rot_scale 1)
    Guard g(ctx);
    const Fr w = host_root_of_unity(k);
    Fr g_r = host_zeta(), w_ext = host_root_of_unity(extended_k);
    for (uint32_t b = part; b; b >>= 1, w_ext = w_ext.sqr())
        if (b & 1) g_r = g_r * w_ext;
    return graph_evaluate_impl(ctx, graph, fixed_dev, n_fixed, advice_dev, n_advice, instance_dev, n_instance, challenges32, n_challenges,
                               beta32, gamma32, theta32, y32, &w, values_dev, k, 1, 0, 1ull << k, g_r);
}

}  // extern "C"
