// BN254 Fr number-theoretic transform for sm_100a.
//
// Device replacement for halo2_proofs::arithmetic::best_fft::<Fr,Fr> and the EvaluationDomain
// transforms built on it (halo2_proofs/src/arithmetic.rs, src/poly/domain.rs @ scroll-tech/halo2
// e5ddf67, pin /root/reference/Cargo.lock:1886-1888): natural order in, natural order out,
// A[j] = sum_i a[i] w^(ij), bit-identical outputs.
//
// Decomposition (DESIGN.md "NTT"): log_n = n_1 + ... + n_P, n_p <= 8.  Pass p transforms digit p of the
// index (most significant first) with a radix-2 DIT butterfly network held in shared memory:
//   input  index i = [I_1][I_2]...[I_P]      output index k = [K_P]...[K_2][K_1]
//   pass p: [K_1..K_{p-1}][I_p][rest] -> [K_1..K_{p-1}][K_p][rest],   in place, strided tile of
//           2^{n_p} digit entries x 8 adjacent "rest" lanes (256 B segments => coalesced);
//   stage s of pass p uses the GLOBAL twiddle  w_{2^(t+s)}^(K*2^t + c),  t = n_1+..+n_{p-1},
//           c = K_1 + K_2 2^{n_1} + ...  (the already-transformed digits), so there are no separate
//           inter-pass twiddle multiplications: exactly (N/2) log N butterfly products in total;
//   the last pass reads 8 rows (adjacent K_1) and stores transposed, 8 consecutive outputs per K_P.
// Twiddles come from one universal per-stage table tab[2^(u-1) + j] = w_{2^u}^j (u <= log_n) that is
// shared by every domain size under the same root (w_{2^u} = ROOT_OF_UNITY^(2^(28-u)) for all k).
// Fused: zero padding + zeta^i coset pre-scaling on load (coeff_to_extended), n^-1 and zeta^-i
// post-scaling on the final store (ifft / extended_to_coeff).
// Part transforms (ntt_part_run, DESIGN.md "Quotient construction") are separate instantiations (Tw = PartTwist) that
// also scale by w_ext^(part*i) on load or by its inverse on store; the plain instantiations (Tw = NoTwist) are unchanged.
#include <type_traits>

#include "common.cuh"

namespace b200zk {

static constexpr int NTT_THREADS = 256;   // 3 blocks/SM: 85 registers per thread, 72 KiB shared memory per block
static constexpr int NTT_MAX_DIGIT = 8;

struct Fr3 {
    Fr c[3];
};

struct NttPass {
    uint32_t log_n, P, p;
    uint32_t dig[4];
    uint32_t t;       // bits above this digit (already transformed)
    uint32_t m;       // this digit
    uint32_t rest;    // bits below this digit
    uint32_t log_in;  // pass 0: source has 2^log_in elements, the rest is implicit zero
    int pre, post;
};

__device__ __forceinline__ Fr sel3(const Fr3& t, uint32_t r) {  // no dynamic indexing of kernel params
    Fr o;
#pragma unroll
    for (int i = 0; i < 8; ++i) o.l.v[i] = r == 0 ? t.c[0].l.v[i] : (r == 1 ? t.c[1].l.v[i] : t.c[2].l.v[i]);
    return o;
}

// The twist of part r of the extended coset: element i is scaled by u^(r*i mod 2^ext_k), u = w_ext on a forward transform's
// load and u = w_ext^-1 on an inverse transform's store.  u^e comes from the level-ext_k run of the universal twiddle table
// of u's family (u^j for j < 2^(ext_k-1); the upper half by u^(j + 2^(ext_k-1)) = -u^j), the table that coeff_to_extended /
// extended_to_coeff keep anyway and whose level-k run is also the n-point transform's: no per-part table is built.
struct NoTwist {};
struct PartTwist {
    const Fr* wtab;   // u^j, j < 2^(ext_k - 1)
    uint64_t mask;    // 2^ext_k - 1
    uint64_t part;
    int pre, post;
};

struct LevelRoots {
    Fr w[29];  // w[u] = primitive 2^u-th root
};

__device__ __forceinline__ Fr ld_fr(const Fr* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = q[0], b = q[1];
    Fr r;
    r.l.v[0] = a.x; r.l.v[1] = a.y; r.l.v[2] = a.z; r.l.v[3] = a.w;
    r.l.v[4] = b.x; r.l.v[5] = b.y; r.l.v[6] = b.z; r.l.v[7] = b.w;
    return r;
}
__device__ __forceinline__ Fr ldg_fr(const Fr* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    Fr r;
    r.l.v[0] = a.x; r.l.v[1] = a.y; r.l.v[2] = a.z; r.l.v[3] = a.w;
    r.l.v[4] = b.x; r.l.v[5] = b.y; r.l.v[6] = b.z; r.l.v[7] = b.w;
    return r;
}
__device__ __forceinline__ Fr part_root(const PartTwist& tw, uint64_t e) {  // u^e, e <= mask
    const uint64_t half = (tw.mask + 1) >> 1;
    Fr w = ldg_fr(tw.wtab + (e & (half - 1)));
    if (e >= half) w = Fr::zero() - w;
    return w;
}
__device__ __forceinline__ void st_fr(Fr* p, const Fr& r) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4(r.l.v[0], r.l.v[1], r.l.v[2], r.l.v[3]);
    q[1] = make_uint4(r.l.v[4], r.l.v[5], r.l.v[6], r.l.v[7]);
}
__device__ __forceinline__ Fr ld_sm(const uint4* lo, const uint4* hi, uint32_t i) {
    uint4 a = lo[i], b = hi[i];
    Fr r;
    r.l.v[0] = a.x; r.l.v[1] = a.y; r.l.v[2] = a.z; r.l.v[3] = a.w;
    r.l.v[4] = b.x; r.l.v[5] = b.y; r.l.v[6] = b.z; r.l.v[7] = b.w;
    return r;
}
__device__ __forceinline__ void st_sm(uint4* lo, uint4* hi, uint32_t i, const Fr& r) {
    lo[i] = make_uint4(r.l.v[0], r.l.v[1], r.l.v[2], r.l.v[3]);
    hi[i] = make_uint4(r.l.v[4], r.l.v[5], r.l.v[6], r.l.v[7]);
}

// tab[e], e = 2^(u-1) + j  ->  w_{2^u}^j
__global__ void ntt_build_table(Fr* tab, LevelRoots roots, uint32_t log_n) {
    uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t total = 1ull << log_n;
    if (e >= total) return;
    if (e == 0) {
        st_fr(tab, Fr::one());
        return;
    }
    uint32_t u = 64 - __clzll(e);  // e in [2^(u-1), 2^u)
    uint32_t j = (uint32_t)(e - (1ull << (u - 1)));
    Fr base = roots.w[u], acc = Fr::one();
    while (j) {
        if (j & 1) acc = acc * base;
        base = base.sqr();
        j >>= 1;
    }
    st_fr(tab + e, acc);
}

// One pass over one tile.  C = lanes per tile (8, or 1 for the single-pass small transform).
template <int C, bool LAST, class Tw = NoTwist>
__global__ void __launch_bounds__(NTT_THREADS, 3)
ntt_pass_kernel(const Fr* __restrict__ in, Fr* __restrict__ out, const Fr* __restrict__ tab, NttPass ps, Fr3 pre_c,
                Fr3 post_c, Tw tw) {
    constexpr bool TWIST = !std::is_same<Tw, NoTwist>::value;
    extern __shared__ uint4 smem[];
    const uint32_t m = ps.m, L = 1u << m, E = L * C;
    uint4* lo = smem;
    uint4* hi = smem + E;
    uint4* twlo = hi + E;   // !LAST only: L entries
    uint4* twhi = twlo + L;
    const uint32_t tid = threadIdx.x, NT = blockDim.x;
    const uint32_t t = ps.t, rest = ps.rest, n = ps.log_n;
    const uint32_t swz_shift = (C == 8 && m >= 3) ? (m - 3) : 31;
    auto idx = [&](uint32_t pos, uint32_t lane) -> uint32_t {
        if (C == 8) return pos * C + (lane ^ ((pos >> swz_shift) & 7u));
        return pos;
    };

    uint64_t base;        // !LAST: global index of (d = 0, lane = 0)
    uint32_t c;           // twist of lane 0
    uint64_t rowstride = 0;
    if (!LAST) {
        uint32_t groups_log = rest - 3;  // 2^rest / 8 lane groups
        uint64_t tile = blockIdx.x;
        uint64_t o = tile >> groups_log, g = tile & ((1ull << groups_log) - 1);
        base = (o << (n - t)) + g * C;
        // c = digit reversal of o: o = [K_1][K_2]..[K_{p}] positionally (K_1 most significant)
        uint32_t sh = t, tq = 0;
        c = 0;
        for (uint32_t q = 0; q < ps.p; ++q) {
            sh -= ps.dig[q];
            uint32_t kq = (uint32_t)(o >> sh) & ((1u << ps.dig[q]) - 1);
            c |= kq << tq;
            tq += ps.dig[q];
        }
    } else {
        c = blockIdx.x * C;  // c0
        // row position of twist c: K_q sits at bit offset n - t_q - n_q
        uint32_t tq = 0;
        uint64_t pos = 0;
        for (uint32_t q = 0; q + 1 < ps.P; ++q) {
            uint32_t kq = (c >> tq) & ((1u << ps.dig[q]) - 1);
            tq += ps.dig[q];
            pos |= (uint64_t)kq << (n - tq);
        }
        base = pos;
        rowstride = (ps.P > 1) ? (1ull << (n - ps.dig[0])) : 0;
    }

    // ---- load (bit-reversed digit position), fused zero padding + coset pre-scaling on pass 0.
    // zskip: coeff_to_extended pads a 2^k vector to 2^(k+2); in pass 0 only digit entries d < L/4 are non-zero and
    // the first two DIT stages merely replicate them 4x, so those entries are written to 4 positions and the
    // butterfly network starts at stage 3 (saves 2 of log_n butterfly stages and 3/4 of the loads).
    const uint64_t in_len = 1ull << ps.log_in;
    const bool zskip = (ps.p == 0) && (ps.log_in + 2 == n) && (m >= 2);
    const uint32_t E_load = zskip ? (E >> 2) : E, L_load = zskip ? (L >> 2) : L;
    for (uint32_t e = tid; e < E_load; e += NT) {
        uint32_t lane, d;
        uint64_t gi;
        if (!LAST) {
            lane = e % C;
            d = e / C;
            gi = base + ((uint64_t)d << rest) + lane;
        } else {
            d = e & (L_load - 1);
            lane = e / L_load;
            gi = base + lane * rowstride + d;
        }
        Fr v;
        if (ps.p == 0 && gi >= in_len) {
            v = Fr::zero();
        } else {
            v = ld_fr(in + gi);
            if (ps.p == 0 && ps.pre) {
                uint32_t r3 = (uint32_t)(gi % 3);
                if (r3) v = v * sel3(pre_c, r3);
            }
            if constexpr (TWIST) {
                if (ps.p == 0 && tw.pre) {
                    const uint64_t e = (tw.part * gi) & tw.mask;
                    if (e) v = v * part_root(tw, e);
                }
            }
        }
        uint32_t pos = __brev(d) >> (32 - m);
        if (zskip) {
#pragma unroll
            for (uint32_t r = 0; r < 4; ++r) st_sm(lo, hi, idx(pos + r, lane), v);
        } else {
            st_sm(lo, hi, idx(pos, lane), v);
        }
    }
    if (!LAST) {
        for (uint32_t j = tid; j < L; j += NT) {
            if (j == 0) continue;
            uint32_t s = 32 - __clz(j);  // j in [2^(s-1), 2^s)
            uint32_t K = j - (1u << (s - 1));
            uint64_t src = (1ull << (t + s - 1)) + ((uint64_t)K << t) + c;
            Fr w = ldg_fr(tab + src);
            st_sm(twlo, twhi, j, w);
        }
    }
    __syncthreads();

    // ---- DIT stages, two per barrier (radix-4 groups held in registers), a final radix-2 stage if m is odd
    auto twiddle = [&](uint32_t s, uint32_t K, uint32_t lane, Fr& w) -> bool {  // false when the twiddle is 1
        if (!LAST) {
            if (K == 0 && c == 0) return false;
            w = ld_sm(twlo, twhi, (1u << (s - 1)) + K);
            return true;
        }
        uint64_t j = ((uint64_t)K << t) + c + lane;
        if (j == 0) return false;
        w = ldg_fr(tab + (1ull << (t + s - 1)) + j);
        return true;
    };
    uint32_t s = zskip ? 3 : 1;
    for (; s + 1 <= m; s += 2) {
        const uint32_t h = 1u << (s - 1);
        const uint32_t ng = (L >> 2) * C;
        for (uint32_t q = tid; q < ng; q += NT) {
            uint32_t lane = q % C, gq = q / C;
            uint32_t K = gq & (h - 1), blk = gq >> (s - 1);
            uint32_t p = (blk << (s + 1)) + K;
            uint32_t i0 = idx(p, lane), i1 = idx(p + h, lane), i2 = idx(p + 2 * h, lane), i3 = idx(p + 3 * h, lane);
            Fr a = ld_sm(lo, hi, i0), b = ld_sm(lo, hi, i1), cc = ld_sm(lo, hi, i2), d = ld_sm(lo, hi, i3);
            Fr w;
            if (twiddle(s, K, lane, w)) {  // stage s: (a,b) and (cc,d) share w_s[K]
                b = b * w;
                d = d * w;
            }
            Fr a1 = a + b, b1 = a - b, c1 = cc + d, d1 = cc - d;
            if (twiddle(s + 1, K, lane, w)) c1 = c1 * w;  // stage s+1: (a1,c1) with w_{s+1}[K]
            twiddle(s + 1, K + h, lane, w);               //            (b1,d1) with w_{s+1}[K+h]  (never 1)
            d1 = d1 * w;
            st_sm(lo, hi, i0, a1 + c1);
            st_sm(lo, hi, i2, a1 - c1);
            st_sm(lo, hi, i1, b1 + d1);
            st_sm(lo, hi, i3, b1 - d1);
        }
        // (measured: replacing this barrier by __syncwarp / 128-thread named barriers for the warp-local early stages
        //  gave -1 % at 2^24 and +5 % at 2^26, so the plain block barrier stays)
        __syncthreads();
    }
    if (s == m) {
        const uint32_t half = 1u << (s - 1);
        const uint32_t nb = (L >> 1) * C;
        for (uint32_t b = tid; b < nb; b += NT) {
            uint32_t lane = b % C, bb = b / C;
            uint32_t K = bb & (half - 1), blk = bb >> (s - 1);
            uint32_t p0 = (blk << s) + K, p1 = p0 + half;
            uint32_t i0 = idx(p0, lane), i1 = idx(p1, lane);
            Fr u = ld_sm(lo, hi, i0), v = ld_sm(lo, hi, i1), w;
            if (twiddle(s, K, lane, w)) v = v * w;
            st_sm(lo, hi, i0, u + v);
            st_sm(lo, hi, i1, u - v);
        }
        __syncthreads();
    }

    // ---- store
    for (uint32_t e = tid; e < E; e += NT) {
        uint32_t lane = e % C, K = e / C;
        Fr v = ld_sm(lo, hi, idx(K, lane));
        uint64_t go;
        if (!LAST) {
            go = base + ((uint64_t)K << rest) + lane;
        } else {
            go = ((uint64_t)K << t) + c + lane;
            if (ps.post) v = v * sel3(post_c, (uint32_t)(go % 3));
            if constexpr (TWIST) {
                if (tw.post) {
                    const uint64_t e = (tw.part * go) & tw.mask;
                    if (e) v = v * part_root(tw, e);
                }
            }
        }
        st_fr(out + go, v);
    }
}

// ---------------------------------------------------------------------------------------------
static Fr host_halve(const Fr& x) {  // x/2 mod r (linear, so valid on Montgomery limbs too)
    Fr r = x;
    uint32_t carry = 0;
    if (x.l.v[0] & 1) {
        uint32_t m[8];
        Fr::modulus(m);
        carry = leaf::add8(r.l.v, x.l.v, m);
    }
    for (int i = 0; i < 8; ++i) {
        uint32_t nxt = (i < 7) ? r.l.v[i + 1] : carry;
        r.l.v[i] = (r.l.v[i] >> 1) | (nxt << 31);
    }
    return r;
}

Fr host_zeta() {  // halo2curves Fr::ZETA in Montgomery form
    Fr z;
    const uint32_t v[8] = {0x55fcd653u, 0x0363f299u, 0x5fc1e200u, 0x73e7950bu,
                           0x576d9d24u, 0xc5fce83eu, 0xa1c3a4d4u, 0x059c805du};
    for (int i = 0; i < 8; ++i) z.l.v[i] = v[i];
    return z;
}

int32_t ntt_get_table(b200zk_ctx* ctx, const Fr& omega, uint32_t log_n, const Fr** out) {
    // level roots w[u] = omega^(2^(log_n-u)); validate primitivity
    LevelRoots roots;
    roots.w[log_n] = omega;
    for (uint32_t u = log_n; u > 0; --u) roots.w[u - 1] = roots.w[u].sqr();
    Fr minus_one = Fr::zero() - Fr::one();
    if (!(roots.w[0] == Fr::one()) || (log_n >= 1 && !(roots.w[1] == minus_one)))
        return fail(ctx, B200ZK_E_INVALID, "omega is not a primitive 2^%u-th root of unity", log_n);
    for (auto& tt : ctx->tables) {
        if (tt.log_n < log_n) continue;
        Fr w = tt.omega;
        for (uint32_t i = tt.log_n; i > log_n; --i) w = w.sqr();
        if (w == omega) {
            *out = tt.dev;
            return B200ZK_OK;
        }
    }
    // build (replace a smaller table of the same family if present)
    for (size_t i = 0; i < ctx->tables.size(); ++i) {
        Fr w = omega;
        bool same = false;
        if (ctx->tables[i].log_n < log_n) {
            for (uint32_t k = log_n; k > ctx->tables[i].log_n; --k) w = w.sqr();
            same = (w == ctx->tables[i].omega);
        }
        if (same) {
            B2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            B2_CUDA(ctx, cudaFree(ctx->tables[i].dev));
            ctx->tables.erase(ctx->tables.begin() + i);
            break;
        }
    }
    for (uint32_t u = log_n + 1; u < 29; ++u) roots.w[u] = Fr::one();
    Fr* dev = nullptr;
    size_t bytes = sizeof(Fr) << log_n;
    cudaError_t e = cudaMalloc(&dev, bytes);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(ctx, B200ZK_E_OOM, "twiddle table cudaMalloc(%zu) failed", bytes);
    }
    uint64_t total = 1ull << log_n;
    uint32_t tpb = 256;
    uint32_t blocks = (uint32_t)((total + tpb - 1) / tpb);
    {
        ProfScope ps(ctx, PROF_NTT_TABLE);
        ntt_build_table<<<blocks, tpb, 0, ctx->stream>>>(dev, roots, log_n);
    }
    B2_LAUNCH_CHECK(ctx);
    ctx->tables.push_back({omega, log_n, dev});
    *out = dev;
    return B200ZK_OK;
}

static void plan_digits(uint32_t log_n, uint32_t* P, uint32_t dig[4]) {
    if (log_n <= NTT_MAX_DIGIT) {
        *P = 1;
        dig[0] = log_n;
        dig[1] = dig[2] = dig[3] = 0;
        return;
    }
    uint32_t p = (log_n + NTT_MAX_DIGIT - 1) / NTT_MAX_DIGIT;
    *P = p;
    uint32_t basebits = log_n / p, extra = log_n % p;
    for (uint32_t i = 0; i < 4; ++i) dig[i] = (i < p) ? basebits + (i < extra ? 1 : 0) : 0;
}

template <int C, bool LAST, class Tw>
static int32_t launch_pass(b200zk_ctx* ctx, const Fr* in, Fr* out, const Fr* tab, const NttPass& ps, const Fr3& pre_c,
                           const Fr3& post_c, const Tw& tw) {
    uint32_t L = 1u << ps.m, E = L * C;
    size_t smem = (size_t)(2 * E + (LAST ? 0 : 2 * L)) * sizeof(uint4);
    // bits 0-3: plain instantiations, bits 9-12: part-twist instantiations (bit 8 is the graph kernel's)
    const uint32_t optin_bit = 1u << ((C == 8 ? 0 : 2) + (LAST ? 1 : 0) + (std::is_same<Tw, NoTwist>::value ? 0 : 9));
    if (!(ctx->smem_optin & optin_bit)) {
        B2_CUDA(ctx, cudaFuncSetAttribute(ntt_pass_kernel<C, LAST, Tw>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)((2 * (1u << NTT_MAX_DIGIT) * C + 2 * (1u << NTT_MAX_DIGIT)) * sizeof(uint4))));
        ctx->smem_optin |= optin_bit;
    }
    uint64_t tiles = (1ull << ps.log_n) / E;
    uint32_t nb = (L >> 2) * C;  // radix-4 groups per double stage
    uint32_t threads = nb >= NTT_THREADS ? NTT_THREADS : (nb < 32 ? 32 : nb);
    {
        ProfScope psc(ctx, PROF_NTT_PASS);
        ntt_pass_kernel<C, LAST, Tw><<<(uint32_t)tiles, threads, smem, ctx->stream>>>(in, out, tab, ps, pre_c, post_c, tw);
    }
    B2_LAUNCH_CHECK(ctx);
    return B200ZK_OK;
}

// the pass sequence of one transform: a single pass up to 2^8 elements, else P passes through ctx->ntt_work
template <class Tw>
static int32_t ntt_passes(b200zk_ctx* ctx, const Fr* in, uint32_t log_in, Fr* out, uint32_t log_n, const Fr* tab, int pre, int post,
                          const Fr3& pre_c, const Fr3& post_c, const Tw& tw) {
    NttPass ps;
    memset(&ps, 0, sizeof ps);
    ps.log_n = log_n;
    plan_digits(log_n, &ps.P, ps.dig);
    if (ps.P == 1) {
        ps.p = 0;
        ps.t = 0;
        ps.m = log_n;
        ps.rest = 0;
        ps.log_in = log_in;
        ps.pre = pre;
        ps.post = post;
        return launch_pass<1, true>(ctx, in, out, tab, ps, pre_c, post_c, tw);
    }
    size_t bytes = sizeof(Fr) << log_n;
    B2_TRY(scratch_reserve(ctx, ctx->ntt_work, bytes));
    Fr* W = (Fr*)ctx->ntt_work.p;
    uint32_t t = 0;
    for (uint32_t p = 0; p < ps.P; ++p) {
        ps.p = p;
        ps.t = t;
        ps.m = ps.dig[p];
        ps.rest = log_n - t - ps.m;
        ps.log_in = (p == 0) ? log_in : log_n;
        ps.pre = (p == 0) ? pre : 0;
        ps.post = (p + 1 == ps.P) ? post : 0;
        if (p + 1 < ps.P)
            B2_TRY((launch_pass<8, false>(ctx, p == 0 ? in : W, W, tab, ps, pre_c, post_c, tw)));
        else
            B2_TRY((launch_pass<8, true>(ctx, W, out, tab, ps, pre_c, post_c, tw)));
        t += ps.m;
    }
    return B200ZK_OK;
}

int32_t ntt_run(b200zk_ctx* ctx, const Fr* in, uint32_t log_in, Fr* out, uint32_t log_n, const Fr& omega,
                int inverse_scale, int coset_mode) {
    if (log_n > 28) return fail(ctx, B200ZK_E_INVALID, "log_n %u exceeds Fr two-adicity 28", log_n);
    if (log_in > log_n) return fail(ctx, B200ZK_E_INVALID, "log_in %u > log_n %u", log_in, log_n);
    if (coset_mode < 0 || coset_mode > 2) return fail(ctx, B200ZK_E_INVALID, "bad coset_mode %d", coset_mode);
    if (log_n == 0) {  // length-1 transform is the identity (times 1)
        if (in != out) B2_CUDA(ctx, cudaMemcpyAsync(out, in, sizeof(Fr), cudaMemcpyDeviceToDevice, ctx->stream));
        return B200ZK_OK;
    }
    const Fr* tab = nullptr;
    B2_TRY(ntt_get_table(ctx, omega, log_n, &tab));

    Fr zeta = host_zeta(), zeta2 = zeta.sqr();
    Fr3 pre_c, post_c;
    pre_c.c[0] = Fr::one();
    pre_c.c[1] = zeta;
    pre_c.c[2] = zeta2;
    Fr scale = Fr::one();
    if (inverse_scale)
        for (uint32_t i = 0; i < log_n; ++i) scale = host_halve(scale);
    post_c.c[0] = scale;
    post_c.c[1] = (coset_mode == B200ZK_COSET_POST) ? scale * zeta2 : scale;
    post_c.c[2] = (coset_mode == B200ZK_COSET_POST) ? scale * zeta : scale;
    const int pre = (coset_mode == B200ZK_COSET_PRE), post = (inverse_scale || coset_mode == B200ZK_COSET_POST);
    return ntt_passes(ctx, in, log_in, out, log_n, tab, pre, post, pre_c, post_c, NoTwist{});
}

Fr host_root_of_unity(uint32_t log_n) {  // halo2curves Fr::ROOT_OF_UNITY^(2^(28 - log_n)): EvaluationDomain's omega of a 2^log_n domain
    Fr w;
    const uint32_t v[8] = {0xb639feb8u, 0x9632c7c5u, 0x0d0ff299u, 0x985ce340u, 0x01b0ecd8u, 0xb2dd8800u, 0x6d98ce29u, 0x1d69070du};
    for (int i = 0; i < 8; ++i) w.l.v[i] = v[i];
    for (uint32_t i = log_n; i < 28; ++i) w = w.sqr();
    return w;
}

// Part `part` of the extended coset zeta * <w_ext> (2^ext_k points), i.e. the n = 2^k points g * w^i, g = zeta * w_ext^part:
//   forward (coeff_to_extended_part):  out[i] = sum_m in[m] g^m w^(im)           (pre-scale by zeta^(m mod 3) w_ext^(part*m))
//   inverse (the first half of extended_parts_to_coeff):  out[m] = scale * g^-m * n^-1 * sum_i in[i] w^(-im)
// Both are one n-point transform with the twist fused into its first load / last store.  in == out is allowed.
int32_t ntt_part_run(b200zk_ctx* ctx, const Fr* in, Fr* out, uint32_t k, uint32_t ext_k, uint32_t part, bool inverse,
                     const Fr& scale) {
    Fr u = host_root_of_unity(ext_k);
    if (inverse) u = u.inv();
    const Fr* tab = nullptr;
    B2_TRY(ntt_get_table(ctx, u, ext_k, &tab));
    PartTwist tw;
    tw.wtab = tab + (1ull << (ext_k - 1));
    tw.mask = (1ull << ext_k) - 1;
    tw.part = part;
    tw.pre = !inverse;
    tw.post = inverse;
    Fr zeta = host_zeta(), zeta2 = zeta.sqr();
    Fr3 pre_c, post_c;
    pre_c.c[0] = Fr::one();
    pre_c.c[1] = zeta;
    pre_c.c[2] = zeta2;
    Fr s = scale;
    if (inverse)
        for (uint32_t i = 0; i < k; ++i) s = host_halve(s);
    post_c.c[0] = s;
    post_c.c[1] = s * zeta2;
    post_c.c[2] = s * zeta;
    return ntt_passes(ctx, in, k, out, k, tab, inverse ? 0 : 1, inverse ? 1 : 0, pre_c, post_c, tw);
}

}  // namespace b200zk
