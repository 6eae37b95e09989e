/*
 * b200zk — C ABI of the B200-native Halo2/KZG polynomial-arithmetic backend.
 *
 * This is the drop-in boundary for the ONE hot path of scroll-prover (SURVEY.md §8(b)): the
 * functions a patched `halo2_proofs` crate binds over FFI in place of its Rayon CPU arithmetic.
 * The reference selects its GPU backend by whole-crate substitution of halo2_proofs
 * (/root/reference/docker/chain-prover/gpu/Dockerfile:7, /root/reference/Cargo.toml:33-45);
 * INTEGRATION.md shows the Rust `extern "C"` stub that replaces each halo2_proofs function body.
 *
 * Conventions
 *  - every entry point returns int32: B200ZK_OK (0) or a negative B200ZK_E_*; it never aborts and
 *    never throws across the boundary; b200zk_last_error(ctx) returns the message of the last
 *    failure on that context (the reference's Rust side turns it into the panic/assert it had).
 *  - field elements are raw Montgomery limbs, memcpy-compatible with halo2curves 0.1.0
 *    `Fr([u64;4])` / `Fq([u64;4])`; points are `G1Affine{x,y}` (64 B, identity = (0,0)) and
 *    `G1{x,y,z}` Jacobian (96 B, identity z = 0)            (pin: /root/reference/Cargo.lock:1911-1913).
 *  - every data pointer may be a host pointer OR a device pointer (detected with
 *    cudaPointerGetAttributes); host inputs are copied to device staging buffers inside the call and are no
 *    longer read once the call returns (pageable or pinned alike), host outputs are complete on return;
 *    results delivered to DEVICE pointers are ordered on the context stream (b200zk_ctx_synchronize to wait).
 *  - one context per process per GPU (one process per GPU is the deployment model); a context is
 *    safe to call from several host threads (calls serialise on the context's stream).
 *  - there is NO CPU fallback: without a CUDA device b200zk_ctx_create fails with B200ZK_E_CUDA.
 */
#ifndef B200ZK_H
#define B200ZK_H
#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define B200ZK_API __attribute__((visibility("default")))
#else
#define B200ZK_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define B200ZK_OK 0
#define B200ZK_E_INVALID (-1)   /* bad argument (the reference would assert/panic) */
#define B200ZK_E_CUDA (-2)      /* CUDA runtime / launch failure, or no device */
#define B200ZK_E_OOM (-3)       /* device or pinned-host allocation failed */
#define B200ZK_E_UNSUPPORTED (-4)

typedef struct b200zk_ctx b200zk_ctx;
typedef struct b200zk_srs b200zk_srs;

/* SRS tags: which ParamsKZG vector the bases are (commit vs commit_lagrange) */
#define B200ZK_SRS_G 0u
#define B200ZK_SRS_G_LAGRANGE 1u

/* coset_mode of b200zk_ntt_fr */
#define B200ZK_COSET_NONE 0      /* plain best_fft */
#define B200ZK_COSET_PRE 1       /* a[i] *= zeta^i before the transform  (coeff_to_extended) */
#define B200ZK_COSET_POST 2      /* a[i] *= zeta^-i after the transform  (extended_to_coeff) */

/* ---- context ------------------------------------------------------------------------------- */
/* devices/n_devices: CUDA ordinals this context drives; this build drives exactly one per context
 * (n_devices == 1).  Multi-GPU = one process and one context per GPU; the contexts of a job are joined into one
 * NCCL communicator with b200zk_ctx_comm_init below (the context owns the communicator). */
B200ZK_API int32_t b200zk_ctx_create(const int* devices, int n_devices, b200zk_ctx** out);
B200ZK_API int32_t b200zk_ctx_destroy(b200zk_ctx* ctx);
B200ZK_API const char* b200zk_last_error(const b200zk_ctx* ctx);
/* Run all work of this context on the caller's CUDA stream (cudaStream_t cast to void*), e.g. the
 * current torch stream, so the caller's CUDA events bracket our kernels.  NULL = own stream. */
B200ZK_API int32_t b200zk_ctx_set_stream(b200zk_ctx* ctx, void* cuda_stream);
B200ZK_API int32_t b200zk_ctx_synchronize(b200zk_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
B200ZK_API int32_t b200zk_ctx_launch_count(const b200zk_ctx* ctx, uint64_t* out);

/* ---- multi-GPU: context-owned NCCL communicator (SURVEY.md §8(b), §8(e)) ------------------------ */
/* Rank 0 obtains a 128-byte NCCL unique id and hands it to the other ranks over whatever channel the caller already
 * has (the prover's RPC, MPI, a shared file ...); every rank then joins with its rank / world size.
 * world == 1 is allowed (no communicator; the sharded entry points degenerate to the single-GPU ones).
 * Collective: all ranks must call b200zk_ctx_comm_init, and later the *_sharded entry points, in the same order. */
B200ZK_API int32_t b200zk_comm_unique_id(void* id128);
B200ZK_API int32_t b200zk_ctx_comm_init(b200zk_ctx* ctx, const void* id128, int rank, int world);
B200ZK_API int32_t b200zk_ctx_comm_info(const b200zk_ctx* ctx, int* rank, int* world);
/* the contiguous slice [first, first + count) of n points that `rank` of `world` owns (sizes differ by <= 1) */
B200ZK_API int32_t b200zk_shard_range(uint64_t n, int rank, int world, uint64_t* first, uint64_t* count);

/* ---- device buffers (lets a caller keep columns resident between calls; SURVEY.md §8(f).1) --- */
B200ZK_API int32_t b200zk_buf_alloc(b200zk_ctx* ctx, uint64_t bytes, void** out_dev);
B200ZK_API int32_t b200zk_buf_free(b200zk_ctx* ctx, void* dev);
B200ZK_API int32_t b200zk_buf_upload(b200zk_ctx* ctx, void* dev, const void* host, uint64_t bytes);
B200ZK_API int32_t b200zk_buf_download(b200zk_ctx* ctx, void* host, const void* dev, uint64_t bytes);

/* ---- SRS ------------------------------------------------------------------------------------ */
/* Replaces holding `ParamsKZG::g` / `g_lagrange` on the host (halo2_proofs/src/poly/kzg/commitment.rs;
 * reference call sites /root/reference/bin/src/trace_prover.rs:35-36, integration/src/prove.rs:12):
 * uploads n affine bases once; they stay resident for the life of the handle. */
B200ZK_API int32_t b200zk_srs_register(b200zk_ctx* ctx, const void* g1_affine, uint64_t n, uint32_t tag, b200zk_srs** out);
/* mode 1 (default): handles of >= 2^16 points also keep the multiples 2^(c*w) P_i of every base (W x the
 * storage, built once at registration) when device memory allows, so all Pippenger windows share one bucket
 * set; mode 0: plain bases only.  Applies to subsequent b200zk_srs_register calls. */
B200ZK_API int32_t b200zk_srs_set_precompute(b200zk_ctx* ctx, int mode);
B200ZK_API int32_t b200zk_srs_release(b200zk_ctx* ctx, b200zk_srs* srs);
B200ZK_API int32_t b200zk_srs_len(const b200zk_srs* srs, uint64_t* out);

/* ---- MSM ------------------------------------------------------------------------------------ */
/* Replaces halo2_proofs::arithmetic::best_multiexp(coeffs, bases) and therefore
 * ParamsKZG::commit / commit_lagrange (halo2_proofs/src/arithmetic.rs, poly/kzg/commitment.rs @ e5ddf67,
 * pin /root/reference/Cargo.lock:1886-1888; reached from /root/reference/integration/src/prove.rs:37-39).
 * result = sum_{i<n} scalars[i] * srs[i] as a normalised Jacobian point (x, y, 1), or (0, 1, 0) for the
 * identity.  n must be <= the SRS length (commit over the first n bases); n == 0 gives the identity. */
B200ZK_API int32_t b200zk_msm_g1(b200zk_ctx* ctx, const b200zk_srs* srs, const void* scalars, uint64_t n, void* out_jacobian96);
/* `count` commitments over the SAME bases in one call: scalars[j] points to n scalars (host or device, independently),
 * out_jacobian96 receives count x 96 B.  Columns go through the Pippenger pipeline in batches whose bucket sets lie side
 * by side, so the latency-bound phases (scans, bucket reduction, final Horner) are paid once per batch -- the case of
 * the several hundred 2^20-row columns of the inner (zkEVM super-circuit) proof.  Same results as count b200zk_msm_g1 calls. */
B200ZK_API int32_t b200zk_msm_g1_batch(b200zk_ctx* ctx, const b200zk_srs* srs, const void* const* scalars, uint32_t count, uint64_t n,
                                       void* out_jacobian96);
/* same with explicit bases (generic best_multiexp; bases are uploaded for the call) */
B200ZK_API int32_t b200zk_msm_g1_bases(b200zk_ctx* ctx, const void* g1_affine, const void* scalars, uint64_t n, void* out_jacobian96);
/* partial MSM over the slice [first, first + n) of the registered bases: sum_{i<n} scalars[i] * srs[first + i]
 * (precomputed tables are used in place -- a slice of them has the same layout).  Building block of the sharded MSM. */
B200ZK_API int32_t b200zk_msm_g1_range(b200zk_ctx* ctx, const b200zk_srs* srs, const void* scalars, uint64_t first, uint64_t n,
                                       void* out_jacobian96);
/* best_multiexp over n_total points SHARDED BY POINT RANGE across the ranks of the context's communicator (BASELINE
 * configs[3]): every rank holds the full SRS handle and passes ONLY its slice of the scalars
 * (b200zk_shard_range(n_total, rank, world)); it computes the partial sum of its slice, the 96-byte partials are
 * exchanged with one ncclAllGather on the context stream and summed locally.  Every rank receives the same normalised
 * point -- the bytes of the single-GPU result. */
B200ZK_API int32_t b200zk_msm_g1_sharded(b200zk_ctx* ctx, const b200zk_srs* srs, const void* scalars_slice, uint64_t n_total,
                                         void* out_jacobian96);
/* sum of `count` Jacobian points (combining per-GPU partial MSMs after the NCCL all-gather) */
B200ZK_API int32_t b200zk_g1_sum(b200zk_ctx* ctx, const void* jacobian_points, uint64_t count, void* out_jacobian96);
/* out[i] = scalars[i] * G1 generator, affine (ParamsKZG::setup's g / g_lagrange generation) */
B200ZK_API int32_t b200zk_g1_generator_mul_batch(b200zk_ctx* ctx, const void* scalars, uint64_t n, void* out_affine);

/* ---- FFT over G1 (SRS tooling) --------------------------------------------------------------- */
/* Replaces halo2_proofs::arithmetic::best_fft::<Fr, G1>(a, omega, log_n): in place on 2^log_n Jacobian points
 * (96 B each, results normalised). */
B200ZK_API int32_t b200zk_fft_g1(b200zk_ctx* ctx, void* jacobian_points, uint32_t log_n, const void* omega32);
/* Replaces poly::kzg::commitment::g_to_lagrange(g, k) as used by Params::downsize
 * (/root/reference/integration/tests/integration.rs:17-18): g_lagrange = iFFT_G1(g) / n, affine in, affine out. */
B200ZK_API int32_t b200zk_g_to_lagrange(b200zk_ctx* ctx, const void* g_affine, uint32_t k, void* out_affine);

/* ---- NTT ------------------------------------------------------------------------------------ */
/* Replaces halo2_proofs::arithmetic::best_fft::<Fr, Fr>(a, omega, log_n) (arithmetic.rs @ e5ddf67):
 * in place, natural order in and out, a.len() == 1 << log_n, A[j] = sum_i a[i] omega^(ij).
 * inverse_scale != 0 additionally multiplies every output by (2^log_n)^-1 (EvaluationDomain::ifft).
 * coset_mode fuses distribute_powers_zeta (poly/domain.rs): PRE for coeff_to_extended, POST for
 * extended_to_coeff.  omega must be a primitive 2^log_n-th root of unity (32 B Montgomery). */
B200ZK_API int32_t b200zk_ntt_fr(b200zk_ctx* ctx, void* data, uint32_t log_n, const void* omega32, int inverse_scale, int coset_mode);
/* Out-of-place form with zero padding: in has 2^log_in elements (log_in <= log_n), out has 2^log_n.
 * EvaluationDomain::coeff_to_extended == (log_in = k, log_n = extended_k, omega = extended_omega, PRE). */
B200ZK_API int32_t b200zk_ntt_fr_ext(b200zk_ctx* ctx, const void* in, uint32_t log_in, void* out, uint32_t log_n,
                          const void* omega32, int inverse_scale, int coset_mode);

/* ---- device-resident column pipeline (the per-column work of plonk::create_proof) ---------------- */
/* For each of `count` columns of 2^k Lagrange values in HOST memory (pinned => the H2D copy of column j+1 overlaps the
 * kernels of column j on an internal copy stream; pageable works too):
 *   mode 0: commit_lagrange / commit only            (commits_out[j] = MSM over the first 2^k bases of `srs`)
 *   mode 1: + lagrange_to_coeff   into coeff_out_dev[j] (device, 2^k elements)  or an internal scratch when NULL
 *   mode 2: + coeff_to_extended   into ext_out_dev[j]   (device, 2^extended_k)  or an internal scratch when NULL
 *   mode 3: lagrange_to_coeff + coeff_to_extended only (no commitment; srs and commits_out may be NULL) -- lets a
 *           multi-GPU caller place a column's MSM and its transforms on different ranks
 * commits_out: count x 96 B normalised Jacobian points (host or device).  No host synchronisation inside the loop;
 * one D2H of the commitments at the end.  Replaces the per-column sequence in halo2_proofs/src/plonk/prover.rs.
 * Jobs are processed in groups (up to 16 small columns): the upload of group g+1 overlaps the kernels of group g, and the
 * commitments of consecutive jobs over the same SRS share one batched MSM pipeline (see b200zk_msm_g1_batch).
 * A values pointer may also be DEVICE memory (a column that is already resident is used in place). */
/* on (default): inside b200zk_run_column_jobs the commitments run on the context stream and the transforms on a second
 * stream, so the MSM's latency/memory-bound phases overlap with NTT butterflies; off: one stream (per-kernel timing). */
B200ZK_API int32_t b200zk_ctx_set_overlap(b200zk_ctx* ctx, int on);
/* Heterogeneous form: every job names its own host buffer, SRS and mode, so one proof phase (Lagrange commits,
 * coefficient-form commits, transforms, and the quotient's extended_to_coeff) is ONE call with a full copy/compute pipeline:
 *   mode 0..3 as above (host_values holds 2^k elements);
 *   mode 4: extended_to_coeff of 2^extended_k host values (inverse coset NTT) into coeff_out_dev or an internal scratch;
 *   mode 5: coeff_to_extended alone: 2^k COEFFICIENTS -> ext_out_dev (fixed / permutation polynomials whose cosets are
 *           not kept, or a polynomial produced on the device).
 * commits_out gets count x 96 B; entries of jobs without a commitment are zero. */
typedef struct b200zk_column_job {
    const void* host_values;
    const b200zk_srs* srs;    /* modes 0, 1, 2 */
    int32_t mode;
    void* coeff_out_dev;      /* optional device output (2^k elements; 2^extended_k for mode 4) */
    void* ext_out_dev;        /* optional device output (2^extended_k elements) */
} b200zk_column_job;
B200ZK_API int32_t b200zk_run_column_jobs(b200zk_ctx* ctx, const b200zk_column_job* jobs, uint32_t count, uint32_t k,
                                          const void* omega_inv32, const void* extended_omega32, const void* extended_omega_inv32,
                                          uint32_t extended_k, void* commits_out);
B200ZK_API int32_t b200zk_commit_columns(b200zk_ctx* ctx, const b200zk_srs* srs, const void* const* host_cols, uint32_t count,
                                         uint32_t k, const void* omega_inv32, const void* extended_omega32, uint32_t extended_k,
                                         void* commits_out, void* const* coeff_out_dev, void* const* ext_out_dev, int mode);

/* ---- polynomial batch ops (halo2_proofs Polynomial +,-,*scalar / parallelize loops) ---------- */
B200ZK_API int32_t b200zk_poly_add(b200zk_ctx* ctx, void* r, const void* a, const void* b, uint64_t n);          /* r = a + b */
B200ZK_API int32_t b200zk_poly_sub(b200zk_ctx* ctx, void* r, const void* a, const void* b, uint64_t n);          /* r = a - b */
B200ZK_API int32_t b200zk_poly_mul(b200zk_ctx* ctx, void* r, const void* a, const void* b, uint64_t n);          /* r = a .* b */
B200ZK_API int32_t b200zk_poly_scale(b200zk_ctx* ctx, void* r, const void* a, const void* s32, uint64_t n);      /* r = s * a */
B200ZK_API int32_t b200zk_poly_axpy(b200zk_ctx* ctx, void* r, const void* a, const void* s32, const void* b, uint64_t n); /* r = s*a + b */
/* arithmetic::eval_polynomial(poly, point) */
B200ZK_API int32_t b200zk_eval_poly(b200zk_ctx* ctx, const void* poly, uint64_t n, const void* point32, void* out32);
/* arithmetic::compute_inner_product(a, b) = sum_i a_i * b_i */
B200ZK_API int32_t b200zk_inner_product(b200zk_ctx* ctx, const void* a, const void* b, uint64_t n, void* out32);
/* ff::BatchInvert on a slice: zeros stay zero */
B200ZK_API int32_t b200zk_batch_invert(b200zk_ctx* ctx, void* data, uint64_t n);
/* arithmetic::kate_division: q (n-1 coeffs) = a (n coeffs) / (X - b) */
B200ZK_API int32_t b200zk_kate_division(b200zk_ctx* ctx, void* q, const void* a, uint64_t n, const void* b32);

/* ---- quotient construction: the work of create_proof BETWEEN the transforms (SURVEY.md §8(f).2) ------------------
 * Upstream: halo2_proofs/src/plonk/{evaluation.rs, permutation/prover.rs, mv_lookup/prover.rs} @ e5ddf67 (pin
 * /root/reference/Cargo.lock:1886-1888; entered from /root/reference/integration/src/prove.rs:37-39).  All column
 * arguments of this group are DEVICE pointers (columns stay resident between b200zk_run_column_jobs and here);
 * scalars, programs and pointer tables are host memory. */

/* Exclusive running product / sum with an initial value: out[0] = init, out[i] = out[i-1] (*|+) in[i-1], i < n.
 * This is the z(X) loop of permutation::Argument::commit (op 0) and the phi(X) loop of the log-derivative lookup
 * (op 1).  in == out is allowed. */
#define B200ZK_SCAN_PRODUCT 0
#define B200ZK_SCAN_SUM 1
B200ZK_API int32_t b200zk_prefix_scan(b200zk_ctx* ctx, int op, const void* in_dev, uint64_t n, const void* init32, void* out_dev);

/* out[i] = sum_j scalars[j] * polys[j][i], i < n: one pass over the inputs (the SHPLONK prover's per-rotation-set
 * sum_i v^i p_i(X) and its final linear combination; poly/kzg/multiopen/shplonk/prover.rs).  out may alias one input. */
B200ZK_API int32_t b200zk_poly_lincomb(b200zk_ctx* ctx, void* out_dev, const void* const* polys_dev, const void* scalars32,
                                       uint32_t count, uint64_t n);

/* One column set of the permutation argument (permutation::Argument::commit, one iteration of its chunk loop):
 *   mv[i]  = prod_j (beta * sigma_j[i] + gamma + v_j[i])            (denominators, then ff::BatchInvert)
 *   mv[i] *= prod_j (delta_omega_j * omega^i * beta + gamma + v_j[i]),  delta_omega_j = delta_omega_start * delta^j
 *   z[0] = z_init, z[i] = z[i-1] * mv[i-1]                          (i < 2^k)
 * values_dev / sigma_dev: n_cols device columns of 2^k Lagrange values each.  The caller overwrites the blinding rows
 * and reads z[2^k - (blinding_factors + 1)] as the next set's z_init, exactly as upstream does on the host. */
B200ZK_API int32_t b200zk_permutation_product(b200zk_ctx* ctx, const void* const* values_dev, const void* const* sigma_dev,
                                              uint32_t n_cols, const void* beta32, const void* gamma32,
                                              const void* delta_omega_start32, const void* delta32, const void* omega32,
                                              uint32_t k, const void* z_init32, void* z_out_dev);

/* Running sum of the log-derivative lookup (mv_lookup::prover, the phi(X) column):
 *   d[i] = sum_j 1 / (inputs_j[i] + beta)  -  m[i] / (table[i] + beta);   phi[0] = phi_init, phi[i] = phi[i-1] + d[i-1]
 * inputs_dev: n_inputs compressed input columns; table_dev: compressed table column; m_dev: multiplicities.
 * Zero denominators invert to zero, as ff::BatchInvert leaves them. */
B200ZK_API int32_t b200zk_logup_running_sum(b200zk_ctx* ctx, const void* const* inputs_dev, uint32_t n_inputs,
                                            const void* table_dev, const void* m_dev, const void* beta32, uint32_t k,
                                            const void* phi_init32, void* phi_out_dev);

/* plonk::evaluation::GraphEvaluator on the device.  A program is the upstream `calculations` list: calculation i
 * writes intermediate i; operands are ValueSources.  Calculation::Horner(start, parts, factor) names its parts as a
 * range of `horner_parts`.  B200ZK_SRC_EXTENDED_X is an addition over upstream: the point zeta * extended_omega^row of
 * the extended coset, so that the permutation / lookup identities (hard-coded loops upstream) are programs too. */
#define B200ZK_SRC_CONSTANT 0u       /* index into the program's constants */
#define B200ZK_SRC_INTERMEDIATE 1u   /* index of an earlier calculation */
#define B200ZK_SRC_FIXED 2u          /* index = column, rotation = index into the program's rotations */
#define B200ZK_SRC_ADVICE 3u
#define B200ZK_SRC_INSTANCE 4u
#define B200ZK_SRC_CHALLENGE 5u      /* index into challenges */
#define B200ZK_SRC_BETA 6u
#define B200ZK_SRC_GAMMA 7u
#define B200ZK_SRC_THETA 8u
#define B200ZK_SRC_Y 9u
#define B200ZK_SRC_PREVIOUS_VALUE 10u
#define B200ZK_SRC_EXTENDED_X 11u
#define B200ZK_CALC_ADD 0u
#define B200ZK_CALC_SUB 1u
#define B200ZK_CALC_MUL 2u
#define B200ZK_CALC_SQUARE 3u
#define B200ZK_CALC_DOUBLE 4u
#define B200ZK_CALC_NEGATE 5u
#define B200ZK_CALC_HORNER 6u        /* a = start value, b = factor, parts = horner_parts[parts_offset .. +parts_len] */
#define B200ZK_CALC_STORE 7u
typedef struct b200zk_value_source {
    uint32_t kind, index, rotation;
} b200zk_value_source;
typedef struct b200zk_calculation {
    uint32_t op;
    b200zk_value_source a, b;
    uint32_t parts_offset, parts_len;
} b200zk_calculation;
typedef struct b200zk_graph b200zk_graph;
/* Validates the program, assigns the live intermediates to on-chip slots and uploads the instruction stream. */
B200ZK_API int32_t b200zk_graph_create(b200zk_ctx* ctx, const b200zk_calculation* calculations, uint32_t n_calculations,
                                       const b200zk_value_source* horner_parts, uint32_t n_parts, const void* constants32,
                                       uint32_t n_constants, const int32_t* rotations, uint32_t n_rotations,
                                       b200zk_graph** out);
/* The validation and lowering of b200zk_graph_create alone -- no context, no device: lets the key-generation side check
 * a program (and read its instruction / slot count) on a machine without a GPU.  message receives the reason on failure. */
B200ZK_API int32_t b200zk_graph_check(const b200zk_calculation* calculations, uint32_t n_calculations,
                                      const b200zk_value_source* horner_parts, uint32_t n_parts, uint32_t n_constants,
                                      uint32_t n_rotations, uint32_t* n_instructions, uint32_t* n_slots, char* message,
                                      uint64_t message_cap);
B200ZK_API int32_t b200zk_graph_destroy(b200zk_ctx* ctx, b200zk_graph* graph);
B200ZK_API int32_t b200zk_graph_info(const b200zk_graph* graph, uint32_t* n_instructions, uint32_t* n_slots);
/* GraphEvaluator::evaluate for every row of the extended domain: values[row] = result of the last calculation, with
 * PreviousValue = the old values[row] (so successive programs chain the way evaluate_h folds gates with y) and
 * column reads at (row + rotations[r] * rot_scale) mod 2^log_size.  extended_omega32 is only read when the program
 * uses B200ZK_SRC_EXTENDED_X (may be NULL otherwise). */
B200ZK_API int32_t b200zk_graph_evaluate(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev,
                                         uint32_t n_fixed, const void* const* advice_dev, uint32_t n_advice,
                                         const void* const* instance_dev, uint32_t n_instance, const void* challenges32,
                                         uint32_t n_challenges, const void* beta32, const void* gamma32, const void* theta32,
                                         const void* y32, const void* extended_omega32, void* values_dev, uint32_t log_size,
                                         int32_t rot_scale);

/* The same for the rows [row_first, row_first + row_count) only: values[row] of the other rows is left untouched.  Column reads
 * still wrap over the whole domain, so the columns must be complete on this device.  This is evaluate_h SHARDED BY ROW RANGE
 * across GPUs (SURVEY.md §8(e)): every rank holds the cosets, evaluates its b200zk_shard_range of the extended domain, and
 * b200zk_allgather_rows makes the quotient numerator complete on every rank. */
B200ZK_API int32_t b200zk_graph_evaluate_rows(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev,
                                              uint32_t n_fixed, const void* const* advice_dev, uint32_t n_advice,
                                              const void* const* instance_dev, uint32_t n_instance, const void* challenges32,
                                              uint32_t n_challenges, const void* beta32, const void* gamma32, const void* theta32,
                                              const void* y32, const void* extended_omega32, void* values_dev, uint32_t log_size,
                                              int32_t rot_scale, uint64_t row_first, uint64_t row_count);
/* Collective over the context's communicator: values_dev holds 2^log_size field elements of which this rank has written its
 * b200zk_shard_range(2^log_size, rank, world) slice; afterwards every rank holds all slices (one in-place ncclAllGather of the
 * 32-byte elements over NVLink, on the context stream).  world must divide 2^log_size (a power of two); world == 1 is a no-op. */
B200ZK_API int32_t b200zk_allgather_rows(b200zk_ctx* ctx, void* values_dev, uint32_t log_size);

/* ---- the extended coset by parts ------------------------------------------------------------------
 * With n = 2^k, J = 2^(extended_k - k) (1 <= k, k <= extended_k <= 28, J <= 16), the extended coset point of row t = r + J*i is
 * zeta * w_ext^t = g_r * w^i, g_r = zeta * w_ext^r (w_ext^J = w).  So the extended domain is J disjoint parts of n points:
 * rotations stay inside a part, X^n - 1 is the constant g_r^n - 1 on part r, and a quotient can be built part by part with
 * n-element columns only.  Same bytes as the full-coset entries. */
/* out_dev[j][i] = p_j(g_part * w^i), i < 2^k: element part + J*i of coeff_to_extended(p_j).  coeffs[j]: 2^k coefficients,
 * host or device; out_dev[j]: device. */
B200ZK_API int32_t b200zk_coeff_to_extended_parts(b200zk_ctx* ctx, const void* const* coeffs, uint32_t count, uint32_t k,
                                                  uint32_t extended_k, uint32_t part, void* const* out_dev);
/* b200zk_graph_evaluate on the 2^k rows of one part: columns hold that part's values, a rotation reads row (i + rot) mod 2^k,
 * B200ZK_SRC_EXTENDED_X is g_part * w^i, PreviousValue is the old values[i].  values_dev: 2^k elements (device). */
B200ZK_API int32_t b200zk_graph_evaluate_part(b200zk_ctx* ctx, const b200zk_graph* graph, const void* const* fixed_dev,
                                              uint32_t n_fixed, const void* const* advice_dev, uint32_t n_advice,
                                              const void* const* instance_dev, uint32_t n_instance, const void* challenges32,
                                              uint32_t n_challenges, const void* beta32, const void* gamma32, const void* theta32,
                                              const void* y32, uint32_t k, uint32_t extended_k, uint32_t part, void* values_dev);
/* parts_dev: 2^extended_k elements, part-major (part r at r * 2^k); consumed (used as scratch).  out_dev receives n_pieces * 2^k
 * coefficients (1 <= n_pieces <= J): extended_to_coeff of the interleaved vector (first passed through divide_by_vanishing_poly
 * when divide_by_vanishing != 0), truncated.  out_dev may equal parts_dev.  With world | J, a rank's
 * b200zk_shard_range(2^extended_k) slice is whole parts, so b200zk_allgather_rows(ctx, parts_dev, extended_k) completes it. */
B200ZK_API int32_t b200zk_extended_parts_to_coeff(b200zk_ctx* ctx, void* parts_dev, uint32_t k, uint32_t extended_k,
                                                  uint32_t n_pieces, int divide_by_vanishing, void* out_dev);

/* ---- diagnostics ----------------------------------------------------------------------------- */
/* element-wise Fr/Fq Montgomery product of two arrays on the device (field-layer parity tests) */
B200ZK_API int32_t b200zk_debug_field_op(b200zk_ctx* ctx, int field /*0 Fr,1 Fq*/, int op /*0 mul,1 add,2 sub,3 inv*/,
                              void* r, const void* a, const void* b, uint64_t n);
/* Per-kernel-class device timing with CUDA events on the context stream (bench.py's roofline):
 * classes: ntt_pass ntt_table msm_count msm_scan msm_scatter msm_accumulate msm_combine msm_reduce msm_finish poly */
B200ZK_API int32_t b200zk_profile_enable(b200zk_ctx* ctx, int on);
B200ZK_API int32_t b200zk_profile_reset(b200zk_ctx* ctx);
B200ZK_API int32_t b200zk_profile_read(b200zk_ctx* ctx, const char* kernel_class, double* total_ms, uint64_t* count);
/* MSM tuning knobs (window bits; 0 = auto) and last-call statistics, for bench/roofline reporting */
B200ZK_API int32_t b200zk_msm_set_window(b200zk_ctx* ctx, uint32_t c);
/* bucket additions actually performed (non-zero signed digits) by all MSMs since the last reset */
B200ZK_API int32_t b200zk_msm_total_adds(b200zk_ctx* ctx, uint64_t* actual_adds, int reset);
B200ZK_API int32_t b200zk_msm_last_stats(const b200zk_ctx* ctx, uint32_t* window_bits, uint32_t* n_windows, uint64_t* n_bucket_adds);

#ifdef __cplusplus
}
#endif
#endif /* B200ZK_H */
