/* rla_b200.h -- C ABI of librla_b200.so, the B200 (sm_100a) sketching engine
 * behind rla4mor's embedding-operator API.
 *
 * Conventions
 *   - every entry point returns 0 on success or a negative rla_status code;
 *     rla_last_error() returns a thread-local message for the last failure;
 *   - a block of m vectors of dimension n is an (m, n) array, ONE VECTOR PER
 *     ROW with n contiguous (the reference's layout: rla/srht.py:142,160 and
 *     `U.to_numpy()` at rla/embeddings.py:169); `ld*` arguments are row
 *     strides in ELEMENTS;
 *   - pointers named *_dev are device pointers owned by the caller (PyTorch
 *     tensors on the host side); nothing here allocates device memory: sizes
 *     of plans and workspaces are queried and the caller provides the buffers;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     all device work is enqueued on it and the call returns without syncing;
 *   - there is no CPU fallback: every compute entry point fails with
 *     RLA_ERR_CUDA when no sm_100 device is usable.
 *
 * Each entry point cites the reference interface it replaces (file:line into
 * alexandre-pasco/rla4mor).  INTEGRATION.md shows the ctypes binding.
 */
#ifndef RLA_B200_H
#define RLA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum rla_status {
    RLA_OK = 0,
    RLA_ERR_INVALID = -1,   /* bad argument (the reference's AssertionError cases) */
    RLA_ERR_CUDA = -2,      /* CUDA runtime / launch failure, or no device */
    RLA_ERR_WORKSPACE = -3, /* workspace too small */
    RLA_ERR_UNSUPPORTED = -4
} rla_status;

int rla_version(void);
const char *rla_last_error(void);
/* number of CUDA kernels this library has launched in this process (bench.py reports
 * the delta over its timed region as "gpu_launches") */
unsigned long long rla_launch_count(void);
/* Adds n to that counter: for kernels of this library replayed from a CUDA graph the caller captured
 * (rla4mor_b200/factorization.py replays the launches of an LU solve that way). */
void rla_launch_count_add(long long n);

/* Pitched host<->device copy on `stream` (cudaMemcpy2DAsync): used to stream column slabs
 * of a row-major host block (pitches and width in BYTES; direction 0 = H2D, 1 = D2H). */
int rla_copy2d_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width_bytes,
                     size_t height, int direction, void *stream);

/* ------------------------------------------------------------------ SRHT ---
 * Replaces srht(x, k, seed, nthreads)            rla/srht.py:136-177
 * as called by SrhtEmbedding.apply               rla/embeddings.py:167-172.
 *
 * The Rademacher signs and the k row indices are drawn ON THE HOST by NumPy's
 * legacy RandomState exactly as rla/srht.py:162-163 does (that is what makes
 * them bit-exact) and handed to rla_srht_plan_create, which turns them into
 * the device-side descriptor the kernel consumes (packed sign bits per tile,
 * de-duplicated / bank-sorted sample descriptors, slot map).  The plan is
 * host-only; rla_srht_plan_upload copies its device image into a caller-owned
 * buffer of rla_srht_plan_device_bytes bytes.
 */
typedef struct rla_srht_plan rla_srht_plan;

int rla_srht_plan_create(rla_srht_plan **plan,
                         const int8_t *signs_host,  /* n entries, +1 / -1   (srht.py:162) */
                         int64_t n,
                         const int64_t *idx_host,   /* k entries in [0, 2**ceil(log2 n))  (srht.py:163) */
                         int64_t k,
                         int elem_bytes);           /* 8 (f64) or 4 (f32): the shared-memory layout depends on it */
void rla_srht_plan_destroy(rla_srht_plan *plan);
size_t rla_srht_plan_device_bytes(const rla_srht_plan *plan);
int rla_srht_plan_upload(rla_srht_plan *plan, void *plan_dev, void *stream);
/* number of passes over x the plan needs (1 unless k has more than 4096 distinct indices) */
int rla_srht_plan_passes(const rla_srht_plan *plan);
/* bytes of scratch needed to sketch m vectors with this plan */
size_t rla_srht_workspace_bytes(const rla_srht_plan *plan, int64_t m);

/* y[c, i] = scale * sum_j (-1)^popcount(idx[i] & j) * signs[j] * x[c, j]
 * (scale = 1/sqrt(k) reproduces srht.py:165-171, see SURVEY.md App. A.1).
 * x is read exactly once per pass and never written (srht.py:156). */
int rla_srht_apply_f64(const rla_srht_plan *plan, const double *x_dev, int64_t m, int64_t ldx,
                       double scale, double *y_dev, int64_t ldy,
                       void *ws_dev, size_t ws_bytes, void *stream);
int rla_srht_apply_f32(const rla_srht_plan *plan, const float *x_dev, int64_t m, int64_t ldx,
                       float scale, float *y_dev, int64_t ldy,
                       void *ws_dev, size_t ws_bytes, void *stream);

/* Explicit rows of the SRHT matrix.  Replaces SrhtEmbedding._get_random_rows,
 * rla/embeddings.py:195-209:
 *   out[i, j] = value * (-1)^popcount(idx[rows[i]] & j) * signs[j],  j < n
 * `value` is computed by the caller as fl(fl(sqrt(n/k)) * fl(1/2**(d/2))) so the
 * result is bit-identical to the reference's. */
int rla_srht_rows_f64(const int8_t *signs_dev, int64_t n, const int64_t *idx_dev,
                      const int64_t *rows_dev, int64_t nrows, double value,
                      double *out_dev, int64_t ldo, void *stream);

/* ------------------------------------------------------------------ FWHT ---
 * Replaces fht_oop(a, nthreads) / fht_ip(a)      rla/srht.py:121-134, 99-118.
 * out = post_scale * H a along each row (H the natural-order Sylvester matrix,
 * n_pow2 = 2**d); out_dev may equal a_dev (in place).  The reference's
 * normalisation is post_scale = 1/2**(d/2) (srht.py:36). */
int rla_fwht_f64(const double *a_dev, int64_t m, int64_t n_pow2, int64_t lda,
                 double *out_dev, int64_t ldo, double post_scale, void *stream);
int rla_fwht_f32(const float *a_dev, int64_t m, int64_t n_pow2, int64_t lda,
                 float *out_dev, int64_t ldo, float post_scale, void *stream);

/* Adjoint of the SRHT rows matrix without materialising it
 * (replaces the dense GEMM of SrhtEmbedding.apply_adjoint, rla/embeddings.py:175-178):
 *   out[c, j] = value * signs[j] * sum_i (-1)^popcount(idx[i] & j) * v[c, i],  j < n
 * order_dev: int32 permutation of [0, k) sorting idx ascending (stable), so duplicate
 * indices are summed in sample order.  scratch: m * 2**d elements
 * (rla_srht_adjoint_workspace_bytes). */
size_t rla_srht_adjoint_workspace_bytes(int64_t m, int64_t n);
int rla_srht_adjoint_f64(const int8_t *signs_dev, int64_t n, const int64_t *idx_dev,
                         const int32_t *order_dev, int64_t k,
                         const double *v_dev, int64_t m, int64_t ldv, double value,
                         double *out_dev, int64_t ldo, void *ws_dev, size_t ws_bytes, void *stream);

/* ---------------------------------------------------- dense embeddings ------
 * Y(m, k) = U(m, n) * Theta(k, n)^T, both operands n-contiguous.
 * Replaces NumpyMatrixOperator(Theta).apply(Q U) = (Theta @ (QU)^T)^T
 *   GaussianEmbedding.apply                      rla/embeddings.py:250-254
 *   BlockGaussianEmbedding.apply (per block)     rla/embeddings.py:425-434
 * FP64 tensor-core (DMMA) GEMM with a deterministic split of the n dimension.
 */
size_t rla_gemm_workspace_bytes(int64_t m, int64_t k, int64_t n);

/* Measured FP64 tensor-pipe peak of the current device in TFLOP/s (independent
 * mma.sync.m8n8k4.f64 issued back to back on every SM): the roofline denominator bench.py
 * uses for the dense sketch.  scratch_dev: >= 1 MiB of device memory.  Synchronises. */
int rla_dmma_peak_tflops(double *tflops, void *scratch_dev, void *stream);

/* Theta materialised in device memory (drawn by the host exactly as
 * rla/embeddings.py:265-270 does). */
/* Philox4x32-10 of Random123 (Salmon et al., SC'11), the generator behind the on-the-fly Theta:
 * `count` items of 6 words {c0, c1, c2, c3, k0, k1} -> 4 output words each.  The host and the
 * device form run the same source (csrc/rng.cuh); tests pin both to the published known-answer
 * vectors. */
int rla_philox4x32_10_host(const uint32_t *ctr_key, int64_t count, uint32_t *out);
int rla_philox4x32_10_device(const uint32_t *ctr_key_dev, int64_t count, uint32_t *out_dev, void *stream);

int rla_gauss_apply_explicit_f64(const double *theta_dev, int64_t k, int64_t n, int64_t ldt,
                                 const double *u_dev, int64_t m, int64_t ldu,
                                 double *y_dev, int64_t ldy,
                                 void *ws_dev, size_t ws_bytes, void *stream);

/* Theta generated on the fly from a counter-based RNG (Philox4x32-10 keyed by
 * `seed`), never materialised: element (row0 + i, col0 + j) of the virtual
 * k_total x n_total matrix is scale * g(seed, row0 + i, col0 + j) with g a
 * standard normal (kind 0, Box-Muller) or a Rademacher +-1 (kind 1).
 * y[c, i] (+)= sum_j theta[row0 + i, col0 + j] * u[c, j]   for i < k_blk, j < n.
 * Reproducibility: the Philox words are exact integer arithmetic (known-answer tested on host
 * and device, rla_philox4x32_10_*), so kind 1 is the same on every device.  Kind 0 turns them
 * into normals with FP32 Box-Muller on the SFU (MUFU lg2 / sin / cos approximations): the map
 * (kind, seed, row, col) -> Theta is bit-stable on sm_100 -- rla_theta_materialize_f64 runs the
 * same device function -- but another architecture may round the last FP32 bits differently.
 * For a Theta that is identical everywhere use options['rng'] = 'mt19937' (host draw, explicit
 * GEMM) or kind 1. */
/* Kinds 0 and 2 (FP32 normals) run on the int8 tensor cores (Ozaki slices, normwise error bound in
 * the header of csrc/gemm_i8.cu; one stream synchronisation per call); kind 1, and blocks with a
 * non-finite entry or one >= 2^900, on the FP64 tensor pipe.
 * ws_dev: rla_gemm_rng_workspace_bytes(m, k_blk, n) (about 8 bytes per element of u more than
 * rla_gemm_workspace_bytes: the int8 slices of u). */
size_t rla_gemm_rng_workspace_bytes(int64_t m, int64_t k, int64_t n);
int rla_embed_apply_rng_f64(uint64_t seed, int kind, double scale,
                            int64_t row0, int64_t k_blk, int64_t col0, int64_t n,
                            const double *u_dev, int64_t m, int64_t ldu,
                            double *y_dev, int64_t ldy, int accumulate,
                            void *ws_dev, size_t ws_bytes, void *stream);
/* The same for a FLOAT32 block (the optional FP32 path of north_star; tolerance 1e-5 relative
 * Frobenius) on the generation-5 tensor cores: tcgen05.mma kind::tf32 with FP32 accumulators in
 * TMEM that are flushed into FP64 every 64 terms, the block split into two TF32 parts (two MMAs
 * per step).  Theta must be exact in TF32: kind 1 (Rademacher) or kind 2 (the normals of kind 0
 * rounded to TF32; rla_embed_apply_rng_f64 / rla_theta_materialize_f64 accept kind 2 too, so
 * Theta is the same matrix for both dtypes).  y is FLOAT64 (the reference's `Theta @ U.T` with a
 * float64 Theta returns float64, rla/embeddings.py:250-254).  col0 must be a multiple of 32,
 * u_dev 16-byte aligned, ldu a multiple of 4.  ws_dev: rla_gemm32_workspace_bytes(m, k_blk, n). */
size_t rla_gemm32_workspace_bytes(int64_t m, int64_t k, int64_t n);
int rla_embed_apply_rng_f32(uint64_t seed, int kind, double scale,
                            int64_t row0, int64_t k_blk, int64_t col0, int64_t n,
                            const float *u_dev, int64_t m, int64_t ldu,
                            double *y_dev, int64_t ldy, int accumulate,
                            void *ws_dev, size_t ws_bytes, void *stream);
/* Export what the on-the-fly generator produces (parity tooling; replaces
 * get_random_matrix / _get_random_block, rla/embeddings.py:87-100, 452-461). */
int rla_theta_materialize_f64(uint64_t seed, int kind, double scale,
                              int64_t row0, int64_t rows, int64_t col0, int64_t cols,
                              double *out_dev, int64_t ldo, void *stream);
/* The adjoint of the on-the-fly Gaussian embeddings, Theta generated in the kernel and never
 * materialised: out(m, n) = V(m, k) * Theta(k, n), all row-major.  Replaces pyMOR's adjoint of the
 * explicit matrix, V @ get_matrix(), of GaussianEmbedding and BlockGaussianEmbedding
 * (rla/embeddings.py:214-270, 373-467; Q^H is applied by the caller).
 * Theta is a stack of nblocks blocks: row_start_dev (nblocks + 1 entries, 0 = row_start[0] <= ... <=
 * row_start[nblocks] = k) and seeds_dev (nblocks entries) are caller-owned device memory.  Rows
 * [row_start[b], row_start[b+1]) of Theta are rows 0 .. size_b - 1 of the virtual matrix
 * scale * g(seeds[b], row, col) of rla_theta_materialize_f64 (kind 0, 1 or 2), each entry formed as
 * fl(scale * g).  The table is read on the device, so ldv >= k is the caller's to ensure.
 * Every element of `out` is one DMMA chain over k in ascending order, four terms at a time: the result
 * equals rla_gemm_nn_f64(V, Theta materialised) bit for bit when that call takes its tensor-pipe path
 * (16-byte aligned operands, even leading dimensions), and is deterministic from run to run.
 * One launch, no workspace. */
int rla_embed_adjoint_rng_f64(int kind, double scale,
                              const uint64_t *seeds_dev, const int64_t *row_start_dev, int64_t nblocks,
                              int64_t n, const double *v_dev, int64_t m, int64_t ldv,
                              double *out_dev, int64_t ldo, void *stream);

/* ------------------------------------------- MT19937 Gaussian Theta ---------
 * The reference draws Theta (and every block of the block embedding) on the host with
 * np.random.RandomState(seed).normal(size=(k, n), loc=0, scale=1/sqrt(k))   rla/embeddings.py:269,458.
 * These entry points produce the same numbers on the device, bit for bit, for a FRESH RandomState
 * (pos = 624, no cached Gaussian).  Output 2p of a stream is scale * f * x2 and output 2p + 1 is
 * scale * f * x1 of its p-th accepted polar attempt (csrc/mt19937.cuh states the arithmetic and the
 * exactness argument: an extended-precision log, with the pairs whose log lies within w ulp of a
 * rounding midpoint finished with the C library's log on the host; w = 1/32 by default, 0.5 sends
 * every pair through the host).
 *
 * Plan (host object + caller-owned device workspace), once per batch of streams:
 *   keys: nstreams x 624 words, RandomState(seed).get_state(legacy=False)['state']['key'];
 *   nseg[i]: segments of rla_mt19937_segment_words() words given to stream i (enough for its
 *   normals: 2 * rla_mt19937_plan_pairs(plan, i) normals are available after the build; the caller
 *   re-plans with more segments if that falls short).
 *   rla_mt19937_plan_build jumps to every segment start (F2 jump-ahead), counts the accepted
 *   attempts of every segment and scans them; it synchronises the stream once.  The workspace must
 *   stay allocated and untouched while the plan is used.
 * Execute: normals [first[i], first[i] + count[i]) of stream i go to out_dev + offset[i]
 *   (out_len elements in all); first may be odd.  ws_dev: rla_mt19937_execute_workspace_bytes(plan,
 *   flag_cap), room for flag_cap flagged pairs; staging_host: flag_cap doubles of pinned host memory
 *   (NULL only if nothing can be flagged).  *nflagged receives the number of flagged pairs; when it
 *   exceeds flag_cap the call returns RLA_ERR_WORKSPACE and the caller retries with a larger one.
 *   Synchronises the stream once after the write pass and, when pairs were flagged, twice more
 *   around the host fix-up (their r2 down, libm's log up). */
typedef struct rla_mt19937_plan rla_mt19937_plan;
int64_t rla_mt19937_segment_words(void);
int rla_mt19937_plan_create(rla_mt19937_plan **plan, const uint32_t *keys, const int64_t *nseg, int64_t nstreams);
void rla_mt19937_plan_destroy(rla_mt19937_plan *plan);
size_t rla_mt19937_plan_workspace_bytes(const rla_mt19937_plan *plan);
int rla_mt19937_plan_build(rla_mt19937_plan *plan, void *ws_dev, size_t ws_bytes, void *stream);
/* accepted pairs available to stream i after the build (-1 before it) */
int64_t rla_mt19937_plan_pairs(const rla_mt19937_plan *plan, int64_t i);
size_t rla_mt19937_execute_workspace_bytes(const rla_mt19937_plan *plan, int64_t flag_cap);
int rla_mt19937_normal_f64(const rla_mt19937_plan *plan, const int64_t *first, const int64_t *count,
                           const int64_t *offset, double scale, double w, double *out_dev, int64_t out_len,
                           void *ws_dev, size_t ws_bytes, int64_t flag_cap, double *staging_host,
                           int64_t *nflagged, void *stream);
/* Host-only hooks of the same code (tests):
 *   rla_mt19937_jump_host: the state `steps` words ahead of key_in (both 624 words, pos = 624);
 *   rla_mt19937_attempts_host: n attempts from 4n output words (tempered, as random_raw gives them)
 *   -> x1, x2, r2, accepted;
 *   rla_mt19937_ext_log_host: the extended log of x in (0, 1) as hi + lo and its midpoint flag;
 *   rla_libm_log_host: the C library's log of n values (several threads, no vector math library). */
int rla_mt19937_jump_host(const uint32_t *key_in, uint64_t steps, uint32_t *key_out);
int rla_mt19937_attempts_host(const uint32_t *words, int64_t n, double *x1, double *x2, double *r2, int8_t *accept);
int rla_mt19937_ext_log_host(const double *x, int64_t n, double w, double *hi, double *lo, int8_t *flag);
int rla_libm_log_host(const double *x, int64_t n, double *out);

/* out(m, n) = V(m, k) * Theta(k, n): the adjoint / explicit-matrix product
 * (SrhtEmbedding.apply_adjoint rla/embeddings.py:175-178, rb.lincomb(T.T)
 * mor/sketched_reductor.py:99-100).  Theta is transposed into scratch and the product
 * runs on the same tensor-core kernel as the sketch. */
size_t rla_gemm_nn_workspace_bytes(int64_t m, int64_t k, int64_t n);
int rla_gemm_nn_f64(const double *v_dev, int64_t m, int64_t k, int64_t ldv,
                    const double *theta_dev, int64_t n, int64_t ldt,
                    double *out_dev, int64_t ldo, void *ws_dev, size_t ws_bytes, void *stream);

/* ------------------------------------------------ sketched reductor ops ----
 * CSR SpMM in the reference's row layout: out[c, i] = sum_j A[i, j] * u[c, j]
 * (the A_q.apply(U) that precedes every sketch, mor/sketched_reductor.py:69-70). */
int rla_spmm_csr_f64(const int64_t *rowptr_dev, const int32_t *col_dev, const double *val_dev,
                     int64_t n_rows, int64_t n_cols,
                     const double *u_dev, int64_t m, int64_t ldu,
                     double *out_dev, int64_t ldo, void *stream);

/* Modified Gram-Schmidt with re-iteration of the r rows (dimension k) of the
 * sketched basis, in place; R (r x r, row-major, ld = r) receives the
 * coefficients as pyMOR's gram_schmidt(..., return_R=True) does
 * (mor/sketched_reductor.py:94).  Rows [0, offset) are assumed orthonormal.
 * flags_dev[i] = 1 when row i was dropped as (numerically) dependent. */
int rla_gram_schmidt_f64(double *a_dev, int64_t r, int64_t k, int64_t lda, int64_t offset,
                         double *R_dev, int32_t *flags_dev,
                         double atol, double rtol, double reiteration_threshold, void *stream);

/* One-sided Jacobi (Hestenes) SVD of a k x m sketch held in the row layout: a_dev is
 * (m, k), row p = column p of the k x m matrix.  On return the rows are u_p * s_p
 * (mutually orthogonal), s_dev holds the m singular values (unsorted) and V_dev (m x m,
 * row p = p-th right singular vector; may be NULL) the accumulated rotations.
 * pairs_dev: round-robin schedule, (me - 1) rounds x (me / 2) int32 pairs with
 * me = m rounded up to even, -1 marking the bye; rot_dev: one int32 of scratch.
 * Synchronises the stream once per sweep to test convergence. */
int rla_svd_jacobi_f64(double *a_dev, int64_t k, int64_t m, int64_t lda,
                       double *s_dev, double *V_dev, const int32_t *pairs_dev, int32_t *rot_dev,
                       int max_sweeps, double tol, int *sweeps_done, void *stream);

/* Many-CTA (cooperative-launch) versions of the two factorisations (csrc/factor.cu).
 * rla_gram_schmidt_ws_f64: same contract as rla_gram_schmidt_f64, rows dealt to many CTAs and kept
 * in registers (right-looking modified Gram-Schmidt, pyMOR's removal / re-iteration tests); a
 * finished row, its decision and the partial corrections of a re-iteration travel between CTAs as
 * tagged 8-byte words in the workspace (no fence, no flag); falls back to the one-CTA kernel when
 * the shape is out of range or ws is too small (rla_gram_schmidt_workspace_bytes returns 0 when
 * the many-CTA kernel does not apply; the workspace holds the hand-over ring, a few MB). */
size_t rla_gram_schmidt_workspace_bytes(int64_t r, int64_t k);
/* Byte offset, inside the workspace, of the int32 status word the grid kernel leaves behind
 * (0 = ok, 1 = a wait on another CTA's flag timed out: the result is NOT usable); -1 when the
 * one-CTA kernel runs for this shape.  Callers read it after the launch and raise. */
int64_t rla_gram_schmidt_status_offset(int64_t r, int64_t k);
int rla_gram_schmidt_ws_f64(double *a_dev, int64_t r, int64_t k, int64_t lda, int64_t offset,
                            double *R_dev, int32_t *flags_dev,
                            double atol, double rtol, double reiteration_threshold,
                            void *ws_dev, size_t ws_bytes, void *stream);
/* Block one-sided Jacobi SVD in ONE launch (same data convention as rla_svd_jacobi_f64):
 * B = rla_svd_jacobi_block_rows(k, m, want_v) rows per block (0: shape not supported, use
 * rla_svd_jacobi_f64); sched_dev: round-robin schedule over nb = ceil(m / B) rounded up to even
 * blocks, (nb - 1) rounds x (nb / 2) int32 pairs, (b, -1) marking the bye of block b;
 * scratch_dev: rla_svd_jacobi_block_scratch_ints(m, B, max_sweeps) int32; on return
 * scratch_dev[0..2] = {sweeps done, converged, timeout}.  No host synchronisation. */
int rla_svd_jacobi_block_rows(int64_t k, int64_t m, int want_v);
size_t rla_svd_jacobi_block_scratch_ints(int64_t m, int B, int max_sweeps);
int rla_svd_jacobi_block_f64(double *a_dev, int64_t k, int64_t m, int64_t lda,
                             double *s_dev, double *V_dev, const int32_t *sched_dev, int B,
                             int32_t *scratch_dev, int max_sweeps, double tol, void *stream);

/* Cluster-resident one-sided Jacobi SVD (csrc/jacobi_cluster.cu; same data convention as
 * rla_svd_jacobi_f64): the whole (m, k [+ m]) row block lives in the distributed shared memory of
 * ONE thread-block cluster of C CTAs for the whole iteration; block rounds of the circle-method
 * tournament end with a DSMEM push and a cluster barrier instead of a trip through global memory.
 * rla_svd_jacobi_cluster_size returns C (2, 4, 8 or 16) or 0 when the shape does not fit (then
 * use rla_svd_jacobi_block_f64 / rla_svd_jacobi_f64).  info_dev: 8 int32, on return {sweeps
 * done, converged, 0, then five phase counters in kilo-cycles of CTA 0: stage load + norms,
 * rotation steps, wait on the stage barrier, push, end-of-round barrier}.  One launch, no host synchronisation, no flags in global memory (the
 * hardware co-schedules the CTAs of a cluster, so there is no timeout path).  This is the SVD
 * of the "thin QR / SVD of the k x m sketch" of BASELINE configs[4]. */
int rla_svd_jacobi_cluster_size(int64_t k, int64_t m, int want_v);
int rla_svd_jacobi_cluster_f64(double *a_dev, int64_t k, int64_t m, int64_t lda,
                               double *s_dev, double *V_dev, int32_t *info_dev,
                               int max_sweeps, double tol, void *stream);

/* T = R^-1 for the upper-triangular r x r factor of Gram-Schmidt (row-major): the reference's
 * T = pinv(R) (mor/sketched_reductor.py:95) when no row was removed. */
int rla_trinv_upper_f64(const double *R_dev, int64_t r, int64_t ldr, double *T_dev, int64_t ldt, void *stream);

/* Sketched residual norm  || sum_q th[q] S_q a - sum_p tr[p] b_p ||_2
 * (ResidualErrorEstimator.estimate_error, mor/sketched_reductor.py:216-219);
 * S_dev is Q contiguous k x r row-major blocks, b_dev P contiguous k-vectors. */
int rla_residual_norm_f64(const double *S_dev, int64_t Q, int64_t k, int64_t r,
                          const double *th_dev, const double *a_dev,
                          const double *b_dev, int64_t P, const double *tr_dev,
                          double *out_dev, void *stream);

/* ------------------------------------------- ROM over a parameter set ------
 * The online half of the sketched ROM for P parameter values mu_p at once (csrc/rom_batch.cu).
 * The affine coefficients are row-major device arrays th_dev (P, Q; row stride ldth) and tf_dev
 * (P, Pf; row stride ldtf); the ROM's data are in its existing layouts.
 *
 * rla_rom_solve_batch_f64 replaces, per mu_p, StationaryModel.solve of the Galerkin ROM
 * (mor/sketched_reductor.py:165-166; SketchedRom.solve): lhs_dev is Q contiguous row-major r x r
 * matrices, rhs_dev Pf contiguous r-vectors.  A_p = sum_q th[p, q] A_q and b_p = sum_j tf[p, j] f_j
 * are assembled in shared memory (ascending q / j, fma), factored by LU with partial pivoting
 * (largest |.|, ties to the smallest row: LAPACK's rule) and solved; row p of a_dev (row stride lda)
 * receives a_p.  info_dev[p] (int32) = 0, or i > 0 when U(i, i) is exactly zero (LAPACK's
 * convention); the row a_p is then NaN.  1 <= r <= rla_rom_solve_batch_max_r() (169: the augmented
 * r x (r + 1) system fits in the shared memory of one CTA).  One launch, no workspace.
 *
 * rla_residual_norm_batch_f64 replaces, per mu_p, ResidualErrorEstimator.estimate_error
 * (mor/sketched_reductor.py:216-219; the single-mu rla_residual_norm_f64):
 *   est[p] = || sum_q th[p, q] S_q a_p - sum_j tf[p, j] g_j ||_2
 * W_dev (N x kp, row stride ldw, N = Q r + Pf) is the stack [S_0^T; ...; S_{Q-1}^T; g_0^T; ...]
 * of the ROM's (r, kp) row blocks and kp-vectors; a_dev (P, r; row stride lda) holds the reduced
 * solutions.  The product X(P, N) W with X[p, q r + i] = th[p, q] a[p, i], X[p, Q r + j] = -tf[p, j]
 * runs on the FP64 tensor pipe with X formed in the kernel; neither X nor the residuals are stored.
 * ws_dev (caller-owned, rla_residual_norm_batch_workspace_bytes(P, kp) = 8 P ceil(kp / 128) bytes)
 * receives the per-tile partial sums, added in tile order: bit-identical from run to run.  A NaN
 * row of a_dev gives a NaN estimate.  Two launches.
 *
 * rla_rom_lstsq_batch_f64 replaces, per mu_p, the solve of the least-squares (minres) ROM
 * (mor/sketched_reductor.py:170-187; LsOperator.apply_inverse, utilities/other_operators.py:12-39):
 *   a_p = argmin_a || sum_q th[p, q] M_q a - sum_j tf[p, j] g_j ||_2,   M_q: ke x r, g_j: ke.
 * W_dev (N x ke, row stride ldw, N = Q r + Pf) is the stack [M_0^T; ...; M_{Q-1}^T; g_0^T; ...], the
 * layout rla_residual_norm_batch_f64 reads (a ROM whose N is below its sketch dimension may pass the
 * transposed triangular factor of the stack instead: the same minimiser, ke = N).  One CTA per mu
 * assembles [M(mu) | b(mu)] in panels of rows (ascending q / j, fma), folds each panel into the
 * r x r triangle by Householder reflections (LAPACK's dlarfg convention) and back-substitutes; row p
 * of a_dev (row stride lda) receives a_p.  info_dev[p] (int32) = 0, or the first i > 0 with R(i, i)
 * exactly zero (dtrtrs' convention, as dgels reports it); the row a_p is then NaN.  Results depend on
 * a mu's own inputs only, not on P: bit-identical from run to run and to a launch with P = 1.
 * 1 <= r <= rla_rom_lstsq_batch_max_r() (R and one panel in the shared memory of one CTA), ke >= r.
 * One launch, no workspace. */
int rla_rom_solve_batch_max_r(void);
int rla_rom_solve_batch_f64(const double *lhs_dev, int64_t Q, int64_t r, const double *rhs_dev, int64_t Pf,
                            const double *th_dev, int64_t ldth, const double *tf_dev, int64_t ldtf, int64_t P,
                            double *a_dev, int64_t lda, int32_t *info_dev, void *stream);
int rla_rom_lstsq_batch_max_r(void);
int rla_rom_lstsq_batch_f64(const double *W_dev, int64_t ldw, int64_t Q, int64_t r, int64_t Pf, int64_t k_eff,
                            const double *th_dev, int64_t ldth, const double *tf_dev, int64_t ldtf, int64_t P,
                            double *a_dev, int64_t lda, int32_t *info_dev, void *stream);
size_t rla_residual_norm_batch_workspace_bytes(int64_t P, int64_t kp);
int rla_residual_norm_batch_f64(const double *W_dev, int64_t ldw, int64_t Q, int64_t r, int64_t Pf, int64_t kp,
                                const double *th_dev, int64_t ldth, const double *tf_dev, int64_t ldtf,
                                const double *a_dev, int64_t lda, int64_t P, double *est_dev,
                                void *ws_dev, size_t ws_bytes, void *stream);

/* ------------------------------------- full-order solves over a parameter set ----
 * Block preconditioned CG for the affine full-order model (csrc/affine_cg.cu): replaces, per mu_p,
 * pyMOR's StationaryModel.solve -> apply_inverse of A(mu_p) = sum_q th[p, q] A_q (symmetric positive
 * definite), with a host-factored SPD preconditioner R applied between the calls (the reductor's
 * InverseLuOperator).  Every (P, n) block is row-major with row stride ld*; row p belongs to mu_p.
 *
 * rla_affine_spmm_f64:  y[p, :] = sum_q th[p, q] A_q x[p, :].  The operator is ONE CSR pattern
 *   (rowptr n + 1 int64, col nnz int32), the union of the terms' patterns, with Q value arrays
 *   val (Q, nnz) (0 where a term has no entry); th (P, Q; row stride ldth), 1 <= Q <= 32.  The
 *   coefficient of an entry is formed per row p in ascending q with fma.  mode (int32 P, may be NULL)
 *   restricts the product to the rows with mode[p] == 2; the other rows of y are not written.  With
 *   ws != NULL the per-tile partial sums of <x_p, y_p> go to ws (see below).  Replaces the Q
 *   MatrixOperator.apply calls and Q scaled additions of LincombOperator.apply.
 * rla_row_dot_partials_f64:  per-tile partial sums of <a_p, b_p> (rows with mode[p] == 2, or all).
 * rla_row_dot_sum_f64:  out[p] = the partials of row p added in tile order.
 *   Workspace: rla_affine_cg_workspace_bytes(n, P) = 8 P ceil(n / 256) bytes, caller-owned; tile t of
 *   row p (entries [256 t, 256 t + 256)) at ws[p ceil(n / 256) + t].  No atomics: the sums depend on
 *   a row's own data only and are bit-identical from run to run.
 *
 * The CG state lives on the device: state (double, 5 x P) = rho, rho_b, alpha, beta, resid;
 * istate (int32, 3 x P) = iterations, info, mode.  mode[p]: 2 = iterating, 1 = the row takes its
 * last step in the coming update_xp, 0 = idle.  info[p]: 0 converged, 1 not converged within
 * maxiter, 2 breakdown (<p, A p> <= 0 or <r, R^-1 r> < 0: A(mu) or R is not SPD; resid NaN).
 * rla_affine_cg_start_f64:  from the partials of <r_0, R^-1 r_0> (ws_r) and <b, R^-1 b> (ws_b; the
 *   same pointer when x_0 = 0) initialises every row: rho_b = 0 (b = 0) and rho_0 <= tol^2 rho_b
 *   finish in 0 iterations, maxiter = 0 gives info 1, the rest iterate.
 * rla_affine_cg_alpha_f64:  from the partials of <p, A p>: alpha = rho / <p, A p>, or breakdown.
 * rla_affine_cg_update_r_f64:  r <- r - alpha A p on iterating rows.
 * rla_affine_cg_beta_f64:  from the partials of <r, z> (z = R^-1 r): converged when
 *   rho' <= tol^2 rho_b (||r||_{R^-1} <= tol ||b||_{R^-1}), out of iterations, breakdown, or
 *   beta = rho' / rho; resid = sqrt(rho' / rho_b).  Rows that took their last step go idle.
 * rla_affine_cg_update_xp_f64:  x <- x + alpha p on rows that took a step; p <- z + beta p on
 *   rows that keep iterating. */
size_t rla_affine_cg_workspace_bytes(int64_t n, int64_t P);
int rla_affine_spmm_f64(const int64_t *rowptr_dev, const int32_t *col_dev, const double *val_dev, int64_t nnz, int64_t Q,
                        int64_t n, const double *th_dev, int64_t ldth, const double *x_dev, int64_t ldx, int64_t P,
                        double *y_dev, int64_t ldy, const int32_t *mode_dev, void *ws_dev, size_t ws_bytes,
                        void *stream);
int rla_row_dot_partials_f64(const double *a_dev, int64_t lda, const double *b_dev, int64_t ldb, int64_t n, int64_t P,
                             const int32_t *mode_dev, void *ws_dev, size_t ws_bytes, void *stream);
int rla_row_dot_sum_f64(const void *ws_dev, size_t ws_bytes, int64_t n, int64_t P, double *out_dev, void *stream);
int rla_affine_cg_start_f64(const void *ws_r_dev, const void *ws_b_dev, size_t ws_bytes, int64_t n, int64_t P,
                            double tol, int64_t maxiter, double *state_dev, int32_t *istate_dev, void *stream);
int rla_affine_cg_alpha_f64(const void *ws_dev, size_t ws_bytes, int64_t n, int64_t P, double *state_dev,
                            int32_t *istate_dev, void *stream);
int rla_affine_cg_update_r_f64(double *r_dev, int64_t ldr, const double *q_dev, int64_t ldq, int64_t n, int64_t P,
                               const double *state_dev, const int32_t *istate_dev, void *stream);
int rla_affine_cg_beta_f64(const void *ws_dev, size_t ws_bytes, int64_t n, int64_t P, double tol, int64_t maxiter,
                           double *state_dev, int32_t *istate_dev, void *stream);
int rla_affine_cg_update_xp_f64(double *x_dev, int64_t ldx, double *p_dev, int64_t ldp, const double *z_dev,
                                int64_t ldz, int64_t n, int64_t P, const double *state_dev, const int32_t *istate_dev,
                                void *stream);

/* --------------------------------------- sparse triangular solves (8f.1) ----
 * Device side of InverseLuOperator.apply / apply_adjoint (utilities/factorization.py:118-132,
 * `slu.solve(V.T).T`): the inverse_product R^-1 in front of the sketch
 * (mor/sketched_reductor.py:69,73).  The factorisation Pr A Pc = L U is SciPy SuperLU's, on the
 * host, as in the reference; L and U are uploaded as CSR.
 * rla_sptrsv_plan_host (HOST arrays in and out, plain C++ on the CPU, once per factor): level of
 * every row (lower != 0: dependencies j < i; else j > i), the processing order of the rows
 * (order_out, inverse pos_out), and -- ALL IN THAT ORDER, i.e. row p = row order_out[p] and
 * external column indices replaced by positions -- the strictly triangular part re-packed as CSR
 * (rowptr2 n + 1, col2 / val2 up to nnz, entries of a row sorted by column), the diagonal (1.0
 * where absent) and split; the solve therefore works on X in schedule order (X[p] = row
 * order_out[p], which rla_sptrsv_transpose_in/out produce with perm = pos[perm_r] etc.).
 * GROUPS (multi-row only): group g = order positions [grp_start[g], grp_start[g] + grp_rows[g]),
 * a chain of at most group_rows <= 128 rows that depend on each other; every dependency of a
 * group outside itself lies in an earlier level of the GROUP dependency graph.  STEPS, up to three
 * per group level: kind 0 / kind 1 = order positions [step_lo, step_hi): each row subtracts its
 * external entries (one warp per row / one CTA of 8 or 16 warps per row for rows of more than 64
 * entries) and a single row divides by its diagonal; kind 2 = groups [step_lo, step_hi) are
 * resolved.  split_out[i] = end of the external entries of row i; behind it the entries that
 * refer to the row's own group, col2 = slot inside the group.  wide_min: levels with more rows
 * stay single rows; max_multi is ignored (kept for ABI stability).  All output arrays hold n
 * entries (rowptr2 n + 1, col2 / val2 nnz).
 * rla_sptrsv_group_inverses_host (HOST): dinv_out + dinv_ptr[g] <- inverse of the triangular
 * block of group g (row-major grp_rows[g]^2 doubles; the caller sizes dinv_ptr as the running
 * sum of grp_rows^2), diag_eff_out[p] <- 1.0 inside groups, the diagonal elsewhere.
 * rla_sptrsv_transpose_in/out: (m, n) block of the reference layout <-> X (n, ldx) with the m
 * right-hand sides contiguous (ldx even, >= m), with the row / column permutation of the
 * factorisation applied on the way (perm_dev may be NULL): X[perm[i], c] = B[c, i] and
 * out[c, i] = X[perm[i], c].
 * rla_sptrsv_solve_f64: in-place T X = X, one launch per step (the step arrays stay on the
 * HOST, everything else on the device); diag_eff_dev NULL = no division (unit diagonal). */
int rla_sptrsv_plan_host(int64_t n, const int64_t *rowptr, const int32_t *col, const double *val,
                         int lower, int wide_min, int group_rows, int max_multi,
                         int32_t *level_out, int32_t *order_out, int32_t *pos_out,
                         int64_t *rowptr2, int32_t *col2, double *val2, double *diag_out,
                         int64_t *split_out, int64_t *grp_start, int32_t *grp_rows, int64_t *ngroups_out,
                         int64_t *step_lo, int64_t *step_mid, int64_t *step_hi, int32_t *step_kind,
                         int64_t *nsteps_out, int32_t *nlevels_out);
int rla_sptrsv_transpose_in_f64(const double *b_dev, int64_t m, int64_t n, int64_t ldb,
                                const int32_t *perm_dev, double *x_dev, int64_t ldx, void *stream);
int rla_sptrsv_transpose_out_f64(const double *x_dev, int64_t m, int64_t n, int64_t ldx,
                                 const int32_t *perm_dev, double *out_dev, int64_t ldo, void *stream);
int rla_sptrsv_group_inverses_host(int64_t n, const int64_t *rowptr2, const int32_t *col2, const double *val2,
                                   const double *diag_in, const int64_t *split, int64_t ngroups,
                                   const int64_t *grp_start, const int32_t *grp_rows,
                                   const int64_t *dinv_ptr, double *dinv_out, double *diag_eff_out);
int rla_sptrsv_solve_f64(const int64_t *rowptr_dev, const int32_t *col_dev, const double *val_dev,
                         const double *diag_eff_dev, const int64_t *split_dev,
                         const int64_t *grp_start_dev, const int32_t *grp_rows_dev,
                         const int64_t *dinv_ptr_dev, const double *dinv_dev,
                         const int64_t *step_lo_host, const int64_t *step_hi_host, const int32_t *step_kind_host,
                         int64_t nsteps, double *x_dev, int64_t m, int64_t ldx, void *stream);
/* out[p, :] = in[map[p], :] on (n, ldx) blocks: re-ordering between the schedules of L and U */
int rla_sptrsv_permute_rows_f64(const double *in_dev, const int32_t *map_dev, double *out_dev,
                                int64_t n, int64_t ldx, void *stream);

/* ------------------------------------------- row-sharded exchange (K5) -----
 * The one exchange step of the row-sharded sketch (SURVEY.md section 8e; no reference
 * analogue: the reference is single-process).  Each rank owns ONE peer buffer (cudaMalloc,
 * zero-filled) that the other ranks of the node map through CUDA IPC:
 *   rla_peer_buffer_create  allocates it and returns the 64-byte IPC handle to hand to the peers,
 *   rla_peer_buffer_open    maps a peer's buffer into this process (NVLink P2P),
 *   rla_peer_buffer_close / _destroy  undo the two.
 * rla_peer_allreduce_f64 sums the (m, k) partial sketches of all ranks in rank order into
 * out_dev (bit-identical on every rank): part_ptrs[p] / flag_ptrs[p] are HOST arrays of this
 * process's device addresses of rank p's partial and of rank p's flag row (>= world uint64,
 * zero before the first call); `epoch` must be 1, 2, 3, ... over successive calls on the same
 * flag rows and the caller alternates between two partial buffers by epoch parity.
 * high_dev (k int32, may be NULL): sample i of rank p's partial is multiplied by
 * (-1)^popcount(high_dev[i] & p), the slab factor of H_{2^d} = H_G (x) H_{2^d/G}.
 * status_dev: one int32 set to 1 if a peer did not publish within timeout_s seconds. */
int rla_peer_buffer_create(size_t bytes, void **dev_ptr, unsigned char *handle64);
int rla_peer_buffer_open(const unsigned char *handle64, void **dev_ptr);
int rla_peer_buffer_close(void *dev_ptr);
int rla_peer_buffer_destroy(void *dev_ptr);
int rla_peer_allreduce_f64(const void *const *part_ptrs, void *const *flag_ptrs, int world, int rank,
                           uint64_t epoch, int64_t m, int64_t k, int64_t ldp,
                           const int32_t *high_dev, double *out_dev, int64_t ldo,
                           int *status_dev, double timeout_s, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RLA_B200_H */
