/*
 * cave_b200.h — C ABI of the B200-native CaVE cone-projection backend (solver='cuda').
 *
 * This is the drop-in boundary for ONE path of khalil-research/CaVE: the batched
 * projection + push-inside + cosine loss + reduction + analytic backward that the
 * reference computes in src/cave.py:55-73 (forward), :121-129 / :197-219
 * (_get_projection), :222-228 (_average_ctrs), :231-264 (_batch_project) and
 * :298-309 (_project_nnls -> scipy.optimize.nnls).  The reference has no FFI of its
 * own (it is pure Python); the seam these entry points replace is the batched early
 * return of _batch_project (src/cave.py:242-244, the `solver == "apgd"` hook), bound
 * from Python with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no C++/torch types; no exceptions.
 *  - Every pointer is a DEVICE pointer unless stated.  The caller owns and allocates every
 *    buffer (including pack and scratch); the library never allocates, frees or keeps a
 *    pointer after the call returns.  Inputs are read-only.
 *  - Calls only enqueue work on `stream` (a cudaStream_t passed as void*) and return
 *    without synchronising.  Re-entrant across streams given distinct pack/scratch.
 *  - Return value: 0 on success, a negative CAVE_E* code otherwise; cave_last_error()
 *    returns a thread-local message for the last failure on the calling thread.
 *  - `A` is the reference's collate_fn layout (src/dataset.py:133-144): float32
 *    [B, m_max, d] row-major contiguous, all-zero rows are padding.  It may be over-read
 *    by < 16 bytes on either side inside the enclosing 16-byte aligned granules.
 */
#ifndef CAVE_B200_H
#define CAVE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CAVE_B200_ABI_VERSION 4

/* error codes */
#define CAVE_OK 0
#define CAVE_EINVAL (-1)    /* bad argument (null pointer, bad enum, size <= 0)          */
#define CAVE_ELIMIT (-2)    /* shape outside the supported range (see cave_limits)         */
#define CAVE_ENOSPC (-3)    /* pack / scratch buffer too small                             */
#define CAVE_ECUDA (-4)     /* a CUDA runtime call failed (message in cave_last_error)     */

/* mode: which target the loss is taken against */
#define CAVE_MODE_EXACT 0      /* exactConeAlignedCosine            (src/cave.py:121-129)          */
#define CAVE_MODE_INNER 1      /* innerConeAlignedCosine QP branch, nnls push-inside (:206-219)    */
#define CAVE_MODE_HEURISTIC 2  /* innerConeAlignedCosine heuristic branch, no solve  (:201-204)    */

/* reduction (optModule._reduce, called at src/cave.py:73) */
#define CAVE_REDUCE_MEAN 0
#define CAVE_REDUCE_SUM 1
#define CAVE_REDUCE_NONE 2

/* dtypes */
#define CAVE_F32 0
#define CAVE_F64 1

/* per-instance status word written by the solver (never a silent NaN) */
#define CAVE_ST_CONVERGED 0
#define CAVE_ST_ITER_CAP 1      /* iteration cap hit; result is the best iterate           */
#define CAVE_ST_STALLED 2       /* line search could not make progress                     */
#define CAVE_ST_NOSPACE 3       /* instance exceeds scratch caps; outputs are NaN          */
#define CAVE_ST_SKIPPED 4       /* heuristic mode or empty cone: no solve was needed       */
#define CAVE_ST_BADINPUT 5      /* NaN / Inf in the prediction: no solve, outputs are NaN  */
#define CAVE_ST_PATH_LH 0x100   /* flag: solved by the Lawson-Hanson path (else Newton)    */
#define CAVE_ST_PATH_GRAM 0x200 /* flag: solved by the dense path (tensor-core Gram + Gram-space Newton) */
#define CAVE_ST_WARM 0x400      /* flag: the Newton solve (structured, or dense with CAVE_ST_PATH_GRAM) started from the
                                   instance's warm-start slot (cave_forward_backward_warm / _warm_ex;
                                   never set without one)                                           */

typedef struct cave_solver_opts {
    int32_t max_iter;        /* Newton iterations / LH pivots cap; <= 0 -> default (200 / 3*m) */
    int32_t max_linesearch;  /* Armijo halvings cap; <= 0 -> default 40                        */
    double tol;              /* KKT tolerance relative to max||a_i||_1 * ||c||; <= 0 -> default
                                1e-12 (the residuals are float64 in both compute modes)        */
    int64_t cap_rows;        /* scratch sizing: max general (non-singleton) rows per instance;
                                <= 0 -> m_max                                                  */
    int64_t cap_nnz;         /* scratch sizing: max non-zeros in those rows; <= 0 -> cap_rows*d */
    int32_t warm_pack;       /* 1: `pack` already holds cave_pack() output for this A          */
    int32_t dense_mode;      /* dense (tensor-core Gram) path for instances without singleton rows and >= 128 rows:
                                0 auto (enabled when 128 <= m_max <= d: structured models always have m > d),
                                1 on (any instance with 128 <= rows <= 2048 and no singleton row), -1 off.
                                When on, cave_scratch_bytes() includes the Gram workspace.                */
    /* Device-resident dataset (optional, needs warm_pack): `pack` was built by cave_pack() over ALL
     * n_packed instances of a dataset ([n_packed, m_max, d]); instance b of this call is dataset instance
     * inst_index[b] (device pointer, int32[B], values in [0, n_packed)).  `A` is then the dataset tensor,
     * or NULL if it is not resident (instances whose general rows did not fit the packed CSR report
     * CAVE_ST_NOSPACE).  Replaces DataLoader + collate_fn re-padding every batch (src/dataset.py:133-144). */
    const int32_t* inst_index;
    int64_t n_packed;        /* 0 / ignored unless inst_index is set                                   */
    int64_t dense_slots;     /* dense path: instances whose Gram workspace is resident at once (the batch is processed
                                in ceil(B / dense_slots) rounds); <= 0 -> default (8 per SM, at most ~24 GiB)      */
} cave_solver_opts;

typedef struct cave_limits {
    int64_t max_d;       /* cost coefficients per instance             */
    int64_t max_m;       /* padded rows per instance                   */
    int64_t max_batch;   /* instances per call                         */
} cave_limits;

int cave_abi_version(void);
/* Kernels this library has launched in the calling process so far (every entry point counts its own launches);
 * bench.py reports the difference over its timed region as `gpu_launches`. */
unsigned long long cave_launch_count(void);
const char* cave_last_error(void);
int cave_get_limits(cave_limits* out);

/* Bytes of the device-resident packed description of A (per-row classes, per-coordinate
 * singleton cone types, average normal).  Replaces what `_average_ctrs` (src/cave.py:222-228)
 * and the row mask of `_project_nnls` (src/cave.py:303) recompute on every call. */
int cave_pack_bytes(int64_t B, int64_t m_max, int64_t d, size_t* out);

/* Diagnostics for the solve kernel's launch plan.  cave_pack() ends with a small kernel that reduces the
 * instances' shared-memory footprints into 8 uint64 statistics stored in the pack at cave_plan_offset(); the solve
 * kernel is enqueued in every candidate configuration and the statistics select one ON THE DEVICE (no host
 * round trip).  cave_plan_choice() applies the same rule to a host copy of those 8 words and returns the index
 * of the configuration that runs (threads per CTA, CTAs per SM, dynamic shared memory per CTA).  Word 5 is the dynamic
 * shared memory of configuration 4 (256 threads, one CTA per SM) when the pack's shape enqueues it (structured
 * instances with d > 2048), 0 otherwise; configuration 4 is chosen only when the largest hot set fits it but not
 * configuration 3. */
int cave_plan_offset(int64_t B, int64_t m_max, int64_t d, size_t* out);
int cave_plan_choice(const uint64_t* plan_host, int64_t d, int io_dtype, int compute_dtype,
                     int* threads, int* ctas_per_sm, int* smem_bytes);

/* Diagnostics for the dense path: offset inside the scratch buffer of its control block: int32[16] ([0] = number of
 * instances of the last call that took the dense path), followed by uint64[16] phase clocks that only builds with
 * -DCAVE_DENSE_PROFILE fill (tools/dense_profile.py). */
int cave_dense_ctrl_offset(int64_t B, int64_t m_max, int64_t d, const cave_solver_opts* opts, size_t* out);

/* Bytes of solver scratch (per-CTA sparse rows, Hessian, vectors, work counter). */
int cave_scratch_bytes(int64_t B, int64_t m_max, int64_t d, int compute_dtype,
                       const cave_solver_opts* opts, size_t* out);

/* One streaming pass over A (HBM bound): classifies every row (padding / singleton +-e_k /
 * general), accumulates the average unit normal, and writes the packed description; two small
 * kernels then add the solve kernel's launch-plan statistics and the cost-ordered instance list.
 * m_rows: optional int32[B] with the number of leading rows that can be non-zero per instance
 * (rows >= m_rows[b] are not read); NULL -> all m_max rows are scanned. */
int cave_pack(const float* A, const int32_t* m_rows, int64_t B, int64_t m_max, int64_t d,
              void* pack, size_t pack_bytes, void* stream);

/* cave_pack with flags: bit 0 = also emit the cached per-instance solver setup (cave_pack() sets it; a pack that is used
 * once does without: the setup kernel costs about what one solve saves). */
int cave_pack_ex(const float* A, const int32_t* m_rows, int64_t B, int64_t m_max, int64_t d, int32_t flags,
                 void* pack, size_t pack_bytes, void* stream);

/* Sparse ingestion: the same pack built from the non-zeros of the binding-constraint rows instead of the dense padded
 * tensor (every shipped model is 0.7 % dense at TSP-50: 90 KB instead of 6.5 MB per instance cross PCIe and HBM).
 * Replaces DataLoader + collate_fn's dense zero padding (src/dataset.py:114-144) for callers that keep `dataset.ctrs`
 * sparse.  Device pointers: rows [inst_off[b], inst_off[b+1]) of row_ptr belong to instance b (at most m_max, in the
 * reference's row order); row r holds the entries [row_ptr[r], row_ptr[r+1]) of col / val, columns ascending, explicit
 * zeros ignored.  flags bit 0: also emit the cached solver setup (worth it when the pack is reused across steps).
 * The pack is then used with opts->warm_pack (and opts->inst_index); A may be NULL in cave_forward_backward, in which
 * case instances that need the dense rows (no singleton row at all, or general rows beyond the packed-CSR capacity)
 * report CAVE_ST_NOSPACE. */
int cave_pack_sparse(const int64_t* inst_off, const int64_t* row_ptr, const int32_t* col, const float* val, int64_t B,
                     int64_t m_max, int64_t d, int32_t flags, void* pack, size_t pack_bytes, void* stream);

/* The hot path.  pred: [B,d] predicted costs (io_dtype).  sign: -1 for EPO.MINIMIZE, +1 for
 * EPO.MAXIMIZE (src/cave.py:62-68).  Outputs (io_dtype unless noted; any of proj, rnorm,
 * status, iters, loss may be NULL):
 *   loss    [1]   reduced loss for MEAN / SUM (ignored for NONE)
 *   loss_i  [B]   per-instance 1 - cos(c, target)                        (required)
 *   grad    [B,d] d(reduced loss)/d pred for an upstream gradient of 1   (required)
 *   proj    [B,d] projection of c = sign*pred onto the cone  (what _batch_project returns)
 *   rnorm   [B]   ||proj - c||_2                               (nnls meaning, src/cave.py:307)
 *   status  [B]   int32 CAVE_ST_*;   iters [B] int32 solver iterations
 * Unless opts->warm_pack is set, cave_pack() is run first on the same stream — in CAVE_MODE_EXACT without the average
 * unit normal, which that mode never reads (the pack is marked: a later warm call with it in another mode reports
 * CAVE_ST_BADINPUT for every instance; build packs that are shared between modes with cave_pack()). */
int cave_forward_backward(const float* A, const int32_t* m_rows, const void* pred,
                          int64_t B, int64_t m_max, int64_t d,
                          double sign, int mode, double inner_ratio, int reduction,
                          int io_dtype, int compute_dtype, const cave_solver_opts* opts,
                          void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                          int32_t* status, int32_t* iters,
                          void* pack, size_t pack_bytes, void* scratch, size_t scratch_bytes,
                          void* stream);

/* Warm start of a resident pack.  The structured Newton solve of pack instance q normally starts from nu = 0; with a
 * warm-start buffer it starts from the multipliers of q's last converged solve, which the call stores back.  The buffer
 * holds one fixed-size slot per pack instance (a header and at most min(m_max, 256) float64 multipliers); an all-zero
 * buffer is a buffer of empty slots, so a reset is a memset.  cave_warm_bytes(): bytes for n_instances (the n_packed of
 * an indexed call, B otherwise).
 * cave_forward_backward_warm(): cave_forward_backward plus the buffer (device pointer, 16-byte aligned).  It needs
 * opts->warm_pack = 1 (CAVE_EINVAL otherwise) and warm_bytes >= cave_warm_bytes() (CAVE_ENOSPC otherwise).  The slot of
 * batch row b is inst_index[b], or b without an index.
 *  - A slot is used only if it holds a solution for the same variables (count and a hash of the structure); its values
 *    are a starting guess (non-finite entries become 0, bounded ones are clamped to >= 0).  Such instances report
 *    CAVE_ST_WARM.  If a warm start ends CAVE_ST_ITER_CAP or CAVE_ST_STALLED, the instance is solved once more from zero
 *    in the same call (iters is the sum; CAVE_ST_WARM is then clear): a warm start never ends worse than a cold one.
 *  - A slot is written only by a structured (Newton) instance that ends CAVE_ST_CONVERGED.  Lawson-Hanson and dense-path
 *    instances, heuristic mode, empty cones, NaN / Inf predictions and instances with more variables than a slot holds
 *    leave it untouched.
 *  - Calls that share one buffer must be ordered (one stream), as calls that share a pack or scratch are.  An index may
 *    hold an instance twice: the slot is then read and written concurrently, which can only change the starting guess. */
int cave_warm_bytes(int64_t n_instances, int64_t m_max, int64_t d, size_t* out);
int cave_forward_backward_warm(const float* A, const int32_t* m_rows, const void* pred,
                               int64_t B, int64_t m_max, int64_t d,
                               double sign, int mode, double inner_ratio, int reduction,
                               int io_dtype, int compute_dtype, const cave_solver_opts* opts,
                               void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                               int32_t* status, int32_t* iters,
                               void* pack, size_t pack_bytes, void* scratch, size_t scratch_bytes,
                               void* warm, size_t warm_bytes, void* stream);

/* Warm start of the dense Gram-space Newton solve (CAVE_ST_PATH_GRAM), with a second buffer of the same kind: one slot per
 * pack instance, a 16-byte header (valid, m, a hash of the rows' indices and lengths, and whether the solve ended with the
 * diagonal metric) and at most min(m_max, 2048) float64 multipliers lambda in the instance's general-row order; all zero =
 * all empty.  cave_dense_warm_bytes(): bytes for n_instances, as cave_warm_bytes().
 * cave_forward_backward_warm_ex(): cave_forward_backward_warm plus warm_dense.  Either buffer may be null, not both
 * (CAVE_EINVAL); it needs opts->warm_pack = 1 (CAVE_EINVAL); each buffer must be 16-byte aligned (CAVE_EINVAL) and hold
 * the pack's instances (CAVE_ENOSPC).  The structured solve uses warm as above; a null warm_dense keeps the dense path cold.
 *  - A dense instance whose slot holds a solution for the same rows starts from it (non-finite and negative values become
 *    0), skips the Gram-space phase and iterates on the true problem at once; it reports CAVE_ST_WARM.  If that ends
 *    CAVE_ST_ITER_CAP or CAVE_ST_STALLED, would hand the instance back to Lawson-Hanson, or starts from a point that fits
 *    worse than lambda = 0, the instance is solved once more from zero in the same call (iters is the sum; CAVE_ST_WARM is
 *    then clear).  Only that cold solve may hand the instance back.
 *  - A slot is written only by a dense instance that ends CAVE_ST_CONVERGED on the dense path.  Instances handed back,
 *    Lawson-Hanson and structured instances, heuristic mode (no dense path) and NaN / Inf predictions leave it untouched.
 *  - Ordering and duplicate indices: as for warm. */
int cave_dense_warm_bytes(int64_t n_instances, int64_t m_max, int64_t d, size_t* out);
int cave_forward_backward_warm_ex(const float* A, const int32_t* m_rows, const void* pred,
                                  int64_t B, int64_t m_max, int64_t d,
                                  double sign, int mode, double inner_ratio, int reduction,
                                  int io_dtype, int compute_dtype, const cave_solver_opts* opts,
                                  void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                                  int32_t* status, int32_t* iters,
                                  void* pack, size_t pack_bytes, void* scratch, size_t scratch_bytes,
                                  void* warm, size_t warm_bytes, void* warm_dense, size_t warm_dense_bytes,
                                  void* stream);

/* Gram cache of a resident dense dataset: G~ = A A^T of every pack instance the dense path could take, computed once, so
 * that later calls with the pack run neither the TF32 split nor the Gram kernel for their dense instances.  A caller-owned
 * buffer over the N instances of a pack built by cave_pack():
 *   [0]     int32 header: valid (1 once built), n_cached, m_pad (m_max rounded up to 128), N
 *   [16]    int32 map[N]: the cache slot of pack instance q, or -1
 *   [base]  base = (16 + 4 N) rounded up to 1024: n_cached slots of float32 [m_pad][m_pad], G~ of the instance's valid
 *           rows in order, both triangles, zero outside the instance's leading square of 128-row blocks.
 * An instance has a slot if it has no singleton row, >= 128 rows that are all general rows, and m_pad <= 2048: every
 * instance that a call with any dense_mode puts on the dense path.
 * cave_gram_cache_count(): the number of such instances of the pack into *n_cached_dev (device memory, on the stream).
 * cave_gram_cache_bytes(): bytes of a cache for N instances with n_cached slots.
 * cave_gram_cache_build(): fills the cache from A and its pack (cave_pack of the same A) with the same prep and Gram kernels
 * a call runs; scratch must hold cave_scratch_bytes(N, ...) with dense_mode = 1 and the same opts (opts->dense_slots
 * instances per round).  The buffer should be zeroed beforehand; it needs at least cave_gram_cache_bytes(N, 0, ...) bytes
 * (CAVE_ENOSPC) and 16-byte alignment (CAVE_EINVAL); one that holds fewer than n_cached slots stays invalid.  Shapes
 * outside the dense path: CAVE_ELIMIT (the count is then 0).
 * cave_forward_backward_resident(): cave_forward_backward_warm_ex plus the cache.  Any of warm, warm_dense and gram may be
 * null, not all three (CAVE_EINVAL); it needs opts->warm_pack = 1 (CAVE_EINVAL); gram needs A and 16-byte alignment
 * (CAVE_EINVAL) and at least cave_gram_cache_bytes(pack instances, 0, ...) bytes (CAVE_ENOSPC).  Results are bit-identical to
 * the same call without the cache.  A dense instance whose cache is not valid for this pack (header, m_pad, N or slot)
 * reports CAVE_ST_BADINPUT | CAVE_ST_PATH_GRAM with NaN outputs.  Calls without the dense path (heuristic mode,
 * dense_mode < 0, or a shape the host gate keeps off it) ignore the cache.  The cache is only read; it stays valid as long
 * as A is not modified. */
int cave_gram_cache_count(const void* pack, size_t pack_bytes, int64_t N, int64_t m_max, int64_t d, int32_t* n_cached_dev,
                          void* stream);
int cave_gram_cache_bytes(int64_t N, int64_t n_cached, int64_t m_max, int64_t d, size_t* out);
int cave_gram_cache_build(const float* A, int64_t N, int64_t m_max, int64_t d, const cave_solver_opts* opts,
                          void* cache, size_t cache_bytes, const void* pack, size_t pack_bytes,
                          void* scratch, size_t scratch_bytes, void* stream);
int cave_forward_backward_resident(const float* A, const int32_t* m_rows, const void* pred,
                                   int64_t B, int64_t m_max, int64_t d,
                                   double sign, int mode, double inner_ratio, int reduction,
                                   int io_dtype, int compute_dtype, const cave_solver_opts* opts,
                                   void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                                   int32_t* status, int32_t* iters,
                                   void* pack, size_t pack_bytes, void* scratch, size_t scratch_bytes,
                                   void* warm, size_t warm_bytes, void* warm_dense, size_t warm_dense_bytes,
                                   const void* gram, size_t gram_bytes, void* stream);

/* Diagnostic for the dense regime (north_star item 1): runs cave_pack() on A and then only the TF32 split and the
 * tensor-core Gram kernel (TMA tiles -> tcgen05.mma, 3xTF32, float32 accumulation in TMEM) for the first
 * min(B, slots) instances, and copies G~ = A A^T of instance i to G_out[i] as a row-major [m_pad, m_pad] float32
 * matrix (m_pad = m_max rounded up to 128; rows are the VALID rows of A in order; entries beyond the valid rows of
 * an instance's last 128-row block are zero, beyond that block unspecified).  Every instance must be dense
 * (no singleton row, >= 128 valid rows).  The parity tests compare it with a float64 product of the same rows.
 * scratch must hold cave_scratch_bytes() with dense_mode = 1. */
int cave_dense_gram(const float* A, int64_t B, int64_t m_max, int64_t d, const cave_solver_opts* opts,
                    float* G_out, int32_t* n_dense_out, void* pack, size_t pack_bytes,
                    void* scratch, size_t scratch_bytes, void* stream);

/* Auxiliary, evaluation only (not on the hot path): exact symmetric TSP by Held-Karp dynamic programming for
 * n_nodes <= 20, one CTA per instance.  Decision regret (BASELINE.json configs[1]; the reference's code_sample.py
 * evaluates with pyepo.metric.regret, which calls Gurobi through src/model/tsp.py) needs optimal tours under predicted
 * and true costs.  cost: [N, n(n-1)/2] float32 edge costs, edges (i<j) in lexicographic order; tour: [N, n_nodes]
 * node sequence starting at 0; obj: [N] float64 tour length.  scratch: cave_tsp_scratch_bytes(). */
int cave_tsp_scratch_bytes(int64_t N, int32_t n_nodes, size_t* out);
int cave_tsp_solve(const float* cost, int64_t N, int32_t n_nodes, int32_t* tour, double* obj, void* scratch, size_t scratch_bytes,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CAVE_B200_H */
