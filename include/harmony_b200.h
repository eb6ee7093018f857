/* harmony_b200.h -- C ABI of the Blackwell-native Harmony inner-loop engine.
 *
 * slowkow/harmonypy has no FFI: its boundary is the Python class ``Harmony``
 * (harmonypy/harmony.py:218-569).  Each entry point below replaces one method (or the
 * device-state part of one method) of that class; the Python host in
 * harmonypy_b200/harmony.py keeps the reference's driver logic (harmonize / cluster loop /
 * check_convergence, harmony.py:419-462, :515-533) verbatim in behaviour and calls these
 * through ctypes.  INTEGRATION.md shows the stub a harmonypy maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; hmy_last_error(ctx) gives
 *     the message (hmy_last_error(NULL) for failures of hmy_create itself);
 *   - "host" pointers are ordinary (pageable or pinned) host memory owned by the caller;
 *     the library owns every device allocation it makes;
 *   - one context per GPU / per rank, not thread-safe; all work is enqueued on the stream
 *     given to hmy_set_stream (default: the legacy default stream);
 *   - matrices cross the boundary CELL-MAJOR: Z is n_cells x d (row stride d), R is
 *     n_cells x K, codes are V x n_cells.  Y is K x d (one centroid per row).  O and E are
 *     K x B (row stride B) like the reference's properties (harmony.py:313-321);
 *   - B = sum(levels_per_var) one-hot rows in pd.get_dummies order (harmony.py:133):
 *     covariate-major, level-minor.  Level codes are 0-based within their covariate.
 *
 * Limits (the reference has none; hmy_create / hmy_set_params fail with the reason, the Python host checks them first):
 *   d <= 128 PCs, 2 <= K <= 256 clusters, <= 8 batch covariates, <= 250 blocks (block_size >= 0.004), B <= 65535 levels.
 *   The tensor-memory round kernel (K <= 128, d <= 64, <= 32 blocks) has no limit on B; the other round kernels keep
 *   two K x B tables per CTA in shared memory (about 250 levels at K = 100) and fail beyond that.
 *   hmy_lisi_compute: 3 * perplexity <= 128 neighbours.
 */
#ifndef HARMONY_B200_H
#define HARMONY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hmy_ctx hmy_ctx;

/* Matrices readable with hmy_get (mirrors the NumPy properties, harmony.py:288-351). */
enum hmy_matrix {
    HMY_Z_CORR = 0, /* float  n_local x d   harmony.py:289-291 */
    HMY_Z_COS  = 1, /* float  n_local x d   harmony.py:299-301 */
    HMY_Z_ORIG = 2, /* float  n_local x d   harmony.py:294-296 */
    HMY_R      = 3, /* float  n_local x K   harmony.py:304-306 */
    HMY_Y      = 4, /* float  K x d (unit rows; transpose of harmony.py:309-311) */
    HMY_O      = 5, /* double K x B         harmony.py:314-316 */
    HMY_E      = 6, /* double K x B         harmony.py:319-321 */
    HMY_W      = 7, /* float  B x K x d  ridge coefficients of the last hmy_ridge_correct */
    HMY_TRACE  = 9  /* uint64 (grid + 1) x 256 timeline stamps of the last round kernel (option "trace") */
};

/* Optional caller-supplied sum-all-reduce over ranks, called at the reduction points of the
 * staged multi-GPU mode with a DEVICE pointer; must enqueue on (or synchronise with)
 * `stream`.  dtype: 0 = float32, 1 = float64. */
typedef int (*hmy_allreduce_fn)(void* user, void* dev_ptr, int64_t count, int dtype, void* stream);

const char* hmy_version(void);
const char* hmy_last_error(const hmy_ctx* ctx);

/* Page-locked ("pinned") host memory, usable from every device of the process.  hmy_set_data and hmy_get recognise
 * arrays that live in page-locked memory (from here, cudaHostAlloc / cudaHostRegister, torch pinned tensors) and move
 * them with ONE DMA; pageable arrays are staged through the context's two pinned 16 MB buffers by a few host threads.
 * hmy_host_alloc returns NULL on failure (no GPU, out of lockable memory); hmy_host_free(NULL) is a no-op. */
void* hmy_host_alloc(int device, size_t bytes);
void  hmy_host_free(void* p);

/* State owner.  Replaces Harmony.__init__ buffers + allocate_buffers (harmony.py:224-271,
 * :357-364).  n_local cells live on this rank; they are cells [cell_offset, cell_offset +
 * n_local) of the n_global cells the permutation indexes. */
int hmy_create(hmy_ctx** out, int device, int64_t n_local, int64_t n_global, int64_t cell_offset,
               int d, int K, int V, const int32_t* levels_per_var);
void hmy_destroy(hmy_ctx* ctx);
int hmy_set_stream(hmy_ctx* ctx, void* cuda_stream);

/* Run parameters (harmony.py:242, :262-271): Pr_b[B], theta[B], sigma[K], lamb[B+1]
 * (lamb[0] is the intercept's 0; ignored when lambda_estimation != 0, harmony.py:541-544). */
int hmy_set_params(hmy_ctx* ctx, const float* Pr_b, const float* theta, const float* sigma,
                   const float* lamb, int lambda_estimation, float alpha, double block_size);

/* Upload this rank's cells: Z (n_local x d, fp32) and level codes (V x n_local, int32).
 * Builds Z_cos (harmony.py:234-238).  Replaces the dense Phi / Phi_moe / batch_index
 * construction (harmony.py:241-256) with integer codes. */
int hmy_set_data(hmy_ctx* ctx, const float* Z_host, const int32_t* codes_host);

/* Tail of init_cluster after sklearn (harmony.py:373-392): normalise the K x d centroids,
 * R = softmax_k(-dist/sigma), O, E, and the three objective sums
 * obj[0] = sum R*dist, obj[1] = sum sigma*R*log R, obj[2] = cross-entropy term
 * (harmony.py:399-411; NOT yet multiplied by 2000/N). */
int hmy_init_from_centroids(hmy_ctx* ctx, const float* Y0_host_Kxd, double obj[3]);

/* Optional replacement of the sklearn call in init_cluster (harmony.py:369-373: KMeans(init="k-means++",
 * n_init=1, max_iter=25) on the unit-length cells) for sizes where it dominates the wall time: k-means++
 * seeding and Lloyd iterations on the resident Z_cos, stopped by sklearn's criterion (squared centre shift <=
 * tol * mean feature variance) or after max_iter iterations.  It cannot reproduce sklearn's random stream:
 * parity configurations keep sklearn and pass the centroids to hmy_init_from_centroids.
 * Y_host: K x d means (feed them to hmy_init_from_centroids); info: iterations run, inertia of the last
 * assignment pass, last squared centre shift (may be NULL).
 *
 * Cells sharded over ranks (n_local < n_global): a COLLECTIVE call -- every rank calls it with the same seed, max_iter
 * and tol, after hmy_set_allreduce and hmy_set_rank (or hmy_comm_attach); it fails before any all-reduce when either is
 * missing.  The ranks' cell ranges must cover the n_global cells exactly once; n_global >= K is required (a shard may
 * hold fewer than K cells), n_global <= 2^32.  The seeds are exactly the cells a single GPU holding all cells picks
 * (the race keys depend on the global cell id only); the Lloyd sums, counts and inertia are summed over ranks.  Every
 * rank returns the same Y_host and info (rank 0's): global inertia and shift.  Cost: 1 all-reduce of 10 x world
 * doubles for the checks, K of world x (2 + d') doubles for the seeding (d' = d rounded up to 4), 2 per Lloyd
 * iteration (K (d' + 1) + 1 doubles and 1 double), 1 of K d' + 3 doubles at the end.  All ranks fail together when any rank's checks or
 * allocations fail, or when they disagree on K, d, n_global or the arguments. */
int hmy_kmeans_init(hmy_ctx* ctx, uint64_t seed, int max_iter, double tol, float* Y_host_Kxd, double info[3]);

/* One iteration of the loop body of cluster() (harmony.py:443-453): centroid update,
 * cosine distances, blockwise update_R (harmony.py:464-513), objective.
 * perm_host: the n_global-long randperm of harmony.py:471 (int64, host) or NULL to draw a
 * device-side pseudo-random permutation from (seed, round counter). */
int hmy_kmeans_round(hmy_ctx* ctx, const int64_t* perm_host, double obj[3]);

/* Contexts with counter "lookahead" = 1: hmy_kmeans_round(ctx, perm, NULL) enqueues the round without waiting for its
 * objective sums, so that the rounds whose objective cannot stop the loop yet (harmony.py:455-458: the first four of a
 * cluster() call) run back to back with no host round trip in between; hmy_objectives then waits once and returns the
 * sums of the last n stages (oldest first, 3 doubles each, n <= 16).  With "lookahead" = 0 obj must not be NULL. */
int hmy_objectives(hmy_ctx* ctx, int n, double* obj_3n);

/* Contexts whose counter "lookahead" is 1 (the tensor-memory round kernel: one GPU, or several with the peer exchange
 * of hmy_comm_attach) run the
 * block permutations ONE ROUND AHEAD: a round already accumulates, per block of the NEXT round, the sums that round
 * will remove from O (harmony.py:491-492), so it must know the next round's blocks.  Call order there:
 *     hmy_queue_perm(perm of round 0)            (omit with device-side permutations)
 *     hmy_init_from_centroids(...)
 *     hmy_kmeans_round(perm of round 1, ...)     runs round 0
 *     hmy_kmeans_round(perm of round 2, ...)     runs round 1 ...
 * i.e. the same stream of torch.randperm draws as harmony.py:471, each handed over one call earlier.  With
 * "lookahead" 0 hmy_kmeans_round takes the permutation of the round it runs and hmy_queue_perm fails. */
int hmy_queue_perm(hmy_ctx* ctx, const int64_t* perm_host);

/* moe_correct_ridge (harmony.py:535-569): per-cluster ridge regression, Z_corr, Z_cos. */
int hmy_ridge_correct(hmy_ctx* ctx);

/* Property reads (harmony.py:288-351).  Cells come back in the caller's original order. */
int hmy_get(hmy_ctx* ctx, int which, void* host_out, int64_t bytes);

int hmy_synchronize(hmy_ctx* ctx);

/* Options (unknown names fail):
 *   "persistent" 0/1   one cooperative kernel per round (default) vs one launch per block step
 *   "seed"       int   seed of the device-side permutation (perm_host == NULL)
 *   "mma"        0/1   tensor-core round kernels (default, d <= 64) vs fp32 SIMT; before hmy_set_params
 *   "ridge_mma"  0/1   tensor-core ridge passes (default, d <= 63) vs fp32 SIMT; before hmy_set_params
 *   "mma_wn"     0/2   force two warps along the cluster axis (A/B runs); before hmy_set_params
 *   "tc5"        -1/0/1 tcgen05 / tensor-memory round kernel (hmy_round_tc5.cuh; K <= 128, d <= 64, <= 32 blocks,
 *                      single-GPU persistent mode): -1 = where it applies (default), 0 = never, 1 = required
 *                      (other shapes FAIL); before hmy_set_params
 *   "write_r"    0/1   lookahead contexts only: the next stages store R to HBM (default 1).  With 0 the rounds skip
 *                      the 4K bytes per cell; hmy_ridge_correct and hmy_get(HMY_R) fail until a stage ran with 1
 *   "relaxed"    0/1   fused multi-GPU mode: exchange the K x B table once per round instead of once
 *                      per block (NOT exact; default 0)
 *   "dbg"        bits  timing experiments on the tensor-memory round kernel (skips parts of its work: results are WRONG
 *                      when non-zero; default 0)
 *   "timing"     0/1   CUDA-event timers around the stages (default 1)
 *   "reset"      1     back to the state right after hmy_set_data (benchmark restarts)
 *   "trace"      1     per-CTA timeline of the round kernel, read with hmy_get(HMY_TRACE) */
int hmy_set_option(hmy_ctx* ctx, const char* name, int64_t value);

/* Counters: "launches" (kernels launched by this library since creation), "rounds",
 * "ridge_passes", "grid", "nblk", "ncombo", "mma", "ridge_mma", "fused", "round_threads",
 * "smem_round", "tc5", "lookahead", "r_valid", "dma_direct" (uploads / read-backs that moved with one DMA because the
 * caller's array is page-locked).  Timers (CUDA events on the context stream, milliseconds, cumulative):
 * "ms_round", "ms_ridge", "ms_init".  Unknown names return -1. */
int64_t hmy_counter(const hmy_ctx* ctx, const char* name);
double hmy_timer_ms(hmy_ctx* ctx, const char* name);

/* ---- multi-GPU (cells sharded over ranks; SURVEY.md section 8e) ---------------------- */

/* Staged mode: the library calls `fn` wherever a small table must be summed over ranks. */
int hmy_set_allreduce(hmy_ctx* ctx, hmy_allreduce_fn fn, void* user);

/* This context's rank among `world` ranks (0 <= rank < world), for the collectives of hmy_kmeans_init on sharded cells.
 * Host-side bookkeeping only: the round kernels and the staged / fused mode do not change.  hmy_comm_attach records
 * the rank too. */
int hmy_set_rank(hmy_ctx* ctx, int rank, int world);

/* Fused mode: ranks exchange the small tables inside the persistent round kernel through
 * peer-mapped device memory.  Each rank exports a 64-byte handle of its exchange buffer;
 * the caller all-gathers the handles (any transport) and hands every rank the full list. */
int hmy_comm_export(hmy_ctx* ctx, void* handle_out_64B);
int hmy_comm_attach(hmy_ctx* ctx, int rank, int world, const void* all_handles_world_x_64B);

/* ---- evaluation metric (SURVEY.md section 8f; not on the harmonize() path) ---------------------- */

/* compute_lisi (harmonypy/lisi.py:24-65): exact k = int(3 * perplexity) nearest neighbours of every cell
 * (Euclidean, fp64, the cell itself dropped afterwards like lisi.py:56-57), per-cell bisection on beta until the
 * entropy of exp(-beta * dist) equals log(perplexity) (lisi.py:68-122), inverse Simpson index of each label
 * column under those weights (lisi.py:127-132, :64).
 * X_host: n x d row-major doubles; codes_host: n_labels x n int32 category codes (pd.Categorical codes);
 * out_host: n x n_labels doubles.  Context-free; failures are reported through hmy_last_error(NULL). */
int hmy_lisi_compute(int device, int64_t n, int d, const double* X_host, int n_labels,
                     const int32_t* codes_host, double perplexity, double* out_host);

#ifdef __cplusplus
}
#endif
#endif /* HARMONY_B200_H */
