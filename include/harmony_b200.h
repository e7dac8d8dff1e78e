/* harmony_b200.h — C ABI of libharmony_b200.so: the B200 (sm_100a) implementation of the Harmony
 * hot loop.  One opaque handle == one instance of the reference's C++ class `harmony`
 * (/root/reference/src/harmony.h:20-70); every entry point below replaces the like-named method /
 * field that the reference exposes to R through its Rcpp module (`RCPP_MODULE(harmony_module)`,
 * /root/reference/src/harmony.cpp:672-709).  INTEGRATION.md shows the Rcpp shim that binds them.
 *
 * Conventions
 *   - plain C types only; the library never throws.  Functions returning `int` give 0 on success,
 *     >0 on error (message via hb_last_error), and hb_cluster additionally -1 for "aborted by
 *     user" exactly like harmony::cluster_cpp (/root/reference/src/harmony.cpp:233-234).
 *   - matrices cross the boundary in the reference's layout: column-major with cells as columns
 *     (Z is d x N, R is K x N, Y is d x K, O/E are K x B, lambda matrix is K x (B+1)), doubles,
 *     i.e. exactly the memory of the R numeric matrices the reference takes and returns.
 *   - the sparse design matrix Phi (B x N dgCMatrix, /root/reference/R/ui.R:210-213) is passed as its
 *     row-index slot: every column has exactly C non-zeros (one level per covariate), so
 *     phi_i[n*C + c] is the (global, 0-based) row of the c-th non-zero of column n.
 *   - all buffers are caller-owned host memory; inputs are copied during the call
 *     (like harmony::setup, harmony.cpp:41,44), outputs are written into caller-allocated arrays.
 *     The *_device entry points take / fill caller-owned DEVICE memory instead (cells as rows, any strides).
 *   - a handle must be driven from one host thread at a time (the reference is single-threaded).
 */
#ifndef HARMONY_B200_H
#define HARMONY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hb_handle hb_handle;

/* ---- lifetime: `new(harmony)` (R/ui.R:269) / the external-pointer finaliser ------------------- */
/* device < 0 selects the current CUDA device. */
int hb_create(hb_handle** out, int device);
void hb_destroy(hb_handle* h);
/* Last error text of this handle ("" if none); valid until the next call on the handle. */
const char* hb_last_error(const hb_handle* h);
/* Pops one pending warning (e.g. "Too few cells. Setting block_size to 0.2", harmony.cpp:86-88) into
 * buf; returns 1 if a warning was written, 0 if none is pending.  The shim turns it into Rcpp::warning. */
int hb_pop_warning(hb_handle* h, char* buf, size_t cap);
/* Library/ABI version: major*10000 + minor*100 + patch. */
int hb_version(void);

/* ---- multi-GPU (one process per GPU; cells sharded contiguously; SURVEY §8e) ------------------- */
/* Size of the opaque communicator id (an ncclUniqueId). */
#define HB_COMM_ID_BYTES 128
/* Rank 0 creates the id and ships it to the other ranks by any host-side means (the Python host uses
 * torch.distributed); every rank then calls hb_comm_init BEFORE hb_setup. */
int hb_comm_unique_id(char id[HB_COMM_ID_BYTES]);
int hb_comm_init(hb_handle* h, int rank, int world_size, const char id[HB_COMM_ID_BYTES]);
/* The communicator stays alive for the life of the process; a later handle of the same (device, rank,
 * world_size) may pass id == NULL to share it instead of paying the ~1 s NCCL set-up again. */
/* Declares that this handle holds cells [cell_offset, cell_offset + n_local) of an N_global-cell
 * problem.  Must precede hb_setup; without it the handle owns all cells. */
int hb_set_shard(hb_handle* h, int64_t N_global, int64_t cell_offset);

/* ---- harmony::setup (harmony.h:25-30, harmony.cpp:29-111; called at R/ui.R:271-275) ---------- */
/* Z: d x N(local) column-major doubles.  lambda: B+1 values, or NULL / lambda[0] == -1 for the
 * reference's automatic estimation (harmony.cpp:75-76).  Errors: N < 6 -> status 1 with the
 * reference's message (harmony.cpp:83-85); 6 <= N < 40 -> warning + block_size 0.2 (:86-88). */
int hb_setup(hb_handle* h, const double* Z, int d, int64_t N, const int32_t* phi_i, const int32_t* B_vec, int C,
             const double* sigma, const double* theta, const double* lambda, double alpha, int max_iter_kmeans,
             double epsilon_kmeans, double epsilon_harmony, int K, double block_size,
             double batch_proportion_cutoff, int verbose);

/* Element types of caller device memory (hb_setup_device, hb_get_field_device). */
enum hb_dtype { HB_F32 = 0, HB_F64 = 1 };

/* harmony::setup with the per-cell inputs in device memory of the handle's device.
 * Z: N cells x d PCs, element (n, c) at Z[n*z_cell_stride + c*z_pc_stride] (elements, not bytes), HB_F32/HB_F64.
 *    Covers a contiguous [N, d] tensor, its [d, N] transpose view and column slices, without a copy.
 * phi_i: device int32, N x C row-major, same meaning as hb_setup's phi_i (global level row).
 * B_vec, sigma, theta, lambda and the scalars: host memory, exactly as in hb_setup.
 * stream: the caller's cudaStream_t on which Z and phi_i are ready (NULL = legacy default stream).
 * The inputs are fully consumed before the call returns, so the caller may free them afterwards.
 * The handle ends in the state hb_setup leaves it in for the same values (Z converted to float as hb_setup does). */
int hb_setup_device(hb_handle* h, const void* Z, int z_dtype, int64_t z_cell_stride, int64_t z_pc_stride, int d,
                    int64_t N, const int32_t* phi_i, const int32_t* B_vec, int C, const double* sigma,
                    const double* theta, const double* lambda, double alpha, int max_iter_kmeans,
                    double epsilon_kmeans, double epsilon_harmony, int K, double block_size,
                    double batch_proportion_cutoff, int verbose, void* stream);

/* Seed of the native generators (k-means initialisation, per-round update orders).  The reference
 * draws both from R's RNG (utils.cpp:10-64, harmony.cpp:272-273); the shim may instead inject them. */
int hb_set_seed(hb_handle* h, uint64_t seed);
/* Polled between clustering rounds like Progress::check_abort() (harmony.cpp:233); non-zero -> -1. */
int hb_set_abort_callback(hb_handle* h, int (*cb)(void*), void* user);

/* ---- harmony::init_cluster_cpp (harmony.cpp:131-156) ------------------------------------------ */
/* Y0: d x K column-major initial centroids (what kmeans_centers returns, harmony.cpp:133), or NULL to
 * run the native GPU k-means initialisation. */
int hb_init_cluster(hb_handle* h, const double* Y0);

/* ---- harmony::cluster_cpp (harmony.cpp:208-262) incl. update_R (:269-342) --------------------- */
/* update_orders: max_iter_kmeans x N_global int64 — row t is the `update_order` that
 * arma::shuffle would produce for the t-th update_R call (harmony.cpp:272-273) — or NULL to draw the
 * orders natively on the device.  Returns 0, -1 (aborted) or >0 (error). */
int hb_cluster(hb_handle* h, const int64_t* update_orders);

/* ---- harmony::moe_correct_ridge_cpp (harmony.cpp:345-638) -------------------------------------- */
int hb_moe_correct_ridge(hb_handle* h);

/* ---- harmony::check_convergence (harmony.cpp:173-205): 1 = converged, 0 = not, <0 = error ----- */
int hb_check_convergence(hb_handle* h, int type);

/* ---- harmony::compute_objective (harmony.cpp:158-170): appends to the four objective traces --- */
int hb_compute_objective(hb_handle* h);

/* ---- fields / getters (harmony.cpp:640-669, 675-696) ------------------------------------------- */
enum hb_field {
  HB_Z_CORR = 0, /* getZcorr(): d x N  */
  HB_Z_ORIG = 1, /* getZorig(): d x N  */
  HB_R = 2,      /* R / getR(): K x N  */
  HB_Y = 3,      /* Y / getCentroids(): d x K */
  HB_O = 4,      /* O: K x B */
  HB_E = 5,      /* E: K x B */
  HB_W = 6,      /* W: (B+1) x d, betas of the last corrected cluster (rows of dropped levels are 0) */
  HB_PR_B = 7,   /* Pr_b: B */
  HB_THETA = 8,  /* theta: B */
  HB_SIGMA = 9,  /* sigma: K */
  HB_LAMBDA = 10,    /* getLambda(): K x (B+1) */
  HB_LAMBDA_VEC = 11 /* lambda field: B+1 (only when not estimating) */
};
/* Number of doubles hb_get_field writes for `field` (0 for an unknown field). */
int64_t hb_field_size(const hb_handle* h, int field);
/* Device -> host copy-out with float -> double conversion (conv_to<RMAT>::from, harmony.cpp:640-650).
 * With a sharded handle the per-cell fields return the local shard. */
int hb_get_field(hb_handle* h, int field, double* out);
/* Writable fields (the Rcpp module's .field() members are read-write): HB_Y, HB_R, HB_O, HB_E,
 * HB_THETA, HB_SIGMA, HB_LAMBDA_VEC, HB_Z_CORR. */
int hb_set_field(hb_handle* h, int field, const double* in);
/* Per-cell fields (HB_Z_CORR, HB_Z_ORIG, HB_R) un-sorted into caller device memory: N_local rows of d (or K)
 * values, row stride ld elements, HB_F32 or HB_F64.  Ordered on `stream`: the library waits for the stream
 * before writing and makes the stream wait for the write, so there is no host synchronisation. */
int hb_get_field_device(hb_handle* h, int field, void* out, int dtype, int64_t ld, void* stream);

enum hb_scalar { HB_N = 0, HB_B = 1, HB_K = 2, HB_D = 3, HB_C = 4, HB_ALPHA = 5, HB_MAX_ITER_KMEANS = 6,
                 HB_BLOCK_SIZE = 7, HB_EPSILON_KMEANS = 8, HB_EPSILON_HARMONY = 9, HB_N_LOCAL = 10,
                 HB_LAMBDA_ESTIMATION = 11, HB_WINDOW_SIZE = 12, HB_LEGACY_CENTROID_STEP = 13, HB_KERNEL_SET = 14,
                 HB_DEVICE = 15 /* CUDA device of the handle (read-only) */ };
/* HB_KERNEL_SET (test hook, default 0, read by the next hb_setup): the library picks its kernels from the problem's
 * shape alone; these bits force the kernels that serve shapes outside the default ones' limits onto ANY shape so that
 * the parity suite can hold them to the same bar (tests/test_gpu_parity.py::test_fallback_kernels_match_oracle). */
enum hb_kernel_set { HB_KS_FFMA_CONTRACTIONS = 1, /* fp32 FFMA assignment / statistics / apply instead of tcgen05 */
                     HB_KS_UPDATE_PER_STEP = 2,   /* three launches per block step (first-generation update_R) */
                     HB_KS_UPDATE_TWO_PASS = 4,   /* first persistent update_R generation (look-ahead + update groups) */
                     HB_KS_NO_PEER_EXCHANGE = 8,  /* sharded cells: one NCCL all-reduce per block step */
                     HB_KS_NO_PLAN_OVERLAP = 16   /* build every call's update plan on the main stream */ };
int hb_get_scalar(const hb_handle* h, int which, double* out);
/* Settable: HB_ALPHA, HB_MAX_ITER_KMEANS (vignettes/detailedWalkthrough.Rmd:364), HB_EPSILON_*, HB_KERNEL_SET and
 * HB_LEGACY_CENTROID_STEP (0/1): run STEP 1 of harmony::cluster_cpp — Y = normalise(Z_corr * R.t()),
 * dist_mat = 2 (1 - Y.t() Z_corr), harmony.cpp:235-238, commented out in 2.0.4 — at the top of every clustering
 * round, as the package version that rendered the reference's vignette did.  Compatibility path: one
 * statistics + assignment pass per round on top of the first-generation update kernels. */
int hb_set_scalar(hb_handle* h, int which, double value);
/* B_vec field (harmony.cpp:683): writes C ints. */
int hb_get_B_vec(const hb_handle* h, int32_t* out);

enum hb_trace_id { HB_OBJECTIVE_KMEANS = 0, HB_OBJECTIVE_KMEANS_DIST = 1, HB_OBJECTIVE_KMEANS_ENTROPY = 2,
                   HB_OBJECTIVE_KMEANS_CROSS = 3, HB_OBJECTIVE_HARMONY = 4, HB_KMEANS_ROUNDS = 5 };
/* Trace vectors (harmony.h:55-56).  Returns the trace length; writes min(length, cap) values if out. */
int64_t hb_trace(const hb_handle* h, int trace, double* out, int64_t cap);

/* ---- instrumentation (src/timer.h regions -> CUDA-event timers) -------------------------------- */
/* Number of kernels this library has launched on the handle since creation. */
int64_t hb_kernel_launches(const hb_handle* h);
/* CUDA stream (cudaStream_t) all work of this handle is ordered on, for callers that time with events. */
void* hb_stream(const hb_handle* h);
/* Blocks until all queued work of the handle has finished; returns the sticky CUDA status as 0/>0. */
int hb_synchronize(hb_handle* h);
/* Accumulated device time (ms) and launch count of a named region ("assign", "update_R",
 * "ridge_stats", "ridge_solve", "ridge_apply", "plan"); returns 0 if the region exists. */
int hb_region_time(hb_handle* h, const char* region, double* ms, int64_t* launches);
/* Enables per-region CUDA-event timing (adds synchronisation; off by default). */
int hb_enable_timing(hb_handle* h, int on);
/* Test hook (host only, no GPU needed): position of cell i (inverse = 0) or the cell at position i
 * (inverse = 1) in the keyed pseudo-random order of n cells that replaces arma::shuffle (harmony.cpp:272-273)
 * when no update order is injected.  Returns ~0 for i >= n. */
uint64_t hb_debug_permute(uint64_t i, uint64_t n, uint64_t key, int inverse);
/* Test hook (host only): the host worker pool of the download path (hb_get_field) widens n floats to
 * doubles; `threads` sizes the pool on first use (<= 0: HB_HOST_THREADS or the core count).  Returns the pool size. */
int hb_debug_widen(double* out, const float* in, int64_t n, int threads);
/* Test hook: the tuple-sort permutation (position -> local cell), N_local int32 values. */
int hb_debug_sort_perm(const hb_handle* h, int32_t* out);
/* Test hooks of the native kmeans_centers (hb_init_cluster(h, NULL); utils.cpp:10-64): the keyed-hash uniform that
 * stands in for arma::randu at (centroid i, global cell g) — i = K addresses the K start-cell draws — and the global
 * cells initialize_centroids chose (returns their number, 0 if the native initialisation has not run). */
double hb_debug_kmeans_uniform(const hb_handle* h, uint64_t i, uint64_t g);
int hb_debug_kmeans_cells(const hb_handle* h, int64_t* out);
/* Test hook (host only): ring geometry of the persistent update_R kernel for rows of KS floats:
 * out = {float4 per lane, row groups per warp ring (a power of two), rows per group, shared-memory bytes, warps per
 * CTA, 0, 0, 0, 0}.  Returns 1 if the shape is supported, 0 if the library would use the other update kernels. */
int hb_debug_update_geometry(int KS, int nb, int64_t out[9]);

#ifdef __cplusplus
}
#endif
#endif /* HARMONY_B200_H */
