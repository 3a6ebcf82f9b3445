/* libgspb200 -- C ABI of the B200-native Chebyshev graph-filtering engine.
 *
 * The reference (PyGSP 0.6.1) has no FFI: its seam for this path is the Python
 * call boundary, below which every operation is a call into SciPy's compiled
 * sparsetools / ARPACK.  Each entry point below replaces one such call; the
 * comment names the reference line it stands in for.  Conventions:
 *
 *   - every array argument is a DEVICE pointer unless its name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     nothing synchronises (the caller owns synchronisation);
 *   - return value 0 = OK, negative = error (-1 bad argument, -2 CUDA error,
 *     -3 unsupported); the message is available from gsp_last_error()
 *     (thread-local).  Nothing throws across the boundary;
 *   - the callee never frees or keeps caller memory.  Outputs whose size is
 *     data dependent come as a *_count / *_fill pair: the count pass writes
 *     the output indptr (whose last element is the nnz to allocate);
 *   - CSR index arrays are int32 (as SciPy's for nnz < 2^31), values are
 *     float (_f32) or double (_f64); the weighted degree `dw` is always double.
 */
#ifndef GSPB200_H_
#define GSPB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSPB200_ABI_VERSION 2

int gsp_abi_version(void);
const char* gsp_last_error(void);
/* number of kernels this library has launched since it was loaded */
uint64_t gsp_launch_count(void);
int gsp_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes);

/* ------------------------------------------------------------------ filter --
 * gsp_cheby_op_*: pygsp/filters/approximations.py:58-114 `cheby_op(G, c, signal)`.
 *   L = (indptr, indices, data) n x n CSR; lmax = G.lmax; coeffs_host is the
 *   (nscales, m) row-major coefficient matrix (m = order + 1 >= 2, else the
 *   reference's TypeError condition is reported as -1); x is (n, nsig)
 *   row-major; r receives (nscales, n, nsig) = the reference's filter-major
 *   (nscales*n, nsig) block; work holds 2*n*nsig elements.  x is not modified.
 *   nnz = number of stored entries of L; plan_host may be NULL (row-group kernel).
 * gsp_cheby_step_*: one fused recurrence step on rows [row_begin, row_end)
 *   x_new = alpha*(L x_cur) + beta*x_cur + gamma*x_old ;  r_i (+)= ck[i]*x_new
 *   (first != 0: r_i = c0[i]/2 * x_cur + ck[i] * x_new, x_old unused).
 *   x_new may alias x_old.  Stands for approximations.py:99-103 (first) and
 *   :107-112 (k >= 2).  Used directly by the vertex-partitioned multi-GPU path,
 *   where column indices address a local x_cur that has halo rows appended.
 * gsp_cheby_clenshaw_*: out = sum_i p_i(L) s_i for nsrc source blocks s_i ((nsrc, n, nsig) in
 *   memory) and coefficient rows c_i ((nsrc, m) row-major), by ONE backward (Clenshaw)
 *   recurrence on an (n, nsig) block: K SpMMs in total and no accumulator.  nsrc = 1 is the
 *   single-filter evaluation; nsrc = Nf is the synthesis of filter.py:313-322 (which runs Nf
 *   forward recurrences).  out is (n, nsig), work 2*n*nsig.  Same value as the forward
 *   recurrence, different rounding.
 * gsp_spmm_*: y = L x, scipy `csr_matrix.dot` (approximations.py:99, graph.py:955).
 */
/* Tiling of the float32 fast path (TMA-staged row tiles, csrc/cheby_tiled.cu).
 * Filled by gsp_cheby_tile_plan() once per (matrix, nsig, nscales); all zeros
 * means "use the row-group kernel".  Plain host struct, owned by the caller. */
typedef struct gsp_tile_plan {
  int rows_per_tile;   /* rows of L per shared-memory stage */
  int slab_capacity;   /* CSR entries a stage can hold (>= the matrix's largest tile) */
  int stages;          /* depth of the TMA ring */
  int consumer_warps;  /* warps that compute (one more warp produces); the two-packet lane
                          mapping of the Clenshaw form runs min(consumer_warps, 8) of them */
  int gather_unroll;   /* reserved (always 4: one LDS.128 group of CSR entries) */
  int blocks_per_sm;   /* 0 = as many as fit */
} gsp_tile_plan;

/* Reads the matrix's largest tile (synchronises `stream` once) and chooses the tiling. */
int gsp_cheby_tile_plan(int64_t n, const int32_t* indptr, int64_t nsig, int nscales,
                        gsp_tile_plan* plan_host_out, void* stream);

/* Halo exchange fused into the tiled float32 step (vertex-partitioned path).  Local rows
 * are ordered boundary-first: rows [0, n_boundary_rows) may reference halo columns
 * (column ids >= n_owned), rows [0, n_push_rows) are needed by some neighbour.  A step is two
 * launches on the caller's stream.  First the tiles that hold such rows ("front" tiles, a few
 * dozen): their warps wait until flags[wait_ids[q]] >= wait_value (the neighbours have stored
 * x_cur's halo rows into this GPU; front tiles gather through L2, never through the
 * non-coherent path), every row < n_push_rows of x_new is stored into
 * peer_base[push_peer[e]][push_row[e], :] for e in [push_ptr[row], push_ptr[row+1]) (peer
 * stores over NVLink) and, with publish != 0, publish_value is written to every
 * peer_flags[q] when the last front tile is done -- at that point the pushed rows are visible
 * and nobody on this GPU reads the halo of x_cur any more, so the neighbours may also
 * overwrite it.  Then all interior tiles, with the plain kernel instantiation (one kernel
 * for both spilled registers into the interior loop: 1.6 x slower steps).  All pointers are
 * device pointers; the struct itself is a host struct.  n_push_tiles / n_wait_tiles are
 * filled in by the library. */
typedef struct gsp_halo_fusion {
  int64_t n_push_rows;
  int64_t n_push_tiles;
  const int32_t* push_ptr;
  const int32_t* push_peer;
  const int64_t* push_row;
  void* const* peer_base;          /* float* const*  : peers' x_new buffers */
  uint64_t* const* peer_flags;     /* my slot in each neighbour's flag array */
  uint64_t* push_counter;          /* one zero-initialised device uint64 */
  const uint64_t* wait_flags;      /* my own flag array */
  const int32_t* wait_ids;         /* neighbour ranks to wait for */
  uint64_t publish_value;
  uint64_t wait_value;
  int32_t n_neighbors;
  int32_t n_wait;
  int64_t n_boundary_rows;         /* rows [0, n_boundary_rows) may read halo columns */
  int64_t n_wait_tiles;
  int64_t n_owned;                 /* columns >= n_owned are halo rows of x_cur */
  int32_t publish;                 /* 0: last step of a call, nothing is published */
  int32_t reserved;
} gsp_halo_fusion;

/* One fused step on the whole local row block with the halo exchange folded in
 * (float32, tiled kernel required: returns -3 when no tile plan applies).  reverse != 0
 * walks the interior tiles from the last to the first (alternate it between steps: the
 * lines a step wrote last are then the first ones the next step reads, still in L2). */
int gsp_cheby_step_halo_f32(int first, int64_t n_rows, int64_t nnz, const int32_t* indptr,
                            const int32_t* indices, const float* data, const float* x_cur,
                            const float* x_old, float* x_new, float* r, int64_t r_rows,
                            int64_t nsig, int nscales, const double* ck_host,
                            const double* c0_host, double alpha, double beta, double gamma,
                            int reverse, const gsp_tile_plan* plan_host,
                            const gsp_halo_fusion* halo_host, void* stream);

#define GSPB200_DECLARE_CHEBY_API(SUF, T)                                                         \
  int gsp_cheby_op_##SUF(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,   \
                         const T* data, double lmax, const double* coeffs_host, int nscales,      \
                         int m, const T* x, int64_t nsig, T* r, T* work,                          \
                         const gsp_tile_plan* plan_host, void* stream);                           \
  int gsp_cheby_step_##SUF(int first, int64_t row_begin, int64_t row_end, int64_t nnz,            \
                           const int32_t* indptr, const int32_t* indices, const T* data,          \
                           const T* x_cur, const T* x_old, T* x_new, T* r, int64_t r_rows,        \
                           int64_t nsig, int nscales, const double* ck_host,                      \
                           const double* c0_host, double alpha, double beta, double gamma,        \
                           const gsp_tile_plan* plan_host, void* stream);                         \
  int gsp_cheby_clenshaw_##SUF(int64_t n, int64_t nnz, const int32_t* indptr,                     \
                               const int32_t* indices, const T* data, double lmax,                \
                               const double* coeffs_host, int nsrc, int m, const T* sources,      \
                               int64_t nsig, T* out, T* work, const gsp_tile_plan* plan_host,     \
                               void* stream);                                                     \
  int gsp_spmm_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices, const T* data,     \
                     const T* x, int64_t nsig, T* y, void* stream);

GSPB200_DECLARE_CHEBY_API(f32, float)
GSPB200_DECLARE_CHEBY_API(f64, double)

/* ------------------------------------------------------------------- lmax ---
 * gsp_spmv_*: y = L x for ONE vector -- scipy's csr_matvec, the product ARPACK calls at
 *   pygsp/graphs/graph.py:911-917 and the one of graph.py:955.  2..32 lanes per row (from the
 *   mean row length), coalesced reads of indices / data, warp-shuffle reduction per row.
 * gsp_lanczos_*: pygsp/graphs/graph.py:911-917 (scipy eigsh -> ARPACK).
 *   Runs Lanczos iterations [j0, j1) on L: two launches per iteration (the SpMV above with
 *   the v'Lv dot product fused in; the three-term update fused with the norm).  V3 holds
 *   3*n elements, scal_dev 2*cap+1+4096 doubles: alpha[0..cap) | beta[-1..cap) | reduction
 *   partials (beta[j] couples v_j and v_{j+1}; beta[-1] is the norm of the start vector).
 *   j0 == 0 seeds the start vector from `seed` (counter-based, reproducible).  The host
 *   reads alpha/beta back and diagonalises the tridiagonal matrix.
 */
int gsp_spmv_f32(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
                 const float* data, const float* x, float* y, void* stream);
int gsp_spmv_f64(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
                 const double* data, const double* x, double* y, void* stream);
int gsp_lanczos_f32(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
                    const float* data, float* V3, int j0, int j1, int cap, uint64_t seed,
                    double* scal_dev, void* stream);
int gsp_lanczos_f64(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
                    const double* data, double* V3, int j0, int j1, int cap, uint64_t seed,
                    double* scal_dev, void* stream);

/* ------------------------------------------------------------------ graph ---
 * gsp_coo_to_csr_*    graph.py:109  sparse.csr_matrix(coo): sort by (row, col), sum duplicates.
 *     indices / data are sized nnz by the caller; the number of distinct entries comes back
 *     in *n_unique_host_out (the call synchronises the stream once).
 * gsp_csr_inspect_*   graph.py:111-122  NaN / Inf / negative / self-loop checks.
 *     stats_dev[8] (int64): [0] NaN [1] Inf [2] negative [3] non-zero diagonal
 *     [4] stored zeros [5] unsorted-or-duplicate columns [6] column out of range.
 * gsp_csr_compact_*   graph.py:128      eliminate_zeros().
 * gsp_csr_asymmetry_* graph.py:403-405  (W != W.T).nnz: entries whose mirror differs.
 * gsp_csr_transpose_* W.T as sorted CSR (needed by the directed-graph branches).
 * gsp_csr_average_*   utils.py:247-248  (A + B)/2, exact zeros dropped.
 * gsp_degree_*        graph.py:772-781, 830-838  d and dw (pass the transpose for
 *     a directed graph, else NULL); d may be NULL.
 * gsp_laplacian_*     graph.py:618-628  lap_type 0 combinatorial, 1 normalized; the
 *     input must be the SYMMETRIC adjacency ((W+W.T)/2 for a directed graph).
 *     indptr/indices of the result are bit-identical to SciPy's.
 * gsp_spectral_bounds_* graph.py:939-958  out5_dev (double): max W, max dw,
 *     max(dw_s+dw_t) over edges, max(dw+(Ws dw)/dw), #NaN terms of the latter.
 * gsp_gather_rows_* / gsp_scatter_rows_*  dst[i,:] = src[idx[i],:] / dst[idx[i],:] = src[i,:]
 *     (vertex reordering in and out, halo packing).
 */
/* ----------------------------------------------------------------- solver ---
 * gsp_cg_*: conjugate gradients for (diag(row_scale) * tau * L + diag(diag)) X = B, a block
 *   of nsig <= 256 right-hand sides advancing together.  Stands for scipy.sparse.linalg.cg
 *   on the operator x -> M x + tau L x of pygsp/learning.py:326-337 (regression_tikhonov,
 *   one solve per column there) and, with row_scale = 1 - M, diag = 0, for the constrained
 *   problem of learning.py:350-365 restricted to the unlabelled vertices.  row_scale / diag
 *   are length-n vectors or NULL (= 1 / = 0).  Runs iterations [it0, it1) (it0 == 0 starts
 *   from X = 0); X, R, P, Q are (n, nsig) state blocks owned by the caller; scal_dev holds
 *   (cap + 1 + 2048) * nsig doubles, its first (cap + 1) x nsig entries are the history of
 *   the squared residual norms per column, which the host reads to test convergence. */
#define GSPB200_DECLARE_CG_API(SUF, T)                                                           \
  int gsp_cg_##SUF(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,       \
                   const T* data, double tau, const T* row_scale, const T* diag, const T* B,     \
                   T* X, T* R, T* P, T* Q, int64_t nsig, int it0, int it1, int cap,              \
                   double* scal_dev, void* stream);

GSPB200_DECLARE_CG_API(f32, float)
GSPB200_DECLARE_CG_API(f64, double)

/* ------------------------------------------------- host <-> device staging ---
 * Filter.filter() takes and returns host arrays (filter.py:146-328).  To overlap the PCIe
 * transfers with the recurrence the signal block is processed in COLUMN chunks; a chunk of a
 * row-major (n, nsig) block is a strided 2-D region (`height` rows of `width_bytes`, row
 * pitches in bytes).
 * gsp_copy2d_async: cudaMemcpy2DAsync on `stream` (copy engines); kind 1 = host to device,
 *   2 = device to host, 3 = device to device.  Host memory must be page-locked.
 * gsp_stage_cols: the same region moved by a kernel of at most max_blocks blocks (0 = one
 *   per SM) that reads / writes PINNED host memory through its unified address; all
 *   pointers, pitches and width_bytes must be multiples of 16. */
int gsp_copy2d_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes,
                     size_t height, int kind, void* stream);
int gsp_stage_cols(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes,
                   size_t height, int max_blocks, void* stream);

/* ------------------------------------------------------------ peer-memory halo ---
 * The vertex-partitioned path (no reference counterpart: PyGSP is single-process).
 * gsp_ipc_alloc / open / close / free: cudaMalloc'ed, zero-filled buffers exported with
 *     CUDA IPC (64-byte handle) so that the other ranks of the node can map them.
 * gsp_halo_push_*: copies rows src[src_row[e], :] into peer_base[dst_peer[e]][dst_row[e], :]
 *     (peer stores over NVLink), fences, then writes `value` to every peer_flags[q]
 *     (the address of this rank's slot in neighbour q's flag array).
 *     done_counter: one zero-initialised device uint32 owned by the caller.
 * gsp_halo_wait: blocks the STREAM (not the host) until flags[neighbor_ids[q]] >= value.
 */
int gsp_ipc_alloc(size_t bytes, void** dev_ptr_out, unsigned char* handle64_out);
int gsp_ipc_open(const unsigned char* handle64, void** dev_ptr_out);
int gsp_ipc_close(void* dev_ptr);
int gsp_ipc_free(void* dev_ptr);
int gsp_halo_push_f32(int64_t n_send, const int64_t* src_row, const int32_t* dst_peer,
                      const int64_t* dst_row, const float* src, float* const* peer_base,
                      int64_t width, uint64_t* const* peer_flags, int n_neighbors,
                      uint64_t value, uint32_t* done_counter, void* stream);
int gsp_halo_push_f64(int64_t n_send, const int64_t* src_row, const int32_t* dst_peer,
                      const int64_t* dst_row, const double* src, double* const* peer_base,
                      int64_t width, uint64_t* const* peer_flags, int n_neighbors,
                      uint64_t value, uint32_t* done_counter, void* stream);
int gsp_halo_wait(const uint64_t* flags, const int32_t* neighbor_ids, int n_neighbors,
                  uint64_t value, void* stream);

/* ------------------------------------------- the partitioned operator, one call ---
 * gsp_cheby_op_dist_*: approximations.py:58-114 on ONE rank's row block of a 1-D vertex
 * partitioned Laplacian (SURVEY.md 8e).  The caller (one process per GPU) builds the plan
 * once -- which of its rows every neighbour needs and where they live in the neighbour's
 * halo, the CUDA-IPC mapped state buffers and flag arrays; that is host-side set-up and
 * needs the job's communicator once (pygsp_b200/distributed.py: HaloPlan, PeerWindow) --
 * and then runs any number of calls without any collective: each of the K recurrence
 * steps waits for the neighbours' flags, computes, stores its boundary rows into the
 * neighbours' halo rows over NVLink and publishes the step (all inside the fused step
 * kernel for float32 with a tile plan; wait / step / push kernels otherwise).
 *
 *   local rows are ordered boundary-first (rows [0, n_boundary_rows) reference halo
 *   columns, rows [0, n_push_rows) are needed by neighbours); local column j < n_local is
 *   local row j, column n_local + h is halo slot h.
 *   buf[b]        : this rank's state buffers, (n_local + n_halo, nsig) each, inside its IPC
 *                   window; buf[2] may be NULL (then the Clenshaw form is not used)
 *   peer_base[b]  : device array of P pointers, entry q = rank q's buf[b] (mapped)
 *   peer_flags[i] : device array, entry i = address of THIS rank's slot in the flag array
 *                   of neighbour neighbor_ids[i]; flags = this rank's own flag array (P slots)
 *   src_row/dst_peer/dst_row (n_send entries): the rows to push as a flat list;
 *   push_ptr/push_peer/push_row: the same list as a CSR over local rows [0, n_push_rows)
 *   push_counter / fused_counter: zero-initialised device counters owned by the caller
 *   x : (n_local, nsig) input (NULL: already in buf[0], local order);
 *   r : (nscales, n_local, nsig) output; x and r are in the CALLER's row order when
 *       plan->perm is given (the gather into local order replaces the copy into buf[0]; the
 *       Clenshaw form stores its last step straight to the caller's rows), else local order;
 *   clenshaw != 0 and nscales == 1: backward (Clenshaw) recurrence, one pass less per order;
 *   seq_host : the rank's sequence counter (starts at 0, advanced by m + 2 per call; all
 *              ranks must make the same calls in the same order).
 * Everything is enqueued on `stream`; nothing synchronises. */
typedef struct gsp_dist_plan {
  int64_t n_local, n_halo, nnz;
  const int32_t* indptr;
  const int32_t* indices;
  const void* data;                  /* float / double values of the local CSR */
  void* buf[3];
  void* const* peer_base[3];
  uint64_t* const* peer_flags;
  uint64_t* flags;
  const int32_t* neighbor_ids;
  int32_t n_neighbors;
  int32_t separate_exchange; /* != 0: never fuse the exchange into the step kernel (wait / step / push kernels) */
  uint32_t* push_counter;
  uint64_t* fused_counter;
  int64_t n_send;
  const int64_t* src_row;
  const int32_t* dst_peer;
  const int64_t* dst_row;
  int64_t n_push_rows;
  const int32_t* push_ptr;
  const int32_t* push_peer;
  const int64_t* push_row;
  int64_t n_boundary_rows;
  const int64_t* perm;               /* local row i = row perm[i] of the caller's blocks; NULL: identity */
} gsp_dist_plan;

int gsp_cheby_op_dist_f32(const gsp_dist_plan* plan_host, const gsp_tile_plan* tile_host,
                          double lmax, const double* coeffs_host, int nscales, int m, const float* x,
                          int64_t nsig, float* r, int clenshaw, uint64_t* seq_host, void* stream);
int gsp_cheby_op_dist_f64(const gsp_dist_plan* plan_host, const gsp_tile_plan* tile_host,
                          double lmax, const double* coeffs_host, int nscales, int m, const double* x,
                          int64_t nsig, double* r, int clenshaw, uint64_t* seq_host, void* stream);

/* ------------------------------------------------------ on-device graph construction ---
 * gsp_grid2d_*: adjacency of pygsp/graphs/grid2d.py:40-89 (n1 x n2 grid, 4 neighbours, unit
 *     weights, row-major numbering) as canonical CSR; count writes indptr (n1*n2 + 1).
 * gsp_knn_grid: k nearest neighbours (self excluded) of n points in 2-D / 3-D by a
 *     uniform cell grid -- the scipy.spatial.KDTree query of nngraph.py:213-216.
 *     points (n, dim) double; lo/hi: bounding box, cells: grid resolution (host arrays
 *     of length dim); outputs (n, k) row-major, ascending distance, ties by index.
 * gsp_knn_to_csr_*: directed k-NN matrix W[i, nn] = exp(-d^2/sigma) as CSR with sorted
 *     rows (nngraph.py:221-226,289); symmetrise with gsp_csr_transpose / _average.
 */
int gsp_grid2d_count(int64_t n1, int64_t n2, int32_t* indptr, void* stream);
int gsp_grid2d_fill_f32(int64_t n1, int64_t n2, const int32_t* indptr, int32_t* indices,
                        float* data, void* stream);
int gsp_grid2d_fill_f64(int64_t n1, int64_t n2, const int32_t* indptr, int32_t* indices,
                        double* data, void* stream);
int gsp_knn_grid(int64_t n, int dim, const double* points, int k, const double* lo_host,
                 const double* hi_host, const int32_t* cells_host, int32_t* nn_idx,
                 double* nn_dist, void* stream);
int gsp_knn_to_csr_f32(int64_t n, int k, const int32_t* nn_idx, const double* nn_dist,
                       double sigma, int32_t* indptr, int32_t* indices, float* data, void* stream);
int gsp_knn_to_csr_f64(int64_t n, int k, const int32_t* nn_idx, const double* nn_dist,
                       double sigma, int32_t* indptr, int32_t* indices, double* data,
                       void* stream);

#define GSPB200_DECLARE_GRAPH_API(SUF, T)                                                        \
  int gsp_csr_inspect_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,            \
                            const T* data, int64_t* stats_dev, void* stream);                    \
  int gsp_csr_compact_count_##SUF(int64_t n, const int32_t* indptr, const T* data,               \
                                  int32_t* out_indptr, void* stream);                            \
  int gsp_csr_compact_fill_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,       \
                                 const T* data, const int32_t* out_indptr, int32_t* out_indices, \
                                 T* out_data, void* stream);                                     \
  int gsp_csr_asymmetry_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,          \
                              const T* data, int64_t* count_dev, void* stream);                  \
  int gsp_csr_transpose_##SUF(int64_t n, int64_t nnz, const int32_t* indptr,                     \
                              const int32_t* indices, const T* data, int32_t* t_indptr,          \
                              int32_t* t_indices, T* t_data, void* stream);                      \
  int gsp_coo_to_csr_##SUF(int64_t n, int64_t nnz, const int32_t* rows, const int32_t* cols,      \
                           const T* vals, int32_t* indptr, int32_t* indices, T* data,             \
                           int64_t* n_unique_host_out, void* stream);                            \
  int gsp_csr_average_count_##SUF(int64_t n, const int32_t* a_indptr, const int32_t* a_indices,  \
                                  const T* a_data, const int32_t* b_indptr,                      \
                                  const int32_t* b_indices, const T* b_data, int32_t* s_indptr,  \
                                  void* stream);                                                 \
  int gsp_csr_average_fill_##SUF(int64_t n, const int32_t* a_indptr, const int32_t* a_indices,   \
                                 const T* a_data, const int32_t* b_indptr,                       \
                                 const int32_t* b_indices, const T* b_data,                      \
                                 const int32_t* s_indptr, int32_t* s_indices, T* s_data,         \
                                 void* stream);                                                  \
  int gsp_degree_##SUF(int64_t n, const int32_t* indptr, const T* data,                          \
                       const int32_t* t_indptr, const T* t_data, double* dw, double* d,          \
                       void* stream);                                                            \
  int gsp_laplacian_count_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,        \
                                const T* data, const double* dw, int lap_type,                   \
                                int32_t* l_indptr, void* stream);                                \
  int gsp_laplacian_fill_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,         \
                               const T* data, const double* dw, int lap_type,                    \
                               const int32_t* l_indptr, int32_t* l_indices, T* l_data,           \
                               void* stream);                                                    \
  int gsp_spectral_bounds_##SUF(int64_t n, const int32_t* w_indptr, const int32_t* w_indices,    \
                                const T* w_data, const int32_t* s_indptr,                        \
                                const int32_t* s_indices, const T* s_data, const double* dw,     \
                                double* out5_dev, void* stream);                                 \
  int gsp_gather_rows_##SUF(int64_t rows, const int64_t* idx, const T* src, int64_t width,       \
                            T* dst, void* stream);                                               \
  int gsp_scatter_rows_##SUF(int64_t rows, const int64_t* idx, const T* src, int64_t width,      \
                             T* dst, void* stream);

GSPB200_DECLARE_GRAPH_API(f32, float)
GSPB200_DECLARE_GRAPH_API(f64, double)

/* ----------------------------------------------------------- differential operator ---
 * D is the N x Ne incidence matrix of pygsp/graphs/difference.py (L = D D^T).  Edge k =
 * (sources[k], targets[k]) with weight weights[k]; column k of D holds -v_s at the source and
 * +v_t at the target, v = sqrt(w) (lap_type 0) or sqrt(w / dw) (lap_type 1), both divided by
 * sqrt(2) when directed != 0; a self-loop's column is empty.  Every value is computed in double
 * with correctly rounded operations and rounded once to T.  Two layouts of D:
 *   edge-major   (d_*): SciPy's CSC arrays of D -- indptr (Ne + 1), row (vertex) indices, values;
 *                       0 entries for a self-loop, 2 for any other edge, the smaller vertex first;
 *   vertex-major (v_*): D as CSR (N x Ne), edge ids ascending within a row.
 * gsp_edge_list_count / _fill_*  graph.py:1022-1029  get_edge_list(): every stored entry of W in
 *     row-major order (directed != 0), else the upper triangle, diagonal included.  The count
 *     writes edge_ptr (n + 1), whose last element is Ne; the fill writes int32 sources and
 *     targets and the weights.
 * gsp_diffop_count / _fill_*  difference.py compute_differential_operator().  The count writes
 *     d_indptr (Ne + 1), whose last element is nnz(D); the fill writes d_indices / d_data and the
 *     vertex-major layout (v_indptr has n + 1 entries).  dw is the weighted degree (double).
 *     2 * Ne must fit int32 (else -1).
 * gsp_grad_*  difference.py grad(): y (Ne, nsig) = D^T x, x (n, nsig), over the edge-major layout.
 * gsp_div_*   difference.py div():  z (n, nsig) = D y, y (Ne, nsig), over the vertex-major layout.
 *     Both start every output at +0.0 and add the products in stored order, multiply and add
 *     rounded separately (no FMA): the result equals SciPy's D.T.dot(x) / D.dot(y) on the same D
 *     bit for bit.
 */
int gsp_edge_list_count(int64_t n, const int32_t* indptr, const int32_t* indices, int directed,
                        int32_t* edge_ptr, void* stream);
int gsp_diffop_count(int64_t n_edges, const int32_t* sources, const int32_t* targets,
                     int32_t* d_indptr, void* stream);

#define GSPB200_DECLARE_DIFFOP_API(SUF, T)                                                       \
  int gsp_edge_list_fill_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,         \
                               const T* data, int directed, const int32_t* edge_ptr,            \
                               int32_t* sources, int32_t* targets, T* weights, void* stream);   \
  int gsp_diffop_fill_##SUF(int64_t n, int64_t n_edges, int64_t nnz, const int32_t* sources,     \
                            const int32_t* targets, const T* weights, const double* dw,          \
                            int lap_type, int directed, const int32_t* d_indptr,                 \
                            int32_t* d_indices, T* d_data, int32_t* v_indptr,                    \
                            int32_t* v_indices, T* v_data, void* stream);                        \
  int gsp_grad_##SUF(int64_t n_edges, const int32_t* d_indptr, const int32_t* d_indices,         \
                     const T* d_data, const T* x, int64_t nsig, T* y, void* stream);            \
  int gsp_div_##SUF(int64_t n, const int32_t* v_indptr, const int32_t* v_indices,                \
                    const T* v_data, const T* y, int64_t nsig, T* z, void* stream);

GSPB200_DECLARE_DIFFOP_API(f32, float)
GSPB200_DECLARE_DIFFOP_API(f64, double)

#ifdef __cplusplus
}
#endif
#endif /* GSPB200_H_ */
