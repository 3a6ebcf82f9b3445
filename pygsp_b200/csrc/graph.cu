// Device-side graph construction: adjacency checks, symmetrisation, weighted
// degree, CSR Laplacian builder (bit-exact indptr/indices vs scipy) and the
// algebraic spectral bounds.
//
// Replaces, for the path pygsp/graphs/graph.py:98-176, 510-630, 783-838, 933-960:
//   * scipy CSR sum / nnz / != / eliminate_zeros      (graph.py:111-135)
//   * utils.symmetrize(W, 'average') = (W + W.T)/2    (utils.py:247-248)
//   * sparse.diags(dw) - W ; I - D*W*D                (graph.py:618-628)
//   * the four bounds of _get_upper_bound             (graph.py:939-958)
//
// All kernels work row-wise on canonical CSR (sorted columns, no duplicates);
// outputs whose size is data dependent use a count pass (row sizes -> scan ->
// indptr) and a fill pass so that the caller allocates the exact nnz.
#include <cub/cub.cuh>

#include "common.cuh"
#include "gspb200.h"

namespace gsp {

constexpr int kRowThreads = 256;

static inline int row_blocks(int64_t n) { return (int)ceil_div(n > 0 ? n : 1, kRowThreads); }

__device__ __forceinline__ void add64(int64_t* p, int64_t v) {
  if (v) atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)v);
}

// order-preserving max of doubles through a CAS loop (one call per warp)
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *p;
  while (__longlong_as_double((long long)old) < v) {
    const unsigned long long seen = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
    if (seen == old) break;
    old = seen;
  }
}

__device__ __forceinline__ double warp_max(double v) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- inclusive scan of row sizes into indptr[1..n] -------------------------
int scan_rows(int32_t* indptr, int64_t n, cudaStream_t st) {
  // indptr[0] = 0 and indptr[1..n] hold row sizes on entry
  if (n == 0) return GSP_OK;
  size_t bytes = 0;
  GSP_CUDA(cub::DeviceScan::InclusiveSum(nullptr, bytes, indptr + 1, indptr + 1, (int)n, st));
  void* tmp = nullptr;
  GSP_CUDA(cudaMallocAsync(&tmp, bytes ? bytes : 16, st));
  cudaError_t e = cub::DeviceScan::InclusiveSum(tmp, bytes, indptr + 1, indptr + 1, (int)n, st);
  cudaFreeAsync(tmp, st);
  return check_cuda(e, "cub::DeviceScan::InclusiveSum");
}

// ---- adjacency inspection (graph.py:111-128) --------------------------------
// stats: [0] NaN  [1] Inf  [2] negative  [3] non-zero diagonal entries
//        [4] stored zeros  [5] order violations (unsorted / duplicate columns)
//        [6] column index out of range
template <typename T>
__global__ void csr_inspect_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                   const int32_t* __restrict__ indices,
                                   const T* __restrict__ data, int64_t* stats) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int64_t c_nan = 0, c_inf = 0, c_neg = 0, c_diag = 0, c_zero = 0, c_ord = 0, c_rng = 0;
  int prev = -1;
  for (int k = indptr[row]; k < indptr[row + 1]; ++k) {
    const int col = indices[k];
    const T v = data[k];
    c_nan += (v != v);
    c_inf += isinf(v) ? 1 : 0;
    c_neg += (v < T(0));
    c_zero += (v == T(0));
    c_diag += (col == row && v != T(0));
    c_ord += (col <= prev);
    c_rng += (col < 0 || col >= n);
    prev = col;
  }
  add64(stats + 0, c_nan); add64(stats + 1, c_inf); add64(stats + 2, c_neg);
  add64(stats + 3, c_diag); add64(stats + 4, c_zero); add64(stats + 5, c_ord);
  add64(stats + 6, c_rng);
}

// ---- eliminate_zeros (graph.py:128) ------------------------------------------
template <typename T>
__global__ void csr_nonzero_count_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                         const T* __restrict__ data, int32_t* out_indptr) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row == 0) out_indptr[0] = 0;
  if (row >= n) return;
  int c = 0;
  for (int k = indptr[row]; k < indptr[row + 1]; ++k) c += (data[k] != T(0));
  out_indptr[row + 1] = c;
}

template <typename T>
__global__ void csr_nonzero_fill_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                        const int32_t* __restrict__ indices,
                                        const T* __restrict__ data,
                                        const int32_t* __restrict__ out_indptr,
                                        int32_t* out_indices, T* out_data) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int o = out_indptr[row];
  for (int k = indptr[row]; k < indptr[row + 1]; ++k)
    if (data[k] != T(0)) { out_indices[o] = indices[k]; out_data[o] = data[k]; ++o; }
}

// ---- directedness: entries whose mirror differs (graph.py:403-405) -----------
template <typename T>
__global__ void csr_asymmetry_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                     const int32_t* __restrict__ indices,
                                     const T* __restrict__ data, int64_t* count) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int64_t bad = 0;
  for (int k = indptr[row]; k < indptr[row + 1]; ++k) {
    const int col = indices[k];
    int lo = indptr[col], hi = indptr[col + 1];
    while (lo < hi) {                      // lower_bound of `row` in row `col`
      const int mid = (lo + hi) >> 1;
      if (indices[mid] < row) lo = mid + 1; else hi = mid;
    }
    const bool found = lo < indptr[col + 1] && indices[lo] == row;
    bad += !(found && data[lo] == data[k]);
  }
  add64(count, bad);
}

// ---- transpose by key sort ------------------------------------------------------
template <typename T>
__global__ void transpose_keys_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                      const int32_t* __restrict__ indices,
                                      uint64_t* keys, int32_t* t_indptr) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n) return;
  for (int k = indptr[row]; k < indptr[row + 1]; ++k) {
    const int col = indices[k];
    keys[k] = (uint64_t(uint32_t(col)) << 32) | uint32_t(row);
    atomicAdd(t_indptr + col + 1, 1);
  }
}

__global__ void transpose_unpack_kernel(int64_t nnz, const uint64_t* __restrict__ keys,
                                        int32_t* t_indices) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k < nnz) t_indices[k] = int32_t(uint32_t(keys[k] & 0xffffffffu));
}

template <typename T>
int csr_transpose(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* indptr,
                  const int32_t* indices, const T* data, int32_t* t_indptr, int32_t* t_indices,
                  T* t_data, cudaStream_t st) {
  GSP_CUDA(cudaMemsetAsync(t_indptr, 0, sizeof(int32_t) * (n_cols + 1), st));
  if (n_rows == 0 || n_cols == 0 || nnz == 0) return GSP_OK;
  uint64_t *keys_in = nullptr, *keys_out = nullptr;
  GSP_CUDA(cudaMallocAsync((void**)&keys_in, sizeof(uint64_t) * nnz, st));
  GSP_CUDA(cudaMallocAsync((void**)&keys_out, sizeof(uint64_t) * nnz, st));
  transpose_keys_kernel<T><<<row_blocks(n_rows), kRowThreads, 0, st>>>(n_rows, indptr, indices,
                                                                        keys_in, t_indptr);
  // keys are (col << 32) | row: the sort covers the low 32 bits and enough high bits for n_cols
  int bits = 33;
  while ((int64_t(1) << (bits - 32)) < n_cols && bits < 64) ++bits;
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys_in, keys_out, data, t_data, (int)nnz, 0,
                                  bits, st);
  void* tmp = nullptr;
  GSP_CUDA(cudaMallocAsync(&tmp, bytes ? bytes : 16, st));
  cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, bytes, keys_in, keys_out, data, t_data,
                                                  (int)nnz, 0, bits, st);
  if (e == cudaSuccess) {
    transpose_unpack_kernel<<<(int)ceil_div(nnz, 256), 256, 0, st>>>(nnz, keys_out, t_indices);
    e = cudaGetLastError();
  }
  cudaFreeAsync(tmp, st);
  cudaFreeAsync(keys_in, st);
  cudaFreeAsync(keys_out, st);
  if (e != cudaSuccess) return check_cuda(e, "csr_transpose");
  return scan_rows(t_indptr, n_cols, st);
}
template int csr_transpose<float>(int64_t, int64_t, int64_t, const int32_t*, const int32_t*,
                                  const float*, int32_t*, int32_t*, float*, cudaStream_t);
template int csr_transpose<double>(int64_t, int64_t, int64_t, const int32_t*, const int32_t*,
                                   const double*, int32_t*, int32_t*, double*, cudaStream_t);

// ---- COO -> canonical CSR (sparse.csr_matrix(coo): duplicates summed, rows sorted) ----
__global__ void coo_keys_kernel(int64_t nnz, const int32_t* __restrict__ rows,
                                const int32_t* __restrict__ cols, int64_t n, uint64_t* keys,
                                int* bad) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  const int r = rows[k], c = cols[k];
  if (r < 0 || r >= n || c < 0 || c >= n) atomicAdd(bad, 1);
  keys[k] = (uint64_t(uint32_t(r)) << 32) | uint32_t(c);
}

__global__ void coo_unpack_kernel(int64_t nuniq, const uint64_t* __restrict__ keys,
                                  int32_t* indices, int32_t* indptr) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= nuniq) return;
  indices[k] = int32_t(uint32_t(keys[k] & 0xffffffffu));
  atomicAdd(indptr + int32_t(keys[k] >> 32) + 1, 1);
}

// Sorts by (row, col), sums duplicates; writes indptr and the first *n_unique_out
// entries of indices / data (both sized nnz by the caller).  Synchronises the stream
// once to return the number of distinct entries.
template <typename T>
static int coo_to_csr(int64_t n, int64_t nnz, const int32_t* rows, const int32_t* cols,
                      const T* vals, int32_t* indptr, int32_t* indices, T* data,
                      int64_t* n_unique_out, cudaStream_t st) {
  GSP_CUDA(cudaMemsetAsync(indptr, 0, sizeof(int32_t) * (n + 1), st));
  *n_unique_out = 0;
  if (nnz == 0) return GSP_OK;
  uint64_t *k0 = nullptr, *k1 = nullptr, *ku = nullptr;
  T* v1 = nullptr;
  int* scal = nullptr;       // [0] bad indices, [1] number of unique keys
  GSP_CUDA(cudaMallocAsync((void**)&k0, 8 * nnz, st));
  GSP_CUDA(cudaMallocAsync((void**)&k1, 8 * nnz, st));
  GSP_CUDA(cudaMallocAsync((void**)&ku, 8 * nnz, st));
  GSP_CUDA(cudaMallocAsync((void**)&v1, sizeof(T) * nnz, st));
  GSP_CUDA(cudaMallocAsync((void**)&scal, 2 * sizeof(int), st));
  GSP_CUDA(cudaMemsetAsync(scal, 0, 2 * sizeof(int), st));
  const int nb = (int)ceil_div(nnz, 256);
  coo_keys_kernel<<<nb, 256, 0, st>>>(nnz, rows, cols, n, k0, scal);
  int bits = 33;
  while ((int64_t(1) << (bits - 32)) < n && bits < 64) ++bits;
  size_t b1 = 0, b2 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b1, k0, k1, vals, v1, (int)nnz, 0, bits, st);
  cub::DeviceReduce::ReduceByKey(nullptr, b2, k1, ku, v1, data, scal + 1, cub::Sum(), (int)nnz, st);
  void* tmp = nullptr;
  const size_t bytes = std::max(b1, b2);
  GSP_CUDA(cudaMallocAsync(&tmp, bytes ? bytes : 16, st));
  cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, b1, k0, k1, vals, v1, (int)nnz, 0, bits, st);
  if (e == cudaSuccess)
    e = cub::DeviceReduce::ReduceByKey(tmp, b2, k1, ku, v1, data, scal + 1, cub::Sum(), (int)nnz, st);
  int host[2] = {0, 0};
  if (e == cudaSuccess) e = cudaMemcpyAsync(host, scal, sizeof(host), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e == cudaSuccess && host[0] == 0) {
    coo_unpack_kernel<<<(int)ceil_div(host[1] > 0 ? host[1] : 1, 256), 256, 0, st>>>(host[1], ku,
                                                                                    indices, indptr);
    e = cudaGetLastError();
    note_launch(2);
  }
  cudaFreeAsync(tmp, st); cudaFreeAsync(k0, st); cudaFreeAsync(k1, st); cudaFreeAsync(ku, st);
  cudaFreeAsync(v1, st); cudaFreeAsync(scal, st);
  if (e != cudaSuccess) return check_cuda(e, "coo_to_csr");
  if (host[0] != 0) return fail(GSP_ERR_ARG, "COO index out of range (%s)", "rows/cols");
  *n_unique_out = host[1];
  return scan_rows(indptr, n, st);
}

// ---- S = (A + B)/2 with exact-zero results dropped (utils.py:247-248) ----------
template <typename T, bool FILL>
__global__ void csr_average_kernel(int64_t n, const int32_t* __restrict__ a_ptr,
                                   const int32_t* __restrict__ a_idx, const T* __restrict__ a_val,
                                   const int32_t* __restrict__ b_ptr,
                                   const int32_t* __restrict__ b_idx, const T* __restrict__ b_val,
                                   int32_t* s_ptr, int32_t* s_idx, T* s_val) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (!FILL && row == 0) s_ptr[0] = 0;
  if (row >= n) return;
  int ia = a_ptr[row], ea = a_ptr[row + 1], ib = b_ptr[row], eb = b_ptr[row + 1];
  int o = FILL ? s_ptr[row] : 0;
  while (ia < ea || ib < eb) {
    const int ca = ia < ea ? a_idx[ia] : INT_MAX;
    const int cb = ib < eb ? b_idx[ib] : INT_MAX;
    const int col = min(ca, cb);
    T sum = T(0);
    if (ca == col) sum += a_val[ia++];
    if (cb == col) sum += b_val[ib++];
    const T v = sum / T(2);
    if (sum != T(0) && v != T(0)) {
      if (FILL) { s_idx[o] = col; s_val[o] = v; }
      ++o;
    }
  }
  if (!FILL) s_ptr[row + 1] = o;
}

// ---- weighted degree / neighbour count (graph.py:772-781, 830-838) -------------
// dw is accumulated in double in stored order (what scipy's column sums do for
// a symmetric matrix); t_* is the transpose for a directed graph, else null.
template <typename T>
__global__ void degree_kernel(int64_t n, const int32_t* __restrict__ indptr,
                              const T* __restrict__ data, const int32_t* __restrict__ t_indptr,
                              const T* __restrict__ t_data, double* dw, double* d) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n) return;
  double out = 0;
  for (int k = indptr[row]; k < indptr[row + 1]; ++k) out += double(data[k]);
  double cnt = double(indptr[row + 1] - indptr[row]);
  if (t_indptr) {
    double in = 0;
    for (int k = t_indptr[row]; k < t_indptr[row + 1]; ++k) in += double(t_data[k]);
    out = (in + out) / 2;
    cnt = (double(t_indptr[row + 1] - t_indptr[row]) + cnt) / 2;
  }
  dw[row] = out;
  if (d) d[row] = cnt;
}

// ---- Laplacian rows (graph.py:618-628) ------------------------------------------
// lap_type 0: L = diag(dw) - W ; 1: L = I - D^-1/2 W D^-1/2 (isolated: empty row).
// The row of L is the row of the symmetric W with the diagonal entry merged in
// at its sorted position; values that are exactly 0 are not stored.
template <typename T>
__device__ __forceinline__ double inv_sqrt_degree(double dw) {
  return dw == 0 ? 0.0 : pow(dw, -0.5);
}

template <typename T, bool FILL>
__global__ void laplacian_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                 const int32_t* __restrict__ indices, const T* __restrict__ data,
                                 const double* __restrict__ dw, int lap_type, int32_t* l_ptr,
                                 int32_t* l_idx, T* l_val) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (!FILL && row == 0) l_ptr[0] = 0;
  if (row >= n) return;
  const int start = indptr[row], end = indptr[row + 1];
  const double dwi = dw[row];
  const double di = lap_type == 1 ? inv_sqrt_degree<T>(dwi) : 0.0;

  // diagonal value
  double loop = 0;
  bool has_loop = false;
  for (int k = start; k < end; ++k)
    if (indices[k] == row) { loop = double(data[k]); has_loop = true; }
  double diag;
  if (lap_type == 0) diag = dwi - loop;
  else diag = (dwi == 0) ? 0.0 : (has_loop ? 1.0 - (di * loop) * di : 1.0);
  const T diag_t = T(diag);
  const bool keep_diag = diag_t != T(0);

  int o = FILL ? l_ptr[row] : 0;
  bool diag_done = false;
  for (int k = start; k < end; ++k) {
    const int col = indices[k];
    if (!diag_done && col >= row) {
      if (keep_diag) { if (FILL) { l_idx[o] = (int)row; l_val[o] = diag_t; } ++o; }
      diag_done = true;
    }
    if (col == row) continue;
    T v;
    if (lap_type == 0) v = -data[k];
    else v = T(-((di * double(data[k])) * inv_sqrt_degree<T>(dw[col])));
    if (v != T(0)) { if (FILL) { l_idx[o] = col; l_val[o] = v; } ++o; }
  }
  if (!diag_done && keep_diag) { if (FILL) { l_idx[o] = (int)row; l_val[o] = diag_t; } ++o; }
  if (!FILL) l_ptr[row + 1] = o;
}

// ---- spectral bounds (graph.py:939-958) -----------------------------------------
// out[0] = max stored W (caller adds the implicit zeros), out[1] = max dw,
// out[2] = max over stored entries of dw_s + dw_t, out[3] = max(dw + (Ws dw)/dw),
// out[4] = number of NaN terms in [3] (np.max propagates NaN).
template <typename T>
__global__ void bounds_kernel(int64_t n, const int32_t* __restrict__ w_ptr,
                              const int32_t* __restrict__ w_idx, const T* __restrict__ w_val,
                              const int32_t* __restrict__ s_ptr, const int32_t* __restrict__ s_idx,
                              const T* __restrict__ s_val, const double* __restrict__ dw,
                              double* out) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const double ninf = -INFINITY;
  double m_w = ninf, m_dw = ninf, m_edge = ninf, m_mer = ninf, nan_cnt = 0;
  if (row < n) {
    const double dwi = dw[row];
    m_dw = dwi;
    for (int k = w_ptr[row]; k < w_ptr[row + 1]; ++k) {
      m_w = fmax(m_w, double(w_val[k]));
      m_edge = fmax(m_edge, dwi + dw[w_idx[k]]);
    }
    double acc = 0;
    for (int k = s_ptr[row]; k < s_ptr[row + 1]; ++k) acc += double(s_val[k]) * dw[s_idx[k]];
    const double t = dwi + acc / dwi;
    if (t != t) nan_cnt = 1; else m_mer = t;
  }
  m_w = warp_max(m_w); m_dw = warp_max(m_dw); m_edge = warp_max(m_edge); m_mer = warp_max(m_mer);
  for (int o = 16; o > 0; o >>= 1) nan_cnt += __shfl_xor_sync(0xffffffffu, nan_cnt, o);
  if ((threadIdx.x & 31) == 0) {
    atomic_max_double(out + 0, m_w);
    atomic_max_double(out + 1, m_dw);
    atomic_max_double(out + 2, m_edge);
    atomic_max_double(out + 3, m_mer);
    if (nan_cnt != 0) atomicAdd(out + 4, nan_cnt);
  }
}

__global__ void bounds_init_kernel(double* out) {
  if (threadIdx.x < 4) out[threadIdx.x] = -INFINITY;
  if (threadIdx.x == 4) out[4] = 0;
}

// ---- row gather: dst[i,:] = src[idx[i],:] (vertex reordering, halo pack) --------
// PACK = int4 when rows are 16-byte multiples and the bases are aligned (one 16-byte packet
// per thread and trip, rows fully coalesced), else the element type.
template <typename PACK, bool SCATTER>
__global__ void move_rows_kernel(int64_t rows, const int64_t* __restrict__ idx,
                                 const PACK* __restrict__ src, int64_t width, PACK* __restrict__ dst) {
  const int64_t total = rows * width;
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; i < total; i += stride) {
    const int64_t r = i / width, c = i - r * width;
    if (SCATTER) dst[idx[r] * width + c] = src[i];
    else dst[i] = src[idx[r] * width + c];
  }
}

// ------------------------------------------------------------------ drivers ------
template <typename T>
int csr_inspect(int64_t n, const int32_t* p, const int32_t* i, const T* d, int64_t* stats,
                cudaStream_t st) {
  GSP_CUDA(cudaMemsetAsync(stats, 0, sizeof(int64_t) * 8, st));
  if (n == 0) return GSP_OK;
  csr_inspect_kernel<T><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, i, d, stats);
  GSP_LAUNCH_CHECK("csr_inspect");
  return GSP_OK;
}

template <typename T>
int csr_compact_count(int64_t n, const int32_t* p, const T* d, int32_t* out_p, cudaStream_t st) {
  csr_nonzero_count_kernel<T><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, d, out_p);
  GSP_LAUNCH_CHECK("csr_compact_count");
  return scan_rows(out_p, n, st);
}

template <typename T>
int csr_compact_fill(int64_t n, const int32_t* p, const int32_t* i, const T* d,
                     const int32_t* out_p, int32_t* out_i, T* out_d, cudaStream_t st) {
  if (n == 0) return GSP_OK;
  csr_nonzero_fill_kernel<T><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, i, d, out_p, out_i,
                                                                     out_d);
  GSP_LAUNCH_CHECK("csr_compact_fill");
  return GSP_OK;
}

template <typename T>
int csr_asymmetry(int64_t n, const int32_t* p, const int32_t* i, const T* d, int64_t* count,
                  cudaStream_t st) {
  GSP_CUDA(cudaMemsetAsync(count, 0, sizeof(int64_t), st));
  if (n == 0) return GSP_OK;
  csr_asymmetry_kernel<T><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, i, d, count);
  GSP_LAUNCH_CHECK("csr_asymmetry");
  return GSP_OK;
}

template <typename T>
int csr_average(bool fill, int64_t n, const int32_t* ap, const int32_t* ai, const T* ad,
                const int32_t* bp, const int32_t* bi, const T* bd, int32_t* sp, int32_t* si,
                T* sd, cudaStream_t st) {
  if (fill) {
    if (n == 0) return GSP_OK;
    csr_average_kernel<T, true><<<row_blocks(n), kRowThreads, 0, st>>>(n, ap, ai, ad, bp, bi, bd,
                                                                       sp, si, sd);
    GSP_LAUNCH_CHECK("csr_average_fill");
    return GSP_OK;
  }
  csr_average_kernel<T, false><<<row_blocks(n), kRowThreads, 0, st>>>(n, ap, ai, ad, bp, bi, bd,
                                                                      sp, nullptr, nullptr);
  GSP_LAUNCH_CHECK("csr_average_count");
  return scan_rows(sp, n, st);
}

template <typename T>
int degree(int64_t n, const int32_t* p, const T* d, const int32_t* tp, const T* td, double* dw,
           double* deg, cudaStream_t st) {
  if (n == 0) return GSP_OK;
  degree_kernel<T><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, d, tp, td, dw, deg);
  GSP_LAUNCH_CHECK("degree");
  return GSP_OK;
}

template <typename T>
int laplacian(bool fill, int64_t n, const int32_t* p, const int32_t* i, const T* d,
              const double* dw, int lap_type, int32_t* lp, int32_t* li, T* ld, cudaStream_t st) {
  GSP_REQUIRE(lap_type == 0 || lap_type == 1, "Unknown Laplacian type");
  if (fill) {
    if (n == 0) return GSP_OK;
    laplacian_kernel<T, true><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, i, d, dw, lap_type, lp,
                                                                     li, ld);
    GSP_LAUNCH_CHECK("laplacian_fill");
    return GSP_OK;
  }
  laplacian_kernel<T, false><<<row_blocks(n), kRowThreads, 0, st>>>(n, p, i, d, dw, lap_type, lp,
                                                                    nullptr, nullptr);
  GSP_LAUNCH_CHECK("laplacian_count");
  return scan_rows(lp, n, st);
}

template <typename T>
int bounds(int64_t n, const int32_t* wp, const int32_t* wi, const T* wd, const int32_t* sp,
           const int32_t* si, const T* sd, const double* dw, double* out, cudaStream_t st) {
  bounds_init_kernel<<<1, 32, 0, st>>>(out);
  if (n > 0) bounds_kernel<T><<<row_blocks(n), kRowThreads, 0, st>>>(n, wp, wi, wd, sp, si, sd, dw, out);
  GSP_LAUNCH_CHECK("bounds");
  return GSP_OK;
}

template <typename T>
int move_rows(bool scatter, int64_t rows, const int64_t* idx, const T* src, int64_t width, T* dst,
              cudaStream_t st) {
  if (rows * width == 0) return GSP_OK;
  const bool vec = (width * sizeof(T)) % 16 == 0 && (reinterpret_cast<uintptr_t>(src) & 15u) == 0 &&
                   (reinterpret_cast<uintptr_t>(dst) & 15u) == 0;
  if (vec) {
    const int64_t w = width * sizeof(T) / 16;
    const int blocks = (int)std::min<int64_t>(ceil_div(rows * w, 256), int64_t(sm_count()) * 32);
    const int4* s4 = reinterpret_cast<const int4*>(src);
    int4* d4 = reinterpret_cast<int4*>(dst);
    if (scatter) move_rows_kernel<int4, true><<<blocks, 256, 0, st>>>(rows, idx, s4, w, d4);
    else move_rows_kernel<int4, false><<<blocks, 256, 0, st>>>(rows, idx, s4, w, d4);
  } else {
    const int blocks = (int)std::min<int64_t>(ceil_div(rows * width, 256), int64_t(sm_count()) * 32);
    if (scatter) move_rows_kernel<T, true><<<blocks, 256, 0, st>>>(rows, idx, src, width, dst);
    else move_rows_kernel<T, false><<<blocks, 256, 0, st>>>(rows, idx, src, width, dst);
  }
  GSP_LAUNCH_CHECK("move_rows");
  return GSP_OK;
}
template int move_rows<float>(bool, int64_t, const int64_t*, const float*, int64_t, float*, cudaStream_t);
template int move_rows<double>(bool, int64_t, const int64_t*, const double*, int64_t, double*, cudaStream_t);

}  // namespace gsp

// ------------------------------- C ABI ------------------------------------
#define GSP_GRAPH_API(SUF, T)                                                                   \
  int gsp_csr_inspect_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,           \
                            const T* data, int64_t* stats_dev, void* stream) {                  \
    return gsp::csr_inspect<T>(n, indptr, indices, data, stats_dev, gsp::as_stream(stream));    \
  }                                                                                             \
  int gsp_csr_compact_count_##SUF(int64_t n, const int32_t* indptr, const T* data,              \
                                  int32_t* out_indptr, void* stream) {                          \
    return gsp::csr_compact_count<T>(n, indptr, data, out_indptr, gsp::as_stream(stream));      \
  }                                                                                             \
  int gsp_csr_compact_fill_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,      \
                                 const T* data, const int32_t* out_indptr, int32_t* out_indices, \
                                 T* out_data, void* stream) {                                   \
    return gsp::csr_compact_fill<T>(n, indptr, indices, data, out_indptr, out_indices,          \
                                    out_data, gsp::as_stream(stream));                          \
  }                                                                                             \
  int gsp_csr_asymmetry_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,         \
                              const T* data, int64_t* count_dev, void* stream) {                \
    return gsp::csr_asymmetry<T>(n, indptr, indices, data, count_dev, gsp::as_stream(stream));  \
  }                                                                                             \
  int gsp_csr_transpose_##SUF(int64_t n, int64_t nnz, const int32_t* indptr,                    \
                              const int32_t* indices, const T* data, int32_t* t_indptr,         \
                              int32_t* t_indices, T* t_data, void* stream) {                    \
    GSP_REQUIRE(nnz < (int64_t(1) << 31), "nnz must fit int32");                                \
    return gsp::csr_transpose<T>(n, n, nnz, indptr, indices, data, t_indptr, t_indices, t_data, \
                                 gsp::as_stream(stream));                                       \
  }                                                                                             \
  int gsp_coo_to_csr_##SUF(int64_t n, int64_t nnz, const int32_t* rows, const int32_t* cols,     \
                           const T* vals, int32_t* indptr, int32_t* indices, T* data,            \
                           int64_t* n_unique_host_out, void* stream) {                           \
    GSP_REQUIRE(nnz < (int64_t(1) << 31) && n_unique_host_out, "nnz must fit int32");            \
    return gsp::coo_to_csr<T>(n, nnz, rows, cols, vals, indptr, indices, data,                   \
                              n_unique_host_out, gsp::as_stream(stream));                        \
  }                                                                                             \
  int gsp_csr_average_count_##SUF(int64_t n, const int32_t* a_indptr, const int32_t* a_indices, \
                                  const T* a_data, const int32_t* b_indptr,                     \
                                  const int32_t* b_indices, const T* b_data, int32_t* s_indptr, \
                                  void* stream) {                                               \
    return gsp::csr_average<T>(false, n, a_indptr, a_indices, a_data, b_indptr, b_indices,      \
                               b_data, s_indptr, nullptr, nullptr, gsp::as_stream(stream));     \
  }                                                                                             \
  int gsp_csr_average_fill_##SUF(int64_t n, const int32_t* a_indptr, const int32_t* a_indices,  \
                                 const T* a_data, const int32_t* b_indptr,                      \
                                 const int32_t* b_indices, const T* b_data,                     \
                                 const int32_t* s_indptr, int32_t* s_indices, T* s_data,        \
                                 void* stream) {                                                \
    return gsp::csr_average<T>(true, n, a_indptr, a_indices, a_data, b_indptr, b_indices,       \
                               b_data, const_cast<int32_t*>(s_indptr), s_indices, s_data,       \
                               gsp::as_stream(stream));                                         \
  }                                                                                             \
  int gsp_degree_##SUF(int64_t n, const int32_t* indptr, const T* data,                         \
                       const int32_t* t_indptr, const T* t_data, double* dw, double* d,         \
                       void* stream) {                                                          \
    return gsp::degree<T>(n, indptr, data, t_indptr, t_data, dw, d, gsp::as_stream(stream));    \
  }                                                                                             \
  int gsp_laplacian_count_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,       \
                                const T* data, const double* dw, int lap_type,                  \
                                int32_t* l_indptr, void* stream) {                              \
    return gsp::laplacian<T>(false, n, indptr, indices, data, dw, lap_type, l_indptr, nullptr,  \
                             nullptr, gsp::as_stream(stream));                                  \
  }                                                                                             \
  int gsp_laplacian_fill_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,        \
                               const T* data, const double* dw, int lap_type,                   \
                               const int32_t* l_indptr, int32_t* l_indices, T* l_data,          \
                               void* stream) {                                                  \
    return gsp::laplacian<T>(true, n, indptr, indices, data, dw, lap_type,                      \
                             const_cast<int32_t*>(l_indptr), l_indices, l_data,                 \
                             gsp::as_stream(stream));                                           \
  }                                                                                             \
  int gsp_spectral_bounds_##SUF(int64_t n, const int32_t* w_indptr, const int32_t* w_indices,   \
                                const T* w_data, const int32_t* s_indptr,                       \
                                const int32_t* s_indices, const T* s_data, const double* dw,    \
                                double* out5_dev, void* stream) {                               \
    return gsp::bounds<T>(n, w_indptr, w_indices, w_data, s_indptr, s_indices, s_data, dw,      \
                          out5_dev, gsp::as_stream(stream));                                    \
  }                                                                                             \
  int gsp_gather_rows_##SUF(int64_t rows, const int64_t* idx, const T* src, int64_t width,      \
                            T* dst, void* stream) {                                             \
    return gsp::move_rows<T>(false, rows, idx, src, width, dst, gsp::as_stream(stream));        \
  }                                                                                             \
  int gsp_scatter_rows_##SUF(int64_t rows, const int64_t* idx, const T* src, int64_t width,     \
                             T* dst, void* stream) {                                            \
    return gsp::move_rows<T>(true, rows, idx, src, width, dst, gsp::as_stream(stream));         \
  }

extern "C" {
GSP_GRAPH_API(f32, float)
GSP_GRAPH_API(f64, double)
}
