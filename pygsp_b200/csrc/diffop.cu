// Graph differential operator: edge list, incidence matrix D, gradient and divergence.
//
// Replaces, for pygsp/graphs/graph.py:962-1029 and pygsp/graphs/difference.py:
//   * W.tocoo() / sparse.triu(W, format="coo")            (get_edge_list)
//   * sparse.csc_matrix((values, (rows, columns))) and
//     eliminate_zeros()                                   (compute_differential_operator)
//   * D.T.dot(x), D.dot(y)                                (grad, div)
//
// D is N x Ne.  Column k of D (edge k = (s, t), weight w) holds -v_s at s and +v_t at t with
// v = sqrt(w) (combinatorial) or sqrt(w / dw) (normalized), both divided by sqrt(2) for a
// directed graph; a self-loop's two entries cancel and its column is empty.  Two layouts:
//   edge-major   : SciPy's CSC arrays of D (= the CSR of D^T, Ne x N), the smaller vertex first;
//   vertex-major : the CSR of D (N x Ne), edge ids ascending in a row (csr_transpose of the first).
// grad is the product over the edge-major layout, div the product over the vertex-major one.
//
// Bit contract: every value is computed in double from the stored weight and dw with correctly
// rounded operations (the reference's float64 operation sequence) and rounded once to T.  Both
// products start each output at +0.0 and add the products in stored order with separately
// rounded multiplies and adds -- scipy's csr_matvec(s) / csc_matvec(s) order, with no
// contraction into FMA -- so that grad and div equal SciPy's on the same D bit for bit.
#include "common.cuh"

namespace gsp {

constexpr int kDiffThreads = 256;

static inline int blocks_for(int64_t n) { return (int)ceil_div(n > 0 ? n : 1, kDiffThreads); }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }

// first entry of a row that belongs to the edge list: the row's start (directed), else the
// first column >= row (the upper triangle, diagonal included)
__device__ __forceinline__ int first_edge_entry(int64_t row, const int32_t* __restrict__ indptr,
                                                const int32_t* __restrict__ indices, int directed) {
  int lo = indptr[row], hi = indptr[row + 1];
  if (directed) return lo;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (indices[mid] < row) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// ---- edge list (graph.py:1022-1029) ------------------------------------------------------
__global__ void edge_count_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                  const int32_t* __restrict__ indices, int directed,
                                  int32_t* edge_ptr) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row == 0) edge_ptr[0] = 0;
  if (row >= n) return;
  edge_ptr[row + 1] = indptr[row + 1] - first_edge_entry(row, indptr, indices, directed);
}

template <typename T>
__global__ void edge_fill_kernel(int64_t n, const int32_t* __restrict__ indptr,
                                 const int32_t* __restrict__ indices, const T* __restrict__ data,
                                 int directed, const int32_t* __restrict__ edge_ptr,
                                 int32_t* sources, int32_t* targets, T* weights) {
  const int64_t row = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int o = edge_ptr[row];
  for (int k = first_edge_entry(row, indptr, indices, directed); k < indptr[row + 1]; ++k, ++o) {
    sources[o] = (int32_t)row;
    targets[o] = indices[k];
    weights[o] = data[k];
  }
}

// ---- D, edge-major (difference.py compute_differential_operator) -------------------------
__global__ void diffop_count_kernel(int64_t ne, const int32_t* __restrict__ sources,
                                    const int32_t* __restrict__ targets, int32_t* d_indptr) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k == 0) d_indptr[0] = 0;
  if (k >= ne) return;
  d_indptr[k + 1] = sources[k] == targets[k] ? 0 : 2;
}

template <typename T>
__global__ void diffop_fill_kernel(int64_t ne, const int32_t* __restrict__ sources,
                                   const int32_t* __restrict__ targets, const T* __restrict__ weights,
                                   const double* __restrict__ dw, int lap_type, int directed,
                                   const int32_t* __restrict__ d_indptr, int32_t* d_indices,
                                   T* d_data) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= ne) return;
  const int s = sources[k], t = targets[k];
  if (s == t) return;                              // -v + v == 0: eliminated, empty column
  const double w = double(weights[k]);
  double vs, vt;
  if (lap_type == 0) {
    vt = __dsqrt_rn(w);
    vs = -vt;
  } else {
    vs = -__dsqrt_rn(__ddiv_rn(w, dw[s]));
    vt = __dsqrt_rn(__ddiv_rn(w, dw[t]));
  }
  if (directed) {
    const double r2 = __dsqrt_rn(2.0);
    vs = __ddiv_rn(vs, r2);
    vt = __ddiv_rn(vt, r2);
  }
  const int p = d_indptr[k];
  const bool s_first = s < t;
  d_indices[p] = s_first ? s : t;
  d_data[p] = T(s_first ? vs : vt);
  d_indices[p + 1] = s_first ? t : s;
  d_data[p + 1] = T(s_first ? vt : vs);
}

// ---- y = A x in exact order (grad: A = D^T edge-major, div: A = D vertex-major) ----------
// Lane mapping of the row-group step kernel (csrc/cheby.cu): G = 2^g lanes own one row, each
// lane a VEC-wide packet of the row's nsig columns; the group loads G CSR entries with one
// coalesced access and broadcasts them with shuffles.  Each lane sums its columns from +0.0 in
// stored order, multiply and add rounded separately.
template <typename T, int VEC, int G>
__global__ void __launch_bounds__(kDiffThreads)
diffop_spmm_kernel(int64_t n_rows, const int32_t* __restrict__ indptr,
                   const int32_t* __restrict__ indices, const T* __restrict__ vals,
                   const T* __restrict__ x, int nsig, T* __restrict__ y) {
  const int lane = threadIdx.x & (G - 1);
  const int64_t row = (int64_t(blockIdx.x) * kDiffThreads + threadIdx.x) / G;
  if (row >= n_rows) return;                       // whole groups leave together (G <= 32)
  const unsigned lane_in_warp = threadIdx.x & 31;
  const unsigned gmask = (G == 32) ? 0xffffffffu
                                   : (((1u << G) - 1u) << (lane_in_warp & ~(G - 1)));
  const int start = __ldg(indptr + row);
  const int end = __ldg(indptr + row + 1);

  for (int cbase = 0; cbase < nsig; cbase += G * VEC) {
    const int c0 = cbase + lane * VEC;
    const bool active = c0 < nsig;
    Vec<T, VEC> acc;
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc.v[v] = T(0);
    for (int base = start; base < end; base += G) {
      const int mine = base + lane;
      int col = 0;
      T val = T(0);
      if (mine < end) {
        col = __ldg(indices + mine);
        val = __ldg(vals + mine);
      }
      const int cnt = min(G, end - base);
      for (int j = 0; j < cnt; ++j) {
        const int cj = __shfl_sync(gmask, col, j, G);
        const T vj = __shfl_sync(gmask, val, j, G);
        if (active) {
          const Vec<T, VEC> xv = load_vec_ro<T, VEC>(x + int64_t(cj) * nsig + c0);
#pragma unroll
          for (int v = 0; v < VEC; ++v) acc.v[v] = add_rn(acc.v[v], mul_rn(vj, xv.v[v]));
        }
      }
    }
    if (active) store_vec_stream<T, VEC>(y + row * nsig + c0, acc);
  }
}

template <typename T, int VEC>
static int launch_spmm(int64_t n_rows, const int32_t* indptr, const int32_t* indices,
                       const T* vals, const T* x, int nsig, T* y, cudaStream_t st) {
  const int packets = (nsig + VEC - 1) / VEC;
#define GSP_GO(GG)                                                                             \
  do {                                                                                         \
    const int64_t blocks = ceil_div(n_rows * GG, kDiffThreads);                                \
    GSP_REQUIRE(blocks < (int64_t(1) << 31), "row range too large for one launch");            \
    diffop_spmm_kernel<T, VEC, GG><<<(unsigned)blocks, kDiffThreads, 0, st>>>(                 \
        n_rows, indptr, indices, vals, x, nsig, y);                                            \
  } while (0)
  if (packets <= 1) GSP_GO(1);
  else if (packets <= 2) GSP_GO(2);
  else if (packets <= 4) GSP_GO(4);
  else if (packets <= 8) GSP_GO(8);
  else if (packets <= 16) GSP_GO(16);
  else GSP_GO(32);
#undef GSP_GO
  GSP_LAUNCH_CHECK("diffop_spmm");
  return GSP_OK;
}

template <typename T>
int exact_spmm(int64_t n_rows, const int32_t* indptr, const int32_t* indices, const T* vals,
               const T* x, int nsig, T* y, cudaStream_t st) {
  if (n_rows == 0) return GSP_OK;
  constexpr int MV = 16 / sizeof(T);
  if (nsig % MV == 0 && aligned16(x) && aligned16(y))
    return launch_spmm<T, MV>(n_rows, indptr, indices, vals, x, nsig, y, st);
  return launch_spmm<T, 1>(n_rows, indptr, indices, vals, x, nsig, y, st);
}

// ------------------------------------------------------------------ drivers ------
int edge_list_count(int64_t n, const int32_t* indptr, const int32_t* indices, int directed,
                    int32_t* edge_ptr, cudaStream_t st) {
  edge_count_kernel<<<blocks_for(n), kDiffThreads, 0, st>>>(n, indptr, indices, directed, edge_ptr);
  GSP_LAUNCH_CHECK("edge_list_count");
  return scan_rows(edge_ptr, n, st);
}

template <typename T>
int edge_list_fill(int64_t n, const int32_t* indptr, const int32_t* indices, const T* data,
                   int directed, const int32_t* edge_ptr, int32_t* sources, int32_t* targets,
                   T* weights, cudaStream_t st) {
  if (n == 0) return GSP_OK;
  edge_fill_kernel<T><<<blocks_for(n), kDiffThreads, 0, st>>>(n, indptr, indices, data, directed,
                                                              edge_ptr, sources, targets, weights);
  GSP_LAUNCH_CHECK("edge_list_fill");
  return GSP_OK;
}

int diffop_count(int64_t ne, const int32_t* sources, const int32_t* targets, int32_t* d_indptr,
                 cudaStream_t st) {
  diffop_count_kernel<<<blocks_for(ne), kDiffThreads, 0, st>>>(ne, sources, targets, d_indptr);
  GSP_LAUNCH_CHECK("diffop_count");
  return scan_rows(d_indptr, ne, st);
}

template <typename T>
int diffop_fill(int64_t n, int64_t ne, int64_t nnz, const int32_t* sources, const int32_t* targets,
                const T* weights, const double* dw, int lap_type, int directed,
                const int32_t* d_indptr, int32_t* d_indices, T* d_data, int32_t* v_indptr,
                int32_t* v_indices, T* v_data, cudaStream_t st) {
  GSP_REQUIRE(lap_type == 0 || lap_type == 1, "Unknown Laplacian type");
  if (ne > 0) {
    diffop_fill_kernel<T><<<blocks_for(ne), kDiffThreads, 0, st>>>(
        ne, sources, targets, weights, dw, lap_type, directed, d_indptr, d_indices, d_data);
    GSP_LAUNCH_CHECK("diffop_fill");
  }
  return csr_transpose<T>(ne, n, nnz, d_indptr, d_indices, d_data, v_indptr, v_indices, v_data,
                          st);
}

}  // namespace gsp

// ------------------------------- C ABI ------------------------------------
#define GSP_DIFFOP_CHECK_EDGES(ne)                                                              \
  GSP_REQUIRE((ne) >= 0 && 2 * (ne) < (int64_t(1) << 31),                                      \
              "2 * n_edges (the entries of D) must fit int32")

#define GSP_DIFFOP_API(SUF, T)                                                                  \
  int gsp_edge_list_fill_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices,        \
                               const T* data, int directed, const int32_t* edge_ptr,           \
                               int32_t* sources, int32_t* targets, T* weights, void* stream) { \
    return gsp::edge_list_fill<T>(n, indptr, indices, data, directed, edge_ptr, sources,        \
                                  targets, weights, gsp::as_stream(stream));                    \
  }                                                                                             \
  int gsp_diffop_fill_##SUF(int64_t n, int64_t n_edges, int64_t nnz, const int32_t* sources,    \
                            const int32_t* targets, const T* weights, const double* dw,         \
                            int lap_type, int directed, const int32_t* d_indptr,                \
                            int32_t* d_indices, T* d_data, int32_t* v_indptr,                   \
                            int32_t* v_indices, T* v_data, void* stream) {                      \
    GSP_DIFFOP_CHECK_EDGES(n_edges);                                                            \
    GSP_REQUIRE(nnz >= 0 && nnz <= 2 * n_edges, "nnz out of range");                            \
    return gsp::diffop_fill<T>(n, n_edges, nnz, sources, targets, weights, dw, lap_type,        \
                               directed, d_indptr, d_indices, d_data, v_indptr, v_indices,      \
                               v_data, gsp::as_stream(stream));                                 \
  }                                                                                             \
  int gsp_grad_##SUF(int64_t n_edges, const int32_t* d_indptr, const int32_t* d_indices,        \
                     const T* d_data, const T* x, int64_t nsig, T* y, void* stream) {           \
    GSP_REQUIRE(nsig >= 1 && nsig <= (1 << 20), "nsig out of range");                           \
    return gsp::exact_spmm<T>(n_edges, d_indptr, d_indices, d_data, x, (int)nsig, y,            \
                              gsp::as_stream(stream));                                          \
  }                                                                                             \
  int gsp_div_##SUF(int64_t n, const int32_t* v_indptr, const int32_t* v_indices,               \
                    const T* v_data, const T* y, int64_t nsig, T* z, void* stream) {            \
    GSP_REQUIRE(nsig >= 1 && nsig <= (1 << 20), "nsig out of range");                           \
    return gsp::exact_spmm<T>(n, v_indptr, v_indices, v_data, y, (int)nsig, z,                  \
                              gsp::as_stream(stream));                                          \
  }

extern "C" {
int gsp_edge_list_count(int64_t n, const int32_t* indptr, const int32_t* indices, int directed,
                        int32_t* edge_ptr, void* stream) {
  return gsp::edge_list_count(n, indptr, indices, directed, edge_ptr, gsp::as_stream(stream));
}

int gsp_diffop_count(int64_t n_edges, const int32_t* sources, const int32_t* targets,
                     int32_t* d_indptr, void* stream) {
  GSP_DIFFOP_CHECK_EDGES(n_edges);
  return gsp::diffop_count(n_edges, sources, targets, d_indptr, gsp::as_stream(stream));
}

GSP_DIFFOP_API(f32, float)
GSP_DIFFOP_API(f64, double)
}
