// Shared helpers for libgspb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <functional>
#include <stdio.h>
#include <string.h>
#include "gspb200.h"

#define GSP_OK 0
#define GSP_ERR_ARG (-1)
#define GSP_ERR_CUDA (-2)
#define GSP_ERR_UNSUPPORTED (-3)

namespace gsp {

// thread-local message returned by gsp_last_error()
char* error_buffer();

inline int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
  snprintf(error_buffer(), 512, fmt, a, b);
  return code;
}

// kernels launched by this library since load (bench.py's gpu_launches)
void note_launch(int n);

inline int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return GSP_OK;
  return fail(GSP_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

#define GSP_CUDA(call)                                        \
  do {                                                        \
    int _rc = gsp::check_cuda((call), #call);                 \
    if (_rc != GSP_OK) return _rc;                            \
  } while (0)

#define GSP_LAUNCH_CHECK(name)                                \
  do {                                                        \
    gsp::note_launch(1);                                      \
    int _rc = gsp::check_cuda(cudaGetLastError(), name);      \
    if (_rc != GSP_OK) return _rc;                            \
  } while (0)

#define GSP_REQUIRE(cond, msg)                                \
  do {                                                        \
    if (!(cond)) return gsp::fail(GSP_ERR_ARG, "%s (%s)", msg, #cond); \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// number of SMs of the current device (cached per device)
int sm_count();

// ----- the fused recurrence step (csrc/cheby.cu, csrc/cheby_tiled.cu) ----------------------
// x_new = alpha (L x_cur) + beta x_cur + gamma x_old;
//   add_source == false: r_i (+)= ck[i] x_new          (reference order, approximations.py:107-109)
//   first              : r_i  = c0[i]/2 x_cur + ck[i] x_new, x_old unused
//   add_source == true : x_new += sum_i ck[i] r_i      (Clenshaw form, r holds read-only sources)
// reverse: the tiled kernel walks the tiles backwards (the lines the previous step wrote last are
// still in L2 and are the first ones this step reads).
template <typename T>
struct Step {
  bool first;
  const T* x_cur;
  const T* x_old;        // may alias x_new (row-local)
  T* x_new;
  T* r;                  // (nscales, r_rows, nsig)
  int nscales;
  const double* ck;
  const double* c0;
  double alpha, beta, gamma;
  bool add_source, reverse;
};

// Step `s` on rows [rb, re) of the CSR (indptr, indices, vals; nnz entries).  float32 with a tile
// plan: the TMA-tiled kernel on the full tiles, the row-group kernel on the remaining rows.  With a
// halo (the partitioned operator's fused exchange, rb == 0) the boundary tiles run first, in a
// launch of their own; a halo without the tiled kernel is GSP_ERR_UNSUPPORTED.
template <typename T>
int run_step(const gsp_tile_plan* plan, const gsp_halo_fusion* halo, const Step<T>& s, int64_t rb,
             int64_t re, int64_t nnz, const int32_t* indptr, const int32_t* indices, const T* vals,
             int64_t r_rows, int nsig, cudaStream_t st,
             const int64_t* out_perm = nullptr);   // x_new row of local row i is out_perm[i]

// The row-group kernel alone (any nsig / nscales; CG's SpMM, the tiled kernel's remainder rows).
template <typename T>
int cheby_step(bool first, int64_t rb, int64_t re, const int32_t* indptr, const int32_t* indices,
               const T* vals, const T* x_cur, const T* x_old, T* x_new, T* r, int64_t r_rows,
               int nsig, int nscales, const double* ck, const double* c0, double alpha,
               double beta, double gamma, cudaStream_t st, bool add_source = false,
               const int64_t* out_perm = nullptr);

// The TMA-tiled kernel on the n_tiles full tiles from row rb (rb % 4 == 0).  halo != NULL: the
// halo-capable instantiation, whose tiles [0, n_front) are boundary tiles (n_wait_tiles /
// n_push_tiles filled in).
int cheby_step_tiled_f32(const Step<float>& s, int64_t rb, int64_t n_tiles,
                         const gsp_halo_fusion* halo, int64_t n_front, int64_t nnz,
                         const int32_t* indptr, const int32_t* indices, const float* vals,
                         int64_t r_rows, int nsig, const gsp_tile_plan& plan, cudaStream_t st,
                         const int64_t* out_perm);

// Step number s = 1..K of a recurrence; the caller runs it on its rows.
template <typename T>
using StepFn = std::function<int(int s, const Step<T>& step)>;

// cheby_op's forward recurrence (approximations.py:99-112) with coefficient rows c ((nscales, m)):
// accumulates into r; T_1 goes to t1, T_2 to t2, T_k (k >= 3) over T_{k-2}.  t2 may be x.
template <typename T>
int cheby_forward(double lmax, const double* c, int nscales, int m, const T* x, T* r, T* t1, T* t2,
                  const StepFn<T>& step);

// Clenshaw's backward recurrence (see cheby_clenshaw in csrc/cheby.cu) for nsrc <= 16 source
// blocks src: out = sum_i p_i(L) s_i.  The b_k rotate through b1 and b2; nsrc > 1 expects
// b_K = sum_i c_iK s_i in b1, nsrc == 1 folds b_K = c_K x into its first step.
template <typename T>
int cheby_backward(double lmax, const double* c, int nsrc, int m, const T* src, T* out, T* b1,
                   T* b2, const StepFn<T>& step);

// gsp_halo_push_* of state buffer b of a partitioned operator (csrc/halo.cu)
template <typename T>
int halo_push(const gsp_dist_plan* p, int64_t n_send, int b, uint64_t value, int64_t width,
              cudaStream_t st);

// dst[i,:] = src[idx[i],:] (scatter: dst[idx[i],:] = src[i,:]) -- csrc/graph.cu
template <typename T>
int move_rows(bool scatter, int64_t rows, const int64_t* idx, const T* src, int64_t width, T* dst,
              cudaStream_t st);

// indptr[1..n] holds row sizes on entry (indptr[0] = 0) and their inclusive scan on exit --
// csrc/graph.cu, the scan of every count / fill pair
int scan_rows(int32_t* indptr, int64_t n, cudaStream_t st);

// Transpose of an n_rows x n_cols CSR as sorted CSR (t_indptr has n_cols + 1 entries); the
// entries of a row of the result keep ascending column order -- csrc/graph.cu
template <typename T>
int csr_transpose(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* indptr,
                  const int32_t* indices, const T* data, int32_t* t_indptr, int32_t* t_indices,
                  T* t_data, cudaStream_t st);

// ----- vector types: 16-byte packets of T --------------------------------
template <typename T, int VEC> struct Pack;
template <> struct Pack<float, 4> { typedef float4 type; };
template <> struct Pack<float, 2> { typedef float2 type; };
template <> struct Pack<float, 1> { typedef float type; };
template <> struct Pack<double, 2> { typedef double2 type; };
template <> struct Pack<double, 1> { typedef double type; };

template <typename T, int VEC>
struct Vec {
  T v[VEC];
};

template <typename T, int VEC>
__device__ __forceinline__ Vec<T, VEC> load_vec(const T* p) {
  typedef typename Pack<T, VEC>::type P;
  union { P p; Vec<T, VEC> v; } u;
  u.p = *reinterpret_cast<const P*>(p);
  return u.v;
}

// read-only (non-coherent) path: data that no thread of this launch writes
template <typename T, int VEC>
__device__ __forceinline__ Vec<T, VEC> load_vec_ro(const T* p) {
  typedef typename Pack<T, VEC>::type P;
  union { P p; Vec<T, VEC> v; } u;
  u.p = __ldg(reinterpret_cast<const P*>(p));
  return u.v;
}

// streaming load: touched once per launch, do not keep in L1
template <typename T, int VEC>
__device__ __forceinline__ Vec<T, VEC> load_vec_stream(const T* p) {
  typedef typename Pack<T, VEC>::type P;
  union { P p; Vec<T, VEC> v; } u;
  u.p = __ldcs(reinterpret_cast<const P*>(p));
  return u.v;
}

template <typename T, int VEC>
__device__ __forceinline__ void store_vec_stream(T* p, const Vec<T, VEC>& v) {
  typedef typename Pack<T, VEC>::type P;
  union { P p; Vec<T, VEC> v; } u;
  u.v = v;
  __stcs(reinterpret_cast<P*>(p), u.p);
}

}  // namespace gsp
