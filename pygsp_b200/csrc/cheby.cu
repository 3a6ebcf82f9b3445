// Chebyshev recurrence on a CSR Laplacian -- the hot path.
//
// Replaces, for the path pygsp/filters/approximations.py:58-114 (cheby_op):
//   * scipy.sparse._sparsetools.csr_matvecs   (approximations.py:99,107)
//   * the dense "- twf_old" temporary          (approximations.py:107)
//   * the fancy-indexed r[tmpN + N*i] += c*T   (approximations.py:108-109)
// by ONE fused kernel per recurrence step:
//   x_new = alpha * (L x_cur) + beta * x_cur + gamma * x_old
//   r_i   = (first ? c_i0/2 * x_cur : r_i) + c_ik * x_new         i < nscales
// with alpha = 4/lmax, beta = -2, gamma = -1 (first step: 2/lmax, -1, 0), so
// the CSR of L is used as stored (the reference builds a second scaled matrix
// "factor", approximations.py:105) and T_{k-2}/T_{k-1}/T_k make exactly one
// trip each through HBM per step.
//
// Layout: signals are (N, nsig) row-major (a vertex's nsig values adjacent),
// r is (nscales, N, nsig) -- the reference's filter-major (Nscales*N, Nsig).
//
// Lane mapping ("row group" kernel): G = 2^g lanes own one row, each lane a
// VEC-wide packet (16 B) of the row's columns.  The group loads G CSR entries
// with one coalesced access and broadcasts them with shuffles; every lane then
// gathers its packet of x_cur[col] -- a 16*G-byte contiguous, fully coalesced
// request per neighbour -- and accumulates in registers.  The accumulation
// order is the stored CSR order, i.e. the order scipy uses.
#include <type_traits>
#include "common.cuh"

namespace gsp {

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

constexpr int kMaxScales = 16;   // coefficients per launch passed by value
constexpr int kStepThreads = 256;

template <typename T>
struct StepCoef {
  T alpha, beta, gamma;
  T half_c0[kMaxScales];   // c[i,0]/2 (first step only)
  T ck[kMaxScales];        // c[i,k]
  // Clenshaw form: `r` holds nscales read-only source blocks s_i and the step is
  // x_new += sum_i ck[i] * s_i; nothing is accumulated into r.
  int add_source;
};

template <typename T, int VEC, int G, bool FIRST, bool SPMM>
__global__ void __launch_bounds__(kStepThreads)
cheby_step_rowgroup(int64_t row_begin, int64_t row_end,
                    const int32_t* __restrict__ indptr,
                    const int32_t* __restrict__ indices,
                    const T* __restrict__ vals,
                    const T* __restrict__ x_cur,   // rows referenced by indices
                    const T* x_old,                // may alias x_new (row-local)
                    T* x_new,
                    T* __restrict__ r,             // (nscales, r_rows, nsig)
                    int64_t r_rows, int nsig, int nscales,
                    StepCoef<T> coef, const int64_t* __restrict__ out_perm) {
  const int lane = threadIdx.x & (G - 1);
  const int64_t group = (int64_t(blockIdx.x) * kStepThreads + threadIdx.x) / G;
  const int64_t row = row_begin + group;
  // all lanes of a group share `row`; groups never straddle a warp (G <= 32)
  if (row >= row_end) return;
  const unsigned lane_in_warp = threadIdx.x & 31;
  const unsigned gmask = (G == 32) ? 0xffffffffu
                                   : (((1u << G) - 1u) << (lane_in_warp & ~(G - 1)));

  const int start = __ldg(indptr + row);
  const int end = __ldg(indptr + row + 1);
  const int64_t out_row = out_perm ? __ldg(out_perm + row) : row;   // x_new only

  // every lane of the group runs the same trip count (the shuffles below need
  // the whole group); lanes past the last column are merely predicated off
  for (int cbase = 0; cbase < nsig; cbase += G * VEC) {
    const int c0 = cbase + lane * VEC;
    const bool active = c0 < nsig;
    Vec<T, VEC> acc, xo, xc;
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc.v[v] = xo.v[v] = xc.v[v] = T(0);

    // streaming operands first: they are in flight while the gather runs
    if (active) {
      if (!FIRST) xo = load_vec_stream<T, VEC>(x_old + row * nsig + c0);
      xc = load_vec_ro<T, VEC>(x_cur + row * nsig + c0);
    }

    if (SPMM) {
      for (int base = start; base < end; base += G) {
        const int mine = base + lane;
        int col = 0;
        T val = T(0);
        if (mine < end) {
          col = __ldg(indices + mine);
          val = __ldg(vals + mine);
        }
        const int cnt = min(G, end - base);
#pragma unroll 4
        for (int j = 0; j < cnt; ++j) {
          const int cj = __shfl_sync(gmask, col, j, G);
          const T vj = __shfl_sync(gmask, val, j, G);
          if (active) {
            const Vec<T, VEC> xn = load_vec_ro<T, VEC>(x_cur + int64_t(cj) * nsig + c0);
#pragma unroll
            for (int v = 0; v < VEC; ++v) acc.v[v] = fma(vj, xn.v[v], acc.v[v]);
          }
        }
      }
    }
    if (!active) continue;

    Vec<T, VEC> xn;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      T t = fma(coef.alpha, acc.v[v], coef.beta * xc.v[v]);
      if (!FIRST) t = fma(coef.gamma, xo.v[v], t);
      xn.v[v] = t;
    }
    if (coef.add_source) {
      for (int i = 0; i < nscales; ++i) {
        const Vec<T, VEC> sv =
            load_vec_stream<T, VEC>(r + (int64_t(i) * r_rows + row) * nsig + c0);
#pragma unroll
        for (int v = 0; v < VEC; ++v) xn.v[v] = fma(coef.ck[i], sv.v[v], xn.v[v]);
      }
      store_vec_stream<T, VEC>(x_new + out_row * nsig + c0, xn);
      continue;
    }
    store_vec_stream<T, VEC>(x_new + out_row * nsig + c0, xn);

    for (int i = 0; i < nscales; ++i) {
      T* rp = r + (int64_t(i) * r_rows + row) * nsig + c0;
      Vec<T, VEC> rv;
      if (FIRST) {
#pragma unroll
        for (int v = 0; v < VEC; ++v)
          rv.v[v] = fma(coef.ck[i], xn.v[v], coef.half_c0[i] * xc.v[v]);
      } else {
        rv = load_vec_stream<T, VEC>(rp);
#pragma unroll
        for (int v = 0; v < VEC; ++v) rv.v[v] = fma(coef.ck[i], xn.v[v], rv.v[v]);
      }
      store_vec_stream<T, VEC>(rp, rv);
    }
  }
}

// r_i += c_ik * x   for filter banks wider than kMaxScales (no SpMM)
template <typename T>
__global__ void cheby_axpy_scales(int64_t count, const T* __restrict__ x,
                                  T* __restrict__ r, int64_t r_stride, int nscales,
                                  StepCoef<T> coef, bool first,
                                  const T* __restrict__ x0) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; i < count; i += stride) {
    const T xv = x[i];
    for (int s = 0; s < nscales; ++s) {
      T* rp = r + int64_t(s) * r_stride + i;
      *rp = first ? fma(coef.ck[s], xv, coef.half_c0[s] * x0[i]) : fma(coef.ck[s], xv, *rp);
    }
  }
}

template <typename T, int VEC, int G>
static int launch_group(bool first, bool spmm, int64_t row_begin, int64_t row_end,
                        const int32_t* indptr, const int32_t* indices, const T* vals,
                        const T* x_cur, const T* x_old, T* x_new, T* r, int64_t r_rows,
                        int nsig, int nscales, const StepCoef<T>& coef, cudaStream_t st,
                        const int64_t* out_perm) {
  const int64_t rows = row_end - row_begin;
  if (rows <= 0) return GSP_OK;
  const int64_t blocks = ceil_div(rows * G, kStepThreads);
  GSP_REQUIRE(blocks < (int64_t(1) << 31), "row range too large for one launch");
  dim3 grid((unsigned)blocks), block(kStepThreads);
#define GSP_GO(F, S)                                                                   \
  cheby_step_rowgroup<T, VEC, G, F, S><<<grid, block, 0, st>>>(                        \
      row_begin, row_end, indptr, indices, vals, x_cur, x_old, x_new, r, r_rows, nsig, \
      nscales, coef, out_perm)
  if (first && spmm) GSP_GO(true, true);
  else if (first) GSP_GO(true, false);
  else if (spmm) GSP_GO(false, true);
  else GSP_GO(false, false);
#undef GSP_GO
  GSP_LAUNCH_CHECK("cheby_step_rowgroup");
  return GSP_OK;
}

template <typename T, int VEC>
static int launch_vec(int groups_needed, bool first, bool spmm, int64_t rb, int64_t re,
                      const int32_t* indptr, const int32_t* indices, const T* vals,
                      const T* x_cur, const T* x_old, T* x_new, T* r, int64_t r_rows,
                      int nsig, int nscales, const StepCoef<T>& coef, cudaStream_t st,
                      const int64_t* out_perm) {
#define GSP_CASE(GG)                                                                     \
  return launch_group<T, VEC, GG>(first, spmm, rb, re, indptr, indices, vals, x_cur,     \
                                  x_old, x_new, r, r_rows, nsig, nscales, coef, st, out_perm)
  if (groups_needed <= 1) GSP_CASE(1);
  if (groups_needed <= 2) GSP_CASE(2);
  if (groups_needed <= 4) GSP_CASE(4);
  if (groups_needed <= 8) GSP_CASE(8);
  if (groups_needed <= 16) GSP_CASE(16);
  GSP_CASE(32);
#undef GSP_CASE
}

template <typename T> struct MaxVec;
template <> struct MaxVec<float> { static constexpr int value = 4; };
template <> struct MaxVec<double> { static constexpr int value = 2; };


// One recurrence step over rows [rb, re).  Handles any nsig / nscales.
template <typename T>
int cheby_step(bool first, int64_t rb, int64_t re, const int32_t* indptr,
               const int32_t* indices, const T* vals, const T* x_cur, const T* x_old,
               T* x_new, T* r, int64_t r_rows, int nsig, int nscales, const double* ck,
               const double* c0, double alpha, double beta, double gamma, cudaStream_t st,
               bool add_source, const int64_t* out_perm) {
  constexpr int MV = MaxVec<T>::value;
  const bool vec_ok = (nsig % MV == 0) && aligned16(x_cur) && aligned16(x_new) &&
                      aligned16(r) && (first || aligned16(x_old));
  for (int s0 = 0; s0 < nscales || s0 == 0; s0 += kMaxScales) {
    const int ns = min(kMaxScales, nscales - s0);
    StepCoef<T> coef;
    coef.alpha = T(alpha);
    coef.beta = T(beta);
    coef.gamma = T(gamma);
    coef.add_source = add_source ? 1 : 0;
    for (int i = 0; i < kMaxScales; ++i) {
      coef.ck[i] = i < ns ? T(ck[s0 + i]) : T(0);
      coef.half_c0[i] = (first && i < ns) ? T(0.5 * c0[s0 + i]) : T(0);
    }
    T* rs = r + int64_t(s0) * r_rows * nsig;
    if (s0 == 0) {
      int rc;
      if (vec_ok)
        rc = launch_vec<T, MV>((nsig + MV - 1) / MV, first, true, rb, re, indptr, indices,
                               vals, x_cur, x_old, x_new, rs, r_rows, nsig, ns, coef, st, out_perm);
      else
        rc = launch_vec<T, 1>(nsig, first, true, rb, re, indptr, indices, vals, x_cur,
                              x_old, x_new, rs, r_rows, nsig, ns, coef, st, out_perm);
      if (rc != GSP_OK) return rc;
    } else {
      // remaining scales of a wide bank: r_i (+)= c_ik * x_new, no second SpMM
      const int64_t count = (re - rb) * nsig;
      if (count > 0) {
        const int blocks = (int)std::min<int64_t>(ceil_div(count, 256), int64_t(sm_count()) * 16);
        cheby_axpy_scales<T><<<blocks, 256, 0, st>>>(
            count, x_new + rb * nsig, rs + rb * nsig, r_rows * nsig, ns, coef, first,
            x_cur + rb * nsig);
        GSP_LAUNCH_CHECK("cheby_axpy_scales");
      }
    }
    if (nscales == 0) break;
  }
  return GSP_OK;
}

template <typename T>
int run_step(const gsp_tile_plan* plan, const gsp_halo_fusion* halo, const Step<T>& s, int64_t rb,
             int64_t re, int64_t nnz, const int32_t* indptr, const int32_t* indices, const T* vals,
             int64_t r_rows, int nsig, cudaStream_t st, const int64_t* out_perm) {
  const bool tiled = std::is_same<T, float>::value && plan && plan->rows_per_tile > 0 &&
                     rb % 4 == 0 && s.nscales <= kMaxScales && aligned16(indptr) &&
                     aligned16(indices) && aligned16(vals) && aligned16(s.x_cur) &&
                     aligned16(s.x_new) && aligned16(s.r) && (s.first || aligned16(s.x_old));
  if (halo && !tiled)
    return fail(GSP_ERR_UNSUPPORTED, "fused halo step needs the tiled kernel (%s)", "plan");
  int64_t done = rb;
  if constexpr (std::is_same<T, float>::value) {
    if (tiled) {
      const int64_t R = plan->rows_per_tile;
      const int64_t tiles = (re - rb) / R;
      int64_t front = 0;
      if (halo) {
        // Two launches on one stream.  (1) The boundary ("front") tiles with the halo-capable
        // instantiation: tiles whose rows read halo columns wait for the neighbours' flags, rows
        // some neighbour needs are pushed into its halo, and the step is published once both sets
        // are done.  (2) The interior tiles with the plain instantiation.  One kernel for both was
        // 1.6 x slower per step: the boundary code's registers spilled inside the interior
        // tiles' gather loop (ptxas, 60-register cap).  The front launch is a few dozen tiles
        // (~10 us) and publishes before the interior runs.
        GSP_REQUIRE(rb == 0, "fused halo push needs the whole row block in one launch");
        GSP_REQUIRE(halo->n_wait <= 32, "at most 32 neighbours");
        GSP_REQUIRE(halo->n_push_rows >= 0 && halo->n_boundary_rows >= 0, "negative row counts");
        gsp_halo_fusion h = *halo;
        h.n_wait_tiles = ceil_div(h.n_boundary_rows, R);
        h.n_push_tiles = h.publish ? ceil_div(std::max(h.n_push_rows, h.n_boundary_rows), R) : 0;
        front = std::max(h.n_wait_tiles, h.n_push_tiles);
        GSP_REQUIRE(front <= tiles, "boundary rows must lie inside the full tiles");
        if (front > 0) {
          Step<float> f = s;
          f.reverse = false;
          int rc = cheby_step_tiled_f32(f, 0, front, &h, front, nnz, indptr, indices, vals, r_rows,
                                        nsig, *plan, st, out_perm);
          if (rc != GSP_OK) return rc;
        }
      }
      int rc = cheby_step_tiled_f32(s, rb + front * R, tiles - front, nullptr, 0, nnz, indptr,
                                    indices, vals, r_rows, nsig, *plan, st, out_perm);
      if (rc != GSP_OK) return rc;
      done = rb + tiles * R;
    }
  }
  return cheby_step<T>(s.first, done, re, indptr, indices, vals, s.x_cur, s.x_old, s.x_new, s.r,
                       r_rows, nsig, s.nscales, s.ck, s.c0, s.alpha, s.beta, s.gamma, st,
                       s.add_source, out_perm);
}

template <typename T>
int cheby_forward(double lmax, const double* c, int nscales, int m, const T* x, T* r, T* t1, T* t2,
                  const StepFn<T>& step) {
  GSP_REQUIRE(nscales <= 1024, "at most 1024 filters per call");
  double ck[1024], c0[1024];
  for (int i = 0; i < nscales; ++i) c0[i] = c[int64_t(i) * m];
  for (int k = 1; k < m; ++k) {
    for (int i = 0; i < nscales; ++i) ck[i] = c[int64_t(i) * m + k];
    // T_1 = (L x - a x)/a = (2/lmax) L x - x ; r_i = c_i0/2 T_0 + c_i1 T_1
    // T_k = (4/lmax) L T_{k-1} - 2 T_{k-1} - T_{k-2}, written over T_{k-2} (row-local) for k >= 3
    const bool first = k == 1;
    T* dst = (k & 1) ? t1 : t2;
    const T* cur = first ? x : ((k & 1) ? t2 : t1);
    const T* old = first ? nullptr : (k == 2 ? x : dst);
    // even k walks the tiles backwards: the lines of T_{k-1} and r that the previous
    // step wrote last are still in L2 and are the first ones this step reads
    int rc = step(k, {first, cur, old, dst, r, nscales, ck, c0, first ? 2.0 / lmax : 4.0 / lmax,
                      first ? -1.0 : -2.0, first ? 0.0 : -1.0, false, (k & 1) == 0});
    if (rc != GSP_OK) return rc;
  }
  return GSP_OK;
}

// Full operator (approximations.py:58-114): K = m-1 fused steps on `stream`.
template <typename T>
int cheby_op(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
             const T* vals, double lmax, const double* coeffs, int nscales, int m, const T* x,
             int nsig, T* r, T* work, const gsp_tile_plan* plan, cudaStream_t st) {
  GSP_REQUIRE(n >= 0 && nsig >= 1 && nscales >= 1, "bad sizes");
  GSP_REQUIRE(m >= 2, "The coefficients have an invalid shape");   // approximations.py:83-84
  GSP_REQUIRE(lmax > 0 && lmax == lmax, "lmax must be positive");
  if (n == 0) return GSP_OK;
  return cheby_forward<T>(lmax, coeffs, nscales, m, x, r, work, work + n * int64_t(nsig),
                          [&](int, const Step<T>& s) {
                            return run_step<T>(plan, nullptr, s, 0, n, nnz, indptr, indices, vals,
                                               n, nsig, st);
                          });
}

// out = sum_i w[i] * src_i   (src: (nsrc, count) blocks) -- the top Clenshaw term S_K
template <typename T>
__global__ void combine_sources(int64_t count, const T* __restrict__ src, int nsrc,
                                StepCoef<T> coef, T* __restrict__ out) {
  int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; i < count; i += stride) {
    T acc = T(0);
    for (int s = 0; s < nsrc; ++s) acc = fma(coef.ck[s], src[int64_t(s) * count + i], acc);
    out[i] = acc;
  }
}

// Chebyshev sums by Clenshaw's recurrence (SURVEY.md 8f ranks 1 and 2).  For source
// blocks s_i (nsrc of them, (nsrc, n, nsig) in memory) and coefficient rows c_i:
//   out = sum_i p_i(L) s_i,   p_i = c_i0/2 + sum_k c_ik T_k(Lt),  Lt = (2/lmax) L - I
// is evaluated as ONE backward recurrence on an (n, nsig) block,
//   S_k = sum_i c_ik s_i ;  b_k = S_k + 2 Lt b_{k+1} - b_{k+2} ;  out = S_0/2 + Lt b_1 - b_2,
// i.e. K SpMMs in total -- the reference's synthesis (filter.py:313-322) runs nsrc
// separate forward recurrences, nsrc*K SpMMs -- and no accumulator block.  With
// nsrc = 1 this is the single-filter Clenshaw evaluation (b_K = c_K x is folded into
// the first step).  work holds 2*n*nsig elements.  Rounding differs from the forward
// recurrence, the value does not (tests: same tolerance against the float64 oracle).
template <typename T>
int cheby_backward(double lmax, const double* c, int nsrc, int m, const T* src, T* out, T* b1,
                   T* b2, const StepFn<T>& step) {
  const int K = m - 1;
  const double a2 = 4.0 / lmax;                  // 2 Lt = a2 L - 2 I
  T* xs = const_cast<T*>(src);                   // read-only source blocks
  double ck[kMaxScales], zero[kMaxScales] = {};
  T* b_cur = b1;                                 // b_{k+1}
  T* b_old = nullptr;                            // b_{k+2}
  int s = 0, k_next = K - 1;
  if (nsrc == 1) {
    if (K == 1)                                  // out = c0/2 x + c1 Lt x
      return step(1, {true, src, nullptr, out, out, 0, zero, zero, c[1] * 2.0 / lmax,
                      0.5 * c[0] - c[1], 0.0, false, false});
    // b_{K-1} = c_{K-1} x + 2 Lt (c_K x): b_K = c_K x is never materialised
    int rc = step(++s, {true, src, nullptr, b1, b1, 0, zero, zero, c[K] * a2,
                        c[K - 1] - 2.0 * c[K], 0.0, false, false});
    if (rc != GSP_OK) return rc;
    k_next = K - 2;
  }
  for (int k = k_next; k >= 0; --k) {
    const bool last = k == 0;
    // middle: b_k = a2 L b_{k+1} - 2 b_{k+1} - b_{k+2} + S_k
    // last  : out = (a2/2) L b_1 - b_1 - b_2 + S_0/2
    const double alpha = last ? 0.5 * a2 : a2, beta = last ? -1.0 : -2.0;
    double gamma = -1.0;
    for (int i = 0; i < nsrc; ++i) ck[i] = (last ? 0.5 : 1.0) * c[int64_t(i) * m + k];
    const T* old = b_old;
    if (!old) {
      // no b_{k+2} buffer yet: it is c_K x (nsrc == 1, folded into the source term) or 0
      if (nsrc == 1) ck[0] -= c[K];
      gamma = 0.0;
      old = b_cur;                                // any valid block, multiplied by 0
    }
    T* dst = last ? out : (b_old ? b_old : b2);
    int rc = step(++s, {false, b_cur, old, dst, xs, nsrc, ck, zero, alpha, beta, gamma, true,
                        (k & 1) == 0});
    if (rc != GSP_OK) return rc;
    b_old = b_cur;
    b_cur = dst;
  }
  return GSP_OK;
}

template <typename T>
int cheby_clenshaw(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,
                   const T* vals, double lmax, const double* c, int nsrc, int m, const T* src,
                   int nsig, T* out, T* work, const gsp_tile_plan* plan, cudaStream_t st) {
  GSP_REQUIRE(n >= 0 && nsig >= 1 && nsrc >= 1 && nsrc <= kMaxScales, "bad sizes");
  GSP_REQUIRE(m >= 2, "The coefficients have an invalid shape");
  GSP_REQUIRE(lmax > 0 && lmax == lmax, "lmax must be positive");
  if (n == 0) return GSP_OK;
  if (nsrc > 1) {
    // b_K = S_K by one combine pass
    StepCoef<T> coef;
    memset(&coef, 0, sizeof(coef));
    for (int i = 0; i < nsrc; ++i) coef.ck[i] = T(c[int64_t(i) * m + m - 1]);
    const int64_t count = n * int64_t(nsig);
    const int blocks = (int)std::min<int64_t>(ceil_div(count, 256), int64_t(sm_count()) * 16);
    combine_sources<T><<<blocks, 256, 0, st>>>(count, src, nsrc, coef, work);
    GSP_LAUNCH_CHECK("combine_sources");
  }
  return cheby_backward<T>(lmax, c, nsrc, m, src, out, work, work + n * int64_t(nsig),
                           [&](int, const Step<T>& s) {
                             return run_step<T>(plan, nullptr, s, 0, n, nnz, indptr, indices,
                                                vals, n, nsig, st);
                           });
}

// y = A x for a block of vectors (no recurrence, no r): used by Lanczos and
// exposed for callers that only need the product (learning.py CG, "next").
template <typename T>
int spmm_plain(int64_t n, const int32_t* indptr, const int32_t* indices, const T* vals,
               const T* x, int nsig, T* y, cudaStream_t st) {
  // x_new = 1 * (A x) + 0 * x ; FIRST form with nscales = 0 touches no r
  double none = 0;
  return cheby_step<T>(true, 0, n, indptr, indices, vals, x, nullptr, y, y, n, nsig, 0, &none,
                       &none, 1.0, 0.0, 0.0, st);
}

#define GSP_INSTANTIATE(T)                                                                      \
  template int cheby_step<T>(bool, int64_t, int64_t, const int32_t*, const int32_t*, const T*,  \
                             const T*, const T*, T*, T*, int64_t, int, int, const double*,      \
                             const double*, double, double, double, cudaStream_t, bool,         \
                             const int64_t*);                                                   \
  template int run_step<T>(const gsp_tile_plan*, const gsp_halo_fusion*, const Step<T>&,        \
                           int64_t, int64_t, int64_t, const int32_t*, const int32_t*, const T*, \
                           int64_t, int, cudaStream_t, const int64_t*);                         \
  template int cheby_forward<T>(double, const double*, int, int, const T*, T*, T*, T*,          \
                                const StepFn<T>&);                                              \
  template int cheby_backward<T>(double, const double*, int, int, const T*, T*, T*, T*,         \
                                 const StepFn<T>&);
GSP_INSTANTIATE(float)
GSP_INSTANTIATE(double)
#undef GSP_INSTANTIATE

}  // namespace gsp

// ------------------------------- C ABI ------------------------------------
extern "C" {

#define GSP_CHEBY_API(SUF, T)                                                                     \
  int gsp_cheby_op_##SUF(int64_t n, int64_t nnz, const int32_t* indptr, const int32_t* indices,   \
                         const T* data, double lmax, const double* coeffs_host, int nscales,      \
                         int m, const T* x, int64_t nsig, T* r, T* work,                          \
                         const gsp_tile_plan* plan_host, void* stream) {                          \
    GSP_REQUIRE(nsig >= 1 && nsig <= (1 << 20), "nsig out of range");                             \
    return gsp::cheby_op<T>(n, nnz, indptr, indices, data, lmax, coeffs_host, nscales, m, x,      \
                            (int)nsig, r, work, plan_host, gsp::as_stream(stream));               \
  }                                                                                               \
  int gsp_cheby_step_##SUF(int first, int64_t row_begin, int64_t row_end, int64_t nnz,            \
                           const int32_t* indptr, const int32_t* indices, const T* data,          \
                           const T* x_cur, const T* x_old, T* x_new, T* r, int64_t r_rows,        \
                           int64_t nsig, int nscales, const double* ck_host,                      \
                           const double* c0_host, double alpha, double beta, double gamma,        \
                           const gsp_tile_plan* plan_host, void* stream) {                        \
    GSP_REQUIRE(nsig >= 1 && nsig <= (1 << 20), "nsig out of range");                             \
    const gsp::Step<T> s = {first != 0, x_cur, x_old, x_new, r, nscales, ck_host, c0_host,        \
                            alpha, beta, gamma, false, false};                                    \
    return gsp::run_step<T>(plan_host, nullptr, s, row_begin, row_end, nnz, indptr, indices,      \
                            data, r_rows, (int)nsig, gsp::as_stream(stream));                     \
  }                                                                                               \
  int gsp_cheby_clenshaw_##SUF(int64_t n, int64_t nnz, const int32_t* indptr,                     \
                               const int32_t* indices, const T* data, double lmax,                \
                               const double* coeffs_host, int nsrc, int m, const T* sources,      \
                               int64_t nsig, T* out, T* work, const gsp_tile_plan* plan_host,     \
                               void* stream) {                                                    \
    GSP_REQUIRE(nsig >= 1 && nsig <= (1 << 20), "nsig out of range");                             \
    return gsp::cheby_clenshaw<T>(n, nnz, indptr, indices, data, lmax, coeffs_host, nsrc, m,      \
                                  sources, (int)nsig, out, work, plan_host,                       \
                                  gsp::as_stream(stream));                                        \
  }                                                                                               \
  int gsp_spmm_##SUF(int64_t n, const int32_t* indptr, const int32_t* indices, const T* data,     \
                     const T* x, int64_t nsig, T* y, void* stream) {                              \
    GSP_REQUIRE(nsig >= 1 && nsig <= (1 << 20), "nsig out of range");                             \
    return gsp::spmm_plain<T>(n, indptr, indices, data, x, (int)nsig, y, gsp::as_stream(stream)); \
  }

GSP_CHEBY_API(f32, float)
GSP_CHEBY_API(f64, double)

int gsp_cheby_step_halo_f32(int first, int64_t n_rows, int64_t nnz, const int32_t* indptr,
                            const int32_t* indices, const float* data, const float* x_cur,
                            const float* x_old, float* x_new, float* r, int64_t r_rows,
                            int64_t nsig, int nscales, const double* ck_host,
                            const double* c0_host, double alpha, double beta, double gamma,
                            int reverse, const gsp_tile_plan* plan_host,
                            const gsp_halo_fusion* halo_host, void* stream) {
  if (!(plan_host && plan_host->rows_per_tile > 0 && halo_host))
    return gsp::fail(GSP_ERR_UNSUPPORTED, "fused halo step needs a tile plan (%s)", "plan");
  GSP_REQUIRE(nscales <= gsp::kMaxScales, "too many filters for the fused step");
  const gsp::Step<float> s = {first != 0, x_cur, x_old, x_new, r, nscales, ck_host, c0_host,
                              alpha, beta, gamma, false, reverse != 0};
  return gsp::run_step<float>(plan_host, halo_host, s, 0, n_rows, nnz, indptr, indices, data,
                              r_rows, (int)nsig, gsp::as_stream(stream));
}

}  // extern "C"
