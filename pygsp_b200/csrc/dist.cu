// The vertex-partitioned cheby_op of ONE rank as a single C entry point.
//
// pygsp/filters/approximations.py:58-114 on rows [lo, hi) of a 1-D partitioned Laplacian
// (SURVEY.md 8e): K fused recurrence steps, each of which also carries this rank's part of
// the halo exchange -- boundary rows of T_k are stored straight into the neighbours' halo
// rows over NVLink peer memory from the step kernel's epilogue, flags order the steps.
// No collective library is involved in the per-step path; the communicator is only needed
// once, on the host side, to build the plan (who needs which rows, IPC handles).
//
// Sequence numbers (one uint64 per rank, advanced by M + 2 per call, identical on all ranks):
//   base+1      entry barrier: nobody writes into a rank that is still in its previous call
//   base+2      halo of T_0 (the input block) is in place
//   base+2+s    halo of the block written by step s is in place, s = 1 .. K-1
#include <type_traits>
#include <vector>
#include <cstdio>
#include "common.cuh"

namespace gsp {

// GSPB200_DIST_TRACE=1: per-step CUDA-event times of one call on stderr (diagnosis; synchronises)
struct StepTrace {
  bool on = false;
  cudaStream_t st = nullptr;
  std::vector<cudaEvent_t> ev;
  explicit StepTrace(cudaStream_t s) : st(s) {
    const char* v = getenv("GSPB200_DIST_TRACE");
    on = v && *v == '1';
  }
  void mark() {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    ev.push_back(e);
  }
  ~StepTrace() {
    if (!on || ev.size() < 2) return;
    cudaEventSynchronize(ev.back());
    fprintf(stderr, "[gspb200 dist trace] ms between marks:");
    for (size_t i = 1; i < ev.size(); ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
      fprintf(stderr, " %.3f", ms);
    }
    fprintf(stderr, "\n");
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};

template <typename T>
int cheby_op_dist(const gsp_dist_plan* p, const gsp_tile_plan* tile, double lmax, const double* c,
                  int nscales, int m, const T* x, int64_t nsig64, T* r, int clenshaw,
                  uint64_t* seq, void* stream) {
  GSP_REQUIRE(p && seq && r, "null argument");
  GSP_REQUIRE(m >= 2, "The coefficients have an invalid shape");        // approximations.py:83-84
  GSP_REQUIRE(nscales >= 1 && nscales <= 16, "1..16 filters per call");
  GSP_REQUIRE(lmax > 0 && lmax == lmax, "lmax must be positive");
  GSP_REQUIRE(nsig64 >= 1 && nsig64 <= (1 << 20), "nsig out of range");
  const int nsig = int(nsig64);
  const int64_t n = p->n_local;
  const int K = m - 1;
  cudaStream_t st = as_stream(stream);
  const uint64_t base = *seq;
  *seq = base + uint64_t(m) + 2;
  T* buf[3] = {static_cast<T*>(p->buf[0]), static_cast<T*>(p->buf[1]), static_cast<T*>(p->buf[2])};
  const T* data = static_cast<const T*>(p->data);
  const bool tiled = std::is_same<T, float>::value && tile && tile->rows_per_tile > 0;
  const bool fused =
      tiled && !p->separate_exchange && p->n_neighbors >= 1 && p->n_neighbors <= 32 &&
      std::max(p->n_push_rows, p->n_boundary_rows) <= (n / tile->rows_per_tile) * tile->rows_per_tile;
  if (clenshaw && (nscales != 1 || K < 2 || !buf[2])) clenshaw = 0;

  StepTrace trace(st);
  trace.mark();
  // entry barrier, input block, halo of T_0
  int rc = halo_push<T>(p, 0, 0, base + 1, nsig, st);
  if (rc != GSP_OK) return rc;
  rc = gsp_halo_wait(p->flags, p->neighbor_ids, p->n_neighbors, base + 1, stream);
  if (rc != GSP_OK) return rc;
  const int64_t* perm = p->perm;      // local row i is row perm[i] of the caller's block
  if (x && perm) {
    rc = move_rows<T>(false, n, perm, x, nsig, buf[0], st);
    if (rc != GSP_OK) return rc;
  } else if (x && x != buf[0]) {
    GSP_CUDA(cudaMemcpyAsync(buf[0], x, sizeof(T) * size_t(n) * nsig, cudaMemcpyDeviceToDevice, st));
  }
  rc = halo_push<T>(p, p->n_send, 0, base + 2, nsig, st);
  if (rc != GSP_OK) return rc;
  trace.mark();

  // Step s waits for the halo of x_cur (base + 1 + s) and, unless it is the last one, publishes
  // the halo of x_new (base + 2 + s).  Fused form (float32 + tile plan): wait, push and publish
  // happen inside the step kernel; otherwise wait kernel -> step -> push kernel.
  const StepFn<T> step = [&](int s, const Step<T>& sp) {
    const bool publish = s < K;
    int b = 0;                          // state buffer x_new is (3: the caller's output)
    while (b < 3 && buf[b] != sp.x_new) ++b;
    const int64_t* out_perm = (clenshaw && s == K) ? perm : nullptr;
    int rc;
    if (fused) {
      gsp_halo_fusion h;
      memset(&h, 0, sizeof(h));
      h.n_push_rows = publish ? p->n_push_rows : 0;
      h.push_ptr = p->push_ptr;
      h.push_peer = p->push_peer;
      h.push_row = p->push_row;
      h.peer_base = b < 3 ? p->peer_base[b] : nullptr;
      h.peer_flags = p->peer_flags;
      h.push_counter = p->fused_counter;
      h.wait_flags = p->flags;
      h.wait_ids = p->neighbor_ids;
      h.publish_value = base + 2 + s;
      h.wait_value = base + 1 + s;
      h.n_neighbors = p->n_neighbors;
      h.n_wait = p->n_neighbors;
      h.n_boundary_rows = p->n_boundary_rows;
      h.n_owned = n;
      h.publish = publish ? 1 : 0;
      rc = run_step<T>(tile, &h, sp, 0, n, p->nnz, p->indptr, p->indices, data, n, nsig, st,
                       out_perm);
    } else {
      rc = gsp_halo_wait(p->flags, p->neighbor_ids, p->n_neighbors, base + 1 + s, stream);
      if (rc == GSP_OK)
        rc = run_step<T>(tile, nullptr, sp, 0, n, p->nnz, p->indptr, p->indices, data, n, nsig, st,
                         out_perm);
      if (rc == GSP_OK && publish) rc = halo_push<T>(p, p->n_send, b, base + 2 + s, nsig, st);
    }
    if (rc == GSP_OK) trace.mark();
    return rc;
  };
  // Clenshaw, single filter: buf[0] keeps x (the source), the b_k rotate through buf[1] and
  // buf[2], the last step writes r
  if (clenshaw) return cheby_backward<T>(lmax, c, 1, m, buf[0], r, buf[1], buf[2], step);
  // forward recurrence, reference order, T_2 over T_0 in buf[0].  With a row permutation the
  // accumulators live in local order in stream-ordered scratch and are scattered to the
  // caller's order at the end.
  T* r_out = r;
  if (perm && n > 0) {
    GSP_CUDA(cudaMallocAsync((void**)&r, sizeof(T) * size_t(nscales) * n * nsig, st));
  }
  rc = cheby_forward<T>(lmax, c, nscales, m, buf[0], r, buf[1], buf[0], step);
  if (r != r_out) {
    for (int i = 0; i < nscales && rc == GSP_OK; ++i)
      rc = move_rows<T>(true, n, perm, r + int64_t(i) * n * nsig, nsig, r_out + int64_t(i) * n * nsig,
                        st);
    cudaFreeAsync(r, st);
  }
  return rc;
}

}  // namespace gsp

extern "C" {
int gsp_cheby_op_dist_f32(const gsp_dist_plan* plan_host, const gsp_tile_plan* tile_host,
                          double lmax, const double* coeffs_host, int nscales, int m, const float* x,
                          int64_t nsig, float* r, int clenshaw, uint64_t* seq_host, void* stream) {
  return gsp::cheby_op_dist<float>(plan_host, tile_host, lmax, coeffs_host, nscales, m, x, nsig, r,
                                   clenshaw, seq_host, stream);
}
int gsp_cheby_op_dist_f64(const gsp_dist_plan* plan_host, const gsp_tile_plan* tile_host,
                          double lmax, const double* coeffs_host, int nscales, int m, const double* x,
                          int64_t nsig, double* r, int clenshaw, uint64_t* seq_host, void* stream) {
  return gsp::cheby_op_dist<double>(plan_host, nullptr, lmax, coeffs_host, nscales, m, x, nsig, r,
                                    clenshaw, seq_host, stream);
}
}
