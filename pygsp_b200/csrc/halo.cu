// Halo exchange over NVLink peer memory (no NCCL in the per-step path).
//
// Each rank owns, for a given signal width, two extended state buffers
// (n_local + n_halo rows) and a flag array; both are cudaMalloc'ed here and
// exported with CUDA IPC so that the neighbours map them.  After a recurrence
// step a rank *pushes* the rows its neighbours need straight into their halo rows
// (peer stores through NVLink / NVSwitch), fences, and publishes the step number
// in the neighbours' flag arrays; before the next step it waits until all of its
// neighbours have published that step.  Stream order + flags are the only
// synchronisation -- the host never blocks.
#include "common.cuh"
#include "gspb200.h"

namespace gsp {

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// dst_base[dst_peer[e]][dst_row[e], :] = src[src_row[e], :]; the last block to
// finish publishes `value` to every neighbour (after a system-scope fence).
template <typename T>
__global__ void halo_push_kernel(int64_t n_send, const int64_t* __restrict__ src_row,
                                 const int32_t* __restrict__ dst_peer,
                                 const int64_t* __restrict__ dst_row, const T* __restrict__ src,
                                 T* const* __restrict__ peer_base, int64_t width,
                                 unsigned long long* const* __restrict__ peer_flags,
                                 int n_neighbors, unsigned long long value,
                                 unsigned int* done_counter) {
  const int64_t total = n_send * width;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t e = i / width, c = i - e * width;
    peer_base[dst_peer[e]][dst_row[e] * width + c] = src[src_row[e] * width + c];
  }
  __threadfence_system();                 // my peer stores are performed system-wide
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int prev = atomicAdd(done_counter, 1u);
    if (prev == gridDim.x - 1) {          // every block has fenced its stores
      *done_counter = 0;                  // ready for the next launch (stream-ordered)
      __threadfence_system();
      for (int q = 0; q < n_neighbors; ++q) st_release_sys(peer_flags[q], value);
    }
  }
}

__global__ void halo_wait_kernel(const unsigned long long* flags, const int32_t* neighbor_ids,
                                 int n_neighbors, unsigned long long value) {
  const int q = threadIdx.x;
  if (q < n_neighbors) {
    const unsigned long long* p = flags + neighbor_ids[q];
    while (ld_acquire_sys(p) < value) __nanosleep(100);
  }
}

template <typename T>
static int push_rows(int64_t n_send, const int64_t* src_row, const int32_t* dst_peer,
                     const int64_t* dst_row, const T* src, T* const* peer_base, int64_t width,
                     uint64_t* const* peer_flags, int n_neighbors, uint64_t value,
                     uint32_t* done_counter, cudaStream_t st) {
  const int64_t total = n_send * width;
  const int blocks =
      (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(total, 256), int64_t(sm_count()) * 4));
  halo_push_kernel<T><<<blocks, 256, 0, st>>>(
      n_send, src_row, dst_peer, dst_row, src, peer_base, width,
      reinterpret_cast<unsigned long long* const*>(peer_flags), n_neighbors,
      (unsigned long long)value, done_counter);
  GSP_LAUNCH_CHECK("halo_push");
  return GSP_OK;
}

template <typename T>
int halo_push(const gsp_dist_plan* p, int64_t n_send, int b, uint64_t value, int64_t width,
              cudaStream_t st) {
  return push_rows<T>(n_send, p->src_row, p->dst_peer, p->dst_row, static_cast<const T*>(p->buf[b]),
                      reinterpret_cast<T* const*>(p->peer_base[b]), width, p->peer_flags,
                      p->n_neighbors, value, p->push_counter, st);
}
template int halo_push<float>(const gsp_dist_plan*, int64_t, int, uint64_t, int64_t, cudaStream_t);
template int halo_push<double>(const gsp_dist_plan*, int64_t, int, uint64_t, int64_t, cudaStream_t);

}  // namespace gsp

extern "C" {

int gsp_ipc_alloc(size_t bytes, void** dev_ptr_out, unsigned char* handle64_out) {
  GSP_REQUIRE(dev_ptr_out && handle64_out, "null output");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  void* p = nullptr;
  GSP_CUDA(cudaMalloc(&p, bytes ? bytes : 256));
  GSP_CUDA(cudaMemset(p, 0, bytes ? bytes : 256));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return gsp::check_cuda(e, "cudaIpcGetMemHandle"); }
  memcpy(handle64_out, &h, 64);
  *dev_ptr_out = p;
  return GSP_OK;
}

int gsp_ipc_open(const unsigned char* handle64, void** dev_ptr_out) {
  GSP_REQUIRE(dev_ptr_out && handle64, "null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  GSP_CUDA(cudaIpcOpenMemHandle(dev_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return GSP_OK;
}

int gsp_ipc_close(void* dev_ptr) {
  GSP_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return GSP_OK;
}

int gsp_ipc_free(void* dev_ptr) {
  GSP_CUDA(cudaFree(dev_ptr));
  return GSP_OK;
}

#define GSP_HALO_API(SUF, T)                                                                     \
  int gsp_halo_push_##SUF(int64_t n_send, const int64_t* src_row, const int32_t* dst_peer,       \
                          const int64_t* dst_row, const T* src, T* const* peer_base,             \
                          int64_t width, uint64_t* const* peer_flags, int n_neighbors,           \
                          uint64_t value, uint32_t* done_counter, void* stream) {                \
    return gsp::push_rows<T>(n_send, src_row, dst_peer, dst_row, src, peer_base, width,          \
                             peer_flags, n_neighbors, value, done_counter,                       \
                             gsp::as_stream(stream));                                            \
  }

GSP_HALO_API(f32, float)
GSP_HALO_API(f64, double)

int gsp_halo_wait(const uint64_t* flags, const int32_t* neighbor_ids, int n_neighbors,
                  uint64_t value, void* stream) {
  if (n_neighbors <= 0) return GSP_OK;
  GSP_REQUIRE(n_neighbors <= 1024, "too many neighbours");
  gsp::halo_wait_kernel<<<1, ((n_neighbors + 31) / 32) * 32, 0, gsp::as_stream(stream)>>>(
      reinterpret_cast<const unsigned long long*>(flags), neighbor_ids, n_neighbors,
      (unsigned long long)value);
  GSP_LAUNCH_CHECK("halo_wait");
  return GSP_OK;
}

}  // extern "C"
