// Tiled, warp-specialised Chebyshev step for sm_100a: the float32 fast path.
//
// Same arithmetic as cheby_step_rowgroup (csrc/cheby.cu) -- and therefore the same
// reference lines, pygsp/filters/approximations.py:99-112 -- but every operand
// that is read *contiguously* no longer passes through registers/L1:
//
//   * a persistent CTA owns row tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...
//   * warp 0 is a producer: for each tile it issues 1-D TMA bulk copies
//     (cp.async.bulk ... mbarrier::complete_tx, L2 evict-first) of the tile's CSR slab
//     (indptr / indices / values) and of the tile's x_old and r rows into a
//     ring of `stages` shared-memory stages; the tile's first/last CSR offsets are
//     fetched one tile ahead so that their latency is off the critical path;
//   * the consumer warps wait on the stage's "full" mbarrier, read the CSR
//     entries from shared memory four at a time (LDS.128, no shuffles), gather x_cur
//     rows with coalesced 16-byte loads through L1/L2 (the only traffic left on that
//     path, so L1 holds nothing but x_cur), accumulate in registers in stored CSR
//     order, apply the three-term recurrence and the coefficient AXPYs and store
//     x_new / r with streaming 16-byte stores; then release the stage ("empty").
//
// Two optional roles of the same kernel:
//   * add_source (Clenshaw form): the r tiles are read-only source blocks,
//     x_new += sum_i ck_i s_i, nothing is written to r  (single-filter Clenshaw and
//     the fused synthesis of Filter.filter);
//   * halo fusion (vertex-partitioned path): wait for the neighbours' flags in the
//     prologue, store boundary rows of x_new into the neighbours' halo rows from
//     the epilogue (peer stores over NVLink), publish the step when the last
//     boundary tile is done  (gsp_halo_fusion in the header).
//
// Lane mapping: G = nsig/4 lanes own one row (a float4 packet each), 32/G rows
// per warp in flight.  A tile's slab must fit `slab_cap` entries: the caller
// obtains the bound from tile_nnz_max() once per matrix (see gsp_cheby_tile_plan).
#include "common.cuh"
#include "gspb200.h"

namespace gsp {

constexpr int kTiledMaxScales = 16;

struct TileArgs {
  int64_t n_tiles;
  int64_t row_begin;   // first row of tile 0 (multiple of 4)
  int64_t r_rows;
  int64_t nnz;
  const int32_t* indptr;
  const int32_t* indices;
  const float* vals;
  const float* x_cur;
  const float* x_old;
  float* x_new;
  float* r;
  int rows_per_tile;   // R, multiple of 4
  int slab_cap;        // entries per stage for indices / values (multiple of 4)
  int stages;
  int consumer_warps;
  int nsig;
  int nscales;
  float alpha, beta, gamma;
  float half_c0[kTiledMaxScales];
  float ck[kTiledMaxScales];
  gsp_halo_fusion halo;   // all zero when the step does not exchange a halo
  int l2_hint;            // evict-first hint on the streamed TMA copies
  int keep_writes;        // plain instead of evict-first stores for x_new / r
  int reverse;            // walk the tiles from the last to the first (see cheby_op)
  int64_t n_front;        // tiles [0, n_front) always run first, in order (halo: boundary tiles)
  int add_source;         // Clenshaw form: x_new += sum_i ck[i] * (tile i of r), r is not written
  const int64_t* out_perm;  // x_new row of local row i is out_perm[i] (NULL: i); last step of a partitioned call
  int vec_direct;           // x_old / r rows are read straight from global memory (not staged by TMA)
};

// ----------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_addr(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
// 1-D TMA bulk copy global -> shared, completion counted on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_addr(dst)),
      "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(smem_addr(bar))
      : "memory");
}

// same, with an L2 eviction-priority hint (streamed operands: read once per step)
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes,
                                              uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1], %2, [%3], %4;" ::"r"(smem_addr(dst)),
      "l"(__cvta_generic_to_global(src)), "r"(bytes), "r"(smem_addr(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}

__device__ __forceinline__ float4 ldg_f4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ void stcs_f4(float* p, const float4& v) {
  __stcs(reinterpret_cast<float4*>(p), v);
}
// x_new / r: streaming (evict-first) stores, or plain ones when the next step walks the
// tiles in the opposite direction and re-reads the lines this step wrote last
__device__ __forceinline__ void store_f4(float* p, const float4& v, bool keep) {
  if (keep) *reinterpret_cast<float4*>(p) = v; else stcs_f4(p, v);
}

// shared-memory carve-up, identical on host and device
struct TileLayout {
  int vec_bytes;      // x_old + r tiles of one stage
  int slab_bytes;     // one of the two CSR slabs
  int ptr_bytes;      // indptr slab + trailing slot
  int stage_bytes;
  int bar_bytes;
  __host__ __device__ TileLayout(int R, int cap, int nsig, int nscales, bool first, int stages) {
    vec_bytes = first ? 0 : (1 + nscales) * R * nsig * 4;
    slab_bytes = (cap + 16) * 4;                // +16: aligned groups may run past the end
    ptr_bytes = (R + 4) * 4;
    stage_bytes = vec_bytes + 2 * slab_bytes + ptr_bytes + 16;   // +16: slab offset, group counter
    bar_bytes = ((2 * stages * 8 + 15) / 16) * 16;
  }
  __host__ __device__ int total(int stages) const { return bar_bytes + stages * stage_bytes; }
};

// Order in which the persistent CTAs visit the tiles.  Tiles [0, n_front) come first, in
// order (vertex-partitioned path: the boundary tiles, whose rows the neighbours wait for);
// the others are walked forwards or backwards (`reverse`: the lines the previous step wrote
// last are still in L2 and are the first ones this step reads).
__device__ __forceinline__ int64_t tile_of_slot(const TileArgs& a, int64_t slot) {
  if (slot < a.n_front) return slot;
  return a.reverse ? a.n_tiles - 1 - (slot - a.n_front) : slot;
}

// Halo rows of x_cur are written by the neighbours (peer stores) while this kernel may
// already be running: a tile whose rows reference halo columns (the boundary tiles of a
// partitioned step, a few per launch) gathers through L2 (ld.global.cg), never through the
// non-coherent path.  Interior tiles only touch rows this GPU owns, which are read-only for the
// whole launch: ld.global.nc.
template <bool COH>
__device__ __forceinline__ float4 gather_f4(const float* __restrict__ xg, int col, int ns) {
  const float* p = xg + int64_t(col) * ns;
  if (COH) return __ldcg(reinterpret_cast<const float4*>(p));
  return ldg_f4(p);
}

// sum_j w_j x_cur[col_j, packets of this lane] over the stored entries [jb, je) of one row
// (slab-relative offsets).  The slab offset is a multiple of 4, so groups of four CSR entries
// are 16-byte aligned in shared memory: one LDS.128 brings four column indices, one four
// weights.  Slots outside [jb, je) (row head / tail) are predicated off, so the sum runs over
// the row's entries in stored order.  A lane owns P float4 packets of the row, 16 G bytes apart
// (P = 1: G lanes cover the row once; P = 2: G lanes cover it twice, so a row group is a quarter
// warp for 64 signals and one LDS.128 of CSR entries serves four rows instead of two -- the
// broadcast read costs one L1 wavefront per quarter warp whatever it delivers).  4 / P entries
// are in flight per lane at a time (the same 64 bytes either way).
// COH: the row may reference halo columns (boundary tiles of a partitioned step) -- the tile
// gathers through L2 then; interior tiles use the plain non-coherent gather only.
template <int G, int P, bool COH>
__device__ __forceinline__ void row_gather_sum(const int32_t* __restrict__ sm_col,
                                               const float* __restrict__ sm_val, int jb, int je,
                                               const float* __restrict__ xg, float4 (&acc)[P]) {
  constexpr int NS = 4 * G * P;
  constexpr int E = 4 / P;                         // entries requested back to back
  const unsigned span = unsigned(je - jb);
#pragma unroll
  for (int p = 0; p < P; ++p) acc[p] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int jj = jb & ~3; jj < je; jj += 4) {
    const int4 c4 = *reinterpret_cast<const int4*>(sm_col + jj);
    const float4 w4 = *reinterpret_cast<const float4*>(sm_val + jj);
    const int base = jj - jb;
    const int cq[4] = {c4.x, c4.y, c4.z, c4.w};
    const float wq[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
    for (int h = 0; h < P; ++h) {
      float4 xv[E][P];
      bool ok[E];
#pragma unroll
      for (int e = 0; e < E; ++e) {
        ok[e] = unsigned(base + h * E + e) < span;
#pragma unroll
        for (int p = 0; p < P; ++p)
          if (ok[e]) xv[e][p] = gather_f4<COH>(xg + p * 4 * G, cq[h * E + e], NS);
      }
#pragma unroll
      for (int e = 0; e < E; ++e) {
        if (ok[e]) {
          const float w = wq[h * E + e];
#pragma unroll
          for (int p = 0; p < P; ++p) {
            acc[p].x = fmaf(w, xv[e][p].x, acc[p].x);
            acc[p].y = fmaf(w, xv[e][p].y, acc[p].y);
            acc[p].z = fmaf(w, xv[e][p].z, acc[p].z);
            acc[p].w = fmaf(w, xv[e][p].w, acc[p].w);
          }
        }
      }
    }
  }
}

// What a consumer lane needs to process one staged tile.
struct TileCtx {
  const float* sm_vec;      // x_old tile, then one r / source tile per scale (empty in direct mode)
  const int32_t* sm_col;    // CSR slab: column indices
  const float* sm_val;      //           values
  const int32_t* sm_ptr;    // indptr[r0 .. r0 + R], slab offset at [R + 4]
  int64_t tile;
  int64_t r0;               // first row of the tile (block-local row index)
  int cw, sub, c0;          // consumer warp, row slot inside the warp, first column of the lane
  bool vd;                  // direct mode: x_old / r rows come straight from global memory
};

__device__ __forceinline__ void fma4(float4& d, float w, const float4& v) {
  d.x = fmaf(w, v.x, d.x);
  d.y = fmaf(w, v.y, d.y);
  d.z = fmaf(w, v.z, d.z);
  d.w = fmaf(w, v.w, d.w);
}

// The rows of one tile: gather + three-term recurrence + coefficient AXPYs + stores.
// COH: the tile's rows may reference halo columns (coherent gathers through L2).
template <int G, bool FIRST, int NSC, bool COH, int P>
__device__ __forceinline__ void tile_rows(const TileArgs& a, const TileCtx t) {
  constexpr int RP = 32 / G;               // rows in flight per warp
  constexpr int NS = 4 * G * P;            // signal columns (compile-time: cheap addressing)
  constexpr int PS = 4 * G;                // column distance between a lane's packets
  const int R = a.rows_per_tile;
  const int NW = a.consumer_warps;
  const int c0 = t.c0;
  const float* __restrict__ xg = a.x_cur + c0;      // this lane's first column packet of x_cur
  const int nscales = NSC >= 0 ? NSC : a.nscales;
  const float alpha = a.alpha, beta = a.beta, gamma = a.gamma;
  const bool keep_writes = a.keep_writes != 0;
  const bool VD = t.vd;
  const float* sm_vec = t.sm_vec;
  const int a0 = t.sm_ptr[R + 4];
  const int64_t r0 = t.r0;
  const float* __restrict__ xc_tile = xg + r0 * NS;
  float* __restrict__ xn_tile = a.x_new + r0 * NS + c0;
  float* __restrict__ r_tile = a.r + r0 * NS + c0;
  const int64_t r_stride = a.r_rows * NS;

  for (int lr = t.cw * RP + t.sub; lr < R; lr += NW * RP) {
    const int off = lr * NS;
    const int jb = t.sm_ptr[lr] - a0;
    const int je = t.sm_ptr[lr + 1] - a0;
    float4 xc[P];
#pragma unroll
    for (int p = 0; p < P; ++p) xc[p] = ldg_f4(xc_tile + off + p * PS);
    // direct mode: this row's x_old and first r / source packets are requested now (streaming
    // loads, no L1 allocation) and consumed after the gather loop, which hides their latency
    float4 xo_d[P], r0_d[P];
#pragma unroll
    for (int p = 0; p < P; ++p) xo_d[p] = r0_d[p] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!FIRST && VD) {
#pragma unroll
      for (int p = 0; p < P; ++p) {
        xo_d[p] = __ldcs(reinterpret_cast<const float4*>(a.x_old + (r0 + lr) * NS + c0 + p * PS));
        if (NSC != 0 && nscales > 0)
          r0_d[p] = __ldcs(reinterpret_cast<const float4*>(a.r + (r0 + lr) * NS + c0 + p * PS));
      }
    }
    float4 acc[P];
    row_gather_sum<G, P, COH>(t.sm_col, t.sm_val, jb, je, xg, acc);
    float4 xn[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
      xn[p].x = fmaf(alpha, acc[p].x, beta * xc[p].x);
      xn[p].y = fmaf(alpha, acc[p].y, beta * xc[p].y);
      xn[p].z = fmaf(alpha, acc[p].z, beta * xc[p].z);
      xn[p].w = fmaf(alpha, acc[p].w, beta * xc[p].w);
      if (!FIRST) {
        const float4 xo =
            VD ? xo_d[p] : *reinterpret_cast<const float4*>(sm_vec + off + c0 + p * PS);
        fma4(xn[p], gamma, xo);
      }
    }
    if (!FIRST && NSC != 0 && a.add_source) {
      // Clenshaw form: the r tiles are read-only source blocks, x_new += sum_i ck_i s_i
#pragma unroll
      for (int i = 0; i < (NSC >= 0 ? NSC : kTiledMaxScales); ++i) {
        if (NSC < 0 && i >= nscales) break;
        const float w = a.ck[i];
#pragma unroll
        for (int p = 0; p < P; ++p) {
          const float4 sv =
              VD ? (i == 0 ? r0_d[p]
                           : __ldcs(reinterpret_cast<const float4*>(
                                 a.r + i * r_stride + (r0 + lr) * NS + c0 + p * PS)))
                 : *reinterpret_cast<const float4*>(sm_vec + (i + 1) * R * NS + off + c0 + p * PS);
          fma4(xn[p], w, sv);
        }
      }
    }
    if (a.out_perm) {    // the caller's row order: local row -> original row (uniform branch)
      float* dst = a.x_new + __ldg(a.out_perm + r0 + lr) * NS + c0;
#pragma unroll
      for (int p = 0; p < P; ++p) store_f4(dst + p * PS, xn[p], keep_writes);
    } else {
#pragma unroll
      for (int p = 0; p < P; ++p) store_f4(xn_tile + off + p * PS, xn[p], keep_writes);
    }
#pragma unroll
    for (int i = 0; i < (NSC >= 0 ? NSC : kTiledMaxScales); ++i) {
      if (NSC < 0 && i >= nscales) break;
      if (!FIRST && a.add_source) break;
      const float ck = a.ck[i];
#pragma unroll
      for (int p = 0; p < P; ++p) {
        float4 rv;
        if (FIRST) {
          const float h0 = a.half_c0[i];
          rv.x = fmaf(ck, xn[p].x, h0 * xc[p].x);
          rv.y = fmaf(ck, xn[p].y, h0 * xc[p].y);
          rv.z = fmaf(ck, xn[p].z, h0 * xc[p].z);
          rv.w = fmaf(ck, xn[p].w, h0 * xc[p].w);
        } else {
          rv = VD ? (i == 0 ? r0_d[p]
                            : __ldcs(reinterpret_cast<const float4*>(
                                  a.r + i * r_stride + (r0 + lr) * NS + c0 + p * PS)))
                  : *reinterpret_cast<const float4*>(sm_vec + (i + 1) * R * NS + off + c0 + p * PS);
          fma4(rv, ck, xn[p]);
        }
        store_f4(r_tile + i * r_stride + off + p * PS, rv, keep_writes);
      }
    }
  }
}

// A boundary ("front") tile of a partitioned step -- a few tiles per launch.  It is a real
// function call on purpose: inlined, its extra state (flags, peer tables, a second copy of
// the gather loop) made ptxas spill registers in the interior tiles' loop as well
// (1.6 x slower steps, measured).  Does, for one consumer warp:
//   wait   : until the neighbours have published the halo of x_cur (they stored it straight
//            into this GPU's memory and released wait_value afterwards);
//   rows   : the tile's rows with coherent gathers;
//   push   : every lane re-reads the packets it has just stored (its own writes, program
//            order) and stores them into the halo rows of the neighbours that reference the
//            row -- peer stores over NVLink;
//   publish: every warp of every CTA checks in once per front tile; when the last one has,
//            (a) all boundary rows of x_new are stored in the neighbours and (b) nobody on this
//            GPU reads the halo of x_cur any more: the step is released to the neighbours,
//            which may then read their halo of x_new and overwrite our halo of x_cur's buffer.
template <int G, bool FIRST, int NSC>
__device__ __noinline__ void boundary_tile(const TileArgs& a, const TileCtx t, int lane) {
  constexpr int RP = 32 / G;
  constexpr int NS = 4 * G;
  const int R = a.rows_per_tile;
  const int NW = a.consumer_warps;
  if (t.tile < a.halo.n_wait_tiles && a.halo.n_wait > 0) {
    if (lane < a.halo.n_wait) {
      const unsigned long long* f =
          reinterpret_cast<const unsigned long long*>(a.halo.wait_flags) + a.halo.wait_ids[lane];
      unsigned long long seen;
      do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(f) : "memory");
      } while (seen < a.halo.wait_value);
    }
    __syncwarp();
  }
  tile_rows<G, FIRST, NSC, true, 1>(a, t);
  if (t.tile >= a.halo.n_push_tiles) return;
  if (!a.out_perm) {
    const float* xn_tile = a.x_new + t.r0 * NS + t.c0;
    for (int lr = t.cw * RP + t.sub; lr < R; lr += NW * RP) {
      const int64_t lrow = t.tile * R + lr;
      if (lrow >= a.halo.n_push_rows) continue;
      const int e0 = a.halo.push_ptr[lrow], e1 = a.halo.push_ptr[lrow + 1];
      if (e0 == e1) continue;
      const float4 xn = *reinterpret_cast<const float4*>(xn_tile + lr * NS);
      for (int e = e0; e < e1; ++e) {
        float* dst = reinterpret_cast<float* const*>(a.halo.peer_base)[a.halo.push_peer[e]] +
                     a.halo.push_row[e] * NS + t.c0;
        *reinterpret_cast<float4*>(dst) = xn;
      }
    }
  }
  __threadfence_system();
  __syncwarp();
  if (lane == 0) {
    const unsigned long long want =
        (unsigned long long)a.halo.n_push_tiles * (unsigned long long)NW;
    const unsigned long long prev =
        atomicAdd(reinterpret_cast<unsigned long long*>(a.halo.push_counter), 1ull);
    if (prev + 1 == want) {
      *reinterpret_cast<volatile unsigned long long*>(a.halo.push_counter) = 0ull;
      __threadfence_system();
      for (int q = 0; q < a.halo.n_neighbors; ++q)
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(
                         reinterpret_cast<unsigned long long* const*>(a.halo.peer_flags)[q]),
                     "l"((unsigned long long)a.halo.publish_value)
                     : "memory");
    }
  }
}

// One packet per lane: 1 + 16 warps per CTA, 2 CTAs per SM (<= 60 registers).  Two packets per
// lane keep twice the state per lane: 1 + 8 warps, 3 CTAs per SM (<= 75 registers).
template <int G, bool FIRST, int NSC, bool HALO, int P>
__global__ void __launch_bounds__(32 * (P == 2 ? 9 : 17), P == 2 ? 3 : 2)
cheby_step_tiled(const __grid_constant__ TileArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int R = a.rows_per_tile;
  const int S = a.stages;
  const int NW = a.consumer_warps;
  const int nsig = a.nsig;
  const bool VD = !FIRST && a.vec_direct != 0;     // CTA-uniform
  const TileLayout lay(R, a.slab_cap, nsig, a.nscales, FIRST || VD, S);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + S;
  unsigned char* stage0 = smem + lay.bar_bytes;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == 0) {
    // ------------------------------------------------------------- producer
    // (nothing the producer stages depends on the halo: CSR slabs, x_old and r rows are local)
    if (lane != 0) return;
    // x_old / r / CSR are touched once per step: mark them evict-first so that the
    // L2 keeps the x_cur lines the gathers re-use (GSPB200_TILE_HINT=0 disables)
    const bool hint = a.l2_hint != 0;
    const uint64_t pol = l2_policy_evict_first();
    int it = 0;
    // the tile's first / last CSR offsets are fetched one tile ahead, so that their
    // DRAM latency is not in series with the wait for a free slot
    int nbegin = 0, nend = 0;
    if (int64_t(blockIdx.x) < a.n_tiles) {
      const int64_t rn = a.row_begin + tile_of_slot(a, blockIdx.x) * R;
      nbegin = __ldg(a.indptr + rn);
      nend = __ldg(a.indptr + rn + R);
    }
    for (int64_t slot = blockIdx.x; slot < a.n_tiles; slot += gridDim.x, ++it) {
      const int64_t tile = tile_of_slot(a, slot);
      const int s = it % S;
      const uint32_t round = uint32_t(it / S);
      const int begin = nbegin, end = nend;
      if (slot + gridDim.x < a.n_tiles) {
        const int64_t rn = a.row_begin + tile_of_slot(a, slot + gridDim.x) * R;
        nbegin = __ldg(a.indptr + rn);
        nend = __ldg(a.indptr + rn + R);
      }
      mbar_wait(empty + s, (round & 1u) ^ 1u);      // slot free (passes at once in round 0)
      unsigned char* st = stage0 + size_t(s) * lay.stage_bytes;
      float* sm_vec = reinterpret_cast<float*>(st);
      int32_t* sm_col = reinterpret_cast<int32_t*>(st + lay.vec_bytes);
      float* sm_val = reinterpret_cast<float*>(st + lay.vec_bytes + lay.slab_bytes);
      int32_t* sm_ptr = reinterpret_cast<int32_t*>(st + lay.vec_bytes + 2 * lay.slab_bytes);
      int32_t* sm_meta = sm_ptr + (R + 4);

      const int64_t r0 = a.row_begin + tile * R;
      const int a0 = begin & ~3;                    // 16-byte aligned slab start
      int a1 = (end + 3) & ~3;
      if (int64_t(a1) > a.nnz) a1 = end & ~3;      // never read past the arrays
      sm_ptr[R] = end;                              // the bulk copy brings indptr[r0 .. r0+R)
      sm_meta[0] = a0;
      for (int k = (a1 > a0 ? a1 : a0); k < end; ++k) {   // <= 3 trailing entries, last tile only
        sm_col[k - a0] = __ldg(a.indices + k);
        sm_val[k - a0] = __ldg(a.vals + k);
      }
      const uint32_t slab = a1 > a0 ? uint32_t(a1 - a0) * 4u : 0u;
      const uint32_t tile_vec = uint32_t(R) * nsig * 4u;
      const bool stage_vec = !FIRST && !VD;
      const uint32_t bytes = uint32_t(R) * 4u + 2u * slab +
                             (stage_vec ? tile_vec * (1 + a.nscales) : 0u);
      mbar_expect_tx(full + s, bytes);
      bulk_g2s(sm_ptr, a.indptr + r0, uint32_t(R) * 4u, full + s);
      if (hint) {
        if (slab) {
          bulk_g2s_hint(sm_col, a.indices + a0, slab, full + s, pol);
          bulk_g2s_hint(sm_val, a.vals + a0, slab, full + s, pol);
        }
        if (stage_vec) {
          bulk_g2s_hint(sm_vec, a.x_old + r0 * nsig, tile_vec, full + s, pol);
          for (int i = 0; i < a.nscales; ++i)
            bulk_g2s_hint(sm_vec + size_t(i + 1) * R * nsig,
                          a.r + (int64_t(i) * a.r_rows + r0) * nsig, tile_vec, full + s, pol);
        }
      } else {
        if (slab) {
          bulk_g2s(sm_col, a.indices + a0, slab, full + s);
          bulk_g2s(sm_val, a.vals + a0, slab, full + s);
        }
        if (stage_vec) {
          bulk_g2s(sm_vec, a.x_old + r0 * nsig, tile_vec, full + s);
          for (int i = 0; i < a.nscales; ++i)
            bulk_g2s(sm_vec + size_t(i + 1) * R * nsig,
                     a.r + (int64_t(i) * a.r_rows + r0) * nsig, tile_vec, full + s);
        }
      }
    }
    return;
  }

  // ---------------------------------------------------------------- consumers
  const int cw = warp - 1;
  const int sub = lane / G;
  const int c0 = (lane % G) * 4;
  int it = 0;
  for (int64_t slot = blockIdx.x; slot < a.n_tiles; slot += gridDim.x, ++it) {
    const int64_t tile = tile_of_slot(a, slot);
    const int s = it % S;
    const uint32_t round = uint32_t(it / S);
    mbar_wait(full + s, round & 1u);
    unsigned char* st = stage0 + size_t(s) * lay.stage_bytes;
    // (the context is built per use and passed BY VALUE: a struct whose address escapes to the
    //  non-inlined boundary routine would live in local memory for the interior path too)
    const TileCtx t = {reinterpret_cast<const float*>(st),
                       reinterpret_cast<const int32_t*>(st + lay.vec_bytes),
                       reinterpret_cast<const float*>(st + lay.vec_bytes + lay.slab_bytes),
                       reinterpret_cast<const int32_t*>(st + lay.vec_bytes + 2 * lay.slab_bytes),
                       tile, a.row_begin + tile * R, cw, sub, c0, VD};
    if (HALO && tile < a.n_front)          // warp-uniform; interior tiles never wait
      boundary_tile<G, FIRST, NSC>(a, t, lane);
    else
      tile_rows<G, FIRST, NSC, false, P>(a, t);
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + s);
  }
}

// max over every window of `rows_per_tile` rows that starts at a multiple of 4 of
// the window's 16-byte-aligned CSR slab length: a bound valid for any tiling of
// any row range [rb, re) with rb % 4 == 0
__global__ void tile_nnz_max_kernel(int64_t n, int rows_per_tile,
                                    const int32_t* __restrict__ indptr, int* out) {
  int best = 0;
  const int64_t windows = (n - rows_per_tile) / 4 + 1;
  for (int64_t w = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; w < windows;
       w += int64_t(gridDim.x) * blockDim.x) {
    const int begin = indptr[4 * w] & ~3;
    const int end = (indptr[4 * w + rows_per_tile] + 3) & ~3;
    best = max(best, end - begin);
  }
  for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, best);
}

static int env_int(const char* name, int fallback) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : fallback;
}

// Decide the tiling for (matrix, nsig, nscales).  Synchronises `st` once.
int tile_plan(int64_t n, const int32_t* indptr, int64_t nsig, int nscales, gsp_tile_plan* plan,
              cudaStream_t st) {
  memset(plan, 0, sizeof(*plan));
  const char* force = getenv("GSPB200_KERNEL");
  if (force && strcmp(force, "rowgroup") == 0) return GSP_OK;
  if (!(nsig == 8 || nsig == 16 || nsig == 32 || nsig == 64 || nsig == 128)) return GSP_OK;
  if (nscales < 0 || nscales > kTiledMaxScales) return GSP_OK;
  // vector tiles per stage: x_old + one r tile per scale; keep a stage near 40 KB
  int R = env_int("GSPB200_TILE_R", nscales <= 1 ? 64 : (nscales <= 2 ? 32 : 16));
  if (nsig == 128) R = std::max(8, R / 2);
  R = std::max(8, (R / 8) * 8);
  const int warps_default = 16;
  // narrow blocks: a warp carries 32 / (nsig/4) rows, a tile should feed every warp
  if (nsig <= 16 && !getenv("GSPB200_TILE_R")) R = std::max(R, warps_default * (128 / (int)nsig));
  const int64_t n_tiles = n / R;
  if (n_tiles < 1) return GSP_OK;
  int* dmax = nullptr;
  GSP_CUDA(cudaMallocAsync((void**)&dmax, sizeof(int), st));
  GSP_CUDA(cudaMemsetAsync(dmax, 0, sizeof(int), st));
  const int blocks = (int)std::min<int64_t>(ceil_div(n / 4 + 1, 256), 2048);
  tile_nnz_max_kernel<<<blocks, 256, 0, st>>>(n, R, indptr, dmax);
  GSP_LAUNCH_CHECK("tile_nnz_max");
  int hmax = 0;
  GSP_CUDA(cudaMemcpyAsync(&hmax, dmax, sizeof(int), cudaMemcpyDeviceToHost, st));
  GSP_CUDA(cudaStreamSynchronize(st));
  cudaFreeAsync(dmax, st);
  const int cap = ((hmax + 8 + 31) / 32) * 32;
  int stages = env_int("GSPB200_TILE_S", nscales <= 1 ? 2 : 3);
  const int warps = std::min(16, std::max(1, env_int("GSPB200_TILE_NW", 16)));
  // keep a CTA's ring within ~100 KB so that L1 keeps room for the x_cur gather
  const int budget = env_int("GSPB200_TILE_SMEM", 100 * 1024);
  const bool vd = env_int("GSPB200_TILE_VDIR", 0) != 0;     // vectors not staged: small stages
  TileLayout lay(R, cap, (int)nsig, nscales, vd, stages);
  while (stages > 2 && lay.total(stages) > budget) { --stages; lay = TileLayout(R, cap, (int)nsig, nscales, vd, stages); }
  if (lay.total(stages) > 200 * 1024) return GSP_OK;        // heavy rows: row-group kernel
  plan->rows_per_tile = R;
  plan->slab_capacity = cap;
  plan->stages = stages;
  plan->consumer_warps = warps;
  plan->gather_unroll = env_int("GSPB200_TILE_U", 4);
  plan->blocks_per_sm = env_int("GSPB200_TILE_BPS", 0);
  return GSP_OK;
}

template <int G, int NSC, bool HALO, int P>
static int launch_tiled_k(bool first, const TileArgs& a, int blocks_per_sm, cudaStream_t st) {
  const TileLayout lay(a.rows_per_tile, a.slab_cap, a.nsig, a.nscales, first || a.vec_direct,
                       a.stages);
  const int smem = lay.total(a.stages);
  const int threads = 32 * (1 + a.consumer_warps);
  GSP_REQUIRE(threads <= 32 * (P == 2 ? 9 : 17), "too many consumer warps for this mapping");
  auto kern = first ? cheby_step_tiled<G, true, NSC, HALO, P> : cheby_step_tiled<G, false, NSC, HALO, P>;
  GSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int per_sm = 0;
  GSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
  if (per_sm < 1) return fail(GSP_ERR_UNSUPPORTED, "tiled kernel does not fit (%s)", "smem");
  if (blocks_per_sm > 0) per_sm = std::min(per_sm, blocks_per_sm);
  const int64_t grid = std::min<int64_t>(a.n_tiles, int64_t(sm_count()) * per_sm);
  kern<<<(unsigned)grid, threads, smem, st>>>(a);
  GSP_LAUNCH_CHECK("cheby_step_tiled");
  return GSP_OK;
}

template <int G, bool HALO, int P>
static int launch_tiled_gh(bool first, const TileArgs& a, int bps, cudaStream_t st) {
  switch (a.nscales) {          // common bank widths get the scale loop unrolled
    case 0: return launch_tiled_k<G, 0, HALO, P>(first, a, bps, st);
    case 1: return launch_tiled_k<G, 1, HALO, P>(first, a, bps, st);
    case 2: return launch_tiled_k<G, 2, HALO, P>(first, a, bps, st);
    default: return launch_tiled_k<G, -1, HALO, P>(first, a, bps, st);
  }
}

// G lanes x P packets x 4 columns = nsig.  The boundary tiles of a partitioned step (halo) always
// take the one-packet mapping; `two` selects the two-packet mapping for the others.
template <int G>
static int launch_tiled_g(bool first, const TileArgs& a, bool halo, bool two, int bps,
                          cudaStream_t st) {
  if (halo) return launch_tiled_gh<G, true, 1>(first, a, bps, st);
  if (two && G >= 8) return launch_tiled_gh<(G >= 8 ? G / 2 : G), false, (G >= 8 ? 2 : 1)>(first, a, bps, st);
  return launch_tiled_gh<G, false, 1>(first, a, bps, st);
}

int cheby_step_tiled_f32(const Step<float>& s, int64_t rb, int64_t n_tiles,
                         const gsp_halo_fusion* halo, int64_t n_front, int64_t nnz,
                         const int32_t* indptr, const int32_t* indices, const float* vals,
                         int64_t r_rows, int nsig, const gsp_tile_plan& plan, cudaStream_t st,
                         const int64_t* out_perm) {
  const bool first = s.first;
  TileArgs a;
  a.out_perm = out_perm;
  a.vec_direct = (!first && env_int("GSPB200_TILE_VDIR", s.add_source ? 1 : 0)) ? 1 : 0;
  a.keep_writes = env_int("GSPB200_TILE_REV", 1);
  a.reverse = (s.reverse && a.keep_writes) ? 1 : 0;
  a.add_source = s.add_source ? 1 : 0;
  a.l2_hint = env_int("GSPB200_TILE_HINT", 1);
  a.n_front = halo ? n_front : 0;
  GSP_REQUIRE(!s.add_source || (s.nscales >= 1 && !first), "add_source needs source blocks");
  memset(&a.halo, 0, sizeof(a.halo));
  gsp_halo_fusion probe;                       // GSPB200_FORCE_HALO=1: run the halo-capable
  if (!halo && rb == 0 && env_int("GSPB200_FORCE_HALO", 0)) {   // variant with no neighbours
    memset(&probe, 0, sizeof(probe));          // (single-GPU A/B of the two instantiations)
    probe.n_owned = 0x7fffffff;
    halo = &probe;
  }
  if (halo) a.halo = *halo;
  a.row_begin = rb;
  a.n_tiles = n_tiles;
  if (a.n_tiles == 0) return GSP_OK;
  a.r_rows = r_rows;
  a.nnz = nnz;
  a.indptr = indptr; a.indices = indices; a.vals = vals;
  a.x_cur = s.x_cur; a.x_old = s.x_old; a.x_new = s.x_new; a.r = s.r;
  a.rows_per_tile = plan.rows_per_tile;
  a.slab_cap = plan.slab_capacity;
  a.stages = plan.stages;
  a.consumer_warps = plan.consumer_warps;
  a.nsig = nsig;
  a.nscales = s.nscales;
  a.alpha = float(s.alpha); a.beta = float(s.beta); a.gamma = float(s.gamma);
  for (int i = 0; i < kTiledMaxScales; ++i) {
    a.ck[i] = i < s.nscales ? float(s.ck[i]) : 0.f;
    a.half_c0[i] = (first && i < s.nscales) ? float(0.5 * s.c0[i]) : 0.f;
  }
  const bool h = halo != nullptr;
  // two packets per lane (32 / 64 / 128 signals): a CSR read in shared memory serves twice
  // as many rows; GSPB200_TILE_P2=0 / 1 forces one / two packets per lane.
  // Measured (profiles/r2_probe_p2_*.jsonl, Clenshaw form with direct vector loads): 64 signals
  // 8.13 -> 6.97 ms per order-30 call, 128 signals 15.9 -> 12.6 ms, 32 signals 4.80 -> 4.73 ms;
  // the forward recurrence with TMA-staged vectors is slower with it (8.8 -> 9.3 ms: only two of
  // the three CTAs fit), so the default follows the form.
  const bool two = !h && nsig >= 32 &&
                   env_int("GSPB200_TILE_P2", (a.add_source && a.vec_direct) ? 1 : 0) != 0;
  if (two) a.consumer_warps = std::min(a.consumer_warps, 8);
  switch (nsig) {
    case 8: return launch_tiled_g<2>(first, a, h, false, plan.blocks_per_sm, st);
    case 16: return launch_tiled_g<4>(first, a, h, false, plan.blocks_per_sm, st);
    case 32: return launch_tiled_g<8>(first, a, h, two, plan.blocks_per_sm, st);
    case 64: return launch_tiled_g<16>(first, a, h, two, plan.blocks_per_sm, st);
    case 128: return launch_tiled_g<32>(first, a, h, two, plan.blocks_per_sm, st);
  }
  return fail(GSP_ERR_UNSUPPORTED, "tiled kernel: nsig must be 8, 16, 32, 64 or 128 (%s)", "nsig");
}

}  // namespace gsp

extern "C" int gsp_cheby_tile_plan(int64_t n, const int32_t* indptr, int64_t nsig, int nscales,
                                   gsp_tile_plan* plan_host_out, void* stream) {
  GSP_REQUIRE(plan_host_out != nullptr, "plan must not be NULL");
  return gsp::tile_plan(n, indptr, nsig, nscales, plan_host_out, gsp::as_stream(stream));
}
