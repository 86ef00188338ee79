// Kernel (a): linear force second-moment Gram  P = sum_{t,d} v v^T,  v = group-summed forces.
//
// Replaces src/aggforce/qp/qplinear.py:66-71 of the reference (two dgemm calls on a
// transposed copy of the force array).  Here the constraint-group sum, the f32->f64
// promotion and the SYRK are one kernel:
//   * frames stream global -> shared memory as 1-D TMA bulk copies (frame_pipe.cuh);
//   * each chunk is converted to an f64 panel  panel[k=(t,d)][x=reduced column]  whose row
//     stride (132 doubles) makes every DMMA fragment load bank-conflict free;
//   * 8 warps run DMMA.8x8x4.  A-fragment of row tile r and B-fragment of column tile c are
//     the SAME shared-memory access pattern (lane (g,q) reads panel[k0+q][8*tile+g]), so a
//     warp loads each needed 8-column fragment once per k-step and reuses it as row and as
//     column operand;
//   * which tiles a warp owns is decided at COMPILE time -- template <NT, warp> static plans
//     over the upper triangle -- so the inner loop is nothing but LDS.64 + DMMA, accumulators
//     live in registers for the whole frame range of the CTA (split-K over frames);
//   * accumulators are added to the global Gram with f64 RED atomics at the end.
// n_red <= 128 (cln025: 97): one CTA shape covers the upper triangle (NT = ceil(n_red/8) tile
// columns).  Larger systems: CTAs enumerate 128x128 block pairs (I <= J) and each warp owns a
// static 2 x 16 tile rectangle; operands are gathered from global memory (compute bound by 60x).
// TMA bulk copies of this file move 16 KB pieces (A/B on the small Gram: 2 / 4 / 8 / 16 KB pieces ->
// 1.342 / 1.293 / 1.270 / 1.266 ms per 1 M frames; the packed-panel SYRK is indifferent).
#ifndef AGF_BULK_PIECE
#define AGF_BULK_PIECE 16384u
#endif
#include "frame_pipe.cuh"
#include "panel.cuh"

#ifndef AGF_TRI_FILL_WARPS
#define AGF_TRI_FILL_WARPS 16
#endif
#ifndef AGF_TRI_UNROLL
#define AGF_TRI_UNROLL 2
#endif
#ifndef AGF_SYRK_WAVES
#define AGF_SYRK_WAVES 12
#endif
#ifndef AGF_TRI_MMA_WARPS
#define AGF_TRI_MMA_WARPS 8
#endif

namespace agf {

constexpr int kGramThreads = 256;
constexpr int kGramWarps = 8;
constexpr int kTriUnroll = AGF_TRI_UNROLL;  // k-steps of the triangular sweep unrolled together
constexpr int kTriMmaWarps = AGF_TRI_MMA_WARPS;  // MMA warps of the single-block kernel (tile plans below)
constexpr int kBlockCols = 128;  // reduced columns per block
constexpr int kStride = 132;     // panel row stride in doubles (132 % 16 == 4: conflict free)

struct GramParams {
  const void* forces;
  int64_t n_frames;
  int32_t n_sites;
  const int32_t* col_ptr;
  const int32_t* col_sites;
  int32_t n_red;
  int32_t n_blocks;  // ceil(n_red / 128)
  int32_t n_pairs;   // n_blocks (n_blocks + 1) / 2
  int32_t k_splits;  // CTAs per block pair
  double* gram;
  const double* weights;  // [n_frames] frame weights (read by the weighted instantiations only)
  ChunkSchedule sch;
};

// ------------------------------------------------------------------ static triangular tile plans
// Tiles of the upper triangle of an NT x NT tile grid in strip (row-major) order; warp w owns
// the contiguous run [tile_begin(w), tile_begin(w+1)) -- balanced to within one tile.
__host__ __device__ constexpr int tri_tiles(int nt) { return nt * (nt + 1) / 2; }
__host__ __device__ constexpr int tile_begin(int nt, int w) {
  const int total = tri_tiles(nt), base = total / kTriMmaWarps, extra = total % kTriMmaWarps;
  return w * base + (w < extra ? w : extra);
}
// Tile order: two tile rows at a time, column by column -- (r,c), (r+1,c), (r,c+1), (r+1,c+1) ... --
// so a warp's contiguous run of ~12 tiles touches 2 row fragments and ~6 column fragments
// (0.67 shared-memory fragment loads per DMMA instead of 1.08 for single-row strips).
__host__ __device__ constexpr int tile_rc(int nt, int t, bool want_row) {
  int idx = 0;
  for (int r0 = 0; r0 < nt; r0 += 2) {
    const int r1 = r0 + 1;
    for (int c = r0; c < nt; ++c) {
      if (idx == t) return want_row ? r0 : c;
      ++idx;
      if (r1 < nt && c >= r1) {
        if (idx == t) return want_row ? r1 : c;
        ++idx;
      }
    }
  }
  return 0;
}
__host__ __device__ constexpr int tile_row(int nt, int t) { return tile_rc(nt, t, true); }
__host__ __device__ constexpr int tile_col(int nt, int t) { return tile_rc(nt, t, false); }
constexpr int kMaxTriSlots = (tri_tiles(16) + kTriMmaWarps - 1) / kTriMmaWarps;

template <int NT, int W, int T, int END>
struct TriTiles {
  static __device__ __forceinline__ void mma(double (&acc)[kMaxTriSlots][2], const double (&frag)[NT]) {
    if constexpr (T < END) {
      constexpr int r = tile_row(NT, T), c = tile_col(NT, T), s = T - tile_begin(NT, W);
      dmma884(acc[s][0], acc[s][1], frag[r], frag[c]);
      TriTiles<NT, W, T + 1, END>::mma(acc, frag);
    }
  }
  static __device__ __forceinline__ void store(const double (&acc)[kMaxTriSlots][2], double* gram, int n_red, int g,
                                               int q) {
    if constexpr (T < END) {
      constexpr int r = tile_row(NT, T), c = tile_col(NT, T), s = T - tile_begin(NT, W);
      const int i = r * 8 + g, j = c * 8 + 2 * q;
      if (i < n_red) {
        double* row = gram + (int64_t)i * n_red;
        if (j < n_red) atomicAdd(row + j, acc[s][0]);
        if (j + 1 < n_red) atomicAdd(row + j + 1, acc[s][1]);
      }
      TriTiles<NT, W, T + 1, END>::store(acc, gram, n_red, g, q);
    }
  }
};

// One chunk: every k-step loads the NT fragments once and feeds this warp's tiles.
template <int NT, int W, int KSTEPS>
__device__ __forceinline__ void tri_sweep(const double* __restrict__ lane_panel, double (&acc)[kMaxTriSlots][2]) {
#pragma unroll kTriUnroll
  for (int kk = 0; kk < KSTEPS; ++kk) {
    const double* pk = lane_panel + kk * 4 * kStride;
    double frag[NT];
#pragma unroll
    for (int i = 0; i < NT; ++i) frag[i] = pk[i * 8];  // fragments this warp never uses are dead code
    TriTiles<NT, W, tile_begin(NT, W), tile_begin(NT, W + 1)>::mma(acc, frag);
  }
}

template <int NT, int KSTEPS>
__device__ __forceinline__ void tri_sweep_warp(int warp, const double* lane_panel, double (&acc)[kMaxTriSlots][2]) {
  switch (warp) {
    case 0: tri_sweep<NT, 0, KSTEPS>(lane_panel, acc); break;
    case 1: tri_sweep<NT, 1, KSTEPS>(lane_panel, acc); break;
    case 2: tri_sweep<NT, 2, KSTEPS>(lane_panel, acc); break;
    case 3: tri_sweep<NT, 3, KSTEPS>(lane_panel, acc); break;
    case 4: tri_sweep<NT, 4, KSTEPS>(lane_panel, acc); break;
    case 5: tri_sweep<NT, 5, KSTEPS>(lane_panel, acc); break;
    case 6: tri_sweep<NT, 6, KSTEPS>(lane_panel, acc); break;
    case 7: tri_sweep<NT, 7, KSTEPS>(lane_panel, acc); break;
    case 8: tri_sweep<NT, 8, KSTEPS>(lane_panel, acc); break;
    case 9: tri_sweep<NT, 9, KSTEPS>(lane_panel, acc); break;
    case 10: tri_sweep<NT, 10, KSTEPS>(lane_panel, acc); break;
    case 11: tri_sweep<NT, 11, KSTEPS>(lane_panel, acc); break;
    case 12: tri_sweep<NT, 12, KSTEPS>(lane_panel, acc); break;
    case 13: tri_sweep<NT, 13, KSTEPS>(lane_panel, acc); break;
    case 14: tri_sweep<NT, 14, KSTEPS>(lane_panel, acc); break;
    default: tri_sweep<NT, kTriMmaWarps - 1, KSTEPS>(lane_panel, acc); break;
  }
}

template <int NT, int W>
__device__ __forceinline__ void tri_store(const double (&acc)[kMaxTriSlots][2], double* gram, int n_red, int g, int q) {
  TriTiles<NT, W, tile_begin(NT, W), tile_begin(NT, W + 1)>::store(acc, gram, n_red, g, q);
}

// ------------------------------------------------------------------ panel fill (group sum + f64 promotion)
// W: the group sums of frame t are scaled by sqrt(weights[t]) (weighted fits; see agf_gram_linear_weighted).
template <typename T, bool GLOBAL, bool W>
__device__ __forceinline__ void fill_panel(const T* __restrict__ frames, int nf, int kf, int n_sites,
                                           const int32_t* __restrict__ col_ptr,
                                           const int32_t* __restrict__ col_sites, int col0, int n_red,
                                           int width_pad, const double* __restrict__ weights,
                                           double* __restrict__ panel) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = warp; t < kf; t += kGramWarps) {
    const T* fr = frames + (int64_t)t * n_sites * 3;
    double sw = 1.0;
    if constexpr (W) sw = t < nf ? sqrt(__ldg(weights + t)) : 0.0;
    for (int x = lane; x < width_pad; x += 32) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
      const int col = col0 + x;
      if (t < nf && col < n_red) {
        const int b = __ldg(col_ptr + col), e = __ldg(col_ptr + col + 1);
        for (int m = b; m < e; ++m) {
          const T* p = fr + 3 * __ldg(col_sites + m);
          if constexpr (GLOBAL) {
            s0 += to_f64(__ldg(p));
            s1 += to_f64(__ldg(p + 1));
            s2 += to_f64(__ldg(p + 2));
          } else {
            s0 += to_f64(p[0]);
            s1 += to_f64(p[1]);
            s2 += to_f64(p[2]);
          }
        }
      }
      if constexpr (W) {
        s0 *= sw;
        s1 *= sw;
        s2 *= sw;
      }
      double* dst = panel + (t * 3) * kStride + x;
      dst[0] = s0;
      dst[kStride] = s1;
      dst[2 * kStride] = s2;
    }
  }
}

// 32-bit shared-memory accessors (no generic-address arithmetic in the fill loop)
template <typename T>
__device__ __forceinline__ double lds_as_f64(uint32_t addr);
template <>
__device__ __forceinline__ double lds_as_f64<float>(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return (double)v;
}
template <>
__device__ __forceinline__ double lds_as_f64<double>(uint32_t addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
  asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

// ------------------------------------------------------------------ single block (n_red <= 128), TMA staged
// Warp-specialised CTA (one per SM): 8 MMA warps sweep panel[j & 1] while 4 fill warps convert
// the next raw chunk into panel[(j+1) & 1] and keep the TMA ring full, so the DMMA pipe never
// waits for a block-wide barrier.
//   raw_full[s]   : TMA bulk copy of a chunk landed            (tx-count mbarrier)
//   panel_full[b] : fill warps finished panel b                (1 arrival, after a named barrier)
//   panel_empty[b]: all 8 MMA warps finished sweeping panel b  (8 arrivals)
constexpr int kMmaWarps = kTriMmaWarps;
constexpr int kFillWarps = AGF_TRI_FILL_WARPS;
constexpr int kTriThreads = (kMmaWarps + kFillWarps) * 32;
constexpr int kFillThreads = kFillWarps * 32;
constexpr int kRawStages = 3;

template <typename T, int KF, int NT, bool W>
__global__ void __launch_bounds__(kTriThreads, 1) gram_tri_kernel(const __grid_constant__ GramParams p) {
  constexpr int KROWS = 3 * KF;
  constexpr int NCOLS = NT * 8;
  static_assert(KROWS % 4 == 0, "k rows must be a multiple of the DMMA k");
  extern __shared__ __align__(128) unsigned char smem[];
  double* panel0 = reinterpret_cast<double*>(smem);
  size_t off = (size_t)2 * KROWS * kStride * sizeof(double);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + off);
  uint64_t* raw_full = bars;                // [kRawStages]
  uint64_t* panel_full = bars + kRawStages; // [2]
  uint64_t* panel_empty = panel_full + 2;   // [2]
  off += 64;
  int32_t* s_ptr = reinterpret_cast<int32_t*>(smem + off);  // CSR copy: [n_red + 1] + [n_sites]
  int32_t* s_sites = s_ptr + (p.n_red + 1);
  off += (size_t)(p.n_red + 1 + p.n_sites) * 4;
  off = (off + 127) / 128 * 128;
  T* raw = reinterpret_cast<T*>(smem + off);
  const int64_t frame_elems = (int64_t)p.n_sites * 3;
  const int64_t stage_elems = ((int64_t)KF * frame_elems * (int64_t)sizeof(T) + 15) / 16 * 16 / (int64_t)sizeof(T);

  for (int i = threadIdx.x; i <= p.n_red; i += blockDim.x) s_ptr[i] = p.col_ptr[i];
  for (int i = threadIdx.x; i < p.col_ptr[p.n_red]; i += blockDim.x) s_sites[i] = p.col_sites[i];
  for (int i = threadIdx.x; i < 2 * KROWS * kStride; i += blockDim.x) panel0[i] = 0.0;  // padding columns stay 0
  if (threadIdx.x == 0) {
    for (int i = 0; i < kRawStages; ++i) mbar_init(&raw_full[i], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&panel_full[i], 1);
      mbar_init(&panel_empty[i], kMmaWarps);
    }
    fence_barrier_init();
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const T* forces = reinterpret_cast<const T*>(p.forces);
  // this CTA's chunks: c_j = first + j * step, skipping the head chunk when it is empty
  const int64_t step = gridDim.x;
  int64_t first = blockIdx.x;
  if (first == 0 && p.sch.head == 0) first += step;
  const int64_t n_mine = p.sch.n_chunks > first ? (p.sch.n_chunks - first + step - 1) / step : 0;

  auto bulkable = [&](int64_t c) {
    const int64_t bytes = (int64_t)p.sch.count(c) * frame_elems * (int64_t)sizeof(T);
    const uintptr_t a = reinterpret_cast<uintptr_t>(forces + p.sch.start(c) * frame_elems);
    return c != 0 && bytes > 0 && (bytes % 16) == 0 && (a % 16) == 0;
  };
  auto issue = [&](int64_t j) {  // one thread: TMA for local chunk j (no-op when not bulk-copyable)
    if (j >= n_mine) return;
    const int64_t c = first + j * step;
    if (!bulkable(c)) return;
    const int stage = (int)(j % kRawStages);
    const uint32_t bytes = (uint32_t)((int64_t)p.sch.count(c) * frame_elems * (int64_t)sizeof(T));
    fence_proxy_async();
    mbar_expect_tx(&raw_full[stage], bytes);
    const char* src = reinterpret_cast<const char*>(forces + p.sch.start(c) * frame_elems);
    char* dst = reinterpret_cast<char*>(raw + (int64_t)stage * stage_elems);
    uint32_t done = 0;
    while (done < bytes) {
      const uint32_t piece = bytes - done < kBulkPiece ? bytes - done : kBulkPiece;
      tma_bulk_g2s(dst + done, src + done, piece, &raw_full[stage]);
      done += piece;
    }
  };

  if (warp >= kMmaWarps) {
    // ------------------------------------------------ fill warps
    const int ft = threadIdx.x - kMmaWarps * 32;  // 0..127
    if (ft == 0) {
      for (int j = 0; j < kRawStages; ++j) issue(j);
    }
    uint32_t raw_phase = 0;  // bit s: parity to wait for on raw_full[s]
    // Work split: fill warp fw owns frames fw, fw+8, ... of every chunk; inside a frame the columns
    // are processed in groups of 32 with lane = column.  Everything a lane needs about its columns
    // (byte offsets of up to 4 member sites, member count, the group's largest count) is loaded
    // once; columns arrive sorted by member count so the lanes of a group mostly agree.
    constexpr int NG = (NCOLS + 31) / 32;
    const int fw = ft >> 5;
    int cnt[NG], wmax[NG];
    uint32_t moff[NG][4], coff[NG];
    bool generic = false;
#pragma unroll
    for (int gi = 0; gi < NG; ++gi) {
      const int x = gi * 32 + lane;
      cnt[gi] = 0;
      coff[gi] = (uint32_t)x * 8u;
#pragma unroll
      for (int m = 0; m < 4; ++m) moff[gi][m] = 0;
      if (x < p.n_red) {
        const int b = s_ptr[x];
        cnt[gi] = s_ptr[x + 1] - b;
#pragma unroll
        for (int m = 0; m < 4; ++m)
          if (m < cnt[gi]) moff[gi][m] = (uint32_t)s_sites[b + m] * 3u * (uint32_t)sizeof(T);
      }
      int wm = cnt[gi];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) wm = max(wm, __shfl_xor_sync(0xffffffffu, wm, o));
      wmax[gi] = wm;
      generic |= wm > 4;
    }
    const uint32_t frame_bytes = (uint32_t)frame_elems * (uint32_t)sizeof(T);
    for (int64_t j = 0; j < n_mine; ++j) {
      const int64_t c = first + j * step;
      const int nf = p.sch.count(c);
      const int stage = (int)(j % kRawStages), pb = (int)(j & 1);
      T* stage_ptr = raw + (int64_t)stage * stage_elems;
      if (bulkable(c)) {
        mbar_wait(&raw_full[stage], (raw_phase >> stage) & 1u);
        raw_phase ^= (1u << stage);
      } else {
        const T* src = forces + p.sch.start(c) * frame_elems;
        for (int64_t i = ft; i < (int64_t)nf * frame_elems; i += kFillThreads) stage_ptr[i] = src[i];
        asm volatile("bar.sync 1, %0;" ::"n"(kFillThreads) : "memory");
      }
      mbar_wait(&panel_empty[pb], (uint32_t)(((j >> 1) & 1) ^ 1));
      double* panel = panel0 + (size_t)pb * KROWS * kStride;
      const uint32_t raw_u32 = smem_u32(stage_ptr), panel_u32 = smem_u32(panel);
      const double* chunk_w = W ? p.weights + p.sch.start(c) : nullptr;
      if (!generic) {
        for (int t = fw; t < KF; t += kFillWarps) {
          const uint32_t rbase = raw_u32 + (uint32_t)t * frame_bytes;
          const uint32_t pbase = panel_u32 + (uint32_t)(t * 3 * kStride * 8);
          const bool live = t < nf;
          double sw = 1.0;  // one multiply per value where the group sum is complete (DMUL, like DADD, shares the DMMA pipe)
          if constexpr (W) sw = live ? sqrt(__ldg(chunk_w + t)) : 0.0;
#pragma unroll
          for (int gi = 0; gi < NG; ++gi) {
            double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              if (m < wmax[gi]) {  // warp-uniform: one conversion sequence per group, not per lane
                if (live && m < cnt[gi]) {
                  const uint32_t a = rbase + moff[gi][m];
                  const double v0 = lds_as_f64<T>(a), v1 = lds_as_f64<T>(a + (uint32_t)sizeof(T)),
                               v2 = lds_as_f64<T>(a + 2u * (uint32_t)sizeof(T));
                  // The first member is assigned, not added: DADD shares the FP64 pipe with DMMA and
                  // loses every arbitration against the MMA warps' DMMA stream (a DADD loop next to
                  // DMMA-streaming warps runs 400x slower, tools/microbench/fill_bench.cu; F2F.F64.F32,
                  // LDS and STS are unaffected), so the fill issues as few DADDs as possible.
                  if (m == 0) {
                    s0 = v0;
                    s1 = v1;
                    s2 = v2;
                  } else {
                    s0 += v0;
                    s1 += v1;
                    s2 += v2;
                  }
                }
              }
            }
            if constexpr (W) {
              s0 *= sw;
              s1 *= sw;
              s2 *= sw;
            }
            if (gi * 32 + lane < p.n_red) {
              const uint32_t d = pbase + coff[gi];
              sts_f64(d, s0);
              sts_f64(d + kStride * 8, s1);
              sts_f64(d + 2 * kStride * 8, s2);
            }
          }
        }
      } else {
        for (int item = ft; item < KF * NCOLS; item += kFillThreads) {
          const int t = item / NCOLS, x = item - t * NCOLS;
          double s0 = 0.0, s1 = 0.0, s2 = 0.0;
          if (t < nf && x < p.n_red) {
            const T* fr = stage_ptr + (int64_t)t * frame_elems;
            for (int m = s_ptr[x]; m < s_ptr[x + 1]; ++m) {
              const T* q = fr + 3 * s_sites[m];
              s0 += to_f64(q[0]);
              s1 += to_f64(q[1]);
              s2 += to_f64(q[2]);
            }
            if constexpr (W) {
              const double sw = sqrt(__ldg(chunk_w + t));
              s0 *= sw;
              s1 *= sw;
              s2 *= sw;
            }
          }
          double* dst = panel + (t * 3) * kStride + x;
          dst[0] = s0;
          dst[kStride] = s1;
          dst[2 * kStride] = s2;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kFillThreads) : "memory");  // panel written, raw stage drained
      if (ft == 0) {
        mbar_arrive(&panel_full[pb]);
        issue(j + kRawStages);
      }
    }
    return;
  }

  // -------------------------------------------------- MMA warps
  const int g = lane >> 2, q = lane & 3;
  double acc[kMaxTriSlots][2];
#pragma unroll
  for (int s = 0; s < kMaxTriSlots; ++s) acc[s][0] = acc[s][1] = 0.0;
  for (int64_t j = 0; j < n_mine; ++j) {
    const int pb = (int)(j & 1);
    mbar_wait(&panel_full[pb], (uint32_t)((j >> 1) & 1));
    const double* lane_panel = panel0 + (size_t)pb * KROWS * kStride + q * kStride + g;
    tri_sweep_warp<NT, KROWS / 4>(warp, lane_panel, acc);
    __syncwarp();
    if (lane == 0) mbar_arrive(&panel_empty[pb]);
  }
  switch (warp) {
    case 0: tri_store<NT, 0>(acc, p.gram, p.n_red, g, q); break;
    case 1: tri_store<NT, 1>(acc, p.gram, p.n_red, g, q); break;
    case 2: tri_store<NT, 2>(acc, p.gram, p.n_red, g, q); break;
    case 3: tri_store<NT, 3>(acc, p.gram, p.n_red, g, q); break;
    case 4: tri_store<NT, 4>(acc, p.gram, p.n_red, g, q); break;
    case 5: tri_store<NT, 5>(acc, p.gram, p.n_red, g, q); break;
    case 6: tri_store<NT, 6>(acc, p.gram, p.n_red, g, q); break;
    case 7: tri_store<NT, 7>(acc, p.gram, p.n_red, g, q); break;
    case 8: tri_store<NT, 8>(acc, p.gram, p.n_red, g, q); break;
    case 9: tri_store<NT, 9>(acc, p.gram, p.n_red, g, q); break;
    case 10: tri_store<NT, 10>(acc, p.gram, p.n_red, g, q); break;
    case 11: tri_store<NT, 11>(acc, p.gram, p.n_red, g, q); break;
    case 12: tri_store<NT, 12>(acc, p.gram, p.n_red, g, q); break;
    case 13: tri_store<NT, 13>(acc, p.gram, p.n_red, g, q); break;
    case 14: tri_store<NT, 14>(acc, p.gram, p.n_red, g, q); break;
    default: tri_store<NT, kTriMmaWarps - 1>(acc, p.gram, p.n_red, g, q); break;
  }
}

// ------------------------------------------------------------------ block pairs (any n_red), global gather
// CTA = block pair (I <= J) x k-split; warp w owns tile rows {2w, 2w+1} x all 16 tile columns.
template <typename T, int KF, bool W>
__global__ void __launch_bounds__(kGramThreads, 1) gram_block_kernel(const __grid_constant__ GramParams p) {
  constexpr int KROWS = 3 * KF;
  extern __shared__ __align__(128) unsigned char smem[];
  const int pair = blockIdx.x % p.n_pairs;
  const int ksplit = blockIdx.x / p.n_pairs;
  int bi = 0, bj = 0;
  {
    int rem = pair, rowlen = p.n_blocks;
    while (rem >= rowlen) {
      rem -= rowlen;
      --rowlen;
      ++bi;
    }
    bj = bi + rem;
  }
  const bool diag = (bi == bj);
  const int col0_i = bi * kBlockCols, col0_j = bj * kBlockCols;
  double* panel_i = reinterpret_cast<double*>(smem);
  double* panel_j = diag ? panel_i : panel_i + KROWS * kStride;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, q = lane & 3;
  const double* lane_i = panel_i + q * kStride + g + warp * 16;
  const double* lane_j = panel_j + q * kStride + g;
  double acc[2][16][2];
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;

  const T* forces = reinterpret_cast<const T*>(p.forces);
  for (int64_t c = ksplit; c < p.sch.n_chunks; c += p.k_splits) {
    const int nf = p.sch.count(c);
    if (nf > 0) {
      const T* src = forces + p.sch.start(c) * (int64_t)p.n_sites * 3;
      const double* w = W ? p.weights + p.sch.start(c) : nullptr;
      fill_panel<T, true, W>(src, nf, KF, p.n_sites, p.col_ptr, p.col_sites, col0_i, p.n_red, kBlockCols, w, panel_i);
      if (!diag)
        fill_panel<T, true, W>(src, nf, KF, p.n_sites, p.col_ptr, p.col_sites, col0_j, p.n_red, kBlockCols, w,
                               panel_j);
    }
    __syncthreads();
    if (nf > 0) {
#pragma unroll 2
      for (int kk = 0; kk < KROWS / 4; ++kk) {
        const double a0 = lane_i[kk * 4 * kStride], a1 = lane_i[kk * 4 * kStride + 8];
#pragma unroll
        for (int cc = 0; cc < 16; ++cc) {
          const double b = lane_j[kk * 4 * kStride + cc * 8];
          dmma884(acc[0][cc][0], acc[0][cc][1], a0, b);
          dmma884(acc[1][cc][0], acc[1][cc][1], a1, b);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int i = col0_i + (warp * 2 + r) * 8 + g;
    if (i >= p.n_red) continue;
    double* row = p.gram + (int64_t)i * p.n_red;
#pragma unroll
    for (int cc = 0; cc < 16; ++cc) {
      const int j = col0_j + cc * 8 + 2 * q;
      if (j < p.n_red) atomicAdd(row + j, acc[r][cc][0]);
      if (j + 1 < p.n_red) atomicAdd(row + j + 1, acc[r][cc][1]);
    }
  }
}

// ------------------------------------------------------------------ any n_red, workspace variant
// Two kernels per slab of frames:
//   gram_pack_kernel : group sums + f64 promotion, written ONCE per frame into a blocked workspace
//                      ws[chunk][block][24 rows][132] -- exactly the shared-memory image of a panel,
//                      so the SYRK kernel moves a whole panel with one TMA bulk copy;
//   gram_syrk_ws_kernel : CTA = block pair (I <= J) x k-split; a producer warp streams the panel
//                      pairs of its chunks through a 4-stage ring (full/empty mbarriers), 8 MMA warps
//                      sweep them (2 x 16 tiles each, accumulators in registers).  No conversion, no
//                      f64 adds and no block-wide barrier beside the DMMA stream.
// The workspace costs 66.5 KB of HBM traffic per frame at n_red = 2600 against 20 Mflop of DMMA
// work: irrelevant for a kernel that is compute bound by 60x.
constexpr int kWsKF = kPanelKF;
constexpr int kWsPanel = kPanelElems;  // doubles per (chunk, block)
static_assert(kStride == kPanelStride && kBlockCols == kPanelCols, "panel geometry");

template <typename T, bool W>
__global__ void __launch_bounds__(256) gram_pack_kernel(const T* __restrict__ forces, int64_t n_frames, int n_sites,
                                                        const int32_t* __restrict__ col_ptr,
                                                        const int32_t* __restrict__ col_sites, int n_red,
                                                        int n_blocks, const double* __restrict__ weights,
                                                        double* __restrict__ ws) {
  const int64_t chunk = blockIdx.x / n_blocks;
  const int blk = blockIdx.x - (int)(chunk * n_blocks);
  const int64_t t0 = chunk * kWsKF;
  const int nf = (int)min((int64_t)kWsKF, n_frames - t0);
  double* panel = ws + ((int64_t)chunk * n_blocks + blk) * kWsPanel;
  for (int item = threadIdx.x; item < kWsKF * kStride; item += blockDim.x) {
    const int t = item / kStride, x = item - t * kStride;
    const int col = blk * kBlockCols + x;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    if (t < nf && x < kBlockCols && col < n_red) {
      const T* fr = forces + (t0 + t) * (int64_t)n_sites * 3;
      const int b = __ldg(col_ptr + col), e = __ldg(col_ptr + col + 1);
      for (int m = b; m < e; ++m) {
        const T* p = fr + 3 * __ldg(col_sites + m);
        s0 += to_f64(__ldg(p));
        s1 += to_f64(__ldg(p + 1));
        s2 += to_f64(__ldg(p + 2));
      }
      if constexpr (W) {
        const double sw = sqrt(__ldg(weights + t0 + t));
        s0 *= sw;
        s1 *= sw;
        s2 *= sw;
      }
    }
    double* dst = panel + (t * 3) * kStride + x;
    dst[0] = s0;
    dst[kStride] = s1;
    dst[2 * kStride] = s2;
  }
}

struct SyrkWsParams {
  const double* ws;
  int64_t n_chunks;
  int32_t n, n_blocks, n_pairs, k_splits, batch;
  double* gram;
};

// Block pair of work item `pair`, heaviest first: off-diagonal pairs of full blocks, then
// diagonal blocks (17/32 of the tiles), then everything touching a narrow last block.
__device__ __forceinline__ void syrk_pair(int pair, int n_blocks, bool last_narrow, int& bi, int& bj) {
  const int nf = last_narrow ? n_blocks - 1 : n_blocks;
  const int n_off = nf * (nf - 1) / 2;
  if (pair < n_off) {
    int rem = pair, rowlen = nf - 1;
    bi = 0;
    while (rem >= rowlen) {
      rem -= rowlen;
      --rowlen;
      ++bi;
    }
    bj = bi + 1 + rem;
  } else if (pair < n_off + nf) {
    bi = bj = pair - n_off;
  } else {
    bi = pair - n_off - nf;  // 0 .. n_blocks-1 against the last block
    bj = n_blocks - 1;
  }
}

__global__ void __launch_bounds__(kPanelThreads, 1) panel_syrk_kernel(const __grid_constant__ SyrkWsParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  // consecutive CTAs = the block pairs of one (k-split, batch item): they stream the same chunks
  // at the same time, so every panel is fetched from HBM once and re-read through L2
  const int pair = blockIdx.x % p.n_pairs;
  const int rest = blockIdx.x / p.n_pairs;
  const int bt = rest % p.batch, ksplit = rest / p.batch;
  const int ct_last = (p.n - (p.n_blocks - 1) * kPanelCols + 7) / 8;
  int bi, bj;
  syrk_pair(pair, p.n_blocks, ct_last < 16, bi, bj);
  const bool diag = bi == bj;
  const int ct_i = bi == p.n_blocks - 1 ? ct_last : 16, ct_j = bj == p.n_blocks - 1 ? ct_last : 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = panel_warp_row(warp);
  const uint32_t m = warp < kPanelMmaWarps ? panel_row_mask(r0, ct_i, ct_j, diag) : 0u;
  PanelStream st;
  const int64_t chunk_step = (int64_t)p.batch * p.n_blocks * kPanelElems;
  const double* base = p.ws + ((int64_t)ksplit * p.batch + bt) * p.n_blocks * kPanelElems;
  st.a = base + (int64_t)bi * kPanelElems;
  st.b = base + (int64_t)bj * kPanelElems;
  st.a_step = st.b_step = chunk_step * p.k_splits;
  st.n = p.n_chunks > ksplit ? (p.n_chunks - ksplit + p.k_splits - 1) / p.k_splits : 0;
  st.same = diag;
  double acc[16][2];
  if (!panel_mainloop<true>(smem, st, m, acc)) return;
  const int g = lane >> 2, q = lane & 3;
  const int i = bi * kPanelCols + r0 * 8 + g;
  if (m == 0u || i >= p.n) return;
  double* row = p.gram + (int64_t)bt * p.n * p.n + (int64_t)i * p.n;
#pragma unroll
  for (int cc = 0; cc < 16; ++cc) {
    if (!((m >> cc) & 1u)) continue;
    const int j2 = bj * kPanelCols + cc * 8 + 2 * q;
    if (j2 < p.n) atomicAdd(row + j2, acc[cc][0]);
    if (j2 + 1 < p.n) atomicAdd(row + j2 + 1, acc[cc][1]);
  }
}

int launch_panel_syrk(const double* ws, int64_t n_chunks, int32_t n, int32_t batch, double* gram,
                      cudaStream_t stream) {
  if (n_chunks <= 0) return AGF_OK;
  SyrkWsParams p;
  p.ws = ws;
  p.n_chunks = n_chunks;
  p.n = n;
  p.n_blocks = panel_blocks(n);
  p.n_pairs = p.n_blocks * (p.n_blocks + 1) / 2;
  p.batch = batch;
  p.gram = gram;
  // Work items differ in cost (full / diagonal 17/32 / narrow) and one CTA occupies an SM, so the
  // launch ends with a tail of about one full item: aim for AGF_SYRK_WAVES waves of CTAs (tail
  // <= 1/waves of the launch) while keeping >= 32 chunks per CTA to amortise the 16 K-atomic epilogue.
  const int64_t items = (int64_t)p.n_pairs * batch;
  int64_t ks = ((int64_t)AGF_SYRK_WAVES * sm_count() + items - 1) / items;
  if (ks < n_chunks / 128) ks = n_chunks / 128;  // long slabs: CTAs of ~128 chunks (~0.45 ms) bound the tail
  if (ks > n_chunks / 32) ks = n_chunks / 32;
  if (ks > n_chunks) ks = n_chunks;
  if (ks < 1) ks = 1;
  p.k_splits = (int32_t)ks;
  AGF_CUDA_TRY(cudaFuncSetAttribute(panel_syrk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPanelSmem));
  panel_syrk_kernel<<<(unsigned)(items * ks), kPanelThreads, kPanelSmem, stream>>>(p);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

__global__ void symmetrize_kernel(double* g, int n) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * n) return;
  int i = (int)(idx / n), j = (int)(idx % n);
  if (i > j) g[idx] = g[(int64_t)j * n + i];
}

template <typename T, int KF, int NT, bool W>
static int launch_tri(GramParams& p, size_t smem, int ctas, cudaStream_t stream) {
  auto kern = gram_tri_kernel<T, KF, NT, W>;
  AGF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<ctas, kTriThreads, smem, stream>>>(p);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

template <typename T, int KF>
static size_t tri_smem_bytes(const GramParams& p) {
  size_t off = (size_t)2 * 3 * KF * kStride * sizeof(double) + 64 + (size_t)(p.n_red + 1 + p.n_sites) * 4;
  off = (off + 127) / 128 * 128;
  size_t stage_bytes = ((size_t)KF * p.n_sites * 3 * sizeof(T) + 15) / 16 * 16;
  return off + kRawStages * stage_bytes;
}

template <typename T, int KF, bool W>
static int dispatch_tri(GramParams& p, cudaStream_t stream) {
  const int sms = sm_count();
  p.sch = make_schedule(p.forces, p.n_frames, (int64_t)p.n_sites * 3 * sizeof(T), KF);
  const size_t smem = tri_smem_bytes<T, KF>(p);
  int64_t want = p.sch.n_chunks;
  int ctas = (int)(want < sms ? (want < 1 ? 1 : want) : sms);
  switch ((p.n_red + 7) / 8) {
    case 1: return launch_tri<T, KF, 1, W>(p, smem, ctas, stream);
    case 2: return launch_tri<T, KF, 2, W>(p, smem, ctas, stream);
    case 3: return launch_tri<T, KF, 3, W>(p, smem, ctas, stream);
    case 4: return launch_tri<T, KF, 4, W>(p, smem, ctas, stream);
    case 5: return launch_tri<T, KF, 5, W>(p, smem, ctas, stream);
    case 6: return launch_tri<T, KF, 6, W>(p, smem, ctas, stream);
    case 7: return launch_tri<T, KF, 7, W>(p, smem, ctas, stream);
    case 8: return launch_tri<T, KF, 8, W>(p, smem, ctas, stream);
    case 9: return launch_tri<T, KF, 9, W>(p, smem, ctas, stream);
    case 10: return launch_tri<T, KF, 10, W>(p, smem, ctas, stream);
    case 11: return launch_tri<T, KF, 11, W>(p, smem, ctas, stream);
    case 12: return launch_tri<T, KF, 12, W>(p, smem, ctas, stream);
    case 13: return launch_tri<T, KF, 13, W>(p, smem, ctas, stream);
    case 14: return launch_tri<T, KF, 14, W>(p, smem, ctas, stream);
    case 15: return launch_tri<T, KF, 15, W>(p, smem, ctas, stream);
    default: return launch_tri<T, KF, 16, W>(p, smem, ctas, stream);
  }
}

// KFBIG / KFSMALL: frames per chunk of the staged kernel (the larger one when it fits in smem).
template <typename T, int KFBIG, int KFSMALL, bool W>
static int launch_gram(GramParams& p, cudaStream_t stream) {
  const int sms = sm_count();
  const size_t budget = 226 * 1024;
  if (p.n_blocks == 1) {
    if (tri_smem_bytes<T, KFBIG>(p) <= budget) return dispatch_tri<T, KFBIG, W>(p, stream);
    if (tri_smem_bytes<T, KFSMALL>(p) <= budget) return dispatch_tri<T, KFSMALL, W>(p, stream);
    // frames too wide to stage in shared memory: use the gather variant
  }
  constexpr int KF = KFSMALL;
  p.sch = make_schedule(p.forces, p.n_frames, (int64_t)p.n_sites * 3 * sizeof(T), KF);
  size_t smem = (size_t)2 * 3 * KF * kStride * sizeof(double);
  int64_t ks = ((int64_t)sms * 2 + p.n_pairs - 1) / p.n_pairs;
  if (ks > p.sch.n_chunks) ks = p.sch.n_chunks;
  if (ks < 1) ks = 1;
  p.k_splits = (int32_t)ks;
  auto kern = gram_block_kernel<T, KF, W>;
  AGF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<p.k_splits * p.n_pairs, kGramThreads, smem, stream>>>(p);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

static int gram_linear_impl(const void* forces, int dtype, int64_t n_frames, int32_t n_sites, const int32_t* col_ptr,
                            const int32_t* col_sites, int32_t n_red, double* gram, const double* weights,
                            void* stream) {
  AGF_REQUIRE(forces && col_ptr && col_sites && gram, "agf_gram_linear: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_red > 0, "agf_gram_linear: bad sizes T=%lld n=%d n_red=%d",
              (long long)n_frames, n_sites, n_red);
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_gram_linear: dtype must be AGF_F32 or AGF_F64");
  if (n_frames == 0) return AGF_OK;
  GramParams p;
  memset(&p, 0, sizeof(p));
  p.forces = forces;
  p.n_frames = n_frames;
  p.n_sites = n_sites;
  p.col_ptr = col_ptr;
  p.col_sites = col_sites;
  p.n_red = n_red;
  p.gram = gram;
  p.weights = weights;
  p.n_blocks = (n_red + kBlockCols - 1) / kBlockCols;
  p.n_pairs = p.n_blocks * (p.n_blocks + 1) / 2;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (weights) {
    if (dtype == AGF_F32) return launch_gram<float, 16, 8, true>(p, s);
    return launch_gram<double, 8, 4, true>(p, s);
  }
  if (dtype == AGF_F32) return launch_gram<float, 16, 8, false>(p, s);
  return launch_gram<double, 8, 4, false>(p, s);
}

template <typename T>
static void launch_pack(const T* forces, int64_t nf, int32_t n_sites, const int32_t* col_ptr, const int32_t* col_sites,
                        int32_t n_red, int n_blocks, const double* weights, double* ws, int64_t grid, cudaStream_t s) {
  if (weights)
    gram_pack_kernel<T, true><<<(unsigned)grid, 256, 0, s>>>(forces, nf, n_sites, col_ptr, col_sites, n_red, n_blocks,
                                                             weights, ws);
  else
    gram_pack_kernel<T, false><<<(unsigned)grid, 256, 0, s>>>(forces, nf, n_sites, col_ptr, col_sites, n_red, n_blocks,
                                                              nullptr, ws);
}

static int gram_linear_ws_impl(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                               const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red, double* gram,
                               void* workspace, size_t workspace_bytes, const double* weights, void* stream) {
  AGF_REQUIRE(forces && col_ptr && col_sites && gram, "agf_gram_linear_ws: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_red > 0, "agf_gram_linear_ws: bad sizes");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_gram_linear_ws: bad dtype");
  const int64_t n_blocks = (n_red + kBlockCols - 1) / kBlockCols;
  const int64_t per_chunk = n_blocks * kWsPanel * (int64_t)sizeof(double);
  if (n_red <= kBlockCols || workspace == nullptr || (int64_t)workspace_bytes < per_chunk)
    return gram_linear_impl(forces, dtype, n_frames, n_sites, col_ptr, col_sites, n_red, gram, weights, stream);
  AGF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) % 16) == 0, "agf_gram_linear_ws: workspace must be 16-byte aligned");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int64_t slab_chunks = (int64_t)workspace_bytes / per_chunk;
  const int64_t slab_frames = slab_chunks * kWsKF;
  const size_t elem = dtype == AGF_F32 ? 4 : 8;
  for (int64_t f0 = 0; f0 < n_frames; f0 += slab_frames) {
    const int64_t nf = n_frames - f0 < slab_frames ? n_frames - f0 : slab_frames;
    const int64_t chunks = (nf + kWsKF - 1) / kWsKF;
    const char* src = reinterpret_cast<const char*>(forces) + (size_t)f0 * n_sites * 3 * elem;
    const double* w = weights ? weights + f0 : nullptr;
    const int64_t pack_grid = chunks * n_blocks;
    AGF_REQUIRE(pack_grid < (int64_t)1 << 31, "agf_gram_linear_ws: slab too large");
    if (dtype == AGF_F32)
      launch_pack(reinterpret_cast<const float*>(src), nf, n_sites, col_ptr, col_sites, n_red, (int)n_blocks, w,
                  reinterpret_cast<double*>(workspace), pack_grid, s);
    else
      launch_pack(reinterpret_cast<const double*>(src), nf, n_sites, col_ptr, col_sites, n_red, (int)n_blocks, w,
                  reinterpret_cast<double*>(workspace), pack_grid, s);
    AGF_CUDA_TRY(cudaGetLastError());
    int rc = launch_panel_syrk(reinterpret_cast<const double*>(workspace), chunks, n_red, 1, gram, s);
    if (rc) return rc;
  }
  return AGF_OK;
}

}  // namespace agf

extern "C" int agf_gram_linear(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                               const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red, double* gram,
                               void* stream) {
  return agf::gram_linear_impl(forces, dtype, n_frames, n_sites, col_ptr, col_sites, n_red, gram, nullptr, stream);
}

extern "C" int agf_gram_linear_weighted(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                                        const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red, double* gram,
                                        const double* frame_weights, void* stream) {
  return agf::gram_linear_impl(forces, dtype, n_frames, n_sites, col_ptr, col_sites, n_red, gram, frame_weights,
                               stream);
}

extern "C" size_t agf_gram_linear_workspace_bytes(int32_t n_sites, int32_t n_red, int64_t n_frames) {
  using namespace agf;
  (void)n_sites;
  if (n_red <= kBlockCols || n_frames <= 0) return 0;
  const int64_t n_blocks = (n_red + kBlockCols - 1) / kBlockCols;
  const int64_t per_chunk = n_blocks * kWsPanel * (int64_t)sizeof(double);
  const int64_t chunks = (n_frames + kWsKF - 1) / kWsKF;
  const int64_t cap = (int64_t)4 << 30;  // slabs of at most 4 GiB
  int64_t want = chunks * per_chunk;
  if (want > cap) want = cap / per_chunk * per_chunk;
  if (want < per_chunk) want = per_chunk;
  return (size_t)want;
}

extern "C" int agf_gram_linear_ws(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                                  const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red, double* gram,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  return agf::gram_linear_ws_impl(forces, dtype, n_frames, n_sites, col_ptr, col_sites, n_red, gram, workspace,
                                  workspace_bytes, nullptr, stream);
}

extern "C" int agf_gram_linear_ws_weighted(const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                                           const int32_t* col_ptr, const int32_t* col_sites, int32_t n_red,
                                           double* gram, void* workspace, size_t workspace_bytes,
                                           const double* frame_weights, void* stream) {
  return agf::gram_linear_ws_impl(forces, dtype, n_frames, n_sites, col_ptr, col_sites, n_red, gram, workspace,
                                  workspace_bytes, frame_weights, stream);
}

extern "C" int agf_symmetrize(double* gram, int32_t n, void* stream) {
  using namespace agf;
  AGF_REQUIRE(gram && n > 0, "agf_symmetrize: bad arguments");
  int64_t total = (int64_t)n * n;
  int blocks = (int)((total + 255) / 256);
  symmetrize_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(gram, n);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}
