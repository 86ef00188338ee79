// Kernel (d): map application  out[t,c,:] = sum_f M[c,f] X[t,f,:], fused with the NaN probe /
// NaN protocol and the residual sum(out^2).
//
// Replaces src/aggforce/util.py:119-124 (einsum), src/aggforce/map/core.py:13-16,219-240
// (NaN probe + protocol) and src/aggforce/agg.py:291-297 (residual) of the reference.
//
// Three paths, chosen by the host from the structure of M:
//   * sparse rows (slice / uniform maps: a few non-zeros per bead): sector-granular gather,
//     only the referenced sites are read from HBM;
//   * dense, small (n_cg <= 64 and the unique-column matrix fits in shared memory): frames
//     stream through a TMA bulk-copy ring fed by a producer warp; consumer warps build DMMA
//     A-fragments (8 frames x 4 unique columns of one xyz component) straight from the raw
//     f32 stage -- the constraint-group sum happens in the fragment build -- and multiply by
//     the register/shared resident map;
//   * dense, large: tiled DFMA fallback with the map read through L2.
// All arithmetic is f64 (the reference promotes f32 points x f64 matrix to f64).
// TMA bulk copies of this file move 16 KB pieces (A/B on the small dense kernel, whose stage is 16.8 KB:
// 4 / 8 / 16 KB pieces -> 0.612 / 0.553 / 0.552 ms per 1 M frames).
#ifndef AGF_BULK_PIECE
#define AGF_BULK_PIECE 16384u
#endif
#include "frame_pipe.cuh"
#include "panel.cuh"

#ifndef AGF_APPLY_TEAMS
#define AGF_APPLY_TEAMS 7
#endif
#ifndef AGF_APPLY_SCRATCH_BUFS
#define AGF_APPLY_SCRATCH_BUFS 1  // 1: two named barriers per octet; 2: one barrier, 21 KB less for the ring
#endif

namespace agf {

constexpr double kNanRtol = 1e-5;  // numpy.allclose default used at map/core.py:230

template <typename TO>
__device__ __forceinline__ void store_out(TO* p, double v) {
  *p = static_cast<TO>(v);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------ sparse
// Gather loads: a slice map touches 12 of every ~2100 bytes, so the L2 is told to fetch no more
// than 64 bytes around a miss (ld.global.nc.L2::64B) instead of a full 128-byte line.
__device__ __forceinline__ double ldg_sparse(const float* p) {
  float v;
  asm volatile("ld.global.nc.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return (double)v;
}
__device__ __forceinline__ double ldg_sparse(const double* p) {
  double v;
  asm volatile("ld.global.nc.L2::64B.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) apply_sparse_kernel(const TI* __restrict__ x, int64_t n_frames, int n_sites,
                                                           const int32_t* __restrict__ row_ptr,
                                                           const int32_t* __restrict__ row_sites,
                                                           const double* __restrict__ row_w, int n_cg,
                                                           TO* __restrict__ out, double* sumsq, int nan_mode,
                                                           double nan_atol, int32_t* nan_flags) {
  const int64_t total = n_frames * n_cg;
  double sq = 0.0;
  bool saw_nan = false, bad = false;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = idx / n_cg;
    const int c = (int)(idx - t * n_cg);
    const TI* fr = x + t * (int64_t)n_sites * 3;
    double a0 = 0, a1 = 0, a2 = 0, w0 = 0, w1 = 0, w2 = 0;
    const int b = __ldg(row_ptr + c), e = __ldg(row_ptr + c + 1);
    for (int m = b; m < e; ++m) {
      const TI* p = fr + 3 * __ldg(row_sites + m);
      const double w = __ldg(row_w + m);
      double v0 = ldg_sparse(p), v1 = ldg_sparse(p + 1), v2 = ldg_sparse(p + 2);
      if (nan_mode) {
        if (v0 != v0) { v0 = 0; w0 += w; saw_nan = true; }
        if (v1 != v1) { v1 = 0; w1 += w; saw_nan = true; }
        if (v2 != v2) { v2 = 0; w2 += w; saw_nan = true; }
      }
      a0 = fma(w, v0, a0);
      a1 = fma(w, v1, a1);
      a2 = fma(w, v2, a2);
    }
    if (nan_mode) {
      bad |= fabs(w0) > nan_atol + kNanRtol * fabs(a0 - w0);
      bad |= fabs(w1) > nan_atol + kNanRtol * fabs(a1 - w1);
      bad |= fabs(w2) > nan_atol + kNanRtol * fabs(a2 - w2);
    }
    TO* o = out + idx * 3;
    store_out(o, a0);
    store_out(o + 1, a1);
    store_out(o + 2, a2);
    // the residual is taken on the values as stored (f32 maps store f32)
    double r0 = (double)static_cast<TO>(a0), r1 = (double)static_cast<TO>(a1), r2 = (double)static_cast<TO>(a2);
    sq += r0 * r0 + r1 * r1 + r2 * r2;
  }
  if (sumsq) {
    sq = warp_sum(sq);
    if ((threadIdx.x & 31) == 0) atomicAdd(sumsq, sq);
  }
  if (nan_mode) {
    if (saw_nan) atomicOr(nan_flags, 1);
    if (bad) atomicOr(nan_flags + 1, 1);
  }
}

// Slice maps (exactly one site per bead, the usual coordinate map): the loads of four (frame, bead)
// items are issued before any of them is used -- the generic kernel above is bound by the latency of
// its one dependent gather per thread (ncu: long-scoreboard stalls, DRAM traffic already at the
// 64-byte minimum), not by bandwidth.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) apply_slice_kernel(const TI* __restrict__ x, int64_t n_frames, int n_sites,
                                                          const int32_t* __restrict__ row_sites,
                                                          const double* __restrict__ row_w, int n_cg,
                                                          TO* __restrict__ out, double* sumsq, int nan_mode,
                                                          double nan_atol, int32_t* nan_flags) {
  constexpr int U = 4;
  const int64_t total = n_frames * n_cg;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double sq = 0.0;
  bool saw_nan = false, bad = false;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; base < total; base += stride * U) {
    double v[U][3], w[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t idx = base + u * stride;
      v[u][0] = v[u][1] = v[u][2] = 0.0;
      w[u] = 0.0;
      if (idx < total) {
        const int64_t t = idx / n_cg;
        const int c = (int)(idx - t * n_cg);
        const TI* p = x + t * (int64_t)n_sites * 3 + 3 * __ldg(row_sites + c);
        w[u] = __ldg(row_w + c);
        v[u][0] = ldg_sparse(p);
        v[u][1] = ldg_sparse(p + 1);
        v[u][2] = ldg_sparse(p + 2);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t idx = base + u * stride;
      if (idx >= total) continue;
      double a[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        double f = v[u][d];
        if (nan_mode && f != f) {  // NaN counts as 0; the result depends on it unless its weight is ~0
          saw_nan = true;
          bad |= fabs(w[u]) > nan_atol + kNanRtol * fabs(w[u]);
          f = 0.0;
        }
        a[d] = w[u] * f;
      }
      TO* o = out + idx * 3;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        store_out(o + d, a[d]);
        const double r = (double)static_cast<TO>(a[d]);
        sq += r * r;
      }
    }
  }
  if (sumsq) {
    sq = warp_sum(sq);
    if ((threadIdx.x & 31) == 0) atomicAdd(sumsq, sq);
  }
  if (nan_mode) {
    if (saw_nan) atomicOr(nan_flags, 1);
    if (bad) atomicOr(nan_flags + 1, 1);
  }
}

// ------------------------------------------------------------------------------------ dense small
// Work item = 8 consecutive frames ("octet").  A producer warp streams octets through a ring
// of shared-memory stages with 1-D TMA bulk copies; each of the 8 consumer warps owns whole
// octets (stage j -> warp j % 8), so there is no block-wide barrier anywhere.  For its octet a
// warp runs, per 4 unique columns, 3 x NT DMMAs (xyz components x bead tiles): lane (g, q)
// builds the A element "frame g, unique column x0+q" for all three components straight from
// the raw stage (constraint-group sum + f64 promotion in registers), B fragments come from the
// shared-memory copy of the map.  NaNs are detected on the OUTPUT (0 * NaN = NaN poisons the
// whole row) and only then is the octet redone with the masking protocol.
struct DenseSmallParams {
  const void* x;
  int64_t n_frames;
  int32_t n_sites;
  const int32_t* ucol_ptr;
  const int32_t* ucol_sites;
  int32_t n_ucol;
  int32_t nnz;
  const double* umat_t;  // [n_ucol, n_cg]
  int32_t n_cg;
  void* out;
  double* sumsq;
  int32_t nan_mode;
  double nan_atol;
  int32_t* nan_flags;
  ChunkSchedule sch;
  int32_t n_stages;
};

constexpr int kApplyConsumers = AGF_APPLY_TEAMS;
constexpr int kOctet = 8;
constexpr int kMaxStages = 16;

template <typename TI>
__device__ __forceinline__ void group_value3(const TI* __restrict__ fr, const int32_t* __restrict__ s_ptr,
                                             const int32_t* __restrict__ s_sites, int x, int n_ucol, bool mask_nan,
                                             double (&v)[3], double (&cnt)[3]) {
  v[0] = v[1] = v[2] = 0.0;
  cnt[0] = cnt[1] = cnt[2] = 0.0;
  if (x >= n_ucol) return;
  for (int m = s_ptr[x]; m < s_ptr[x + 1]; ++m) {
    const TI* p = fr + 3 * s_sites[m];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      double f = to_f64(p[d]);
      if (mask_nan && f != f) {
        f = 0.0;
        cnt[d] += 1.0;
      }
      v[d] += f;
    }
  }
}

// SPLIT = warps per octet: with SPLIT == 2 the two warps of a team each contract half of the unique
// columns and the partial accumulators are combined through a double-buffered shared-memory
// scratch (one 64-thread named barrier per octet).  The per-octet chain LDS -> F2F -> DADD -> DMMA is
// latency bound; twice the warps per SM hide twice the latency.
template <typename TI, typename TO, int NT, int SPLIT>
__global__ void __launch_bounds__((kApplyConsumers * SPLIT + 1) * 32, 1)
    apply_dense_small_kernel(const __grid_constant__ DenseSmallParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int n_cg_pad = NT * 8;
  const int su = panel_stride(n_cg_pad);
  const int xpad = (p.n_ucol + 3) & ~3;
  // carve-up: U^T panel | member table | CSR | barriers | raw ring
  double* s_u = reinterpret_cast<double*>(smem);
  size_t off = (size_t)xpad * su * sizeof(double);
  int4* s_tab = reinterpret_cast<int4*>(smem + off);  // up to 4 member offsets (site*3) per unique column, -1 = none
  off += (size_t)xpad * sizeof(int4);
  int32_t* s_ptr = reinterpret_cast<int32_t*>(smem + off);
  off += (size_t)(p.n_ucol + 1) * 4;
  int32_t* s_sites = reinterpret_cast<int32_t*>(smem + off);
  off += (size_t)p.nnz * 4;
  off = (off + 15) / 16 * 16;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + off);
  uint64_t* empty = full + kMaxStages;
  off += 2 * kMaxStages * sizeof(uint64_t);
  off = (off + 127) / 128 * 128;
  constexpr int kAccDoubles = 3 * NT * 2;  // per lane
  double* s_scratch = reinterpret_cast<double*>(smem + off);  // [team][2][kAccDoubles][32], SPLIT == 2 only
  if (SPLIT == 2) off += (size_t)kApplyConsumers * AGF_APPLY_SCRATCH_BUFS * kAccDoubles * 32 * sizeof(double);
  TI* raw = reinterpret_cast<TI*>(smem + off);
  const int64_t frame_elems = (int64_t)p.n_sites * 3;
  const int64_t stage_elems = ((int64_t)kOctet * frame_elems * (int64_t)sizeof(TI) + 15) / 16 * 16 / (int64_t)sizeof(TI);
  const int n_stages = p.n_stages;

  for (int i = threadIdx.x; i < xpad * su; i += blockDim.x) {
    const int xx = i / su, c = i - xx * su;
    s_u[i] = (xx < p.n_ucol && c < p.n_cg) ? p.umat_t[(int64_t)xx * p.n_cg + c] : 0.0;
  }
  for (int i = threadIdx.x; i <= p.n_ucol; i += blockDim.x) s_ptr[i] = p.ucol_ptr[i];
  for (int i = threadIdx.x; i < p.nnz; i += blockDim.x) s_sites[i] = p.ucol_sites[i];
  __shared__ int s_generic;  // some unique column has more than 4 member sites -> CSR walk
  if (threadIdx.x == 0) s_generic = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < xpad; i += blockDim.x) {
    int m[4] = {-1, -1, -1, -1};
    if (i < p.n_ucol) {
      const int b = p.ucol_ptr[i], e = p.ucol_ptr[i + 1];
      for (int k = 0; k < 4 && b + k < e; ++k) m[k] = 3 * p.ucol_sites[b + k];
      if (e - b > 4) s_generic = 1;
    }
    s_tab[i] = make_int4(m[0], m[1], m[2], m[3]);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    fence_barrier_init();
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TI* base = reinterpret_cast<const TI*>(p.x);
  const int64_t first = blockIdx.x, step = gridDim.x;
  const int64_t n_mine = p.sch.n_chunks > first ? (p.sch.n_chunks - first + step - 1) / step : 0;

  if (warp == kApplyConsumers * SPLIT) {
    // ---------------- producer warp
    for (int64_t j = 0; j < n_mine; ++j) {
      const int64_t c = first + j * step;
      const int stage = (int)(j % n_stages);
      const uint32_t parity = (uint32_t)((j / n_stages) & 1);
      mbar_wait(&empty[stage], parity ^ 1u);
      const int nf = p.sch.count(c);
      const int64_t bytes = (int64_t)nf * frame_elems * (int64_t)sizeof(TI);
      const TI* src = base + p.sch.start(c) * frame_elems;
      TI* dst = raw + (int64_t)stage * stage_elems;
      const bool bulk = c != 0 && bytes > 0 && (bytes % 16) == 0 && (reinterpret_cast<uintptr_t>(src) % 16) == 0;
      if (bulk) {
        if (lane == 0) {
          fence_proxy_async();
          mbar_expect_tx(&full[stage], (uint32_t)bytes);
          uint32_t done = 0;
          while (done < (uint32_t)bytes) {
            const uint32_t piece = (uint32_t)bytes - done < kBulkPiece ? (uint32_t)bytes - done : kBulkPiece;
            tma_bulk_g2s(reinterpret_cast<char*>(dst) + done, reinterpret_cast<const char*>(src) + done, piece,
                         &full[stage]);
            done += piece;
          }
        }
      } else {
        const int64_t n = (int64_t)nf * frame_elems;
        for (int64_t i = lane; i < n; i += 32) dst[i] = src[i];
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[stage]);
      }
      __syncwarp();
    }
    return;
  }

  // ---------------- consumer warps
  const int g = lane >> 2, q = lane & 3;
  const bool nan_mode = p.nan_mode != 0;
  const bool generic_groups = s_generic != 0;
  TO* out = reinterpret_cast<TO*>(p.out);
  double sq = 0.0;
  bool saw_nan = false, bad = false;
  // A waiter can tell the current mbarrier phase from the previous one only, so at most n_stages
  // warps may consume (then the stage a warp waits for is never two phases ahead of its fill).
  const int n_cons = n_stages < kApplyConsumers ? n_stages : kApplyConsumers;
  const int team = warp / SPLIT, half = warp % SPLIT;
  if (team >= n_cons) return;
  // this warp's share of the unique columns
  const int xmid = SPLIT == 2 ? ((xpad / 4 + 1) / 2) * 4 : xpad;
  const int x_begin = half == 0 ? 0 : xmid, x_end = (SPLIT == 2 && half == 0) ? xmid : xpad;
  int it = 0;
  for (int64_t j = team; j < n_mine; j += n_cons) {
    const int64_t c = first + j * step;
    const int stage = (int)(j % n_stages);
    const uint32_t parity = (uint32_t)((j / n_stages) & 1);
    mbar_wait(&full[stage], parity);
    const int nf = p.sch.count(c);
    if (nf > 0) {
      const int64_t t0 = p.sch.start(c);
      const bool valid = g < nf;
      const TI* fr = raw + (int64_t)stage * stage_elems + (int64_t)(valid ? g : 0) * frame_elems;
      double acc[3][NT][2];
#pragma unroll
      for (int d = 0; d < 3; ++d)
#pragma unroll
        for (int n = 0; n < NT; ++n) acc[d][n][0] = acc[d][n][1] = 0.0;
      if (!generic_groups) {
#pragma unroll 2
        for (int x0 = x_begin; x0 < x_end; x0 += 4) {
          const int4 mem = s_tab[x0 + q];
          double a0 = 0.0, a1 = 0.0, a2 = 0.0;
          if (mem.x >= 0) { a0 = to_f64(fr[mem.x]); a1 = to_f64(fr[mem.x + 1]); a2 = to_f64(fr[mem.x + 2]); }
          if (mem.y >= 0) { a0 += to_f64(fr[mem.y]); a1 += to_f64(fr[mem.y + 1]); a2 += to_f64(fr[mem.y + 2]); }
          if (mem.z >= 0) { a0 += to_f64(fr[mem.z]); a1 += to_f64(fr[mem.z + 1]); a2 += to_f64(fr[mem.z + 2]); }
          if (mem.w >= 0) { a0 += to_f64(fr[mem.w]); a1 += to_f64(fr[mem.w + 1]); a2 += to_f64(fr[mem.w + 2]); }
          if (!valid) a0 = a1 = a2 = 0.0;
          const double* bp = s_u + (x0 + q) * su + g;
#pragma unroll
          for (int n = 0; n < NT; ++n) {
            const double b = bp[n * 8];
            dmma884(acc[0][n][0], acc[0][n][1], a0, b);
            dmma884(acc[1][n][0], acc[1][n][1], a1, b);
            dmma884(acc[2][n][0], acc[2][n][1], a2, b);
          }
        }
      } else {
        for (int x0 = x_begin; x0 < x_end; x0 += 4) {
          double v[3], cnt[3];
          group_value3<TI>(fr, s_ptr, s_sites, x0 + q, p.n_ucol, false, v, cnt);
          if (!valid) v[0] = v[1] = v[2] = 0.0;
          const double* bp = s_u + (x0 + q) * su + g;
#pragma unroll
          for (int n = 0; n < NT; ++n) {
            const double b = bp[n * 8];
            dmma884(acc[0][n][0], acc[0][n][1], v[0], b);
            dmma884(acc[1][n][0], acc[1][n][1], v[1], b);
            dmma884(acc[2][n][0], acc[2][n][1], v[2], b);
          }
        }
      }
      if (SPLIT == 2) {
        // combine the two halves: warp 1 of the team publishes, warp 0 adds and finishes the octet
        double* scr = s_scratch + ((size_t)(team * AGF_APPLY_SCRATCH_BUFS + (it & (AGF_APPLY_SCRATCH_BUFS - 1))) *
                                   kAccDoubles) * 32 + lane;
        ++it;
        if (half == 1) {
#pragma unroll
          for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int n = 0; n < NT; ++n) {
              scr[((d * NT + n) * 2) * 32] = acc[d][n][0];
              scr[((d * NT + n) * 2 + 1) * 32] = acc[d][n][1];
            }
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + team) : "memory");
        if (half == 0) {
#pragma unroll
          for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int n = 0; n < NT; ++n) {
              acc[d][n][0] += scr[((d * NT + n) * 2) * 32];
              acc[d][n][1] += scr[((d * NT + n) * 2 + 1) * 32];
            }
        }
        if (AGF_APPLY_SCRATCH_BUFS == 1)  // single buffer: warp 1 may not overwrite it before warp 0 has read it
          asm volatile("bar.sync %0, 64;" ::"r"(1 + team) : "memory");
        if (half == 1) continue;  // the raw stage is released by warp 0 (which may still redo it)
      }
      if (nan_mode) {
        bool has_nan = false;
#pragma unroll
        for (int d = 0; d < 3; ++d)
#pragma unroll
          for (int n = 0; n < NT; ++n) has_nan |= (acc[d][n][0] != acc[d][n][0]) | (acc[d][n][1] != acc[d][n][1]);
        if (__any_sync(0xffffffffu, has_nan)) {
          // rare path: redo the octet with NaN -> 0 and accumulate the weight mass on NaN entries
          double nw[3][NT][2];
#pragma unroll
          for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int n = 0; n < NT; ++n) acc[d][n][0] = acc[d][n][1] = nw[d][n][0] = nw[d][n][1] = 0.0;
          bool any_cnt = false;
          for (int x0 = 0; x0 < xpad; x0 += 4) {
            double v[3], cnt[3];
            group_value3<TI>(fr, s_ptr, s_sites, x0 + q, p.n_ucol, true, v, cnt);
            if (!valid) v[0] = v[1] = v[2] = cnt[0] = cnt[1] = cnt[2] = 0.0;
            any_cnt |= (cnt[0] + cnt[1] + cnt[2]) != 0.0;
            const double* bp = s_u + (x0 + q) * su + g;
#pragma unroll
            for (int n = 0; n < NT; ++n) {
              const double b = bp[n * 8];
#pragma unroll
              for (int d = 0; d < 3; ++d) {
                dmma884(acc[d][n][0], acc[d][n][1], v[d], b);
                dmma884(nw[d][n][0], nw[d][n][1], cnt[d], b);
              }
            }
          }
          saw_nan |= __any_sync(0xffffffffu, any_cnt);
#pragma unroll
          for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int n = 0; n < NT; ++n) {
              bad |= fabs(nw[d][n][0]) > p.nan_atol + kNanRtol * fabs(acc[d][n][0] - nw[d][n][0]);
              bad |= fabs(nw[d][n][1]) > p.nan_atol + kNanRtol * fabs(acc[d][n][1] - nw[d][n][1]);
            }
        }
      }
      // C[g][2q], C[g][2q+1] of component d: frame t0+g, beads n*8+2q (+1) -> 6 consecutive outputs
      if (valid) {
        TO* orow = out + (t0 + g) * (int64_t)p.n_cg * 3;
#pragma unroll
        for (int n = 0; n < NT; ++n) {
          const int cb = n * 8 + 2 * q;
          if (cb < p.n_cg) {
#pragma unroll
            for (int d = 0; d < 3; ++d) {
              store_out(orow + (int64_t)cb * 3 + d, acc[d][n][0]);
              const double r = (double)static_cast<TO>(acc[d][n][0]);
              sq += r * r;
            }
          }
          if (cb + 1 < p.n_cg) {
#pragma unroll
            for (int d = 0; d < 3; ++d) {
              store_out(orow + (int64_t)(cb + 1) * 3 + d, acc[d][n][1]);
              const double r = (double)static_cast<TO>(acc[d][n][1]);
              sq += r * r;
            }
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0 && half == 0) mbar_arrive(&empty[stage]);  // one arrival per stage (also for empty chunks)
  }
  if (p.sumsq) {
    sq = warp_sum(sq);
    if (lane == 0) atomicAdd(p.sumsq, sq);
  }
  if (nan_mode) {
    if (saw_nan) atomicOr(p.nan_flags, 1);
    if (bad) atomicOr(p.nan_flags + 1, 1);
  }
}

// ------------------------------------------------------------------------------------ dense large: packed-panel GEMM
// out[(t,d), c] = sum_x Xg[(t,d), x] U^T[x, c]  as a DMMA GEMM over packed panels (panel.cuh):
//   apply_pack_kernel     : group sums + f64 promotion of 128 frames x 24 unique columns, one panel
//                           per xyz component:  wsA[(frame block, d)][k-chunk][24 x][132 frames];
//                           also the NaN probe (map/core.py:13-16) -- it reads every referenced value;
//   apply_pack_map_kernel : U^T as  wsB[bead block][k-chunk][24 x][132 beads];
//   apply_gemm_kernel     : CTA = (frame block, d) x bead block, contraction over all unique columns.
// If the probe saw a NaN the slab is redone by the masking fallback kernel below (gated on the
// workspace header), which implements the NaN protocol (map/core.py:219-240).
struct ApplyWsHeader {
  int32_t redo;   // a referenced input value was NaN
  int32_t pad;
  double sumsq;   // sum(out^2) of the GEMM result
};
constexpr size_t kApplyWsHeaderBytes = 256;

template <typename TI>
__global__ void __launch_bounds__(256) apply_pack_kernel(const TI* __restrict__ x, int64_t n_frames, int n_sites,
                                                         const int32_t* __restrict__ ucol_ptr,
                                                         const int32_t* __restrict__ ucol_sites, int n_ucol,
                                                         int n_kchunks, double* __restrict__ ws_a,
                                                         ApplyWsHeader* header, int nan_mode) {
  const int fb = blockIdx.x / n_kchunks, kc = blockIdx.x - fb * n_kchunks;
  const int64_t t0 = (int64_t)fb * kPanelCols;
  bool saw_nan = false;
  double* pan0 = ws_a + ((int64_t)(fb * 3) * n_kchunks + kc) * kPanelElems;
  const int64_t dstep = (int64_t)n_kchunks * kPanelElems;
  for (int item = threadIdx.x; item < kPanelRows * kPanelCols; item += blockDim.x) {
    const int kr = item >> 7, m = item & 127;
    const int u = kc * kPanelRows + kr;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    if (u < n_ucol && t0 + m < n_frames) {
      const TI* fr = x + (t0 + m) * (int64_t)n_sites * 3;
      const int b = __ldg(ucol_ptr + u), e = __ldg(ucol_ptr + u + 1);
      for (int k = b; k < e; ++k) {
        const TI* q = fr + 3 * __ldg(ucol_sites + k);
        s0 += to_f64(__ldg(q));
        s1 += to_f64(__ldg(q + 1));
        s2 += to_f64(__ldg(q + 2));
      }
      saw_nan |= (s0 != s0) | (s1 != s1) | (s2 != s2);
    }
    double* dst = pan0 + kr * kPanelStride + m;
    dst[0] = s0;
    dst[dstep] = s1;
    dst[2 * dstep] = s2;
  }
  if (saw_nan && nan_mode) atomicOr(&header->redo, 1);
}

__global__ void apply_pack_map_kernel(const double* __restrict__ umat_t, int n_ucol, int n_cg, int n_kchunks,
                                      double* __restrict__ ws_b) {
  const int nbk = blockIdx.x / n_kchunks, kc = blockIdx.x - nbk * n_kchunks;
  double* pan = ws_b + (int64_t)blockIdx.x * kPanelElems;
  for (int item = threadIdx.x; item < kPanelRows * kPanelCols; item += blockDim.x) {
    const int kr = item >> 7, n = item & 127;
    const int u = kc * kPanelRows + kr, c = nbk * kPanelCols + n;
    pan[kr * kPanelStride + n] = (u < n_ucol && c < n_cg) ? __ldg(umat_t + (int64_t)u * n_cg + c) : 0.0;
  }
}

struct ApplyGemmParams {
  const double* ws_a;
  const double* ws_b;
  int64_t n_frames;
  int32_t n_cg, n_kchunks, n_nblocks;
  void* out;
  ApplyWsHeader* header;
};

template <typename TO>
__global__ void __launch_bounds__(kPanelThreads, 1) apply_gemm_kernel(const __grid_constant__ ApplyGemmParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  // adjacent CTAs = the bead blocks of one (frame block, d): the A panels are fetched from HBM once
  const int nbk = blockIdx.x % p.n_nblocks, mb = blockIdx.x / p.n_nblocks;
  const int fb = mb / 3, d = mb - fb * 3;
  const int64_t t0 = (int64_t)fb * kPanelCols;
  const int64_t left = p.n_frames - t0;
  const int ct_rows = left >= kPanelCols ? 16 : (int)((left + 7) / 8);
  const int cols_left = p.n_cg - nbk * kPanelCols;
  const int ct_cols = cols_left >= kPanelCols ? 16 : (cols_left + 7) / 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = panel_warp_row(warp);
  const uint32_t m = warp < kPanelMmaWarps ? panel_row_mask(r0, ct_rows, ct_cols, false) : 0u;
  PanelStream st;
  st.a = p.ws_a + (int64_t)mb * p.n_kchunks * kPanelElems;
  st.b = p.ws_b + (int64_t)nbk * p.n_kchunks * kPanelElems;
  st.a_step = st.b_step = kPanelElems;
  st.n = p.n_kchunks;
  st.same = false;
  double acc[16][2];
  if (!panel_mainloop<false>(smem, st, m, acc)) return;
  const int g = lane >> 2, q = lane & 3;
  TO* out = reinterpret_cast<TO*>(p.out);
  double sq = 0.0;
  const int64_t t = t0 + r0 * 8 + g;
  if (m != 0u && t < p.n_frames) {
    TO* orow = out + t * (int64_t)p.n_cg * 3 + d;
#pragma unroll
    for (int cc = 0; cc < 16; ++cc) {
      if (!((m >> cc) & 1u)) continue;
      const int c = nbk * kPanelCols + cc * 8 + 2 * q;
      if (c < p.n_cg) {
        store_out(orow + (int64_t)c * 3, acc[cc][0]);
        const double v = (double)static_cast<TO>(acc[cc][0]);
        sq += v * v;
      }
      if (c + 1 < p.n_cg) {
        store_out(orow + (int64_t)(c + 1) * 3, acc[cc][1]);
        const double v = (double)static_cast<TO>(acc[cc][1]);
        sq += v * v;
      }
    }
  }
  sq = warp_sum(sq);
  if (lane == 0 && sq != 0.0) atomicAdd(&p.header->sumsq, sq);
}

// ------------------------------------------------------------------------------------ dense large (NaN fallback / no workspace)
// CTA = 8 frames (24 rows); thread = one bead c (strided); unique columns processed in
// blocks of 64 whose group sums are staged in shared memory as xg[x][row].
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) apply_dense_big_kernel(const TI* __restrict__ x, int64_t n_frames, int n_sites,
                                                              const int32_t* __restrict__ ucol_ptr,
                                                              const int32_t* __restrict__ ucol_sites, int n_ucol,
                                                              const double* __restrict__ umat_t, int n_cg,
                                                              TO* __restrict__ out, double* sumsq, int nan_mode,
                                                              double nan_atol, int32_t* nan_flags,
                                                              const ApplyWsHeader* gate) {
  constexpr int FR = 8, ROWS = FR * 3, XB = 64;
  if (gate != nullptr && gate->redo == 0) {
    // the packed-panel GEMM already produced this slab: only publish its residual sum
    if (blockIdx.x == 0 && threadIdx.x == 0 && sumsq) atomicAdd(sumsq, gate->sumsq);
    return;
  }
  __shared__ double xg[XB][ROWS];
  __shared__ double xn[XB][ROWS];
  __shared__ int s_has_nan;
  double sq = 0.0;
  bool saw_nan = false, bad = false;
  const int64_t n_groups = (n_frames + FR - 1) / FR;
  for (int64_t grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const int64_t t0 = grp * FR;
    const int nf = (int)min((int64_t)FR, n_frames - t0);
    for (int cb = 0; cb < n_cg; cb += blockDim.x) {
      const int c = cb + threadIdx.x;
      double acc[ROWS], nw[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) acc[r] = nw[r] = 0.0;
      bool any_nan_blocks = false;
      for (int xb = 0; xb < n_ucol; xb += XB) {
        __syncthreads();
        if (threadIdx.x == 0) s_has_nan = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < XB * ROWS; i += blockDim.x) {
          const int xx = i / ROWS, r = i - xx * ROWS;
          const int t = r / 3, d = r - t * 3;
          double v = 0.0, nc = 0.0;
          if (xb + xx < n_ucol && t < nf) {
            const TI* fr = x + (t0 + t) * (int64_t)n_sites * 3 + d;
            const int b = __ldg(ucol_ptr + xb + xx), e = __ldg(ucol_ptr + xb + xx + 1);
            for (int m = b; m < e; ++m) {
              double f = to_f64(__ldg(fr + 3 * __ldg(ucol_sites + m)));
              if (nan_mode && f != f) {
                f = 0.0;
                nc += 1.0;
              }
              v += f;
            }
          }
          xg[xx][r] = v;
          xn[xx][r] = nc;
          if (nc != 0.0) s_has_nan = 1;
        }
        __syncthreads();
        const bool has_nan = s_has_nan != 0;
        any_nan_blocks |= has_nan;
        if (c < n_cg) {
          const int lim = min(XB, n_ucol - xb);
          for (int xx = 0; xx < lim; ++xx) {
            const double u = __ldg(umat_t + (int64_t)(xb + xx) * n_cg + c);
#pragma unroll
            for (int r = 0; r < ROWS; ++r) acc[r] = fma(u, xg[xx][r], acc[r]);
            if (has_nan) {
#pragma unroll
              for (int r = 0; r < ROWS; ++r) nw[r] = fma(u, xn[xx][r], nw[r]);
            }
          }
        }
      }
      saw_nan |= any_nan_blocks;
      if (c < n_cg) {
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
          const int t = r / 3, d = r - t * 3;
          if (t < nf) {
            store_out(out + ((t0 + t) * (int64_t)n_cg + c) * 3 + d, acc[r]);
            double v = (double)static_cast<TO>(acc[r]);
            sq += v * v;
            if (any_nan_blocks) bad |= fabs(nw[r]) > nan_atol + kNanRtol * fabs(acc[r] - nw[r]);
          }
        }
      }
    }
  }
  if (sumsq) {
    sq = warp_sum(sq);
    if ((threadIdx.x & 31) == 0) atomicAdd(sumsq, sq);
  }
  if (nan_mode) {
    if (saw_nan) atomicOr(nan_flags, 1);
    if (bad) atomicOr(nan_flags + 1, 1);
  }
}

// Shared-memory footprint of the small dense kernel before its raw ring; 0 = does not apply.
static int small_split(int ntk) { return ntk <= 2 ? 2 : 1; }  // warps per octet (scratch grows with NT)

static size_t small_fixed_bytes(int n_ucol, int nnz, int n_cg) {
  const int nt = (n_cg + 7) / 8;
  if (n_cg > 64 || nt < 1) return 0;
  const int ntk = nt <= 4 ? nt : (nt <= 6 ? 6 : 8);
  const int su = panel_stride(ntk * 8);
  const int xpad = (n_ucol + 3) & ~3;
  size_t off = (size_t)xpad * su * sizeof(double) + (size_t)xpad * 16 + (size_t)(n_ucol + 1) * 4 + (size_t)nnz * 4;
  off = (off + 15) / 16 * 16 + 2 * kMaxStages * sizeof(uint64_t);
  off = (off + 127) / 128 * 128;
  if (small_split(ntk) == 2) off += (size_t)kApplyConsumers * AGF_APPLY_SCRATCH_BUFS * (3 * ntk * 2) * 32 * sizeof(double);
  return off;
}
static bool small_fits(int n_sites, int n_ucol, int nnz, int n_cg, size_t elem) {
  const size_t off = small_fixed_bytes(n_ucol, nnz, n_cg);
  const size_t stage_bytes = ((size_t)kOctet * n_sites * 3 * elem + 15) / 16 * 16;
  return off != 0 && off + 4 * stage_bytes <= (size_t)224 * 1024;
}

template <typename TI, typename TO, int NT>
static int launch_small(DenseSmallParams& p, cudaStream_t stream) {
  p.sch = make_schedule(p.x, p.n_frames, (int64_t)p.n_sites * 3 * sizeof(TI), kOctet);
  const size_t off = small_fixed_bytes(p.n_ucol, p.nnz, p.n_cg);
  size_t stage_bytes = ((size_t)kOctet * p.n_sites * 3 * sizeof(TI) + 15) / 16 * 16;
  const size_t budget = 224 * 1024;
  if (!small_fits(p.n_sites, p.n_ucol, p.nnz, p.n_cg, sizeof(TI))) return 1;  // caller uses the GEMM path
  int n_stages = (int)((budget - off) / stage_bytes);
  if (n_stages > kMaxStages) n_stages = kMaxStages;
  p.n_stages = n_stages;
  size_t smem = off + (size_t)n_stages * stage_bytes;
  constexpr int SPLIT = NT <= 2 ? 2 : 1;
  auto kern = apply_dense_small_kernel<TI, TO, NT, SPLIT>;
  AGF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t ctas = sm_count();
  int64_t want = (p.sch.n_chunks + kApplyConsumers - 1) / kApplyConsumers;
  if (ctas > want) ctas = want;
  if (ctas < 1) ctas = 1;
  kern<<<(int)ctas, (kApplyConsumers * SPLIT + 1) * 32, smem, stream>>>(p);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

template <typename TI, typename TO>
static int dispatch_small(DenseSmallParams& p, cudaStream_t stream) {
  const int nt = (p.n_cg + 7) / 8;
  switch (nt) {
    case 1: return launch_small<TI, TO, 1>(p, stream);
    case 2: return launch_small<TI, TO, 2>(p, stream);
    case 3: return launch_small<TI, TO, 3>(p, stream);
    case 4: return launch_small<TI, TO, 4>(p, stream);
    case 5:
    case 6: return launch_small<TI, TO, 6>(p, stream);
    case 7:
    case 8: return launch_small<TI, TO, 8>(p, stream);
    default: return 1;
  }
}

// Bytes of packed A panels per block of 128 frames, and of the packed map.
static int64_t gemm_kchunks(int n_ucol) { return (n_ucol + kPanelRows - 1) / kPanelRows; }
static int64_t gemm_fb_bytes(int n_ucol) { return 3 * gemm_kchunks(n_ucol) * (int64_t)kPanelBytes; }
static int64_t gemm_map_bytes(int n_ucol, int n_cg) {
  return (int64_t)panel_blocks(n_cg) * gemm_kchunks(n_ucol) * (int64_t)kPanelBytes;
}

template <typename TI, typename TO>
static int launch_big(const TI* x, int64_t n_frames, int n_sites, const int32_t* ucol_ptr, const int32_t* ucol_sites,
                      int n_ucol, const double* umat_t, int n_cg, TO* out, double* sumsq, int nan_mode,
                      double nan_atol, int32_t* nan_flags, const ApplyWsHeader* gate, cudaStream_t stream) {
  int64_t groups = (n_frames + 7) / 8;
  int blocks = (int)(groups < (int64_t)sm_count() * 4 ? groups : (int64_t)sm_count() * 4);
  if (blocks < 1) blocks = 1;
  apply_dense_big_kernel<TI, TO><<<blocks, 256, 0, stream>>>(x, n_frames, n_sites, ucol_ptr, ucol_sites, n_ucol, umat_t,
                                                             n_cg, out, sumsq, nan_mode, nan_atol, nan_flags, gate);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

template <typename TI, typename TO>
static int apply_typed(const void* points, int64_t n_frames, int32_t n_sites, const int32_t* ucol_ptr,
                       const int32_t* ucol_sites, int32_t n_ucol, int32_t nnz, const double* umat_t, int32_t n_cg,
                       void* out, double* sumsq, int nan_mode, double nan_atol, int32_t* nan_flags, void* workspace,
                       size_t workspace_bytes, cudaStream_t stream) {
  DenseSmallParams p;
  memset(&p, 0, sizeof(p));
  p.x = points;
  p.n_frames = n_frames;
  p.n_sites = n_sites;
  p.ucol_ptr = ucol_ptr;
  p.ucol_sites = ucol_sites;
  p.n_ucol = n_ucol;
  p.nnz = nnz;
  p.umat_t = umat_t;
  p.n_cg = n_cg;
  p.out = out;
  p.sumsq = sumsq;
  p.nan_mode = nan_mode;
  p.nan_atol = nan_atol;
  p.nan_flags = nan_flags;
  int rc = 1;
  if (n_cg <= 64 && nnz >= 0) rc = dispatch_small<TI, TO>(p, stream);
  if (rc <= 0) return rc;
  const TI* x = reinterpret_cast<const TI*>(points);
  TO* o = reinterpret_cast<TO*>(out);
  const int64_t fixed = (int64_t)kApplyWsHeaderBytes + gemm_map_bytes(n_ucol, n_cg);
  const int64_t fb_bytes = gemm_fb_bytes(n_ucol);
  if (workspace == nullptr || (int64_t)workspace_bytes < fixed + fb_bytes)
    return launch_big<TI, TO>(x, n_frames, n_sites, ucol_ptr, ucol_sites, n_ucol, umat_t, n_cg, o, sumsq, nan_mode,
                              nan_atol, nan_flags, nullptr, stream);
  // ---- packed-panel GEMM over slabs of frames
  char* wsp = reinterpret_cast<char*>(workspace);
  ApplyWsHeader* header = reinterpret_cast<ApplyWsHeader*>(wsp);
  double* ws_b = reinterpret_cast<double*>(wsp + kApplyWsHeaderBytes);
  double* ws_a = reinterpret_cast<double*>(wsp + fixed);
  const int n_kchunks = (int)gemm_kchunks(n_ucol), n_nblocks = panel_blocks(n_cg);
  apply_pack_map_kernel<<<n_nblocks * n_kchunks, 256, 0, stream>>>(umat_t, n_ucol, n_cg, n_kchunks, ws_b);
  AGF_CUDA_TRY(cudaGetLastError());
  AGF_CUDA_TRY(cudaFuncSetAttribute(apply_gemm_kernel<TO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPanelSmem));
  const int64_t slab_fb = ((int64_t)workspace_bytes - fixed) / fb_bytes;
  const int64_t slab_frames = slab_fb * kPanelCols;
  for (int64_t f0 = 0; f0 < n_frames; f0 += slab_frames) {
    const int64_t nf = n_frames - f0 < slab_frames ? n_frames - f0 : slab_frames;
    const int64_t fbs = (nf + kPanelCols - 1) / kPanelCols;
    const TI* xs = x + f0 * (int64_t)n_sites * 3;
    TO* os = o + f0 * (int64_t)n_cg * 3;
    AGF_CUDA_TRY(cudaMemsetAsync(header, 0, sizeof(ApplyWsHeader), stream));
    AGF_REQUIRE(fbs * n_kchunks < (int64_t)1 << 31 && fbs * 3 * n_nblocks < (int64_t)1 << 31, "agf_map_apply: slab too large");
    apply_pack_kernel<TI><<<(unsigned)(fbs * n_kchunks), 256, 0, stream>>>(xs, nf, n_sites, ucol_ptr, ucol_sites, n_ucol,
                                                                         n_kchunks, ws_a, header, nan_mode);
    AGF_CUDA_TRY(cudaGetLastError());
    ApplyGemmParams gp;
    gp.ws_a = ws_a;
    gp.ws_b = ws_b;
    gp.n_frames = nf;
    gp.n_cg = n_cg;
    gp.n_kchunks = n_kchunks;
    gp.n_nblocks = n_nblocks;
    gp.out = os;
    gp.header = header;
    apply_gemm_kernel<TO><<<(unsigned)(fbs * 3 * n_nblocks), kPanelThreads, kPanelSmem, stream>>>(gp);
    AGF_CUDA_TRY(cudaGetLastError());
    // publishes the residual sum, or redoes the slab with the NaN protocol if the probe fired
    if (sumsq != nullptr || nan_mode != 0) {
      rc = launch_big<TI, TO>(xs, nf, n_sites, ucol_ptr, ucol_sites, n_ucol, umat_t, n_cg, os, sumsq, nan_mode, nan_atol,
                              nan_flags, header, stream);
      if (rc) return rc;
    }
  }
  return AGF_OK;
}

}  // namespace agf

extern "C" size_t agf_map_apply_workspace_bytes(int in_dtype, int32_t n_sites, int32_t n_ucol, int32_t nnz,
                                                int32_t n_cg, int64_t n_frames) {
  using namespace agf;
  if (n_sites <= 0 || n_ucol <= 0 || n_cg <= 0 || n_frames <= 0) return 0;
  if (small_fits(n_sites, n_ucol, nnz, n_cg, in_dtype == AGF_F32 ? 4 : 8)) return 0;
  const int64_t fixed = (int64_t)kApplyWsHeaderBytes + gemm_map_bytes(n_ucol, n_cg);
  const int64_t fb_bytes = gemm_fb_bytes(n_ucol);
  int64_t fbs = (n_frames + kPanelCols - 1) / kPanelCols;
  const int64_t cap = ((int64_t)2 << 30) / fb_bytes;  // slabs of at most 2 GiB
  if (fbs > cap) fbs = cap < 1 ? 1 : cap;
  return (size_t)(fixed + fbs * fb_bytes);
}

extern "C" int agf_map_apply_ws(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                                const int32_t* ucol_ptr, const int32_t* ucol_sites, int32_t n_ucol, int32_t nnz,
                                const double* umat_t, int32_t n_cg, void* out, int out_dtype, double* sumsq,
                                int nan_mode, double nan_atol, int32_t* nan_flags, void* workspace,
                                size_t workspace_bytes, void* stream) {
  using namespace agf;
  AGF_REQUIRE(points && ucol_ptr && ucol_sites && umat_t && out, "agf_map_apply: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_ucol > 0 && n_cg > 0 && nnz > 0, "agf_map_apply: bad sizes");
  AGF_REQUIRE(nan_mode == 0 || nan_flags != nullptr, "agf_map_apply: nan_mode 1 needs nan_flags");
  AGF_REQUIRE((in_dtype == AGF_F32 || in_dtype == AGF_F64) && (out_dtype == AGF_F32 || out_dtype == AGF_F64),
              "agf_map_apply: bad dtype");
  AGF_REQUIRE(workspace == nullptr || (reinterpret_cast<uintptr_t>(workspace) % 256) == 0,
              "agf_map_apply: workspace must be 256-byte aligned");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
#define AGF_APPLY(TI, TO)                                                                                      \
  return apply_typed<TI, TO>(points, n_frames, n_sites, ucol_ptr, ucol_sites, n_ucol, nnz, umat_t, n_cg, out, \
                             sumsq, nan_mode, nan_atol, nan_flags, workspace, workspace_bytes, s)
  if (in_dtype == AGF_F32 && out_dtype == AGF_F64) AGF_APPLY(float, double);
  if (in_dtype == AGF_F32 && out_dtype == AGF_F32) AGF_APPLY(float, float);
  if (in_dtype == AGF_F64 && out_dtype == AGF_F64) AGF_APPLY(double, double);
  AGF_APPLY(double, float);
#undef AGF_APPLY
}

extern "C" int agf_map_apply(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                             const int32_t* ucol_ptr, const int32_t* ucol_sites, int32_t n_ucol, int32_t nnz,
                             const double* umat_t, int32_t n_cg, void* out, int out_dtype, double* sumsq,
                             int nan_mode, double nan_atol, int32_t* nan_flags, void* stream) {
  return agf_map_apply_ws(points, in_dtype, n_frames, n_sites, ucol_ptr, ucol_sites, n_ucol, nnz, umat_t, n_cg, out,
                          out_dtype, sumsq, nan_mode, nan_atol, nan_flags, nullptr, 0, stream);
}

extern "C" int agf_map_apply_sparse(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                                    const int32_t* row_ptr, const int32_t* row_sites, const double* row_weights,
                                    int32_t n_cg, void* out, int out_dtype, double* sumsq, int nan_mode,
                                    double nan_atol, int32_t* nan_flags, void* stream) {
  using namespace agf;
  AGF_REQUIRE(points && row_ptr && row_sites && row_weights && out, "agf_map_apply_sparse: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_cg > 0, "agf_map_apply_sparse: bad sizes");
  AGF_REQUIRE(nan_mode == 0 || nan_flags != nullptr, "agf_map_apply_sparse: nan_mode 1 needs nan_flags");
  AGF_REQUIRE((in_dtype == AGF_F32 || in_dtype == AGF_F64) && (out_dtype == AGF_F32 || out_dtype == AGF_F64),
              "agf_map_apply_sparse: bad dtype");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int64_t total = n_frames * n_cg;
  int64_t want = (total + 255) / 256;
  int blocks = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
#define AGF_SP(TI, TO)                                                                                          \
  apply_sparse_kernel<TI, TO><<<blocks, 256, 0, s>>>(reinterpret_cast<const TI*>(points), n_frames, n_sites,    \
                                                     row_ptr, row_sites, row_weights, n_cg,                     \
                                                     reinterpret_cast<TO*>(out), sumsq, nan_mode, nan_atol,     \
                                                     nan_flags)
  if (in_dtype == AGF_F32 && out_dtype == AGF_F64) AGF_SP(float, double);
  else if (in_dtype == AGF_F32 && out_dtype == AGF_F32) AGF_SP(float, float);
  else if (in_dtype == AGF_F64 && out_dtype == AGF_F64) AGF_SP(double, double);
  else AGF_SP(double, float);
#undef AGF_SP
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

extern "C" int agf_map_apply_slice(const void* points, int in_dtype, int64_t n_frames, int32_t n_sites,
                                   const int32_t* row_sites, const double* row_weights, int32_t n_cg, void* out,
                                   int out_dtype, double* sumsq, int nan_mode, double nan_atol, int32_t* nan_flags,
                                   void* stream) {
  using namespace agf;
  AGF_REQUIRE(points && row_sites && row_weights && out, "agf_map_apply_slice: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_cg > 0, "agf_map_apply_slice: bad sizes");
  AGF_REQUIRE(nan_mode == 0 || nan_flags != nullptr, "agf_map_apply_slice: nan_mode 1 needs nan_flags");
  AGF_REQUIRE((in_dtype == AGF_F32 || in_dtype == AGF_F64) && (out_dtype == AGF_F32 || out_dtype == AGF_F64),
              "agf_map_apply_slice: bad dtype");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int64_t total = n_frames * n_cg;
  const int64_t want = (total + 256 * 4 - 1) / (256 * 4);
  const int blocks = (int)(want < (int64_t)sm_count() * 8 ? (want < 1 ? 1 : want) : (int64_t)sm_count() * 8);
#define AGF_SL(TI, TO)                                                                                        \
  apply_slice_kernel<TI, TO><<<blocks, 256, 0, s>>>(reinterpret_cast<const TI*>(points), n_frames, n_sites,   \
                                                    row_sites, row_weights, n_cg, reinterpret_cast<TO*>(out), \
                                                    sumsq, nan_mode, nan_atol, nan_flags)
  if (in_dtype == AGF_F32 && out_dtype == AGF_F64) AGF_SL(float, double);
  else if (in_dtype == AGF_F32 && out_dtype == AGF_F32) AGF_SL(float, float);
  else if (in_dtype == AGF_F64 && out_dtype == AGF_F64) AGF_SL(double, double);
  else AGF_SL(double, float);
#undef AGF_SL
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

// ------------------------------------------------------------------ weighted residual
// sumsq += sum_t w_t sum_e x[t, e]^2 over a mapped array [n_frames, per_frame]: warp = frame, lanes stride its
// elements; one float64 atomic per block.
namespace agf {
template <typename T>
__global__ void __launch_bounds__(256) weighted_sumsq_kernel(const T* __restrict__ x, int64_t n_frames, int per_frame,
                                                             const double* __restrict__ w, double* sumsq) {
  __shared__ double s_part[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double acc = 0.0;
  for (int64_t t = (int64_t)blockIdx.x * 8 + warp; t < n_frames; t += (int64_t)gridDim.x * 8) {
    const T* row = x + t * per_frame;
    double s = 0.0;
    for (int e = lane; e < per_frame; e += 32) {
      const double v = to_f64(row[e]);
      s += v * v;
    }
    acc += __ldg(w + t) * s;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) s_part[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double b = 0.0;
    for (int i = 0; i < 8; ++i) b += s_part[i];
    atomicAdd(sumsq, b);
  }
}
}  // namespace agf

extern "C" int agf_weighted_sumsq(const void* x, int dtype, int64_t n_frames, int32_t per_frame,
                                  const double* frame_weights, double* sumsq, void* stream) {
  using namespace agf;
  AGF_REQUIRE(x && frame_weights && sumsq, "agf_weighted_sumsq: null pointer");
  AGF_REQUIRE(n_frames >= 0 && per_frame > 0, "agf_weighted_sumsq: bad sizes");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_weighted_sumsq: bad dtype");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int64_t want = (n_frames + 7) / 8;
  const int blocks = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
  if (dtype == AGF_F32)
    weighted_sumsq_kernel<float><<<blocks, 256, 0, s>>>(reinterpret_cast<const float*>(x), n_frames, per_frame,
                                                        frame_weights, sumsq);
  else
    weighted_sumsq_kernel<double><<<blocks, 256, 0, s>>>(reinterpret_cast<const double*>(x), n_frames, per_frame,
                                                         frame_weights, sumsq);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}
