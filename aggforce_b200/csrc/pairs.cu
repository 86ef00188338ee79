// Kernel (c): pair-distance moments for guess_pairwise_constraints.
//
// Replaces src/aggforce/util.py:64-70 + src/aggforce/constraints/constfinder.py:47 of the
// reference, which materialise a (T, n, n, 3) displacement array.  Here
//   * agf_pair_screen  does the literal all-pairs pass over a SHORT frame prefix and returns the
//     partial sum of squared deviations per pair (exact pruning bound, see agf_b200.h);
//   * agf_pair_moments streams ALL frames once for the surviving pairs only: frames arrive in
//     shared memory through the TMA bulk-copy ring, every consumer thread owns one
//     (pair, frame-slot) and keeps its two running sums in registers; distances and sums
//     are float64 (SURVEY Q10: the parity target is the float64 evaluation).
#include "frame_pipe.cuh"

namespace agf {

constexpr int kPairConsumers = 8;
constexpr int kPairThreads = (kPairConsumers + 1) * 32;
constexpr int kPairStages = 3;
constexpr int kPairsPerCta = kPairConsumers * 32;

template <typename T>
__device__ __forceinline__ double pair_dist(const T* __restrict__ a, const T* __restrict__ b) {
  const double dx = to_f64(b[0]) - to_f64(a[0]);
  const double dy = to_f64(b[1]) - to_f64(a[1]);
  const double dz = to_f64(b[2]) - to_f64(a[2]);
  return sqrt(fma(dx, dx, fma(dy, dy, dz * dz)));
}

struct PairParams {
  const void* xyz;
  int64_t n_frames;
  int32_t n_sites;
  const int32_t* pairs;
  int64_t n_pairs;
  const double* shift;
  double* acc;
  ChunkSchedule sch;
  int32_t pair_blocks;  // ceil(n_pairs / kPairsPerCta)
  int32_t k_splits;
};

// self mode (other == xyz): staged ring
template <typename T, int KF>
__global__ void __launch_bounds__(kPairThreads, 1) pair_moments_ring_kernel(const __grid_constant__ PairParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  T* raw = reinterpret_cast<T*>(smem + 128);
  FrameRing<T, kPairStages> ring;
  ring.init(raw, bars, reinterpret_cast<const T*>(p.xyz), (int64_t)p.n_sites * 3, p.sch, kPairConsumers);
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pb = blockIdx.x % p.pair_blocks;
  const int64_t first = blockIdx.x / p.pair_blocks, step = p.k_splits;
  if (warp == kPairConsumers) {
    ring.produce(first, step);
    return;
  }
  // pairs of this CTA: [pb*256, ...); with fewer than 256 pairs several threads share a pair
  // and split the frames of each chunk between them ("slots").
  const int64_t p0 = (int64_t)pb * kPairsPerCta;
  const int np = (int)min((int64_t)kPairsPerCta, p.n_pairs - p0);
  const int slots = max(1, kPairsPerCta / np);
  const int tid = threadIdx.x;
  const int my_pair = tid % np, my_slot = tid / np;
  const bool active = my_slot < slots;
  int ia = 0, ib = 0;
  double c = 0.0;
  if (active) {
    ia = 3 * __ldg(p.pairs + 2 * (p0 + my_pair));
    ib = 3 * __ldg(p.pairs + 2 * (p0 + my_pair) + 1);
    c = __ldg(p.shift + p0 + my_pair);
  }
  double s1 = 0.0, s2 = 0.0;
  RingCursor<kPairStages> cur;
  const int64_t fstride = (int64_t)p.n_sites * 3;
  for (int64_t ch = first; ch < p.sch.n_chunks; ch += step) {
    const int nf = p.sch.count(ch);
    if (nf == 0) continue;
    mbar_wait(&ring.full[cur.stage], cur.phase);
    if (active) {
      const T* stage = ring.stage_ptr(cur.stage);
      for (int t = my_slot; t < nf; t += slots) {
        const T* fr = stage + t * fstride;
        const double d = pair_dist<T>(fr + ia, fr + ib) - c;
        s1 += d;
        s2 = fma(d, d, s2);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&ring.empty[cur.stage]);
    cur.advance();
  }
  if (active) {
    atomicAdd(p.acc + 2 * (p0 + my_pair), s1);
    atomicAdd(p.acc + 2 * (p0 + my_pair) + 1, s2);
  }
}

// cross mode / generic: direct gather from global memory
template <typename T>
__global__ void __launch_bounds__(256) pair_moments_gather_kernel(const T* __restrict__ xyz, const T* __restrict__ other,
                                                                  int64_t n_frames, int n_sites, int n_other,
                                                                  const int32_t* __restrict__ pairs, int64_t n_pairs,
                                                                  const double* __restrict__ shift,
                                                                  double* __restrict__ acc, int frames_per_cta) {
  const int64_t pidx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pidx >= n_pairs) return;
  const int64_t t0 = (int64_t)blockIdx.y * frames_per_cta;
  const int64_t t1 = min(n_frames, t0 + frames_per_cta);
  const int i = __ldg(pairs + 2 * pidx), j = __ldg(pairs + 2 * pidx + 1);
  const double c = __ldg(shift + pidx);
  double s1 = 0.0, s2 = 0.0;
  for (int64_t t = t0; t < t1; ++t) {
    const T* a = other + (t * n_other + i) * 3;
    const T* b = xyz + (t * n_sites + j) * 3;
    const double d = pair_dist<T>(a, b) - c;
    s1 += d;
    s2 = fma(d, d, s2);
  }
  atomicAdd(acc + 2 * pidx, s1);
  atomicAdd(acc + 2 * pidx + 1, s2);
}

template <typename T>
__global__ void pair_first_kernel(const T* __restrict__ xyz, const T* __restrict__ other, int n_sites, int n_other,
                                  const int32_t* __restrict__ pairs, int64_t n_pairs, double* __restrict__ shift) {
  const int64_t pidx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pidx >= n_pairs) return;
  const int i = pairs[2 * pidx], j = pairs[2 * pidx + 1];
  shift[pidx] = pair_dist<T>(other + (int64_t)i * 3, xyz + (int64_t)j * 3);
}

// all pairs over a short frame prefix.  Block = one site i of `other` x 32 sites j of `xyz` (coalesced
// reads of xyz[t, j]) x 8 frame slices: the eight warps of a block split the frames of the prefix and
// combine their (s1, s2) through shared memory, so a longer prefix costs latency, not a longer serial loop.
template <typename T>
__global__ void __launch_bounds__(256) pair_screen_kernel(const T* __restrict__ xyz, const T* __restrict__ other,
                                                          int64_t n_frames, int n_sites, int n_other, bool self,
                                                          double* __restrict__ m2) {
  __shared__ double red[2][8][32];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int i = blockIdx.y;
  const int n_jb = (n_sites + 31) / 32;
  // self pairs: only j > i is visited.  The blocks of row i walk the column blocks from the one holding i + 1
  // (a block per (i, column block) meant 785 000 blocks at 5 000 sites, half of them empty: the launch rate of
  // the blocks, not the arithmetic, set the time); block 0 of the row marks what lies to the left.
  const int first_jb = self ? (i + 1) / 32 : 0;
  if (blockIdx.x == 0) {
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    for (int j = threadIdx.x; j < min(first_jb * 32, n_sites); j += blockDim.x) m2[(int64_t)i * n_sites + j] = inf;
  }
  for (int jb = first_jb + blockIdx.x; jb < n_jb; jb += gridDim.x) {
    const int j = jb * 32 + lane;
    const bool live = j < n_sites && !(self && i >= j);
    double s1 = 0.0, s2 = 0.0;
    if (live) {
      const double c = pair_dist<T>(other + (int64_t)i * 3, xyz + (int64_t)j * 3);  // frame 0
      for (int64_t t = slice; t < n_frames; t += 8) {
        const double e = pair_dist<T>(other + (t * n_other + i) * 3, xyz + (t * n_sites + j) * 3) - c;
        s1 += e;
        s2 = fma(e, e, s2);
      }
    }
    __syncthreads();  // the previous column block's sums have been read
    red[0][slice][lane] = s1;
    red[1][slice][lane] = s2;
    __syncthreads();
    if (slice == 0 && j < n_sites) {
      double* dst = m2 + (int64_t)i * n_sites + j;
      if (!live) {
        *dst = __longlong_as_double(0x7ff0000000000000LL);
      } else {
#pragma unroll
        for (int k = 1; k < 8; ++k) {
          s1 += red[0][k][lane];
          s2 += red[1][k][lane];
        }
        *dst = s2 - s1 * s1 / (double)n_frames;
      }
    }
  }
}

// Ordered compaction of the screened pair matrix by ONE CTA (small systems: n_other * n_sites <= 2^18):
// pairs with m2 <= bound, in row-major order (what a host-side nonzero() returns, so every rank of a
// sharded run builds the same list), their frame-0 distance (the shift of the streaming pass) and
// zeroed accumulators.  count[0] = number of survivors, or -(number) when it exceeds `cap` (nothing
// beyond cap is written; the caller takes the general path).
constexpr int kSelectThreads = 1024;

template <typename T>
__global__ void __launch_bounds__(kSelectThreads) pair_select_kernel(const double* __restrict__ m2, double bound,
                                                                     const double* __restrict__ counts, int n_counts,
                                                                     const T* __restrict__ xyz0,
                                                                     const T* __restrict__ other0, int n_sites,
                                                                     int n_other, int cap, int32_t* __restrict__ pairs,
                                                                     double* __restrict__ shift,
                                                                     double* __restrict__ acc,
                                                                     int32_t* __restrict__ count) {
  __shared__ int warp_tot[kSelectThreads / 32];
  __shared__ int total_s;
  const int total = n_sites * n_other;
  const int per = (total + kSelectThreads - 1) / kSelectThreads;
  const int lo = min(total, (int)threadIdx.x * per), hi = min(total, lo + per);
  // sharded runs: `bound` holds threshold^2 and the (reduced) per-rank frame counts follow the matrix
  double b = bound;
  if (counts) {
    double total = 0.0;
    for (int r = 0; r < n_counts; ++r) total += __ldg(counts + r);
    b = bound * total * (1.0 + 1e-6) + 1e-300;
  }
  int mine = 0;
  for (int e = lo; e < hi; ++e) mine += (__ldg(m2 + e) <= b) ? 1 : 0;
  // block-wide exclusive scan of `mine`
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += v;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = warp_tot[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, w, d);
      if (lane >= d) w += v;
    }
    warp_tot[lane] = w;  // inclusive totals of warps 0..lane
    if (lane == 31) total_s = w;
  }
  __syncthreads();
  int pos = incl - mine + (warp ? warp_tot[warp - 1] : 0);
  const int n_found = total_s;
  if (threadIdx.x == 0) *count = n_found <= cap ? n_found : -n_found;
  if (n_found > cap) return;
  for (int e = lo; e < hi; ++e) {
    if (__ldg(m2 + e) <= b) {
      const int i = e / n_sites, j = e - i * n_sites;
      pairs[2 * pos] = i;
      pairs[2 * pos + 1] = j;
      shift[pos] = pair_dist<T>(other0 + (int64_t)i * 3, xyz0 + (int64_t)j * 3);
      acc[2 * pos] = 0.0;
      acc[2 * pos + 1] = 0.0;
      ++pos;
    }
  }
}

template <typename T>
static int pair_moments_typed(const void* xyz, const void* other, int64_t n_frames, int32_t n_sites, int32_t n_other,
                              const int32_t* pairs, int64_t n_pairs, const double* shift, double* acc,
                              cudaStream_t stream) {
  constexpr int KF = sizeof(T) == 4 ? 16 : 8;
  // the pairs are listed explicitly, so other == xyz (the same data) may take the self-mode ring
  const bool self = (other == nullptr || other == xyz);
  size_t stage_bytes = ((size_t)KF * n_sites * 3 * sizeof(T) + 15) / 16 * 16;
  size_t smem = 128 + kPairStages * stage_bytes;
  if (self && smem <= 200 * 1024) {
    PairParams p;
    memset(&p, 0, sizeof(p));
    p.xyz = xyz;
    p.n_frames = n_frames;
    p.n_sites = n_sites;
    p.pairs = pairs;
    p.n_pairs = n_pairs;
    p.shift = shift;
    p.acc = acc;
    p.sch = make_schedule(xyz, n_frames, (int64_t)n_sites * 3 * sizeof(T), KF);
    p.pair_blocks = (int32_t)((n_pairs + kPairsPerCta - 1) / kPairsPerCta);
    int64_t ks = (2LL * sm_count() + p.pair_blocks - 1) / p.pair_blocks;
    if (ks > p.sch.n_chunks) ks = p.sch.n_chunks;
    if (ks < 1) ks = 1;
    p.k_splits = (int32_t)ks;
    auto kern = pair_moments_ring_kernel<T, KF>;
    AGF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<p.pair_blocks * p.k_splits, kPairThreads, smem, stream>>>(p);
    AGF_CUDA_TRY(cudaGetLastError());
    return AGF_OK;
  }
  const T* o = reinterpret_cast<const T*>(self ? xyz : other);
  const int n_o = self ? n_sites : n_other;
  int bx = (int)((n_pairs + 255) / 256);
  int64_t want_y = (4LL * sm_count() + bx - 1) / bx;
  int64_t fpc = (n_frames + want_y - 1) / want_y;
  if (fpc < 64) fpc = 64;
  int by = (int)((n_frames + fpc - 1) / fpc);
  if (by > 65535) {
    by = 65535;
    fpc = (n_frames + by - 1) / by;
  }
  pair_moments_gather_kernel<T><<<dim3(bx, by), 256, 0, stream>>>(reinterpret_cast<const T*>(xyz), o, n_frames, n_sites,
                                                                 n_o, pairs, n_pairs, shift, acc, (int)fpc);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

}  // namespace agf

extern "C" int agf_pair_moments(const void* xyz, const void* other, int dtype, int64_t n_frames, int32_t n_sites,
                                int32_t n_other, const int32_t* pairs, int64_t n_pairs, const double* shift,
                                double* acc, void* stream) {
  using namespace agf;
  AGF_REQUIRE(xyz && pairs && shift && acc, "agf_pair_moments: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_pairs >= 0, "agf_pair_moments: bad sizes");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_pair_moments: bad dtype");
  if (n_frames == 0 || n_pairs == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == AGF_F32)
    return pair_moments_typed<float>(xyz, other, n_frames, n_sites, n_other, pairs, n_pairs, shift, acc, s);
  return pair_moments_typed<double>(xyz, other, n_frames, n_sites, n_other, pairs, n_pairs, shift, acc, s);
}

extern "C" int agf_pair_first(const void* xyz, const void* other, int dtype, int32_t n_sites, int32_t n_other,
                              const int32_t* pairs, int64_t n_pairs, double* shift, void* stream) {
  using namespace agf;
  AGF_REQUIRE(xyz && pairs && shift, "agf_pair_first: null pointer");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_pair_first: bad dtype");
  if (n_pairs == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const bool self = (other == nullptr || other == xyz);  // explicit pair list: the same array reads the same
  int blocks = (int)((n_pairs + 255) / 256);
  if (dtype == AGF_F32)
    pair_first_kernel<float><<<blocks, 256, 0, s>>>(reinterpret_cast<const float*>(xyz),
                                                    reinterpret_cast<const float*>(self ? xyz : other), n_sites,
                                                    self ? n_sites : n_other, pairs, n_pairs, shift);
  else
    pair_first_kernel<double><<<blocks, 256, 0, s>>>(reinterpret_cast<const double*>(xyz),
                                                     reinterpret_cast<const double*>(self ? xyz : other), n_sites,
                                                     self ? n_sites : n_other, pairs, n_pairs, shift);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

extern "C" int agf_pair_screen(const void* xyz, const void* other, int dtype, int64_t n_frames, int32_t n_sites,
                               int32_t n_other, double* m2, void* stream) {
  using namespace agf;
  AGF_REQUIRE(xyz && m2, "agf_pair_screen: null pointer");
  AGF_REQUIRE(n_frames > 0 && n_sites > 0, "agf_pair_screen: bad sizes");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_pair_screen: bad dtype");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  // self mode is other == NULL only: the same array passed as `other` is a cross-mode request, which
  // also visits the diagonal and both orders of every pair
  const bool self = other == nullptr;
  const int n_o = self ? n_sites : n_other;
  const int n_jb = (n_sites + 31) / 32;
  dim3 grid(n_jb < 8 ? n_jb : 8, n_o);  // up to eight blocks per row share its column blocks
  AGF_REQUIRE(grid.y <= 65535, "agf_pair_screen: too many sites in `other` (%d)", n_o);
  if (dtype == AGF_F32)
    pair_screen_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(xyz),
                                                   reinterpret_cast<const float*>(self ? xyz : other), n_frames,
                                                   n_sites, n_o, self, m2);
  else
    pair_screen_kernel<double><<<grid, 256, 0, s>>>(reinterpret_cast<const double*>(xyz),
                                                    reinterpret_cast<const double*>(self ? xyz : other), n_frames,
                                                    n_sites, n_o, self, m2);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

extern "C" int agf_pair_select(const double* m2, double bound, const double* counts, int32_t n_counts, const void* xyz,
                               const void* other, int dtype, int32_t n_sites, int32_t n_other, int32_t cap,
                               int32_t* pairs, double* shift, double* acc, int32_t* count, void* stream) {
  using namespace agf;
  AGF_REQUIRE(m2 && xyz && pairs && shift && acc && count, "agf_pair_select: null pointer");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_pair_select: bad dtype");
  const bool self = other == nullptr;  // as in agf_pair_screen: the same array as `other` is cross mode
  const int n_o = self ? n_sites : n_other;
  AGF_REQUIRE(n_sites > 0 && n_o > 0 && cap > 0 && (int64_t)n_sites * n_o <= (1 << 18),
              "agf_pair_select: at most 2^18 candidate pairs (got %d x %d)", n_o, n_sites);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (dtype == AGF_F32)
    pair_select_kernel<float><<<1, kSelectThreads, 0, s>>>(m2, bound, counts, n_counts, reinterpret_cast<const float*>(xyz),
                                                           reinterpret_cast<const float*>(self ? xyz : other),
                                                           n_sites, n_o, cap, pairs, shift, acc, count);
  else
    pair_select_kernel<double><<<1, kSelectThreads, 0, s>>>(m2, bound, counts, n_counts, reinterpret_cast<const double*>(xyz),
                                                            reinterpret_cast<const double*>(self ? xyz : other),
                                                            n_sites, n_o, cap, pairs, shift, acc, count);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}
