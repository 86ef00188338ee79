// Kernel (a), Blackwell tensor-core path: the linear Gram through int8 slices on tcgen05 (Ozaki scheme).
//
// Same result as agf_gram_linear (src/aggforce/qp/qplinear.py:66-71 of the reference:
// P = (R C)' (R C) in float64) for float32 forces and n_red <= 97, but the contraction runs on the
// 5th-generation tensor cores, which have no float64 kind:
//   * every reduced column x gets a power-of-two scale 2^E_x from a sample of the frames; a group
//     sum v (float64, exact) becomes the 39-bit fixed-point number q = rint(v 2^(39 - E_x)) and q is
//     split into five signed 8-bit digits d_0..d_4 (most significant first).  One add and one xor
//     produce all five digits: the bytes of (q + B) ^ B with B = 0x8080808080;
//   * digit planes D_s[k][x] (k = (frame, xyz) rows) are written to shared memory in the canonical
//     MN-major no-swizzle UMMA layout; ONE thread issues tcgen05.mma.kind::i8 (M 128, N 96, K 32):
//     15 products D_s' D_t with s + t <= 4 per block of 32 rows, accumulated EXACTLY in int32 in
//     five TMEM accumulators (one per level l = s + t, 5 x 96 = 480 of the 512 columns);
//   * at the end  G[x][y] = 2^(E_x + E_y - 14) sum_l 2^(-8 l) acc_l[x][y]  in float64.  The dropped
//     products (s + t >= 5) are below 2^-40 of the column scales: 2e-12 relative Frobenius error on
//     cln025 (tools/ozaki/ozaki_numerics.py; bar 1e-9).
//   * N = 96 keeps five accumulators inside TMEM; column 96 (n_red = 97) rides along as row 96 of the
//     M = 128 operand (G is symmetric), its diagonal element is a scalar side sum.
//   * a frame with a value outside the fixed-point range (|v| >= 2^(E_x - 1), or not finite) is left
//     out of the digit planes and appended to a list; gram_leftover_kernel adds those frames in
//     float64 afterwards, so the result does not depend on the sample being representative.
// Roles in the CTA (one per SM): 16 frame warps (raw frame -> digits of its three rows), 1 load warp (1-D TMA
// ring of raw frames), 1 MMA warp (TMEM allocation, MMA issue, tcgen05.commit onto the panel barriers);
// frame warps 0-3 read the accumulators back (tcgen05.ld).  All hand-offs are mbarriers -- no block-wide
// barrier in the main loop, so the frame warps drift apart and their conversion (XU pipe), integer and
// shared-memory phases overlap instead of running in lock step.
#ifndef AGF_BULK_PIECE
#define AGF_BULK_PIECE 16384u
#endif
#include "frame_pipe.cuh"
#include "i8.cuh"

namespace agf {

constexpr int kI8Slices = 5;
constexpr int kI8M = 128, kI8N = 96, kI8K = 32;
constexpr int kI8Cols = 112;                                       // columns stored per k-row: 7 blocks of 16
constexpr int kI8BlockBytes = 144;                                 // one core matrix (8 k-rows x 16 B) + 16 B: SBO.  The
                                                                   // pad rotates the banks, so the six words a k-row
                                                                   // store writes per plane (one per block) never collide
constexpr int kI8GroupBytes = 7 * kI8BlockBytes;                   // 8 k-rows of one plane (LBO)
constexpr int kI8SubFrames = 16;                                   // frames per raw stage
constexpr int kI8PanelRows = 96;                                   // 32 frames = 3 MMA k-blocks
constexpr int kI8PlaneBytes = (kI8PanelRows / 8) * kI8GroupBytes;  // 10 752
constexpr int kI8PanelBytes = (kI8Slices * kI8PlaneBytes + kI8BlockBytes + 1023) / 1024 * 1024;  // + the block A reads past the end
constexpr int kI8RawStages = 3;
constexpr int kI8FrameWarps = 16;                    // one frame of the sub-chunk each
constexpr int kI8LoadWarp = kI8FrameWarps;            // TMA producer of the raw-frame ring
constexpr int kI8MmaWarp = kI8FrameWarps + 1;         // TMEM allocation, MMA issue
constexpr int kI8Threads = (kI8FrameWarps + 2) * 32;
constexpr int kI8MaxFramesPerCta = 8192;  // 5 products of at most 2^14 per row and level: 24 576 rows stay below 2^31
constexpr int kI8SampleFrames = 4096;
constexpr uint32_t kI8Idesc = umma_idesc_i8(kI8M, kI8N);

struct GramI8Params {
  const float* forces;
  int64_t n_frames;
  int64_t frame0;  // index of forces[0] in the caller's array (for the leftover list)
  int32_t n_sites;
  const int32_t* col_ptr;
  const int32_t* col_sites;
  int32_t n_red;
  double* gram;
  const unsigned long long* colmax_bits;  // [n_red] max |group sum| of the sample, as double bits
  int32_t* leftover_count;
  int32_t* leftover;  // frame indices
  long long* sums;    // [2][n_red][n_red] exact integer partial sums (see the epilogue), zeroed per call
  double* side_slots; // [gridDim.x][kI8FrameWarps] partial sums of the (96, 96) element
  ChunkSchedule sch;
};

__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t addr) {
  // MN blocks kI8BlockBytes apart (SBO), groups of 8 k-rows kI8GroupBytes apart (LBO)
  return umma_desc_mn_i8(addr, kI8GroupBytes, kI8BlockBytes);
}

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
  umma_i8_issue(tmem_d, da, db, kI8Idesc, accumulate);
}

// not volatile: the compiler may batch these loads (the mbarrier waits around them carry memory clobbers)
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
// byte offset of (row k, column x) inside one digit plane
__device__ __forceinline__ uint32_t plane_off(int k, int x) {
  return (uint32_t)((k >> 3) * kI8GroupBytes + (x >> 4) * kI8BlockBytes + (k & 7) * 16 + (x & 15));
}

// W0..W3: members visited for slot 0..3 of a column quad (the largest group size of that slot over all
// quads; lanes with fewer members multiply by a 0 mask).  Compile-time trip counts: straight-line fill.
template <int W0, int W1, int W2, int W3>
__global__ void __launch_bounds__(kI8Threads, 1) gram_i8_kernel(const __grid_constant__ GramI8Params p) {
  constexpr int kW[4] = {W0, W1, W2, W3};
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* panels = smem;                                       // 2 digit panels
  size_t off = (size_t)2 * kI8PanelBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + off);
  uint64_t* ring_bars = bars;                          // [2 * kI8RawStages]: raw stage full / empty
  uint64_t* panel_full = ring_bars + 2 * kI8RawStages; // [2]
  uint64_t* panel_empty = panel_full + 2;              // [2]
  uint64_t* acc_done = panel_empty + 2;                // [1]
  off += 128;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + off);
  off += 16;
  int32_t* s_exp = reinterpret_cast<int32_t*>(smem + off);       // [kI8Cols]
  off += kI8Cols * 4;
  int32_t* s_ptr = reinterpret_cast<int32_t*>(smem + off);       // CSR copy
  int32_t* s_sites = s_ptr + (p.n_red + 1);
  off += (size_t)(p.n_red + 1 + p.n_sites) * 4;
  off = (off + 127) / 128 * 128;
  float* raw = reinterpret_cast<float*>(smem + off);
  const int64_t frame_elems = (int64_t)p.n_sites * 3;

  for (int i = threadIdx.x; i <= p.n_red; i += blockDim.x) s_ptr[i] = p.col_ptr[i];
  for (int i = threadIdx.x; i < p.col_ptr[p.n_red]; i += blockDim.x) s_sites[i] = p.col_sites[i];
  for (int i = threadIdx.x; i < 2 * kI8PanelBytes / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(panels)[i] = make_uint4(0, 0, 0, 0);  // columns >= n_red and the pad stay zero
  for (int i = threadIdx.x; i < kI8Cols; i += blockDim.x) s_exp[i] = i < p.n_red ? column_exponent(p.colmax_bits[i]) : 0;
  FrameRing<float, kI8RawStages> ring;
  ring.init(raw, ring_bars, p.forces, frame_elems, p.sch, kI8FrameWarps);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&panel_full[i], 2 * kI8FrameWarps);  // every frame warp arrives once per half panel
      mbar_init(&panel_empty[i], 1);
    }
    mbar_init(acc_done, 1);
    fence_barrier_init();
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kI8MmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  fence_proxy_async();  // the zero fill above must be visible to the tensor core's reads
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *s_tmem;

  // this CTA's sub-chunks: c_j = first + j * step, skipping an empty head chunk
  const int64_t step = gridDim.x;
  int64_t first = blockIdx.x;
  if (first == 0 && p.sch.head == 0) first += step;
  const int64_t n_mine = p.sch.n_chunks > first ? (p.sch.n_chunks - first + step - 1) / step : 0;
  const int64_t n_panels = (n_mine + 1) / 2;

  if (warp == kI8MmaWarp) {
    // ------------------------------------------------ MMA warp: one thread issues
    if (lane == 0) {
      const uint32_t pbase = smem_u32(panels);
      for (int64_t pj = 0; pj < n_panels; ++pj) {
        const int pb = (int)(pj & 1);
        mbar_wait(&panel_full[pb], (uint32_t)((pj >> 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t panel = pbase + (uint32_t)pb * kI8PanelBytes;
#pragma unroll
        for (int kb = 0; kb < kI8PanelRows / kI8K; ++kb) {
          uint32_t started = (pj > 0 || kb > 0) ? 0x1Fu : 0u;  // bit l: accumulator l already holds a product
#pragma unroll
          for (int s = 0; s < kI8Slices; ++s) {
#pragma unroll
            for (int t = 0; t < kI8Slices - s; ++t) {
              const int l = s + t;
              const uint64_t da = umma_desc_mn(panel + s * kI8PlaneBytes + kb * 4 * kI8GroupBytes);
              const uint64_t db = umma_desc_mn(panel + t * kI8PlaneBytes + kb * 4 * kI8GroupBytes);
              umma_i8(tmem_base + (uint32_t)(l * kI8N), da, db, (started >> l) & 1u);
              started |= 1u << l;
            }
          }
        }
        umma_commit(&panel_empty[pb]);  // arrives when the tensor core has finished reading the panel
      }
      umma_commit(acc_done);
    }
  } else if (warp == kI8LoadWarp) {
    // ------------------------------------------------ load warp: keeps the ring of raw frames full
    ring.produce(first, step);
  } else {
    // ------------------------------------------------ frame warps.  No block-wide barrier in the loop: a warp
    // waits for its raw stage and its panel, fills the three rows of ITS frame and arrives on the two
    // mbarriers, so the warps drift apart and their conversion (XU), integer and store phases overlap.
    //
    // warp = frame of the sub-chunk; lane q owns the COLUMN QUAD 4q..4q+3 (24 quads = columns 0..95, quad 24
    // = column 96 when n_red = 97), one xyz component per pass, so the four digits of a plane form one
    // 32-bit word and every store is an STS.32.  The host orders the columns so that SLOT c of every quad
    // holds columns of similar group size (slot 0 the largest groups ... slot 3 single sites): the member
    // loop of a slot then has a warp-uniform trip count and lanes without that member multiply by a 0
    // mask -- no divergence.
    // Fixed point in ONE instruction: t = fma(v, 2^(39-E), 1.5 * 2^52 + B) holds q + B in its low 40 bits
    // (round to nearest), and its upper 24 bits are a known constant exactly when |q| is in range.
    const int n_quads = p.n_red > kI8N ? kI8N / 4 + 1 : kI8N / 4;
    // The first member is loaded without a mask.  A column with no sites (empty, or past n_red) keeps scale 0, so
    // the value it loads gives digit 0, and it loads the first listed site: a non-finite value there sends the
    // frame to the float64 pass whatever this column does.  (With the exponent of an all-zero column, -900, any
    // non-zero value would leave the fixed-point range and the frame would be added in float64 for nothing.)
    const uint32_t idle_off = s_ptr[p.n_red] > 0 ? (uint32_t)s_sites[0] * 12u : 0u;
    uint32_t moff[4][4];
    float mask[4][4];
    double scale[4];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      const int x = 4 * lane + cc;
      scale[cc] = 0.0;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        moff[cc][m] = m == 0 ? idle_off : 0u;
        mask[cc][m] = 0.f;
      }
      if (lane < n_quads && x < p.n_red) {
        const int b = s_ptr[x];
        const int n = s_ptr[x + 1] - b;
#pragma unroll
        for (int m = 0; m < 4; ++m)
          if (m < n) {
            moff[cc][m] = (uint32_t)s_sites[b + m] * 12u;
            mask[cc][m] = 1.f;
          }
        if (n > 0) scale[cc] = ldexp(1.0, 39 - s_exp[x]);
      }
    }
    const double magic = 6755399441055744.0 + 551911719040.0;  // 1.5 * 2^52 + 0x8080808080
    const uint32_t hi_expect = 0x43380000u;                    // upper word of 1.5 * 2^52 (low byte: digit 0)
    const uint32_t lane_off = (uint32_t)((lane >> 2) * kI8BlockBytes + (lane & 3) * 4);  // block and byte of x = 4 lane
    const bool side_lane = p.n_red > kI8N && lane == kI8N / 4;  // owns column 96: its diagonal element is a side sum
    double side = 0.0;
    const uint32_t frame_bytes = (uint32_t)frame_elems * 4u;
    const int t = warp;
    RingCursor<kI8RawStages> cur;
    int64_t c = first;
    for (int64_t j = 0; j < n_mine; ++j, c += step) {
      const int nf = p.sch.count(c);
      const int pb = (int)((j >> 1) & 1), half = (int)(j & 1);
      const int64_t pj = j >> 1;
      mbar_wait(&ring.full[cur.stage], cur.phase);
      if (half == 0) mbar_wait(&panel_empty[pb], (uint32_t)(((pj >> 1) & 1) ^ 1));
      const uint32_t panel = smem_u32(panels) + (uint32_t)pb * kI8PanelBytes;

      // group sums -> fixed point -> digits, written at once; a frame with a value out of range is
      // cleared again below and listed for the float64 pass (rare)
      const bool live = t < nf;
      const uint32_t fbase = smem_u32(ring.stage_ptr(cur.stage)) + (uint32_t)(live ? t : 0) * frame_bytes;
      const double live_scale = live ? 1.0 : 0.0;
      uint32_t range = 0;  // any bit above the low byte set: some value left the fixed-point range
      double sq = 0.0;
      if (lane < n_quads) {
        uint32_t lo[3][4], hi[3][4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const uint32_t a0 = fbase + moff[cc][0];
          double v0 = (double)lds_f32(a0), v1 = (double)lds_f32(a0 + 4u), v2 = (double)lds_f32(a0 + 8u);
#pragma unroll
          for (int m = 1; m < 4; ++m) {
            if (m < kW[cc]) {
              const uint32_t a = fbase + moff[cc][m];
              const float k = mask[cc][m];
              v0 += (double)(lds_f32(a) * k);
              v1 += (double)(lds_f32(a + 4u) * k);
              v2 += (double)(lds_f32(a + 8u) * k);
            }
          }
          const double sc = scale[cc] * live_scale;
          const double t0 = fma(v0, sc, magic), t1 = fma(v1, sc, magic), t2 = fma(v2, sc, magic);
          if (cc == 0) {  // q = t - magic exactly: the values the tensor core sees, so that row and column 96 agree
            const double q0 = t0 - magic, q1 = t1 - magic, q2 = t2 - magic;
            sq = fma(q0, q0, fma(q1, q1, q2 * q2));
          }
          lo[0][cc] = (uint32_t)__double2loint(t0);
          hi[0][cc] = (uint32_t)__double2hiint(t0);
          lo[1][cc] = (uint32_t)__double2loint(t1);
          hi[1][cc] = (uint32_t)__double2hiint(t1);
          lo[2][cc] = (uint32_t)__double2loint(t2);
          hi[2][cc] = (uint32_t)__double2hiint(t2);
          range |= (hi[0][cc] ^ hi_expect) | (hi[1][cc] ^ hi_expect) | (hi[2][cc] ^ hi_expect);
        }
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const int k = half * 48 + t * 3 + d;
          const uint32_t dst = panel + (uint32_t)((k >> 3) * kI8GroupBytes + (k & 7) * 16) + lane_off;
          // plane s holds digit s (most significant first) = byte 4 - s of q + B, top bit flipped (offset binary ->
          // two's complement), gathered from the four columns
          sts_u32(dst + 0 * kI8PlaneBytes, gather_bytes(hi[d][0], hi[d][1], hi[d][2], hi[d][3], 0) ^ 0x80808080u);
          sts_u32(dst + 1 * kI8PlaneBytes, gather_bytes(lo[d][0], lo[d][1], lo[d][2], lo[d][3], 3) ^ 0x80808080u);
          sts_u32(dst + 2 * kI8PlaneBytes, gather_bytes(lo[d][0], lo[d][1], lo[d][2], lo[d][3], 2) ^ 0x80808080u);
          sts_u32(dst + 3 * kI8PlaneBytes, gather_bytes(lo[d][0], lo[d][1], lo[d][2], lo[d][3], 1) ^ 0x80808080u);
          sts_u32(dst + 4 * kI8PlaneBytes, gather_bytes(lo[d][0], lo[d][1], lo[d][2], lo[d][3], 0) ^ 0x80808080u);
        }
      }
      // the raw frame has been read (its values sit in the digits): hand the stage back to the load warp
      const bool ovf = __any_sync(0xffffffffu, (range & 0xFFFFFF00u) != 0);
      if (lane == 0) mbar_arrive(&ring.empty[cur.stage]);
      if (ovf) {  // warp-uniform: this warp's frame goes to the float64 pass; clear its rows, list it
        __syncwarp();
        for (int i = lane; i < kI8Slices * 3 * (kI8Cols / 4); i += 32) {
          const int sidx = i / (3 * (kI8Cols / 4)), r = i - sidx * 3 * (kI8Cols / 4);
          const int d = r / (kI8Cols / 4), x = 4 * (r - d * (kI8Cols / 4));
          sts_u32(panel + sidx * kI8PlaneBytes + plane_off(half * 48 + t * 3 + d, x), 0u);
        }
        if (live && lane == 0) {
          const int slot = atomicAdd(p.leftover_count, 1);
          p.leftover[slot] = (int32_t)(p.frame0 + p.sch.start(c) + t);
        }
      } else if (side_lane) {
        side += sq;
      }
      const bool tail_half = half == 0 && j == n_mine - 1;  // odd number of sub-chunks: the other half stays empty
      if (tail_half) {
        for (int i = lane; i < kI8Slices * 3 * (kI8Cols / 4); i += 32) {
          const int sidx = i / (3 * (kI8Cols / 4)), r = i - sidx * 3 * (kI8Cols / 4);
          const int d = r / (kI8Cols / 4), x = 4 * (r - d * (kI8Cols / 4));
          sts_u32(panel + sidx * kI8PlaneBytes + plane_off(48 + t * 3 + d, x), 0u);
        }
      }
      fence_proxy_async();  // digit stores (generic proxy) -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&panel_full[pb]);
        if (tail_half) mbar_arrive(&panel_full[pb]);
      }
      cur.advance();
    }

    // ------------------------------------------------ epilogue: fill warps 0..3 own TMEM lanes 32 w .. 32 w + 31
    if (warp < 4 && n_panels > 0) {
      mbar_wait(acc_done, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int x = warp * 32 + lane;
      for (int c0 = 0; c0 < kI8N; c0 += 16) {
        // The CTA's int32 accumulators are EXACT, and so are integer sums over CTAs and launches: the levels are
        // packed into two int64 per element -- hi = 2^8 acc_0 + acc_1, lo = 2^16 acc_2 + 2^8 acc_3 + acc_4 -- and
        // added with integer atomics, whose result does not depend on the order.  gram_i8_finalize_kernel turns
        // them into float64 once per call: the Gram is bit-identical from run to run.
        long long hi[16], lo[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) hi[i] = lo[i] = 0;
#pragma unroll
        for (int l = 0; l < kI8Slices; ++l) {
          uint32_t r[16];
          const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(l * kI8N + c0);
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
              "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
              : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
              : "r"(taddr));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const long long a = (long long)(int32_t)r[i];
            if (l < 2) hi[i] = hi[i] * 256 + a;
            else lo[i] = lo[i] * 256 + a;
          }
        }
        if (x < p.n_red) {
          const int64_t nn = (int64_t)p.n_red * p.n_red;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int y = c0 + i;
            if (y >= p.n_red) continue;
            int64_t e;
            if (x < kI8N) {
              if (y < x) continue;
              e = (int64_t)x * p.n_red + y;
            } else {
              e = (int64_t)y * p.n_red + x;  // row 96 of the operand = column 96 of the Gram
            }
            atomicAdd(reinterpret_cast<unsigned long long*>(p.sums + e), (unsigned long long)hi[i]);
            atomicAdd(reinterpret_cast<unsigned long long*>(p.sums + nn + e), (unsigned long long)lo[i]);
          }
        }
      }
    }
    if (side_lane) p.side_slots[blockIdx.x * kI8FrameWarps + warp] += side;  // this warp's slot: plain add
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == kI8MmaWarp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base));
}

// Integer partial sums -> float64, once per call (thread = element of the upper triangle).  The LAST block sums the
// per-warp side slots of the (96, 96) element in a fixed order (strided partial sums per thread, then thread 0 over
// the 256 partials): deterministic like the rest.
__global__ void __launch_bounds__(256) gram_i8_finalize_kernel(const long long* __restrict__ sums,
                                                               const double* __restrict__ side_slots, int n_slots,
                                                               const unsigned long long* __restrict__ colmax_bits,
                                                               int n_red, double* __restrict__ gram) {
  if (blockIdx.x == gridDim.x - 1) {
    if (n_red <= kI8N) return;
    __shared__ double part[256];
    double acc = 0.0;
    for (int i = threadIdx.x; i < n_slots; i += 256) acc += side_slots[i];
    part[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double side = 0.0;
      for (int i = 0; i < 256; ++i) side += part[i];
      gram[(int64_t)kI8N * n_red + kI8N] += ldexp(side, 2 * column_exponent(colmax_bits[kI8N]) - 78);
    }
    return;
  }
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_red * n_red) return;
  const int x = e / n_red, y = e - x * n_red;
  if (y < x || (x == kI8N && y == kI8N)) return;
  const int ex = column_exponent(colmax_bits[x]), ey = column_exponent(colmax_bits[y]);
  const double g = (double)sums[e] * (1.0 / 256.0) + (double)sums[(int64_t)n_red * n_red + e] * (1.0 / 4294967296.0);
  gram[e] += ldexp(g, ex + ey - 14);
}

// Column maxima of the group sums over a sample of frames (thread = (frame, column)).
__global__ void __launch_bounds__(256) gram_i8_sample_kernel(const float* __restrict__ forces, int64_t n_frames, int n_sites,
                                                             const int32_t* __restrict__ col_ptr,
                                                             const int32_t* __restrict__ col_sites, int n_red,
                                                             unsigned long long* __restrict__ colmax_bits) {
  const int64_t total = n_frames * n_red;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = idx / n_red;
    const int x = (int)(idx - t * n_red);
    const float* fr = forces + t * (int64_t)n_sites * 3;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
    for (int m = __ldg(col_ptr + x); m < __ldg(col_ptr + x + 1); ++m) {
      const float* q = fr + 3 * __ldg(col_sites + m);
      s0 += (double)__ldg(q);
      s1 += (double)__ldg(q + 1);
      s2 += (double)__ldg(q + 2);
    }
    const double m = fmax(fabs(s0), fmax(fabs(s1), fabs(s2)));
    if (m < 1.0e300) atomicMax(colmax_bits + x, (unsigned long long)__double_as_longlong(m));  // bits of x >= 0 order like x
  }
}

// Frames the fixed-point pass declined: exact float64 rank-3 updates of the upper triangle.
__global__ void __launch_bounds__(256) gram_leftover_kernel(const float* __restrict__ forces, int64_t frame0, int n_sites,
                                                            const int32_t* __restrict__ col_ptr,
                                                            const int32_t* __restrict__ col_sites, int n_red,
                                                            const int32_t* __restrict__ count,
                                                            const int32_t* __restrict__ frames, double* __restrict__ gram) {
  __shared__ double v[3][128];
  const int n = *count;
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    const float* fr = forces + ((int64_t)frames[i] - frame0) * (int64_t)n_sites * 3;
    __syncthreads();
    for (int x = threadIdx.x; x < n_red; x += blockDim.x) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
      for (int m = col_ptr[x]; m < col_ptr[x + 1]; ++m) {
        const float* q = fr + 3 * col_sites[m];
        s0 += (double)q[0];
        s1 += (double)q[1];
        s2 += (double)q[2];
      }
      v[0][x] = s0;
      v[1][x] = s1;
      v[2][x] = s2;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < n_red * n_red; e += blockDim.x) {
      const int x = e / n_red, y = e - x * n_red;
      if (y >= x) atomicAdd(gram + e, v[0][x] * v[0][y] + v[1][x] * v[1][y] + v[2][x] * v[2][y]);
    }
  }
}

constexpr int kI8SideSlots = 1024 * kI8FrameWarps;  // (CTA, frame warp) slots of the (96, 96) side sum: up to 1 024 SMs
static size_t i8_ws_sums_offset(int64_t n_frames) { return (1024 + (size_t)n_frames * sizeof(int32_t) + 15) / 16 * 16; }

static size_t gram_i8_smem(int n_sites, int n_red) {
  size_t off = (size_t)2 * kI8PanelBytes + 128 + 16 + kI8Cols * 4 + (size_t)(n_red + 1 + n_sites) * 4;
  off = (off + 127) / 128 * 128;
  const size_t stage = ((size_t)kI8SubFrames * n_sites * 12 + 15) / 16 * 16;
  return off + kI8RawStages * stage;
}

}  // namespace agf

extern "C" size_t agf_gram_linear_i8_workspace_bytes(int32_t n_sites, int32_t n_red, int64_t n_frames) {
  using namespace agf;
  if (n_red < 1 || n_red > kI8N + 1 || n_frames < 1 || n_frames >= ((int64_t)1 << 31)) return 0;
  if (gram_i8_smem(n_sites, n_red) > (size_t)226 * 1024) return 0;
  return i8_ws_sums_offset(n_frames) + (size_t)2 * n_red * n_red * sizeof(long long) + kI8SideSlots * sizeof(double);
}

extern "C" int agf_gram_linear_i8(const void* forces, int dtype, int64_t n_frames, int32_t n_sites, const int32_t* col_ptr,
                                  const int32_t* col_sites, int32_t n_red, int32_t max_group, uint32_t slot_members,
                                  double* gram, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace agf;
  AGF_REQUIRE(forces && col_ptr && col_sites && gram && workspace, "agf_gram_linear_i8: null pointer");
  AGF_REQUIRE(dtype == AGF_F32, "agf_gram_linear_i8: float32 forces only (float64 input takes agf_gram_linear)");
  AGF_REQUIRE(n_red >= 1 && n_red <= kI8N + 1 && max_group >= 1 && max_group <= 4,
              "agf_gram_linear_i8: needs n_red <= %d and constraint groups of at most 4 sites (got %d, %d)", kI8N + 1, n_red,
              max_group);
  const size_t need = agf_gram_linear_i8_workspace_bytes(n_sites, n_red, n_frames);
  AGF_REQUIRE(need != 0 && workspace_bytes >= need, "agf_gram_linear_i8: shape not supported or workspace too small");
  AGF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) % 16) == 0, "agf_gram_linear_i8: workspace must be 16-byte aligned");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  unsigned long long* colmax = reinterpret_cast<unsigned long long*>(workspace);  // [128]
  int32_t* count = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(workspace) + 1024 - 16);
  int32_t* leftover = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(workspace) + 1024);
  long long* sums = reinterpret_cast<long long*>(reinterpret_cast<char*>(workspace) + i8_ws_sums_offset(n_frames));
  double* side_slots = reinterpret_cast<double*>(sums + (size_t)2 * n_red * n_red);
  AGF_CUDA_TRY(cudaMemsetAsync(workspace, 0, 1024, s));
  AGF_CUDA_TRY(cudaMemsetAsync(sums, 0, (size_t)2 * n_red * n_red * sizeof(long long) +
                                            (size_t)sm_count() * kI8FrameWarps * sizeof(double), s));
  const float* f = reinterpret_cast<const float*>(forces);
  const int64_t sample = n_frames < kI8SampleFrames ? n_frames : kI8SampleFrames;
  gram_i8_sample_kernel<<<(int)((sample * n_red + 255) / 256), 256, 0, s>>>(f, sample, n_sites, col_ptr, col_sites, n_red,
                                                                         colmax);
  AGF_CUDA_TRY(cudaGetLastError());
  const size_t smem = gram_i8_smem(n_sites, n_red);
  // members visited per quad slot: the caller passes them packed in max_group's upper bytes
  // (slot c in bits 8 (c + 1) .. 8 (c + 1) + 7); 0 = unknown -> visit max_group members everywhere
  const int w0 = (slot_members >> 0) & 0xff, w1 = (slot_members >> 8) & 0xff, w2 = (slot_members >> 16) & 0xff,
            w3 = (slot_members >> 24) & 0xff;
  void (*kern)(GramI8Params) = gram_i8_kernel<4, 4, 4, 4>;
  if (w0 >= 1 && w0 <= 4 && w1 == 2 && w2 == 2 && w3 == 1) kern = gram_i8_kernel<4, 2, 2, 1>;
  else if (w0 == 1 && w1 == 1 && w2 == 1 && w3 == 1) kern = gram_i8_kernel<1, 1, 1, 1>;
  else if (w0 >= 1 && w0 <= 2 && w1 >= 1 && w1 <= 2 && w2 >= 1 && w2 <= 2 && w3 >= 1 && w3 <= 2) kern = gram_i8_kernel<2, 2, 2, 2>;
  AGF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int sms = sm_count();
  AGF_REQUIRE(sms * kI8FrameWarps <= kI8SideSlots, "agf_gram_linear_i8: more SMs than side slots");
  const int64_t slab = (int64_t)sms * kI8MaxFramesPerCta;  // int32 accumulators: bounded rows per CTA and launch
  for (int64_t f0 = 0; f0 < n_frames; f0 += slab) {
    GramI8Params p;
    memset(&p, 0, sizeof(p));
    p.n_frames = n_frames - f0 < slab ? n_frames - f0 : slab;
    p.forces = f + f0 * (int64_t)n_sites * 3;
    p.frame0 = f0;
    p.n_sites = n_sites;
    p.col_ptr = col_ptr;
    p.col_sites = col_sites;
    p.n_red = n_red;
    p.gram = gram;
    p.colmax_bits = colmax;
    p.leftover_count = count;
    p.leftover = leftover;
    p.sums = sums;
    p.side_slots = side_slots;
    p.sch = make_schedule(p.forces, p.n_frames, (int64_t)n_sites * 12, kI8SubFrames);
    const int64_t want = (p.sch.n_chunks + 1) / 2;
    const int ctas = (int)(want < sms ? (want < 1 ? 1 : want) : sms);
    kern<<<ctas, kI8Threads, smem, s>>>(p);
    AGF_CUDA_TRY(cudaGetLastError());
  }
  gram_i8_finalize_kernel<<<(n_red * n_red + 255) / 256 + 1, 256, 0, s>>>(sums, side_slots, sms * kI8FrameWarps, colmax, n_red, gram);
  AGF_CUDA_TRY(cudaGetLastError());
  gram_leftover_kernel<<<sms, 256, 0, s>>>(f, 0, n_sites, col_ptr, col_sites, n_red, count, leftover, gram);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}
