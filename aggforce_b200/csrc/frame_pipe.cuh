// Frame-chunk streaming: global [n_frames, frame_elems] -> shared-memory stages via 1-D TMA
// bulk copies (cp.async.bulk + mbarrier).  Frames of a trajectory array are contiguous, so a
// chunk of KF frames is ONE contiguous span; no tensor map is needed and the 12-byte xyz
// inner extent (which rules out tiled TMA boxes, SURVEY section 7) does not matter.
//
// Alignment: bulk copies need 16-byte aligned source/size.  With frame_bytes = 12*n (f32) a
// chunk start is aligned every 4 frames, so the schedule is
//     chunk 0      = the first `head` frames (0..3) needed to reach an aligned address,
//     chunk c >= 1 = KF frames each (KF % 4 == 0), the last one possibly short.
// Chunks that are not bulk-copyable (the head, a short tail whose byte count is not a
// multiple of 16) are loaded cooperatively with plain loads; there are at most two per launch.
#pragma once
#include "common.cuh"

namespace agf {

struct ChunkSchedule {
  int64_t n_frames;
  int64_t n_chunks;  // including the (possibly empty) head chunk 0
  int32_t head;      // frames in chunk 0
  int32_t kf;        // frames per regular chunk

  __host__ __device__ int64_t start(int64_t c) const { return c == 0 ? 0 : head + (c - 1) * (int64_t)kf; }
  __host__ __device__ int32_t count(int64_t c) const {
    if (c == 0) return head;
    int64_t s = start(c);
    int64_t r = n_frames - s;
    return (int32_t)(r < kf ? (r < 0 ? 0 : r) : kf);
  }
};

// Host: builds the schedule for an array whose first frame lives at `base`.
inline ChunkSchedule make_schedule(const void* base, int64_t n_frames, int64_t frame_bytes, int kf) {
  ChunkSchedule s;
  s.n_frames = n_frames;
  s.kf = kf;
  int head = 0;
  uintptr_t a = reinterpret_cast<uintptr_t>(base);
  while (head < 16 && head < n_frames && ((a + (uintptr_t)head * (uintptr_t)frame_bytes) % 16) != 0) ++head;
  // hopeless alignment: everything cooperative.  With fewer than 16 frames the search also ends at n_frames, which
  // may be more frames than a chunk (a stage) holds.
  if (head >= 16 || head > kf) head = (int)(n_frames < kf ? n_frames : kf);
  s.head = head;
  int64_t rest = n_frames - head;
  s.n_chunks = 1 + (rest + kf - 1) / kf;
  return s;
}

template <typename T, int STAGES>
struct FrameStager {
  T* raw;               // STAGES * stage_elems
  uint64_t* full;       // STAGES mbarriers
  const T* base;        // global
  int64_t frame_elems;  // elements per frame (3 * n_sites)
  int64_t stage_elems;  // kf * frame_elems rounded up to 16 bytes
  ChunkSchedule sch;
  uint32_t phase_bits;

  __device__ void init(T* raw_, uint64_t* full_, const T* base_, int64_t frame_elems_, const ChunkSchedule& s) {
    raw = raw_;
    full = full_;
    base = base_;
    frame_elems = frame_elems_;
    sch = s;
    stage_elems = ((int64_t)s.kf * frame_elems * (int64_t)sizeof(T) + 15) / 16 * 16 / (int64_t)sizeof(T);
    phase_bits = 0;
    if (threadIdx.x == 0) {
      for (int i = 0; i < STAGES; ++i) mbar_init(&full[i], 1);
      fence_barrier_init();
    }
  }

  __device__ bool bulkable(int64_t c) const {
    if (c == 0) return false;
    int64_t bytes = (int64_t)sch.count(c) * frame_elems * (int64_t)sizeof(T);
    uintptr_t a = reinterpret_cast<uintptr_t>(base + sch.start(c) * frame_elems);
    return bytes > 0 && (bytes % 16) == 0 && (a % 16) == 0;
  }

  __device__ T* stage_ptr(int stage) const { return raw + (int64_t)stage * stage_elems; }

  // One thread: start the async copy of chunk c into `stage` (no-op for cooperative chunks).
  // The caller guarantees (via __syncthreads) that every thread finished reading the stage.
  __device__ void issue(int64_t c, int stage) {
    if (c >= sch.n_chunks || !bulkable(c)) return;
    fence_proxy_async();
    uint32_t bytes = (uint32_t)((int64_t)sch.count(c) * frame_elems * (int64_t)sizeof(T));
    mbar_expect_tx(&full[stage], bytes);
    const char* src = reinterpret_cast<const char*>(base + sch.start(c) * frame_elems);
    char* dst = reinterpret_cast<char*>(stage_ptr(stage));
    // split into <= 64 KiB pieces (all multiples of 16 bytes)
    uint32_t off = 0;
    while (off < bytes) {
      uint32_t piece = bytes - off < kBulkPiece ? bytes - off : kBulkPiece;
      tma_bulk_g2s(dst + off, src + off, piece, &full[stage]);
      off += piece;
    }
  }

  // All threads: block until chunk c is resident in `stage`.
  __device__ void wait(int64_t c, int stage) {
    if (bulkable(c)) {
      mbar_wait(&full[stage], (phase_bits >> stage) & 1u);
      phase_bits ^= (1u << stage);
    } else {
      int64_t n = (int64_t)sch.count(c) * frame_elems;
      const T* src = base + sch.start(c) * frame_elems;
      T* dst = stage_ptr(stage);
      for (int64_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
      __syncthreads();
    }
  }
};

}  // namespace agf

namespace agf {

// Producer/consumer variant: one producer warp keeps a ring of STAGES chunk buffers full,
// consumer warps signal per-stage "empty" barriers when they are done with a chunk, so
// no block-wide barrier sits between loading and computing.
template <typename T, int STAGES>
struct FrameRing {
  T* raw;
  uint64_t* full;   // STAGES, 1 arrival (+ tx bytes)
  uint64_t* empty;  // STAGES, n_consumer_warps arrivals
  const T* base;
  int64_t frame_elems;
  int64_t stage_elems;
  ChunkSchedule sch;

  __device__ static size_t barrier_bytes() { return 2 * STAGES * sizeof(uint64_t); }

  __device__ void init(T* raw_, uint64_t* bars, const T* base_, int64_t frame_elems_, const ChunkSchedule& s,
                       int n_consumer_warps) {
    raw = raw_;
    full = bars;
    empty = bars + STAGES;
    base = base_;
    frame_elems = frame_elems_;
    sch = s;
    stage_elems = ((int64_t)s.kf * frame_elems * (int64_t)sizeof(T) + 15) / 16 * 16 / (int64_t)sizeof(T);
    if (threadIdx.x == 0) {
      for (int i = 0; i < STAGES; ++i) {
        mbar_init(&full[i], 1);
        mbar_init(&empty[i], n_consumer_warps);
      }
      fence_barrier_init();
    }
  }

  __device__ T* stage_ptr(int stage) const { return raw + (int64_t)stage * stage_elems; }

  __device__ bool bulkable(int64_t c) const {
    if (c == 0) return false;
    int64_t bytes = (int64_t)sch.count(c) * frame_elems * (int64_t)sizeof(T);
    uintptr_t a = reinterpret_cast<uintptr_t>(base + sch.start(c) * frame_elems);
    return bytes > 0 && (bytes % 16) == 0 && (a % 16) == 0;
  }

  // Whole producer warp: stream chunks first, first+step, ... through the ring.
  __device__ void produce(int64_t first, int64_t step) {
    const int lane = threadIdx.x & 31;
    int stage = 0;
    uint32_t phase = 0;
    for (int64_t c = first; c < sch.n_chunks; c += step) {
      if (sch.count(c) == 0) continue;
      mbar_wait(&empty[stage], phase ^ 1u);
      if (bulkable(c)) {
        if (lane == 0) {
          fence_proxy_async();
          uint32_t bytes = (uint32_t)((int64_t)sch.count(c) * frame_elems * (int64_t)sizeof(T));
          mbar_expect_tx(&full[stage], bytes);
          const char* src = reinterpret_cast<const char*>(base + sch.start(c) * frame_elems);
          char* dst = reinterpret_cast<char*>(stage_ptr(stage));
          uint32_t off = 0;
          while (off < bytes) {
            uint32_t piece = bytes - off < kBulkPiece ? bytes - off : kBulkPiece;
            tma_bulk_g2s(dst + off, src + off, piece, &full[stage]);
            off += piece;
          }
        }
      } else {
        int64_t n = (int64_t)sch.count(c) * frame_elems;
        const T* src = base + sch.start(c) * frame_elems;
        T* dst = stage_ptr(stage);
        for (int64_t i = lane; i < n; i += 32) dst[i] = src[i];
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[stage]);
      }
      __syncwarp();
      if (++stage == STAGES) {
        stage = 0;
        phase ^= 1u;
      }
    }
  }
};

// Consumer-side cursor over the same chunk sequence.
template <int STAGES>
struct RingCursor {
  int stage = 0;
  uint32_t phase = 0;
  __device__ void advance() {
    if (++stage == STAGES) {
      stage = 0;
      phase ^= 1u;
    }
  }
};

}  // namespace agf
