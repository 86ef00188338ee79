// Kernel (b): featurised Gram for qp_feat_linear_map with Multifeaturize([id_feat, gb_feat]).
//
// Replaces src/aggforce/qp/featlinearmap.py:361-370 of the reference together with the feature
// generators it consumes (id_feat featlinearmap.py:553-627; gb_feat jaxfeat.py:20-567), which
// materialise a (T, n_fg, n_feat) float32 tensor per bead (475 KB per frame at cln025).  Both
// feature families are one-hot in the atom's constraint group, so the atom contraction
// collapses to GROUP forces and the regression row of bead c, frame t, component d is
//     v[g]               = Fg[t,g,d]                                              g < G
//     v[G + ch*nb + k]   = g_k(d_ch) Fg[t,ch,d] + kbt m_ch g_k'(d_ch) u_ch[d]     ch < n_ch
// with d_ch = |mean position of group ch - bead position|, u_ch the unit vector, m_ch the
// group size, g_k the clipped Gaussian (jaxfeat.py:272-276) and g_k' its derivative (the
// "reorder" divergence, jaxfeat.py:544-565, with the bead held fixed).  Nothing but the
// trajectory itself is read from HBM: every CTA regenerates, in float64 and in shared memory,
// the 128-column slabs of v it needs for its 128x128 block of  P_c = sum_{t,d} v v^T  and feeds
// them to DMMA.8x8x4 (2 x 16 output tiles per warp, accumulators in registers across the CTA's
// frame range, RED.ADD.F64 at the end).
//
// Also here: agf_feat_rows (the equality-constraint rows of featlinearmap.py:446-450 for a
// handful of frames) and agf_feat_apply (application of the fitted map, featlinearmap.py:
// 512-520 + map/core.py:428-430, without materialising per-frame weights).
#include "common.cuh"
#include "i8_digits.cuh"
#include "panel.cuh"

namespace agf {

constexpr int kFgThreads = 256;
constexpr int kFgBlock = 128;   // feature columns per block
constexpr int kFgStride = 132;  // panel stride (conflict-free DMMA fragment loads)
constexpr int kFgKF = 8;        // frames per chunk -> 24 panel rows, 6 k-steps

struct FeatParams {
  const void* coords;
  const void* forces;
  int64_t n_frames;
  int32_t n_sites;
  const int32_t* grp_ptr;    // [G+1] label -> member sites (CSR)
  const int32_t* grp_sites;
  int32_t n_groups;          // G (id features)
  int32_t n_channels;        // gb channels (G or G-1: SURVEY Q5)
  const int32_t* bead_ptr;   // [n_cg+1] CSR rows of the coordinate map
  const int32_t* bead_sites;
  const double* bead_w;
  int32_t n_cg;
  const double* centers;     // [nb]
  int32_t nb;
  double inv_width;
  double clip;
  double ln_inv_clip;        // -log(clip): Gaussian is exactly 0 once z^2 exceeds it
  double kbt;
  int32_t n_feat;            // G + nb * n_channels
  int32_t n_blocks, n_pairs, k_splits;
  double* gram;              // [n_cg, n_feat, n_feat] (+=), upper block triangle
  const double* frame_w;     // [n_frames] frame weights, frame-aligned with forces (weighted Grams only)
};

template <typename T>
__device__ __forceinline__ void group_sum(const T* __restrict__ frame, const int32_t* __restrict__ ptr,
                                          const int32_t* __restrict__ sites, int g, double (&s)[3], double& m) {
  s[0] = s[1] = s[2] = 0.0;
  const int b = __ldg(ptr + g), e = __ldg(ptr + g + 1);
  for (int i = b; i < e; ++i) {
    const T* p = frame + 3 * __ldg(sites + i);
    s[0] += to_f64(__ldg(p));
    s[1] += to_f64(__ldg(p + 1));
    s[2] += to_f64(__ldg(p + 2));
  }
  m = (double)(e - b);
}

// Gaussian bin k of a distance and its derivative (jaxfeat.py:235-236, 272-276).
__device__ __forceinline__ void clipped_gauss(double d, double mu, double inv_w, double clip, double ln_inv_clip,
                                              double& g, double& gp) {
  const double z = (d - mu) * inv_w;
  const double zz = z * z;
  if (zz > ln_inv_clip + 1e-9) {  // exp(-zz) < clip: clipped to exactly zero (NaN falls through)
    g = 0.0;
    gp = 0.0;
    return;
  }
  const double e = exp(-zz);
  g = fmax(e, clip) - clip;
  gp = (e > clip) ? -2.0 * z * inv_w * e : 0.0;
  if (e != e) g = e;  // fmax drops NaN; keep it
}

// Fills panel rows (t,d) x 128 feature columns [col0, col0+128) for the chunk [t0, t0+nf).
// W: the rows of frame t are multiplied by sqrt(frame_w[t]) once complete (weighted fits).
template <typename T, bool W>
__device__ __forceinline__ void fill_feat_panel(const FeatParams& p, const T* __restrict__ coords,
                                                const T* __restrict__ forces, int64_t t0, int nf, int col0,
                                                const double (*__restrict__ bead_pos)[3], double* __restrict__ panel) {
  const int G = p.n_groups, nb = p.nb;
  const int col1 = min(col0 + kFgBlock, p.n_feat);
  // id columns of this block: [col0, min(col1, G))
  const int id_lo = min(col0, G), id_hi = min(col1, G);
  const int n_id = id_hi - id_lo;
  // gb channels intersecting the block
  int ch_lo = 0, ch_hi = 0;
  if (col1 > G) {
    ch_lo = (max(col0, G) - G) / nb;
    ch_hi = (col1 - G + nb - 1) / nb;
  }
  const int n_ch = ch_hi - ch_lo;
  const int per_frame = n_id + n_ch;
  const int64_t fstride = (int64_t)p.n_sites * 3;
  // zero padding: columns beyond n_feat, rows beyond nf
  const int width = col1 - col0;
  for (int i = threadIdx.x; i < kFgKF * 3 * kFgBlock; i += blockDim.x) {
    const int r = i / kFgBlock, x = i - r * kFgBlock;
    if (x >= width || r >= nf * 3) panel[r * kFgStride + x] = 0.0;
  }
  for (int item = threadIdx.x; item < nf * per_frame; item += blockDim.x) {
    const int t = item / per_frame, u = item - t * per_frame;
    const T* fr_f = forces + (t0 + t) * fstride;
    double* row = panel + (t * 3) * kFgStride;
    double sw = 1.0;
    if constexpr (W) sw = sqrt(__ldg(p.frame_w + t0 + t));
    if (u < n_id) {
      const int g = id_lo + u;
      double f[3], m;
      group_sum<T>(fr_f, p.grp_ptr, p.grp_sites, g, f, m);
      if constexpr (W) {
        f[0] *= sw;
        f[1] *= sw;
        f[2] *= sw;
      }
      const int x = g - col0;
      row[x] = f[0];
      row[kFgStride + x] = f[1];
      row[2 * kFgStride + x] = f[2];
    } else {
      const int ch = ch_lo + (u - n_id);
      const T* fr_c = coords + (t0 + t) * fstride;
      double f[3], pos[3], m;
      group_sum<T>(fr_f, p.grp_ptr, p.grp_sites, ch, f, m);
      group_sum<T>(fr_c, p.grp_ptr, p.grp_sites, ch, pos, m);
      const double dx = pos[0] / m - bead_pos[t][0], dy = pos[1] / m - bead_pos[t][1],
                   dz = pos[2] / m - bead_pos[t][2];
      const double dist = sqrt(dx * dx + dy * dy + dz * dz);
      const double ux = dx / dist, uy = dy / dist, uz = dz / dist;  // NaN at dist == 0 (SURVEY Q6)
      const int fbase = G + ch * nb;
      for (int k = 0; k < nb; ++k) {
        const int col = fbase + k;
        if (col < col0 || col >= col1) continue;
        double g, gp;
        clipped_gauss(dist, __ldg(p.centers + k), p.inv_width, p.clip, p.ln_inv_clip, g, gp);
        const double c = p.kbt * m * gp;
        const int x = col - col0;
        double v0 = g * f[0] + c * ux, v1 = g * f[1] + c * uy, v2 = g * f[2] + c * uz;
        if constexpr (W) {
          v0 *= sw;
          v1 *= sw;
          v2 *= sw;
        }
        row[x] = v0;
        row[kFgStride + x] = v1;
        row[2 * kFgStride + x] = v2;
      }
    }
  }
}

template <typename T>
__device__ __forceinline__ void bead_positions(const FeatParams& p, const T* __restrict__ coords, int64_t t0, int nf,
                                               int bead, double (*bead_pos)[3]) {
  const int64_t fstride = (int64_t)p.n_sites * 3;
  for (int i = threadIdx.x; i < kFgKF * 3; i += blockDim.x) {
    const int t = i / 3, d = i - t * 3;
    double s = 0.0;
    if (t < nf) {
      const T* fr = coords + (t0 + t) * fstride;
      for (int k = __ldg(p.bead_ptr + bead); k < __ldg(p.bead_ptr + bead + 1); ++k)
        s = fma(__ldg(p.bead_w + k), to_f64(__ldg(fr + 3 * __ldg(p.bead_sites + k) + d)), s);
    }
    bead_pos[t][d] = s;
  }
}

template <typename T, bool W>
__global__ void __launch_bounds__(kFgThreads, 1) feat_gram_kernel(const __grid_constant__ FeatParams p) {
  constexpr int KROWS = 3 * kFgKF;
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ double bead_pos[kFgKF][3];
  // work item: (bead, block pair, k-split)
  const int per_bead = p.n_pairs * p.k_splits;
  const int bead = blockIdx.x / per_bead;
  const int rem0 = blockIdx.x - bead * per_bead;
  const int pair = rem0 % p.n_pairs, ksplit = rem0 / p.n_pairs;
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
  const bool diag = bi == bj;
  double* panel_i = reinterpret_cast<double*>(smem);
  double* panel_j = diag ? panel_i : panel_i + KROWS * kFgStride;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const double* lane_i = panel_i + q * kFgStride + g + warp * 16;
  const double* lane_j = panel_j + q * kFgStride + g;
  double acc[2][16][2];
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;

  const T* coords = reinterpret_cast<const T*>(p.coords);
  const T* forces = reinterpret_cast<const T*>(p.forces);
  const int64_t n_chunks = (p.n_frames + kFgKF - 1) / kFgKF;
  for (int64_t c = ksplit; c < n_chunks; c += p.k_splits) {
    const int64_t t0 = c * kFgKF;
    const int nf = (int)min((int64_t)kFgKF, p.n_frames - t0);
    bead_positions<T>(p, coords, t0, nf, bead, bead_pos);
    __syncthreads();
    fill_feat_panel<T, W>(p, coords, forces, t0, nf, bi * kFgBlock, bead_pos, panel_i);
    if (!diag) fill_feat_panel<T, W>(p, coords, forces, t0, nf, bj * kFgBlock, bead_pos, panel_j);
    __syncthreads();
#pragma unroll 2
    for (int kk = 0; kk < KROWS / 4; ++kk) {
      const double a0 = lane_i[kk * 4 * kFgStride], a1 = lane_i[kk * 4 * kFgStride + 8];
#pragma unroll
      for (int cc = 0; cc < 16; ++cc) {
        const double b = lane_j[kk * 4 * kFgStride + cc * 8];
        dmma884(acc[0][cc][0], acc[0][cc][1], a0, b);
        dmma884(acc[1][cc][0], acc[1][cc][1], a1, b);
      }
    }
    __syncthreads();
  }
  double* gram = p.gram + (int64_t)bead * p.n_feat * p.n_feat;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int i = bi * kFgBlock + (warp * 2 + r) * 8 + g;
    if (i >= p.n_feat) continue;
    double* row = gram + (int64_t)i * p.n_feat;
#pragma unroll
    for (int cc = 0; cc < 16; ++cc) {
      const int j = bj * kFgBlock + cc * 8 + 2 * q;
      if (j < p.n_feat) atomicAdd(row + j, acc[r][cc][0]);
      if (j + 1 < p.n_feat) atomicAdd(row + j + 1, acc[r][cc][1]);
    }
  }
}

// ---------------------------------------------------------------------------- workspace variant
// feat_pack_kernel evaluates every regression row ONCE -- group sums, group mean positions,
// distance to the bead, clipped Gaussians and their derivative, all in float64 -- and writes it as
// packed DMMA panels  ws[chunk][bead][block][24 rows][132]  (panel.cuh); the batched panel SYRK
// (gram.cu: panel_syrk_kernel, batch = beads) then contracts them.  Against the fused kernel
// above this removes the 7x re-evaluation of every feature slab, skips the mirrored half of the
// diagonal blocks and all but one tile column of the nearly empty last block (n_feat 769 = 6*128+1).
// Phase 1 (thread per (frame, group)): group force, distance to the bead and unit vector into
// shared memory.  Phase 2 (thread per (frame, feature column)): one clipped Gaussian each, stores
// of consecutive threads fall on consecutive addresses of a panel row.
template <typename T, bool W>
__global__ void __launch_bounds__(256) feat_pack_kernel(const __grid_constant__ FeatParams p, double* __restrict__ ws) {
  extern __shared__ __align__(16) unsigned char fp_smem[];
  __shared__ double bead_pos[kPanelKF][3];
  double* s_grp = reinterpret_cast<double*>(fp_smem);  // [kPanelKF][G][8]: f[3], dist, m*u[3], pad
  const int64_t chunk = blockIdx.x / p.n_cg;
  const int bead = blockIdx.x - (int)(chunk * p.n_cg);
  const int64_t t0 = chunk * kPanelKF;
  const int nf = (int)min((int64_t)kPanelKF, p.n_frames - t0);
  const T* coords = reinterpret_cast<const T*>(p.coords);
  const T* forces = reinterpret_cast<const T*>(p.forces);
  const int64_t fstride = (int64_t)p.n_sites * 3;
  double* slab = ws + ((int64_t)chunk * p.n_cg + bead) * p.n_blocks * kPanelElems;  // [block][24][132]
  bead_positions<T>(p, coords, t0, nf, bead, bead_pos);
  // rows of frames past the end contribute nothing
  if (nf < kPanelKF) {
    const int rows0 = nf * 3, nrows = kPanelRows - rows0;
    for (int i = threadIdx.x; i < p.n_blocks * nrows * kPanelCols; i += blockDim.x) {
      const int blk = i / (nrows * kPanelCols), rem = i - blk * nrows * kPanelCols;
      const int r = rows0 + rem / kPanelCols, x = rem % kPanelCols;
      slab[(int64_t)blk * kPanelElems + r * kPanelStride + x] = 0.0;
    }
  }
  __syncthreads();
  const int G = p.n_groups, nb = p.nb;
  for (int item = threadIdx.x; item < nf * G; item += blockDim.x) {
    const int t = item / G, g = item - t * G;
    double f[3], m;
    group_sum<T>(forces + (t0 + t) * fstride, p.grp_ptr, p.grp_sites, g, f, m);
    double* rec = s_grp + (size_t)item * 8;
    rec[0] = f[0];
    rec[1] = f[1];
    rec[2] = f[2];
    if (g < p.n_channels) {
      double pos[3];
      group_sum<T>(coords + (t0 + t) * fstride, p.grp_ptr, p.grp_sites, g, pos, m);
      const double dx = pos[0] / m - bead_pos[t][0], dy = pos[1] / m - bead_pos[t][1],
                   dz = pos[2] / m - bead_pos[t][2];
      const double dist = sqrt(dx * dx + dy * dy + dz * dz);
      rec[3] = dist;
      rec[4] = m * (dx / dist);  // NaN at dist == 0 (SURVEY Q6)
      rec[5] = m * (dy / dist);
      rec[6] = m * (dz / dist);
    }
  }
  __syncthreads();
  const int n_feat = p.n_feat;
  for (int item = threadIdx.x; item < nf * n_feat; item += blockDim.x) {
    const int t = item / n_feat, col = item - t * n_feat;
    double v0, v1, v2;
    if (col < G) {
      const double* rec = s_grp + (size_t)(t * G + col) * 8;
      v0 = rec[0];
      v1 = rec[1];
      v2 = rec[2];
    } else {
      const int ch = (col - G) / nb, k = (col - G) - ch * nb;
      const double* rec = s_grp + (size_t)(t * G + ch) * 8;
      double gk, gp;
      clipped_gauss(rec[3], __ldg(p.centers + k), p.inv_width, p.clip, p.ln_inv_clip, gk, gp);
      const double c = p.kbt * gp;
      v0 = gk * rec[0] + c * rec[4];
      v1 = gk * rec[1] + c * rec[5];
      v2 = gk * rec[2] + c * rec[6];
    }
    if constexpr (W) {
      const double sw = sqrt(__ldg(p.frame_w + t0 + t));
      v0 *= sw;
      v1 *= sw;
      v2 *= sw;
    }
    double* dst = slab + (int64_t)(col >> 7) * kPanelElems + (t * 3) * kPanelStride + (col & 127);
    dst[0] = v0;
    dst[kPanelStride] = v1;
    dst[2 * kPanelStride] = v2;
  }
}

__global__ void symmetrize_batch_kernel(double* g, int n, int batch) {
  const int64_t per = (int64_t)n * n;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= per * batch) return;
  const int64_t b = idx / per, r = idx - b * per;
  const int i = (int)(r / n), j = (int)(r % n);
  if (i > j) g[idx] = g[b * per + (int64_t)j * n + i];
}

// ---------------------------------------------------------------------------- equality rows
// rows[s, c', f] = sum_a cmap[c', a] phi_c[frame_s, a, f]   (featlinearmap.py:446-450) for ONE bead c.
// phi_c[t, a, :] is one-hot: id column label(a) = 1, gb columns label(a)*nb + k = g_k(d_label(a)).
template <typename T>
__global__ void feat_rows_kernel(const FeatParams p, const int64_t* __restrict__ frames, int n_sel, int bead,
                                 const int32_t* __restrict__ label_of_site, double* __restrict__ rows) {
  const int64_t total = (int64_t)n_sel * p.n_cg;
  const T* coords = reinterpret_cast<const T*>(p.coords);
  const int64_t fstride = (int64_t)p.n_sites * 3;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(idx / p.n_cg), cp = (int)(idx - (int64_t)s * p.n_cg);
    const T* fr = coords + frames[s] * fstride;
    double bp[3] = {0, 0, 0};
    for (int k = p.bead_ptr[bead]; k < p.bead_ptr[bead + 1]; ++k)
      for (int d = 0; d < 3; ++d) bp[d] = fma(p.bead_w[k], to_f64(fr[3 * p.bead_sites[k] + d]), bp[d]);
    double* out = rows + idx * p.n_feat;
    for (int f = 0; f < p.n_feat; ++f) out[f] = 0.0;
    for (int k = p.bead_ptr[cp]; k < p.bead_ptr[cp + 1]; ++k) {
      const double w = p.bead_w[k];
      const int lab = label_of_site[p.bead_sites[k]];
      out[lab] += w;
      if (lab < p.n_channels) {
        double pos[3], m;
        group_sum<T>(fr, p.grp_ptr, p.grp_sites, lab, pos, m);
        const double dx = pos[0] / m - bp[0], dy = pos[1] / m - bp[1], dz = pos[2] / m - bp[2];
        const double dist = sqrt(dx * dx + dy * dy + dz * dz);
        for (int kb = 0; kb < p.nb; ++kb) {
          double g, gp;
          clipped_gauss(dist, p.centers[kb], p.inv_width, p.clip, p.ln_inv_clip, g, gp);
          out[p.n_groups + lab * p.nb + kb] += w * g;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------- featurised map application
// mapped[t,c,:] = sum_g (coef_c[g] + sum_k coef_c[G+g*nb+k] g_k(d_g)) Fg[t,g,:]
//               + sum_{g,k} coef_c[G+g*nb+k] m_g g_k'(d_g) u_g          (no kbt: SURVEY Q7)
template <typename T, typename TO>
__global__ void __launch_bounds__(256) feat_apply_kernel(const FeatParams p, const double* __restrict__ coefs,
                                                         TO* __restrict__ out, double* sumsq) {
  const int64_t total = p.n_frames * p.n_cg;
  const T* coords = reinterpret_cast<const T*>(p.coords);
  const T* forces = reinterpret_cast<const T*>(p.forces);
  const int64_t fstride = (int64_t)p.n_sites * 3;
  double sq = 0.0;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = idx / p.n_cg;
    const int c = (int)(idx - t * p.n_cg);
    const T* fc = coords + t * fstride;
    const T* ff = forces + t * fstride;
    const double* co = coefs + (int64_t)c * p.n_feat;
    double bp[3] = {0, 0, 0};
    for (int k = __ldg(p.bead_ptr + c); k < __ldg(p.bead_ptr + c + 1); ++k)
      for (int d = 0; d < 3; ++d) bp[d] = fma(__ldg(p.bead_w + k), to_f64(__ldg(fc + 3 * __ldg(p.bead_sites + k) + d)), bp[d]);
    double o[3] = {0, 0, 0};
    for (int g = 0; g < p.n_groups; ++g) {
      double f[3], m;
      group_sum<T>(ff, p.grp_ptr, p.grp_sites, g, f, m);
      double w = __ldg(co + g);
      if (g < p.n_channels) {
        double pos[3];
        group_sum<T>(fc, p.grp_ptr, p.grp_sites, g, pos, m);
        const double dx = pos[0] / m - bp[0], dy = pos[1] / m - bp[1], dz = pos[2] / m - bp[2];
        const double dist = sqrt(dx * dx + dy * dy + dz * dz);
        double tr = 0.0;
        for (int kb = 0; kb < p.nb; ++kb) {
          double gg, gp;
          clipped_gauss(dist, __ldg(p.centers + kb), p.inv_width, p.clip, p.ln_inv_clip, gg, gp);
          const double ck = __ldg(co + p.n_groups + g * p.nb + kb);
          w = fma(ck, gg, w);
          tr = fma(ck, gp, tr);
        }
        tr *= m;  // NaN when the group sits exactly on the bead, as in the reference (SURVEY Q6)
        o[0] += tr * (dx / dist);
        o[1] += tr * (dy / dist);
        o[2] += tr * (dz / dist);
      }
      o[0] = fma(w, f[0], o[0]);
      o[1] = fma(w, f[1], o[1]);
      o[2] = fma(w, f[2], o[2]);
    }
    for (int d = 0; d < 3; ++d) {
      out[idx * 3 + d] = static_cast<TO>(o[d]);
      const double r = (double)static_cast<TO>(o[d]);
      sq += r * r;
    }
  }
  if (sumsq) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, s);
    if ((threadIdx.x & 31) == 0) atomicAdd(sumsq, sq);
  }
}


// ------------------------------------------------------------------------------------------------
// Featurised Gram on the Blackwell tensor cores (agf_gram_feat_i8): the regression rows v (one set of n_feat
// columns per bead) go through the same int8 digit planes as the linear Gram (i8_digits.cuh, gram_i8t.cu) and the
// tiled SYRK runs batched over the beads.  feat_digits_kernel evaluates the rows exactly like feat_pack_kernel
// (float64, per-frame group records in shared memory) and either records the column maxima of a sample of frame
// groups (SAMPLE) or writes the digits.
struct FeatDigits {
  int64_t n_frames;       // frames of the slab (digits) or of the whole call (sample)
  int64_t group_stride;   // SAMPLE: frame groups between consecutive sampled groups
  int32_t n_xb;           // 16-column blocks per bead
  const double* scales;   // [n_cg][n_xb * 16]
  unsigned char* digits;  // bead-major buffers, bead_stride bytes apart
  int64_t bead_stride;
  int32_t* flags;         // [frames of the slab, rounded up to 32]
  double* gmax;           // SAMPLE: [sample group][n_cg * n_xb * 16], or NULL: ...
  unsigned long long* colmax_bits;  // ... maxima over ALL sampled groups (bits of a non-negative double), [n_cg * n_xb * 16]
};

template <typename T, bool SAMPLE>
__global__ void __launch_bounds__(256) feat_digits_kernel(const __grid_constant__ FeatParams p, const __grid_constant__ FeatDigits q) {
  extern __shared__ __align__(16) unsigned char fd_smem[];
  __shared__ double bead_pos[kPanelKF][3];
  __shared__ unsigned long long s_max[kT_PanelCols];
  unsigned char* tiles = fd_smem;                                             // 2 staging tiles (digits only)
  double* s_grp = reinterpret_cast<double*>(fd_smem + (SAMPLE ? 0 : 2 * kT_TileBytes));  // [8][G][8]: f[3], dist, m*u[3], pad
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bead = blockIdx.y;
  const int64_t fg = SAMPLE ? (int64_t)blockIdx.x * q.group_stride : (int64_t)blockIdx.x;
  const int64_t t0 = fg * kT_ItemFrames;
  const int nf = (int)max((int64_t)0, min((int64_t)kT_ItemFrames, q.n_frames - t0));
  const T* coords = reinterpret_cast<const T*>(p.coords);
  const T* forces = reinterpret_cast<const T*>(p.forces);
  const int64_t fstride = (int64_t)p.n_sites * 3;
  const int n_pad = q.n_xb * 16;
  bead_positions<T>(p, coords, t0, nf, bead, bead_pos);
  __syncthreads();
  const int G = p.n_groups, nb = p.nb;
  for (int item = threadIdx.x; item < nf * G; item += blockDim.x) {
    const int t = item / G, g = item - t * G;
    double f[3], m;
    group_sum<T>(forces + (t0 + t) * fstride, p.grp_ptr, p.grp_sites, g, f, m);
    double* rec = s_grp + (size_t)item * 8;
    rec[0] = f[0];
    rec[1] = f[1];
    rec[2] = f[2];
    if (g < p.n_channels) {
      double pos[3];
      group_sum<T>(coords + (t0 + t) * fstride, p.grp_ptr, p.grp_sites, g, pos, m);
      const double dx = pos[0] / m - bead_pos[t][0], dy = pos[1] / m - bead_pos[t][1],
                   dz = pos[2] / m - bead_pos[t][2];
      const double dist = sqrt(dx * dx + dy * dy + dz * dz);
      rec[3] = dist;
      rec[4] = m * (dx / dist);  // NaN at dist == 0 (SURVEY Q6)
      rec[5] = m * (dy / dist);
      rec[6] = m * (dz / dist);
    }
  }
  __syncthreads();
  const bool live = warp < nf;  // warp = frame of the group
  const int fb = (int)(fg >> 2), kg = (int)(fg & 3);
  int buf = 0;
  for (int pass = 0; pass < (n_pad + kT_PanelCols - 1) / kT_PanelCols; ++pass, buf ^= 1) {
    if (SAMPLE) {
      if (threadIdx.x < kT_PanelCols) s_max[threadIdx.x] = 0ull;
      __syncthreads();
    }
    uint32_t lo_w[3][4], hi_w[3][4];
    uint32_t range = 0;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      const int col = pass * kT_PanelCols + 4 * lane + cc;
      double v0 = 0.0, v1 = 0.0, v2 = 0.0;
      if (live && col < p.n_feat) {
        if (col < G) {
          const double* rec = s_grp + (size_t)(warp * G + col) * 8;
          v0 = rec[0];
          v1 = rec[1];
          v2 = rec[2];
        } else {
          const int ch = (col - G) / nb, k = (col - G) - ch * nb;
          const double* rec = s_grp + (size_t)(warp * G + ch) * 8;
          double gk, gp;
          clipped_gauss(rec[3], __ldg(p.centers + k), p.inv_width, p.clip, p.ln_inv_clip, gk, gp);
          const double c = p.kbt * gp;
          v0 = gk * rec[0] + c * rec[4];
          v1 = gk * rec[1] + c * rec[5];
          v2 = gk * rec[2] + c * rec[6];
        }
      }
      if (SAMPLE) {
        const double m = fmax(fabs(v0), fmax(fabs(v1), fabs(v2)));
        if (m > 0.0 && m < 1.0e300) atomicMax(&s_max[4 * lane + cc], (unsigned long long)__double_as_longlong(m));
      } else {
        const double sc = (live && col < p.n_feat) ? __ldg(q.scales + (size_t)bead * n_pad + col) : 0.0;
        const double t0d = fma(v0, sc, kI8Magic), t1d = fma(v1, sc, kI8Magic), t2d = fma(v2, sc, kI8Magic);
        lo_w[0][cc] = (uint32_t)__double2loint(t0d);
        hi_w[0][cc] = (uint32_t)__double2hiint(t0d);
        lo_w[1][cc] = (uint32_t)__double2loint(t1d);
        hi_w[1][cc] = (uint32_t)__double2hiint(t1d);
        lo_w[2][cc] = (uint32_t)__double2loint(t2d);
        hi_w[2][cc] = (uint32_t)__double2hiint(t2d);
        range |= (hi_w[0][cc] ^ kI8HiExpect) | (hi_w[1][cc] ^ kI8HiExpect) | (hi_w[2][cc] ^ kI8HiExpect);
      }
    }
    if (SAMPLE) {
      __syncthreads();
      if (threadIdx.x < kT_PanelCols && pass * kT_PanelCols + (int)threadIdx.x < n_pad) {
        const size_t x = (size_t)bead * n_pad + pass * kT_PanelCols + threadIdx.x;
        if (q.gmax != nullptr)
          q.gmax[(size_t)blockIdx.x * p.n_cg * n_pad + x] = __longlong_as_double((long long)s_max[threadIdx.x]);
        else if (s_max[threadIdx.x] != 0ull)
          atomicMax(q.colmax_bits + x, s_max[threadIdx.x]);
      }
      __syncthreads();
      continue;
    }
    if (__any_sync(0xffffffffu, (range & 0xFFFFFF00u) != 0) && lane == 0) q.flags[t0 + warp] = 1;
    const uint32_t tbase = smem_u32(tiles) + (uint32_t)buf * kT_TileBytes;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const uint32_t dst = tbase + (uint32_t)((d * kT_Slices) * (kT_PanelCols / 16) + (lane >> 2)) * kT_TileXb +
                           (uint32_t)(warp * 16 + (lane & 3) * 4);
      constexpr uint32_t ps = (kT_PanelCols / 16) * kT_TileXb;  // plane stride inside the tile
      sts_u32(dst + 0 * ps, gather_bytes(hi_w[d][0], hi_w[d][1], hi_w[d][2], hi_w[d][3], 0) ^ 0x80808080u);
      sts_u32(dst + 1 * ps, gather_bytes(lo_w[d][0], lo_w[d][1], lo_w[d][2], lo_w[d][3], 3) ^ 0x80808080u);
      sts_u32(dst + 2 * ps, gather_bytes(lo_w[d][0], lo_w[d][1], lo_w[d][2], lo_w[d][3], 2) ^ 0x80808080u);
      sts_u32(dst + 3 * ps, gather_bytes(lo_w[d][0], lo_w[d][1], lo_w[d][2], lo_w[d][3], 1) ^ 0x80808080u);
      sts_u32(dst + 4 * ps, gather_bytes(lo_w[d][0], lo_w[d][1], lo_w[d][2], lo_w[d][3], 0) ^ 0x80808080u);
    }
    __syncthreads();  // also: everyone has left the copy-out of the pass before the previous one (same buffer)
    const unsigned char* tile = tiles + (size_t)buf * kT_TileBytes;
    unsigned char* out = q.digits + (size_t)bead * q.bead_stride;
    for (int idx = threadIdx.x; idx < 3 * kT_Slices * (kT_PanelCols / 16) * kT_ItemFrames; idx += blockDim.x) {
      const int qq = idx & (kT_ItemFrames - 1);
      const int xb = (idx >> 3) & (kT_PanelCols / 16 - 1), ds = idx >> 6;
      const int gxb = pass * (kT_PanelCols / 16) + xb;
      if (gxb >= q.n_xb) continue;  // n_pad need not be a multiple of 128 (e.g. 288 for 200 columns)
      const uint4 v = *reinterpret_cast<const uint4*>(tile + (size_t)(ds * (kT_PanelCols / 16) + xb) * kT_TileXb + qq * 16);
      const int d = ds / kT_Slices, s = ds - d * kT_Slices;
      *reinterpret_cast<uint4*>(out + i8t_row_offset<kGramLayout>(q.n_xb, fb, d, s, gxb, kg) + qq * 16) = v;
    }
  }
}

// Column scales of the featurised rows.  id columns (group forces): the robust upper quartile of 64 sampled
// group maxima, as for the linear Gram.  gb columns  v = g_k F + kbt m g_k' u  are heavy-tailed (a distance
// wandering through the flank of a Gaussian bin changes g_k by orders of magnitude), so neither a quantile nor the
// maximum of a few hundred frames predicts their range: too little headroom sends frames to the float64 pass by
// the hundred, too much costs the gb x gb block of the Gram its precision (the dropped digit products are
// relative to the SCALES; seven spare bits showed up as 1e-6 in the fitted coefficients of an ill-conditioned
// featurised QP).  They take the maximum over EVERY FOURTH group of 8 frames (a second, denser sampling pass:
// one more evaluation of a quarter of the rows) with 4-8x headroom, capped by the a-priori bound
// |v| <= |F| + kbt m max|g'|  (|g_k| < 1, max|g'| = sqrt(2/e) / width) at the id column's range -- a frame whose
// group forces are in range can then not overflow a capped column, and a stray huge force cannot coarsen a gb
// column beyond that bound.  Columns that barely leave the clip (maximum below 2^-15 of the bound; g - clip starts
// from zero there) get a floor of 2^-12 of the bound: their absolute error stays 2^-51 of the bound.
__global__ void feat_scale_kernel(const double* __restrict__ gmax, int n_groups,
                                  const unsigned long long* __restrict__ colmax_bits, FeatParams p, int n_pad,
                                  int32_t* __restrict__ exps, double* __restrict__ scales, double* __restrict__ pow2) {
  const int x = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // warp = column
  const int lane = threadIdx.x & 31;
  const int cols = p.n_cg * n_pad;
  if (x >= cols) return;
  const int bead = x / n_pad, col = x - bead * n_pad;
  int e = 0;
  const bool live = col < p.n_feat;
  if (live) {
    const int G = p.n_groups;
    const int g = col < G ? col : (col - G) / p.nb;
    const int e_id = column_exponent_robust(i8t_group_quartile(gmax, n_groups, cols, bead * n_pad + g));
    if (col < G) {
      e = e_id;
    } else {
      const double m = (double)(__ldg(p.grp_ptr + g + 1) - __ldg(p.grp_ptr + g));
      const double bound = ldexp(1.0, e_id - 1) + p.kbt * m * 0.8577638849607068 * p.inv_width;
      const int e_cap = ilogb(bound) + 2;
      const double best = __longlong_as_double((long long)colmax_bits[x]);  // over a quarter of all frames
      e = (best > 0.0 && best < 1.0e300) ? max(min(ilogb(best) + 3, e_cap), e_cap - 12) : e_cap;
      e = e < -900 ? -900 : (e > 900 ? 900 : e);
    }
  }
  if (lane != 0) return;
  exps[x] = e;
  scales[x] = live ? ldexp(1.0, 39 - e) : 0.0;
  pow2[x] = ldexp(1.0, e - 7);
}

// Flagged frames of the featurised fit: clear their rows in every bead's planes, list the ones that exist.
__global__ void __launch_bounds__(256) feat_scrub_kernel(const int32_t* __restrict__ flags, int n_flags, int64_t n_frames,
                                                         int64_t frame0, int n_xb, int n_cg, unsigned char* __restrict__ digits,
                                                         int64_t bead_stride, int32_t* __restrict__ leftover_count,
                                                         int32_t* __restrict__ leftover) {
  const int lane = threadIdx.x & 31;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  for (int base = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32; base < n_flags; base += n_warps * 32) {
    const int mine = base + lane < n_flags ? flags[base + lane] : 0;
    uint32_t mask = __ballot_sync(0xffffffffu, mine != 0);
    while (mask) {
      const int f = base + __ffs(mask) - 1;
      mask &= mask - 1;
      const int fb = f / kT_ChunkFrames, r = f - fb * kT_ChunkFrames;
      for (int idx = lane; idx < n_cg * 3 * kT_Slices * n_xb; idx += 32) {
        const int gxb = idx % n_xb, rest = idx / n_xb;
        const int ds = rest % (3 * kT_Slices), bead = rest / (3 * kT_Slices);
        const int d = ds / kT_Slices, s = ds - d * kT_Slices;
        unsigned char* dst = digits + (size_t)bead * bead_stride + i8t_row_offset<kGramLayout>(n_xb, fb, d, s, gxb, r >> 3) + (r & 7) * 16;
        *reinterpret_cast<uint4*>(dst) = make_uint4(0, 0, 0, 0);
      }
      if (lane == 0 && f < n_frames) {
        const int slot = atomicAdd(leftover_count, 1);
        leftover[slot] = (int32_t)(frame0 + f);
      }
    }
  }
}

// Frames the fixed-point pass declined, in float64: CTA = (listed frame, bead), rank-3 update of the upper triangle.
template <typename T>
__global__ void __launch_bounds__(256) feat_leftover_kernel(const __grid_constant__ FeatParams p, const int32_t* __restrict__ count,
                                                            const int32_t* __restrict__ frames) {
  extern __shared__ double fl_v[];  // [3][n_feat]
  __shared__ double bead_pos[kPanelKF][3];
  const T* coords = reinterpret_cast<const T*>(p.coords);
  const T* forces = reinterpret_cast<const T*>(p.forces);
  const int64_t fstride = (int64_t)p.n_sites * 3;
  const int G = p.n_groups, nb = p.nb, n = *count;
  for (int item = blockIdx.x; item < n * p.n_cg; item += gridDim.x) {
    const int64_t t = frames[item / p.n_cg];
    const int bead = item % p.n_cg;
    __syncthreads();
    bead_positions<T>(p, coords, t, 1, bead, bead_pos);
    __syncthreads();
    for (int col = threadIdx.x; col < p.n_feat; col += blockDim.x) {
      const int g = col < G ? col : (col - G) / nb;
      double f[3], m, v0, v1, v2;
      group_sum<T>(forces + t * fstride, p.grp_ptr, p.grp_sites, g, f, m);
      if (col < G) {
        v0 = f[0];
        v1 = f[1];
        v2 = f[2];
      } else {
        double pos[3];
        group_sum<T>(coords + t * fstride, p.grp_ptr, p.grp_sites, g, pos, m);
        const double dx = pos[0] / m - bead_pos[0][0], dy = pos[1] / m - bead_pos[0][1], dz = pos[2] / m - bead_pos[0][2];
        const double dist = sqrt(dx * dx + dy * dy + dz * dz);
        double gk, gp;
        clipped_gauss(dist, __ldg(p.centers + (col - G - g * nb)), p.inv_width, p.clip, p.ln_inv_clip, gk, gp);
        const double c = p.kbt * gp * m;
        v0 = gk * f[0] + c * (dx / dist);
        v1 = gk * f[1] + c * (dy / dist);
        v2 = gk * f[2] + c * (dz / dist);
      }
      fl_v[col] = v0;
      fl_v[p.n_feat + col] = v1;
      fl_v[2 * p.n_feat + col] = v2;
    }
    __syncthreads();
    double* gram = p.gram + (int64_t)bead * p.n_feat * p.n_feat;
    for (int64_t e = threadIdx.x; e < (int64_t)p.n_feat * p.n_feat; e += blockDim.x) {
      const int x = (int)(e / p.n_feat), y = (int)(e - (int64_t)x * p.n_feat);
      if (y >= x)
        atomicAdd(gram + e, fl_v[x] * fl_v[y] + fl_v[p.n_feat + x] * fl_v[p.n_feat + y] +
                                fl_v[2 * p.n_feat + x] * fl_v[2 * p.n_feat + y]);
    }
  }
}

struct FeatI8Layout {
  size_t gmax, colmax, exps, scales, pow2, count, leftover, flags, digits, total;
  int64_t slab, bead_stride;
  int n_pad;
};

static FeatI8Layout feat_i8_layout(int n_feat, int n_cg, int64_t n_frames) {
  FeatI8Layout L;
  auto up = [](size_t v) { return (v + 1023) / 1024 * 1024; };
  L.n_pad = i8t_pad(n_feat);
  const size_t cols = (size_t)n_cg * L.n_pad;
  L.gmax = 0;
  L.colmax = up(cols * 8 * kT_MaxSampleGroups);
  L.exps = L.colmax + up(cols * 8);
  L.scales = L.exps + up(cols * 4);
  L.pow2 = L.scales + up(cols * 8);
  L.count = L.pow2 + up(cols * 8);
  L.leftover = L.count + 1024;
  const int64_t rounded = (n_frames + kT_ChunkFrames - 1) / kT_ChunkFrames * kT_ChunkFrames;
  L.slab = rounded < kT_SlabFrames ? rounded : kT_SlabFrames;
  L.flags = L.leftover + up((size_t)n_frames * 4);
  L.digits = L.flags + up((size_t)L.slab * 4);
  L.bead_stride = (int64_t)(L.slab / kT_ChunkFrames) * 3 * kT_Slices * (L.n_pad / 16) * kT_XbBytes;
  L.total = L.digits + (size_t)n_cg * L.bead_stride;
  return L;
}

static int fill_params(FeatParams& p, const void* coords, const void* forces, int64_t n_frames, int32_t n_sites,
                       const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups, int32_t n_channels,
                       const int32_t* bead_ptr, const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                       const double* centers, int32_t nb, double width, double clip, double kbt) {
  AGF_REQUIRE(coords && grp_ptr && grp_sites && bead_ptr && bead_sites && bead_w && centers, "feat: null pointer");
  AGF_REQUIRE(n_frames >= 0 && n_sites > 0 && n_groups > 0 && n_channels >= 0 && n_channels <= n_groups && n_cg > 0 &&
                  nb > 0 && width > 0 && clip > 0 && clip < 1,
              "feat: bad sizes/parameters");
  memset(&p, 0, sizeof(p));
  p.coords = coords;
  p.forces = forces;
  p.n_frames = n_frames;
  p.n_sites = n_sites;
  p.grp_ptr = grp_ptr;
  p.grp_sites = grp_sites;
  p.n_groups = n_groups;
  p.n_channels = n_channels;
  p.bead_ptr = bead_ptr;
  p.bead_sites = bead_sites;
  p.bead_w = bead_w;
  p.n_cg = n_cg;
  p.centers = centers;
  p.nb = nb;
  p.inv_width = 1.0 / width;
  p.clip = clip;
  p.ln_inv_clip = -log(clip);
  p.kbt = kbt;
  p.n_feat = n_groups + nb * n_channels;
  p.n_blocks = (p.n_feat + kFgBlock - 1) / kFgBlock;
  p.n_pairs = p.n_blocks * (p.n_blocks + 1) / 2;
  return AGF_OK;
}

}  // namespace agf

namespace agf {

template <typename T, bool W>
static int launch_feat_gram(const FeatParams& p, int grid, size_t smem, cudaStream_t s) {
  AGF_CUDA_TRY(cudaFuncSetAttribute(feat_gram_kernel<T, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  feat_gram_kernel<T, W><<<grid, kFgThreads, smem, s>>>(p);
  return AGF_OK;
}

// Both public forms of each Gram share one host path: frame_weights == NULL is the unweighted Gram.
static int gram_feat_impl(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                          const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups, int32_t n_channels,
                          const int32_t* bead_ptr, const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                          const double* centers, int32_t nb, double width, double clip, double kbt, double* gram,
                          const double* frame_weights, void* stream) {
  FeatParams p;
  int rc = fill_params(p, coords, forces, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                       bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt);
  if (rc) return rc;
  AGF_REQUIRE(forces && gram, "agf_gram_feat: null pointer");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_gram_feat: bad dtype");
  if (n_frames == 0) return AGF_OK;
  p.gram = gram;
  p.frame_w = frame_weights;
  const int64_t n_chunks = (n_frames + kFgKF - 1) / kFgKF;
  int64_t items = (int64_t)n_cg * p.n_pairs;
  int64_t ks = (2LL * sm_count() + items - 1) / items;
  if (ks > n_chunks) ks = n_chunks;
  if (ks < 1) ks = 1;
  p.k_splits = (int32_t)ks;
  const size_t smem = (size_t)2 * 3 * kFgKF * kFgStride * sizeof(double);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int grid = (int)(items * ks);
  if (dtype == AGF_F32)
    rc = frame_weights ? launch_feat_gram<float, true>(p, grid, smem, s) : launch_feat_gram<float, false>(p, grid, smem, s);
  else
    rc = frame_weights ? launch_feat_gram<double, true>(p, grid, smem, s)
                       : launch_feat_gram<double, false>(p, grid, smem, s);
  if (rc) return rc;
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

template <typename T, bool W>
static int launch_feat_pack(const FeatParams& p, int64_t grid, size_t smem, double* ws, cudaStream_t s) {
  AGF_CUDA_TRY(cudaFuncSetAttribute(feat_pack_kernel<T, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  feat_pack_kernel<T, W><<<(unsigned)grid, 256, smem, s>>>(p, ws);
  return AGF_OK;
}

static int gram_feat_ws_impl(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                             const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups, int32_t n_channels,
                             const int32_t* bead_ptr, const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                             const double* centers, int32_t nb, double width, double clip, double kbt, double* gram,
                             void* workspace, size_t workspace_bytes, const double* frame_weights, void* stream) {
  FeatParams p;
  int rc = fill_params(p, coords, forces, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                       bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt);
  if (rc) return rc;
  AGF_REQUIRE(forces && gram, "agf_gram_feat_ws: null pointer");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_gram_feat_ws: bad dtype");
  const int64_t per_chunk = (int64_t)n_cg * p.n_blocks * kPanelBytes;
  const size_t pack_smem = (size_t)kPanelKF * n_groups * 8 * sizeof(double);
  if (workspace == nullptr || (int64_t)workspace_bytes < per_chunk)
    return gram_feat_impl(coords, forces, dtype, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                          bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt, gram, frame_weights, stream);
  AGF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) % 16) == 0, "agf_gram_feat_ws: workspace must be 16-byte aligned");
  if (n_frames == 0) return AGF_OK;
  if (pack_smem > (size_t)200 * 1024)  // > 3200 constraint groups: per-frame records do not fit in shared memory
    return gram_feat_impl(coords, forces, dtype, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                          bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt, gram, frame_weights, stream);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int64_t slab_chunks = (int64_t)workspace_bytes / per_chunk;
  const int64_t slab_frames = slab_chunks * kPanelKF;
  const size_t elem = dtype == AGF_F32 ? 4 : 8;
  const size_t frame_bytes = (size_t)n_sites * 3 * elem;
  for (int64_t f0 = 0; f0 < n_frames; f0 += slab_frames) {
    const int64_t nf = n_frames - f0 < slab_frames ? n_frames - f0 : slab_frames;
    const int64_t chunks = (nf + kPanelKF - 1) / kPanelKF;
    p.coords = reinterpret_cast<const char*>(coords) + (size_t)f0 * frame_bytes;
    p.forces = reinterpret_cast<const char*>(forces) + (size_t)f0 * frame_bytes;
    p.frame_w = frame_weights ? frame_weights + f0 : nullptr;
    p.n_frames = nf;
    const int64_t grid = chunks * n_cg;
    AGF_REQUIRE(grid < (int64_t)1 << 31, "agf_gram_feat_ws: slab too large");
    double* ws = reinterpret_cast<double*>(workspace);
    if (dtype == AGF_F32)
      rc = frame_weights ? launch_feat_pack<float, true>(p, grid, pack_smem, ws, s)
                         : launch_feat_pack<float, false>(p, grid, pack_smem, ws, s);
    else
      rc = frame_weights ? launch_feat_pack<double, true>(p, grid, pack_smem, ws, s)
                         : launch_feat_pack<double, false>(p, grid, pack_smem, ws, s);
    if (rc) return rc;
    AGF_CUDA_TRY(cudaGetLastError());
    rc = launch_panel_syrk(reinterpret_cast<const double*>(workspace), chunks, p.n_feat, n_cg, gram, s);
    if (rc) return rc;
  }
  return AGF_OK;
}

}  // namespace agf

extern "C" int agf_gram_feat(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                             const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups,
                             int32_t n_channels, const int32_t* bead_ptr, const int32_t* bead_sites,
                             const double* bead_w, int32_t n_cg, const double* centers, int32_t nb, double width,
                             double clip, double kbt, double* gram, void* stream) {
  return agf::gram_feat_impl(coords, forces, dtype, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels,
                             bead_ptr, bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt, gram, nullptr, stream);
}

extern "C" int agf_gram_feat_weighted(const void* coords, const void* forces, int dtype, int64_t n_frames,
                                      int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                                      int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                                      const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                                      const double* centers, int32_t nb, double width, double clip, double kbt,
                                      double* gram, const double* frame_weights, void* stream) {
  return agf::gram_feat_impl(coords, forces, dtype, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels,
                             bead_ptr, bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt, gram, frame_weights,
                             stream);
}

extern "C" size_t agf_gram_feat_workspace_bytes(int32_t n_groups, int32_t n_channels, int32_t nb, int32_t n_cg,
                                                int64_t n_frames) {
  using namespace agf;
  if (n_groups <= 0 || n_channels < 0 || nb <= 0 || n_cg <= 0 || n_frames <= 0) return 0;
  const int64_t n_feat = (int64_t)n_groups + (int64_t)nb * n_channels;
  const int64_t per_chunk = (int64_t)n_cg * panel_blocks((int)n_feat) * kPanelBytes;
  const int64_t chunks = (n_frames + kPanelKF - 1) / kPanelKF;
  const int64_t cap = (int64_t)8 << 30;  // slabs of at most 8 GiB
  int64_t want = chunks * per_chunk;
  if (want > cap) want = cap / per_chunk * per_chunk;
  if (want < per_chunk) want = per_chunk;
  return (size_t)want;
}

extern "C" int agf_gram_feat_ws(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                                const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups,
                                int32_t n_channels, const int32_t* bead_ptr, const int32_t* bead_sites,
                                const double* bead_w, int32_t n_cg, const double* centers, int32_t nb, double width,
                                double clip, double kbt, double* gram, void* workspace, size_t workspace_bytes,
                                void* stream) {
  return agf::gram_feat_ws_impl(coords, forces, dtype, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels,
                                bead_ptr, bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt, gram, workspace,
                                workspace_bytes, nullptr, stream);
}

extern "C" int agf_gram_feat_ws_weighted(const void* coords, const void* forces, int dtype, int64_t n_frames,
                                         int32_t n_sites, const int32_t* grp_ptr, const int32_t* grp_sites,
                                         int32_t n_groups, int32_t n_channels, const int32_t* bead_ptr,
                                         const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                                         const double* centers, int32_t nb, double width, double clip, double kbt,
                                         double* gram, void* workspace, size_t workspace_bytes,
                                         const double* frame_weights, void* stream) {
  return agf::gram_feat_ws_impl(coords, forces, dtype, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels,
                                bead_ptr, bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt, gram, workspace,
                                workspace_bytes, frame_weights, stream);
}

extern "C" size_t agf_gram_feat_i8_workspace_bytes(int32_t n_groups, int32_t n_channels, int32_t nb, int32_t n_cg,
                                                   int64_t n_frames) {
  using namespace agf;
  if (n_groups <= 0 || n_channels < 0 || nb <= 0 || n_cg <= 0 || n_frames <= 0 || n_frames >= ((int64_t)1 << 31)) return 0;
  const int64_t n_feat = (int64_t)n_groups + (int64_t)nb * n_channels;
  if (n_feat > 8192 || (size_t)kPanelKF * n_groups * 64 + 2 * kT_TileBytes > (size_t)200 * 1024) return 0;
  return feat_i8_layout((int)n_feat, n_cg, n_frames).total;
}

extern "C" int agf_gram_feat_i8(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                                const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups, int32_t n_channels,
                                const int32_t* bead_ptr, const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                                const double* centers, int32_t nb, double width, double clip, double kbt, double* gram,
                                void* workspace, size_t workspace_bytes, void* stream) {
  using namespace agf;
  FeatParams p;
  int rc = fill_params(p, coords, forces, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                       bead_sites, bead_w, n_cg, centers, nb, width, clip, kbt);
  if (rc) return rc;
  AGF_REQUIRE(forces && gram && workspace, "agf_gram_feat_i8: null pointer");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_gram_feat_i8: bad dtype");
  const size_t need = agf_gram_feat_i8_workspace_bytes(n_groups, n_channels, nb, n_cg, n_frames);
  AGF_REQUIRE(need != 0 && workspace_bytes >= need, "agf_gram_feat_i8: shape not supported or workspace too small");
  AGF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) % 16) == 0, "agf_gram_feat_i8: workspace must be 16-byte aligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  p.gram = gram;
  const FeatI8Layout L = feat_i8_layout(p.n_feat, n_cg, n_frames);
  char* ws = reinterpret_cast<char*>(workspace);
  double* gmax = reinterpret_cast<double*>(ws + L.gmax);
  unsigned long long* colmax = reinterpret_cast<unsigned long long*>(ws + L.colmax);
  int32_t* exps = reinterpret_cast<int32_t*>(ws + L.exps);
  double* scales = reinterpret_cast<double*>(ws + L.scales);
  double* pow2 = reinterpret_cast<double*>(ws + L.pow2);
  int32_t* count = reinterpret_cast<int32_t*>(ws + L.count);
  int32_t* leftover = reinterpret_cast<int32_t*>(ws + L.leftover);
  int32_t* flags = reinterpret_cast<int32_t*>(ws + L.flags);
  unsigned char* digits = reinterpret_cast<unsigned char*>(ws + L.digits);
  const int n_xb = L.n_pad / 16, cols = n_cg * L.n_pad;
  const size_t elem = dtype == AGF_F32 ? 4 : 8;
  const size_t frame_bytes = (size_t)n_sites * 3 * elem;
  const size_t grp_smem = (size_t)kPanelKF * n_groups * 8 * sizeof(double);
  AGF_CUDA_TRY(cudaMemsetAsync(ws, 0, L.leftover, s));
  FeatDigits q;
  memset(&q, 0, sizeof(q));
  q.n_xb = n_xb;
  q.scales = scales;
  q.digits = digits;
  q.bead_stride = L.bead_stride;
  q.flags = flags;
  q.gmax = gmax;
#define AGF_FEAT_DIGITS(SAMPLE, grid, smem)                                                                       \
  do {                                                                                                            \
    if (dtype == AGF_F32) {                                                                                       \
      AGF_CUDA_TRY(cudaFuncSetAttribute(feat_digits_kernel<float, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem))); \
      feat_digits_kernel<float, SAMPLE><<<grid, 256, smem, s>>>(p, q);                                          \
    } else {                                                                                                      \
      AGF_CUDA_TRY(cudaFuncSetAttribute(feat_digits_kernel<double, SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem))); \
      feat_digits_kernel<double, SAMPLE><<<grid, 256, smem, s>>>(p, q);                                         \
    }                                                                                                             \
    AGF_CUDA_TRY(cudaGetLastError());                                                                             \
  } while (0)
  {  // column scales: up to 64 groups of 8 frames spread over the call's frames
    const int64_t all_groups = (n_frames + kT_ItemFrames - 1) / kT_ItemFrames;
    const int n_sg = (int)(all_groups < kT_MaxSampleGroups ? all_groups : kT_MaxSampleGroups);
    q.n_frames = n_frames;
    q.group_stride = all_groups / n_sg;
    AGF_FEAT_DIGITS(true, dim3(n_sg, n_cg), grp_smem);
    // the denser pass for the gb columns: every fourth group, maxima merged with atomicMax (colmax is zeroed above)
    const int64_t dense_stride = all_groups >= 8 ? 4 : 1;
    q.gmax = nullptr;
    q.colmax_bits = colmax;
    q.group_stride = dense_stride;
    AGF_FEAT_DIGITS(true, dim3((unsigned)((all_groups + dense_stride - 1) / dense_stride), n_cg), grp_smem);
    q.gmax = gmax;
    feat_scale_kernel<<<(cols + 7) / 8, 256, 0, s>>>(gmax, n_sg, colmax, p, L.n_pad, exps, scales, pow2);
    AGF_CUDA_TRY(cudaGetLastError());
  }
  const int sms = sm_count();
  for (int64_t f0 = 0; f0 < n_frames; f0 += L.slab) {
    const int64_t nf = n_frames - f0 < L.slab ? n_frames - f0 : L.slab;
    const int n_fb = (int)((nf + kT_ChunkFrames - 1) / kT_ChunkFrames);
    const int n_flags = n_fb * kT_ChunkFrames;
    p.coords = reinterpret_cast<const char*>(coords) + (size_t)f0 * frame_bytes;
    p.forces = reinterpret_cast<const char*>(forces) + (size_t)f0 * frame_bytes;
    p.n_frames = nf;
    q.n_frames = nf;
    AGF_CUDA_TRY(cudaMemsetAsync(flags, 0, (size_t)n_flags * 4, s));
    AGF_FEAT_DIGITS(false, dim3(n_fb * (kT_ChunkFrames / kT_ItemFrames), n_cg), grp_smem + 2 * kT_TileBytes);
    feat_scrub_kernel<<<(n_flags + 255) / 256 < sms ? (n_flags + 255) / 256 : sms, 256, 0, s>>>(
        flags, n_flags, nf, f0, n_xb, n_cg, digits, L.bead_stride, count, leftover);
    AGF_CUDA_TRY(cudaGetLastError());
    I8tSyrkLaunch l;
    l.digits = digits;
    l.n_chunks = 3 * n_fb;
    l.n_red = p.n_feat;
    l.slice_chunks = 0;  // default (256): measured 17.1 / 15.5 / 14.8 / 14.4 ms per 50 k frames at 32 / 64 / 128 / 256
    l.n_batch = n_cg;
    l.digits_batch_stride = L.bead_stride;
    l.pow2 = pow2;
    l.gram = gram;
    l.gram_batch_stride = (int64_t)p.n_feat * p.n_feat;
    rc = i8t_launch_syrk(l, s);
    if (rc) return rc;
  }
#undef AGF_FEAT_DIGITS
  p.coords = coords;
  p.forces = forces;
  p.n_frames = n_frames;
  const size_t lsmem = (size_t)3 * p.n_feat * sizeof(double);
  if (dtype == AGF_F32) {
    AGF_CUDA_TRY(cudaFuncSetAttribute(feat_leftover_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsmem));
    feat_leftover_kernel<float><<<sms, 256, lsmem, s>>>(p, count, leftover);
  } else {
    AGF_CUDA_TRY(cudaFuncSetAttribute(feat_leftover_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsmem));
    feat_leftover_kernel<double><<<sms, 256, lsmem, s>>>(p, count, leftover);
  }
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

extern "C" int agf_symmetrize_batch(double* gram, int32_t n, int32_t batch, void* stream) {
  using namespace agf;
  AGF_REQUIRE(gram && n > 0 && batch > 0, "agf_symmetrize_batch: bad arguments");
  const int64_t total = (int64_t)n * n * batch;
  symmetrize_batch_kernel<<<(int)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(gram, n,
                                                                                                        batch);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

extern "C" int agf_feat_rows(const void* coords, int dtype, int32_t n_sites, const int64_t* frames, int32_t n_sel,
                             int32_t bead, const int32_t* label_of_site, const int32_t* grp_ptr,
                             const int32_t* grp_sites, int32_t n_groups, int32_t n_channels,
                             const int32_t* bead_ptr, const int32_t* bead_sites, const double* bead_w, int32_t n_cg,
                             const double* centers, int32_t nb, double width, double clip, double* rows,
                             void* stream) {
  using namespace agf;
  FeatParams p;
  int rc = fill_params(p, coords, nullptr, 1, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                       bead_sites, bead_w, n_cg, centers, nb, width, clip, 0.0);
  if (rc) return rc;
  AGF_REQUIRE(frames && label_of_site && rows && n_sel > 0 && bead >= 0 && bead < n_cg, "agf_feat_rows: bad arguments");
  AGF_REQUIRE(dtype == AGF_F32 || dtype == AGF_F64, "agf_feat_rows: bad dtype");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int total = n_sel * n_cg;
  const int blocks = (total + 63) / 64;
  if (dtype == AGF_F32) feat_rows_kernel<float><<<blocks, 64, 0, s>>>(p, frames, n_sel, bead, label_of_site, rows);
  else feat_rows_kernel<double><<<blocks, 64, 0, s>>>(p, frames, n_sel, bead, label_of_site, rows);
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}

extern "C" int agf_feat_apply(const void* coords, const void* forces, int dtype, int64_t n_frames, int32_t n_sites,
                              const int32_t* grp_ptr, const int32_t* grp_sites, int32_t n_groups,
                              int32_t n_channels, const int32_t* bead_ptr, const int32_t* bead_sites,
                              const double* bead_w, int32_t n_cg, const double* centers, int32_t nb, double width,
                              double clip, const double* coefs, void* out, int out_dtype, double* sumsq,
                              void* stream) {
  using namespace agf;
  FeatParams p;
  int rc = fill_params(p, coords, forces, n_frames, n_sites, grp_ptr, grp_sites, n_groups, n_channels, bead_ptr,
                       bead_sites, bead_w, n_cg, centers, nb, width, clip, 0.0);
  if (rc) return rc;
  AGF_REQUIRE(forces && coefs && out, "agf_feat_apply: null pointer");
  AGF_REQUIRE((dtype == AGF_F32 || dtype == AGF_F64) && (out_dtype == AGF_F32 || out_dtype == AGF_F64),
              "agf_feat_apply: bad dtype");
  if (n_frames == 0) return AGF_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int64_t total = n_frames * n_cg;
  const int64_t want = (total + 255) / 256;
  const int blocks = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
#define AGF_FA(TI, TO) \
  feat_apply_kernel<TI, TO><<<blocks, 256, 0, s>>>(p, coefs, reinterpret_cast<TO*>(out), sumsq)
  if (dtype == AGF_F32 && out_dtype == AGF_F64) AGF_FA(float, double);
  else if (dtype == AGF_F32) AGF_FA(float, float);
  else if (out_dtype == AGF_F64) AGF_FA(double, double);
  else AGF_FA(double, float);
#undef AGF_FA
  AGF_CUDA_TRY(cudaGetLastError());
  return AGF_OK;
}
