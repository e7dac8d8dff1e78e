// kernels.cuh — CUDA kernels of the Harmony hot loop (sm_100a).  FFMA generation ("v1"): every
// contraction is a shared-memory-tiled fp32 kernel; they double as the in-repo correctness anchor
// for the tcgen05 versions.
//
// Device data layout (all fp32, row-major, one row per cell; cells are stored sorted by their joint
// covariate tuple so that a tile of consecutive cells shares its levels):
//   Zo[n][d]  original embedding (Z_orig, harmony.h:50)     Zc[n][d]  corrected embedding (Z_corr)
//   U [n][K]  logits -dist/sigma of the current centroids    R [n][K]  soft assignments
//   Y [K][d]  centroids                                       O,E[B][K] observed / expected counts
// The reference's dist_mat (K x N, harmony.h:64) is never materialised: dist = -sigma*U.
#pragma once
#include "common.cuh"

namespace hb {

constexpr int TM = 64;           // cells per tile in every tiled kernel
constexpr int ASSIGN_THREADS = 256;
constexpr int ROW_THREADS = 256;  // 8 warps, one row per warp at a time
constexpr int NWARP = ROW_THREADS / 32;

// ------------------------------------------------------------------------------------------------
// setup helpers
// ------------------------------------------------------------------------------------------------
// dst[dst_row[r0 + r]][c] = (float)src[r * src_rs + c * src_cs]   (double / float -> float conversion of
// harmony.cpp:41 fused with the scatter into tuple-sorted order).  Strides in elements: (cols, 1) for the host path's
// staging rows, any pair for a caller's device tensor; consecutive threads walk the source's smaller stride.
template <typename T>
__global__ void k_upload_rows(const T* __restrict__ src, int64_t src_rs, int64_t src_cs, float* __restrict__ dst,
                              const int* __restrict__ dst_row, int64_t r0, int64_t rows, int cols, int ld) {
  const bool along_row = src_cs <= src_rs;
  int64_t total = rows * cols;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t r;
    int c;
    if (along_row) {
      r = idx / cols;
      c = (int)(idx - r * cols);
    } else {
      c = (int)(idx / rows);
      r = idx - (int64_t)c * rows;
    }
    dst[(int64_t)dst_row[r0 + r] * ld + c] = (float)src[r * src_rs + (int64_t)c * src_cs];
  }
}
// out[r * out_ld + c] = (T) src[src_row[r0 + r]][c]   (conv_to<RMAT>::from of harmony.cpp:640-650 + un-sort).  T = double:
// the host path's staging rows; T = float: its threaded variant (the host workers widen while they scatter) and
// device outputs of either type.
template <typename T>
__global__ void k_download_rows(const float* __restrict__ src, T* __restrict__ out, int64_t out_ld,
                                const int* __restrict__ src_row, int64_t r0, int64_t rows, int cols, int ld) {
  int64_t total = rows * cols;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = idx / cols;
    int c = (int)(idx - r * cols);
    out[r * out_ld + c] = (T)src[(int64_t)src_row[r0 + r] * ld + c];
  }
}
// Legacy centroid step (harmony.cpp:235-238, commented out in 2.0.4): Y_k = normalise(sum_i R_ik z_i) from the
// per-tuple sums S[q][k][0..d) of the statistics kernels run on Z_corr.  One block per cluster.
__global__ void k_centroids_from_stats(const float* __restrict__ S, float* __restrict__ Y, int J, int K, int d) {
  extern __shared__ float ysum[];  // [d]
  const int k = blockIdx.x, D1 = d + 1;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float t = 0.f;
    for (int q = 0; q < J; ++q) t += S[((size_t)q * K + k) * D1 + c];
    ysum[c] = t;
  }
  __syncthreads();
  float ss = 0.f;
  for (int c = 0; c < d; ++c) ss += ysum[c] * ysum[c];  // every thread: d is small
  float nrm = sqrtf(ss);
  if (nrm == 0.f) nrm = 1.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) Y[(size_t)k * d + c] = ysum[c] / nrm;
}
__global__ void k_fill_f(float* __restrict__ out, int64_t n, float v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = v;
}
// compact a padded [rows][ld] table into [rows][cols]
__global__ void k_compact(const float* __restrict__ src, float* __restrict__ out, int rows, int cols, int ld) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < rows * cols) out[idx] = src[(idx / cols) * ld + (idx % cols)];
}
__global__ void k_expand(const float* __restrict__ src, float* __restrict__ out, int rows, int cols, int ld) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < rows * cols) out[(idx / cols) * ld + (idx % cols)] = src[idx];
}

// arma::normalise(X, 2, 0) on the rows of X[n][d] (= columns of the reference's d x N matrix); a zero
// norm divides by 1.  One warp per row.  dst may alias src.
__global__ void k_normalise_rows(const float* __restrict__ src, float* __restrict__ dst, int64_t n, int d, int ld) {
  int lane = threadIdx.x & 31;
  int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = w; r < n; r += nw) {
    const float* x = src + r * ld;
    float s = 0.f;
    for (int c = lane; c < d; c += 32) {
      float v = x[c];
      s += v * v;
    }
    s = warp_sum(s);
    float nrm = sqrtf(s);
    if (nrm == 0.f) nrm = 1.f;
    for (int c = lane; c < d; c += 32) dst[r * ld + c] = x[c] / nrm;
  }
}

// ------------------------------------------------------------------------------------------------
// native k-means initialisation (stand-in for kmeans_centers, utils.cpp:10-64; outside the timed loop)
// ------------------------------------------------------------------------------------------------
// initialize_centroids (utils.cpp:10-49).  The reference draws K start cells floor(u N'), N' = N - 1, and then,
// for every centroid i in turn, replaces it by the cell j that minimises -log(u_ij) / |2 (1 - y_i . x_j)| (a race of
// exponentials: cell j wins with probability proportional to its distance from the START cell i), skipping cells
// that were already taken.  R's random stream cannot be replayed; here u is a keyed hash of (seed, i, global cell),
// so the rule itself is the reference's and tests replay it exactly (tests/numpy_restatement.py).
__host__ __device__ __forceinline__ float kmeans_uniform(uint64_t seed, uint64_t i, uint64_t g) {
  const uint64_t h = hb_mix64(seed ^ hb_mix64((i << 40) ^ g ^ 0x6b6d2b2b00000000ull));
  return ((float)(h >> 40) + 0.5f) * (1.0f / 16777216.0f);  // 24 random bits, strictly inside (0, 1)
}
// Y[k] <- the (cosine-normalised) cell with GLOBAL index cells[k]; each rank writes the rows it owns, the rest
// stay 0 (the caller zeroes Y and all-reduces it).  only >= 0: just that centroid.
__global__ void k_kmeans_gather(const float* __restrict__ Zc, const int* __restrict__ inv_sort, float* __restrict__ Y,
                                const int64_t* __restrict__ cells, int K, int d, int DS, int64_t cell_offset,
                                int64_t n_local, int only) {
  const int k = blockIdx.x;
  if (k >= K || (only >= 0 && k != only)) return;
  const int64_t l = cells[k] - cell_offset;
  if (l < 0 || l >= n_local) return;
  const float* z = Zc + (size_t)inv_sort[l] * DS;
  for (int c = threadIdx.x; c < d; c += blockDim.x) Y[(size_t)k * d + c] = z[c];
}
// One pass over the local cells: best[i] = min over cells of (float bits of -log(u_ij) / dist_ij) << 32 | global cell
// for the centroids i in [i0, i1) (all values are >= 0, so the bit patterns order like the floats; ties go to the
// smaller cell index).  Cells listed in `taken` (ntaken global indices) do not take part.  Thread per cell, start
// centroids in shared memory.
__global__ void __launch_bounds__(128) k_kmeans_race(const float* __restrict__ Zc, const int* __restrict__ sort_perm,
                                                     const float* __restrict__ Y, unsigned long long* __restrict__ best,
                                                     const int64_t* __restrict__ taken, int ntaken, int64_t n, int K, int d,
                                                     int DS, int64_t cell_offset, uint64_t seed, int i0, int i1) {
  extern __shared__ __align__(16) float smem[];
  float* Ys = smem;  // [i1 - i0][d]
  for (int i = threadIdx.x; i < (i1 - i0) * d; i += blockDim.x) Ys[i] = Y[(size_t)i0 * d + i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = blockIdx.x * (int64_t)blockDim.x; base < n; base += stride) {  // whole warps stay in the loop
    const int64_t s = base + threadIdx.x;
    const bool on = s < n;
    const float* z = Zc + (size_t)(on ? s : 0) * DS;
    const uint64_t g = (uint64_t)(cell_offset + (on ? sort_perm[s] : 0));
    bool free_cell = on;
    for (int e = 0; e < ntaken && free_cell; ++e) free_cell = (uint64_t)taken[e] != g;
    for (int i = i0; i < i1; ++i) {
      const float* y = Ys + (size_t)(i - i0) * d;
      float acc = 0.f;
      for (int c = 0; c < d; ++c) acc = fmaf(z[c], y[c], acc);
      const float dist = fabsf(2.f * (1.f - acc));
      const float p = -logf(kmeans_uniform(seed, (uint64_t)i, g)) / dist;  // dist == 0: +inf, never the minimum
      unsigned long long key = free_cell ? (((unsigned long long)__float_as_uint(p) << 32) | (unsigned long long)(g & 0xffffffffull))
                                         : 0xffffffffffffffffull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other < key ? other : key;
      }
      if (lane == 0 && key != 0xffffffffffffffffull) atomicMin(best + i, key);
    }
  }
}
// ---- the same two steps fed by tensor-core logits U[i][k] = 2 (z_i . y_k - 1) (k_logits_tc with sigma = 1) ----
// Race of initialize_centroids from the logits of the START cells: |U[i][k]| is the distance |2 (1 - y_k . x_i)| of
// utils.cpp:27.  One warp per row (lane l owns the 16-byte pieces l, l + 32, ..), running minima per column in
// registers, one atomicMin per column and warp at the end.  Centroids outside [i0, i1) and cells in `taken` sit out.
template <int NV>
__global__ void __launch_bounds__(256) k_kmeans_race_u(const float* __restrict__ U, const int* __restrict__ sort_perm,
                                                       unsigned long long* __restrict__ best, const int64_t* __restrict__ taken,
                                                       int ntaken, int64_t n, int K, int KS, int64_t cell_offset, uint64_t seed,
                                                       int i0, int i1) {
  const int lane = threadIdx.x & 31;
  const int64_t gw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int KS4 = KS >> 2;
  unsigned long long mn[NV][4];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int c = 0; c < 4; ++c) mn[v][c] = ~0ull;
  for (int64_t s = gw; s < n; s += nw) {
    const uint64_t g = (uint64_t)(cell_offset + sort_perm[s]);
    bool free_cell = true;
    for (int e = 0; e < ntaken && free_cell; ++e) free_cell = (uint64_t)taken[e] != g;
    if (!free_cell) continue;  // warp-uniform
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      if (lane + 32 * v >= KS4) continue;
      const float4 u = ld_stream4(reinterpret_cast<const float4*>(U + (size_t)s * KS) + lane + 32 * v);
      const float uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int i = 4 * (lane + 32 * v) + c;
        if (i >= i0 && i < i1 && i < K) {
          const float p = -logf(kmeans_uniform(seed, (uint64_t)i, g)) / fabsf(uu[c]);  // dist == 0: +inf, never the minimum
          const unsigned long long key = ((unsigned long long)__float_as_uint(p) << 32) | (unsigned long long)(g & 0xffffffffull);
          mn[v][c] = key < mn[v][c] ? key : mn[v][c];
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int i = 4 * (lane + 32 * v) + c;
      if (i < K && mn[v][c] != ~0ull) atomicMin(best + i, mn[v][c]);
    }
}
// |y_k|^2 of the current means
__global__ void k_kmeans_norms(const float* __restrict__ Y, float* __restrict__ yy, int K, int d) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  float s = 0.f;
  for (int c = 0; c < d; ++c) s = fmaf(Y[(size_t)k * d + c], Y[(size_t)k * d + c], s);
  yy[k] = s;
}
// Lloyd assignment from the logits: nearest mean in Euclidean distance = argmax_k (2 z.y_k - |y_k|^2) = argmax_k
// (U[i][k] - |y_k|^2) (ties: the lower k), written as a one-hot row of R — the statistics kernel (K3) then yields the
// members' sums and counts of every mean on the tensor cores.  One warp per row.
template <int NV>
__global__ void __launch_bounds__(256) k_kmeans_pick(const float* __restrict__ U, const float* __restrict__ yy,
                                                     float* __restrict__ R, int64_t n, int K, int KS) {
  const int lane = threadIdx.x & 31;
  const int64_t gw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int KS4 = KS >> 2;
  float ny[NV][4];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int k = 4 * (lane + 32 * v) + c;
      ny[v][c] = (k < K) ? yy[k] : 0.f;
    }
  for (int64_t s = gw; s < n; s += nw) {
    float bv = -3.0e38f;
    int bk = 0x7fffffff;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      if (lane + 32 * v >= KS4) continue;
      const float4 u = ld_stream4(reinterpret_cast<const float4*>(U + (size_t)s * KS) + lane + 32 * v);
      const float uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int k = 4 * (lane + 32 * v) + c;
        const float sc = uu[c] - ny[v][c];
        if (k < K && sc > bv) {  // ascending k within the lane: a tie keeps the lower k
          bv = sc;
          bk = k;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
      if (ov > bv || (ov == bv && ok < bk)) {
        bv = ov;
        bk = ok;
      }
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      if (lane + 32 * v >= KS4) continue;
      const int k0 = 4 * (lane + 32 * v);
      *reinterpret_cast<float4*>(R + (size_t)s * KS + k0) =
          make_float4(bk == k0 ? 1.f : 0.f, bk == k0 + 1 ? 1.f : 0.f, bk == k0 + 2 ? 1.f : 0.f, bk == k0 + 3 ? 1.f : 0.f);
    }
  }
}
// means from the statistics S[q][k][0..d] (sums of the members per tuple, column d = their number): means without
// members stay where they are (arma::kmeans keep_existing; Armadillo's dead-mean heuristic is not restated)
__global__ void k_kmeans_means_from_stats(const float* __restrict__ S, float* __restrict__ Y, int J, int K, int d) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= K * d) return;
  const int k = idx / d, c = idx - k * d;
  const int D1 = d + 1;
  float sum = 0.f, cnt = 0.f;
  for (int q = 0; q < J; ++q) {
    sum += S[((size_t)q * K + k) * D1 + c];
    cnt += S[((size_t)q * K + k) * D1 + d];
  }
  if (cnt > 0.f) Y[idx] = sum / cnt;
}

// one Lloyd assignment pass on the cosine-normalised cells: nearest centroid by largest dot product,
// accumulate per-cluster sums and counts.  Thread per cell, centroids in shared memory.
__global__ void __launch_bounds__(128) k_kmeans_assign(const float* __restrict__ Zc, const float* __restrict__ Y,
                                                       float* __restrict__ Ysum, float* __restrict__ cnt,
                                                       int64_t n, int K, int d, int DS) {
  extern __shared__ __align__(16) float smem[];
  float* Ys = smem;  // [K][d]
  for (int i = threadIdx.x; i < K * d; i += blockDim.x) Ys[i] = Y[i];
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float* z = Zc + (size_t)i * DS;
    int best = 0;
    float bv = -3.0e38f;
    for (int k = 0; k < K; ++k) {
      float acc = 0.f;
      const float* y = Ys + (size_t)k * d;
      for (int c = 0; c < d; ++c) acc = fmaf(z[c], y[c], acc);
      // squared Euclidean distance to the (un-normalised) centroid: |z|^2 - 2 z.y + |y|^2 with |z| = 1
      float yy = 0.f;
      for (int c = 0; c < d; ++c) yy = fmaf(y[c], y[c], yy);
      float score = 2.f * acc - yy;
      if (score > bv) {
        bv = score;
        best = k;
      }
    }
    atomicAdd(cnt + best, 1.f);
    for (int c = 0; c < d; ++c) atomicAdd(Ysum + (size_t)best * d + c, z[c]);
  }
}
__global__ void k_kmeans_update(float* __restrict__ Y, const float* __restrict__ Ysum, const float* __restrict__ cnt,
                                int K, int d) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= K * d) return;
  float c = cnt[idx / d];
  if (c > 0.f) Y[idx] = Ysum[idx] / c;  // empty clusters keep their centroid (arma::kmeans keep_existing)
}

// ------------------------------------------------------------------------------------------------
// K1: assignment from the centroids — harmony.cpp:141-150 (init) and :220-227 (cold start)
//   Zc <- L2-normalised rows (cold start only), dist = 2(1 - Y^T z), U = -dist/sigma,
//   R = exp(U)/sum_k exp(U), O[b] += column sums of R per level, rs += row sums (for E),
//   objective partials sum(R*dist), sum(sigma*R*log R).
// One CTA = one tile of <= TM consecutive cells that share a covariate tuple.
// ------------------------------------------------------------------------------------------------
struct AssignArgs {
  float* Zc;
  const float* Y;       // [K][d]
  const float* sigma;   // [K]
  float* U;
  float* R;
  const int* tile_cell0;  // [ntiles]
  const int* tile_len;
  const int* tile_tuple;
  const int* tuple_levels;  // [J][C]
  float* O_acc;             // [B][K]
  float* rs_acc;            // [K]
  double* obj_acc;          // [0] = sum R*dist, [1] = sum sigma R log R
  int ntiles, d, K, C, KP;  // KP = K rounded up to a multiple of 64
  int DS, KS;               // row strides of Z and of U/R/O (multiples of 4 floats)
  int normalise;
};

template <int KQ>
__global__ void __launch_bounds__(ASSIGN_THREADS) k_assign(AssignArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int d = a.d, K = a.K, KP = a.KP, LS = KP + 4;
  const int DP4 = (d + 3) & ~3;
  float* Ys = smem;                     // [DP4][KP]  (rows >= d are zero)
  float* Zs = Ys + (size_t)DP4 * KP;    // [TM][DP4]  (columns >= d are zero)
  float* Ls = Zs + (size_t)TM * DP4;    // [TM][LS]   dist tile
  float* sig = Ls + (size_t)TM * LS;    // [KP]
  float* part = sig + KP;               // [NWARP][KP]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (int idx = tid; idx < DP4 * KP; idx += ASSIGN_THREADS) {
    int dd = idx / KP, k = idx - dd * KP;
    Ys[idx] = (k < K && dd < d) ? a.Y[(size_t)k * d + dd] : 0.f;
  }
  for (int k = tid; k < KP; k += ASSIGN_THREADS) sig[k] = (k < K) ? a.sigma[k] : 1.f;

  float okd = 0.f, oent = 0.f;
  for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const int cell0 = a.tile_cell0[tile], len = a.tile_len[tile], q = a.tile_tuple[tile];
    __syncthreads();  // previous tile's epilogue is done with Zs/Ls/part (and Ys/sig are filled)
    // ---- load (+ normalise) the Z tile into Zs[cell][dd]
    for (int r = warp; r < TM; r += NWARP) {
      if (r < len) {
        float* zrow = a.Zc + (size_t)(cell0 + r) * a.DS;
        float nrm = 1.f;
        if (a.normalise) {
          float s = 0.f;
          for (int c = lane; c < d; c += 32) {
            float v = zrow[c];
            s += v * v;
          }
          s = warp_sum(s);
          nrm = sqrtf(s);
          if (nrm == 0.f) nrm = 1.f;
        }
        for (int c = lane; c < DP4; c += 32) {
          float v = 0.f;
          if (c < d) {
            v = zrow[c];
            if (a.normalise) {
              v = v / nrm;
              zrow[c] = v;
            }
          }
          Zs[r * DP4 + c] = v;
        }
      } else {
        for (int c = lane; c < DP4; c += 32) Zs[r * DP4 + c] = 0.f;
      }
    }
    __syncthreads();
    // ---- dist tile: Ls[cell][k] = 2 * (1 - z . y_k); thread = 4 cells x 4 clusters per 64-cluster chunk
    {
      const int ty = tid >> 4, tx = tid & 15;
      for (int kc = 0; kc < KP; kc += 64) {
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        const float* zp = Zs + (size_t)(ty * 4) * DP4;
        const float* yp = Ys + kc + tx * 4;
        for (int dd = 0; dd < DP4; dd += 4) {
          float4 z4[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) z4[i] = *reinterpret_cast<const float4*>(zp + (size_t)i * DP4 + dd);
#pragma unroll
          for (int jd = 0; jd < 4; ++jd) {
            float4 y4 = *reinterpret_cast<const float4*>(yp + (size_t)(dd + jd) * KP);
            float yy[4] = {y4.x, y4.y, y4.z, y4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float zz = (jd == 0) ? z4[i].x : (jd == 1) ? z4[i].y : (jd == 2) ? z4[i].z : z4[i].w;
#pragma unroll
              for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(zz, yy[j], acc[i][j]);
            }
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 o;
          o.x = 2.f * (1.f - acc[i][0]);
          o.y = 2.f * (1.f - acc[i][1]);
          o.z = 2.f * (1.f - acc[i][2]);
          o.w = 2.f * (1.f - acc[i][3]);
          *reinterpret_cast<float4*>(Ls + (size_t)(ty * 4 + i) * LS + kc + tx * 4) = o;
        }
      }
    }
    __syncthreads();
    // ---- row epilogue: one warp per row, lanes over clusters
    float cs[KQ];
#pragma unroll
    for (int qq = 0; qq < KQ; ++qq) cs[qq] = 0.f;
    for (int r = warp; r < len; r += NWARP) {
      const size_t row = (size_t)(cell0 + r);
      float u[KQ], e[KQ], dist[KQ];
      float s = 0.f;
#pragma unroll
      for (int qq = 0; qq < KQ; ++qq) {
        int k = lane + 32 * qq;
        if (k < K) {
          dist[qq] = Ls[(size_t)r * LS + k];
          u[qq] = -dist[qq] / sig[k];
          e[qq] = expf(u[qq]);
        } else {
          dist[qq] = 0.f;
          u[qq] = 0.f;
          e[qq] = 0.f;
        }
        s += e[qq];
      }
      s = warp_sum(s);
      const float ls = logf(s);
#pragma unroll
      for (int qq = 0; qq < KQ; ++qq) {
        int k = lane + 32 * qq;
        if (k < K) {
          float rv = e[qq] / s;  // R.each_row() /= sum(R, 0): no zero guard in the reference
          a.U[row * a.KS + k] = u[qq];
          a.R[row * a.KS + k] = rv;
          cs[qq] += rv;
          okd += rv * dist[qq];
          if (rv > 0.f) oent += sig[k] * rv * (u[qq] - ls);
        }
      }
    }
#pragma unroll
    for (int qq = 0; qq < KQ; ++qq) {
      int k = lane + 32 * qq;
      if (k < KP) part[warp * KP + k] = cs[qq];
    }
    __syncthreads();
    for (int k = tid; k < K; k += ASSIGN_THREADS) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < NWARP; ++w) t += part[w * KP + k];
      atomicAdd(a.rs_acc + k, t);
      for (int c = 0; c < a.C; ++c) atomicAdd(a.O_acc + (size_t)a.tuple_levels[q * a.C + c] * a.KS + k, t);
    }
  }
  okd = warp_sum(okd);
  oent = warp_sum(oent);
  if (lane == 0) {
    atomicAdd(a.obj_acc + 0, (double)okd);
    atomicAdd(a.obj_acc + 1, (double)oent);
  }
}

// E = sum(R,1) * Pr_b^T (harmony.cpp:149,226) and O from the accumulators.
__global__ void k_assign_finalize(const float* __restrict__ O_acc, const float* __restrict__ rs_acc,
                                  const float* __restrict__ Pr_b, float* __restrict__ O, float* __restrict__ E,
                                  int B, int K, int KS) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < B * KS) {
    int b = idx / KS, k = idx - b * KS;
    O[idx] = (k < K) ? O_acc[idx] : 0.f;
    E[idx] = (k < K) ? rs_acc[k] * Pr_b[b] : 0.f;
  }
}

// Assignment step in plan order: the tiles' column sums went to the rem halves of the update kernel's accumulator
// slots (slot(j) at (j + 1) * SL: [add | rem_O B*KS | rem_rs KS]); O = sum_j rem_O(j), E = (sum_j rem_rs(j)) Pr_b^T.
__global__ void k_assign_finalize_plan(const float* __restrict__ acc, int nb, const float* __restrict__ Pr_b,
                                       float* __restrict__ O, float* __restrict__ E, int B, int K, int KS) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < B * KS) {
    const size_t XH = (size_t)B * KS + KS;
    int b = idx / KS, k = idx - b * KS;
    float o = 0.f, rs = 0.f;
    if (k < K)
      for (int j = 0; j < nb; ++j) {
        const float* rem = acc + (size_t)(j + 1) * 2 * XH + XH;
        o += rem[idx];
        rs += rem[(size_t)B * KS + k];
      }
    O[idx] = o;
    E[idx] = rs * Pr_b[b];
  }
}

// ------------------------------------------------------------------------------------------------
// update-order plan (replaces the physical shuffles of harmony.cpp:272-291)
// ------------------------------------------------------------------------------------------------
// Injected order: for global position p, cell update_order[p] belongs to block min(p/cpb, nb-1).
__global__ void k_plan_block_injected(const int64_t* __restrict__ update_order, int64_t N_global, int64_t cell_offset,
                                      int64_t n_local, const int* __restrict__ inv_sort, uint32_t cpb, int nb,
                                      int* __restrict__ blk_of, int* __restrict__ err_flag) {
  update_order += (size_t)blockIdx.y * (size_t)N_global;  // blockIdx.y: round of the call
  blk_of += (size_t)blockIdx.y * (size_t)n_local;
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < N_global;
       p += (int64_t)gridDim.x * blockDim.x) {
    int64_t g = update_order[p];
    if (g < 0 || g >= N_global) {
      atomicExch(err_flag, 1);
      continue;
    }
    int64_t l = g - cell_offset;
    if (l < 0 || l >= n_local) continue;
    int64_t b = p / cpb;
    if (b > nb - 1) b = nb - 1;
    blk_of[inv_sort[l]] = (int)b;
  }
}
// Native order: position of global cell g is hb_permute(g) (a keyed bijection of [0, N)); the key of a round
// depends on (seed, round counter) only.  blockIdx.y: round of the call.
__host__ __device__ __forceinline__ uint64_t plan_round_key(uint64_t seed, uint64_t round_counter) {
  return hb_mix64(seed ^ hb_mix64(round_counter + 0x1234567ull));
}
__global__ void k_plan_block_native(int64_t N_global, int64_t cell_offset, int64_t n_local,
                                    const int* __restrict__ sort_perm, uint32_t cpb, int nb, int half_bits,
                                    uint64_t seed, uint64_t round_counter0, int* __restrict__ blk_of) {
  const uint64_t key = plan_round_key(seed, round_counter0 + blockIdx.y);
  blk_of += (size_t)blockIdx.y * (size_t)n_local;
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < n_local;
       s += (int64_t)gridDim.x * blockDim.x) {
    uint64_t g = (uint64_t)(cell_offset + sort_perm[s]);
    uint64_t pos = hb_permute(g, (uint64_t)N_global, half_bits, key);
    uint64_t b = pos / cpb;
    if (b > (uint64_t)(nb - 1)) b = nb - 1;
    blk_of[s] = (int)b;
  }
}
// Sort key of a cell in round t: (block in round t, tuple, block in round t+1, chunk, cell).  Chunks are runs of
// consecutive (tuple-sorted) cells of one tuple, so with the histogram laid out as
//   H[blk][ nsub * cq0[c] + sub * cnq[c] + (c - cq0[c]) ]      (cq0 / cnq: first chunk / #chunks of c's tuple)
// one plain exclusive scan of H yields the offsets of that order (nsub = nb, sub = next-round block; nsub = 1
// switches the third key off).
__device__ __forceinline__ size_t plan_hidx(int blk, int sub, int c, int nchunks, int nsub, const int* __restrict__ cq0,
                                            const int* __restrict__ cnq) {
  const int c0 = cq0[c];
  return (size_t)blk * nsub * nchunks + (size_t)nsub * c0 + (size_t)sub * cnq[c] + (c - c0);
}
// One warp per chunk: H[..] = #cells of the chunk with (block, next-round block) = (blk, sub).
__global__ void k_plan_hist(const int* __restrict__ blk_of, const int* __restrict__ blk_next,
                            const int* __restrict__ chunk_start, const int* __restrict__ cq0, const int* __restrict__ cnq,
                            int nchunks, int nb, int nsub, int* __restrict__ H, int* __restrict__ err_flag, int64_t n_local,
                            int rounds_with_next) {
  extern __shared__ int sh[];
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* cnt = sh + warp * nb * nsub;
  int c = blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= nchunks) return;
  // blockIdx.y: round of the batch (rounds are n_local apart in blk_of; blk_next of round y is blk_of of round y + 1)
  blk_of += (size_t)blockIdx.y * (size_t)n_local;
  blk_next = ((int)blockIdx.y < rounds_with_next) ? blk_of + n_local : nullptr;
  H += (size_t)blockIdx.y * (size_t)nb * nsub * nchunks;
  for (int j = lane; j < nb * nsub; j += 32) cnt[j] = 0;
  __syncwarp();
  int s0 = chunk_start[c], s1 = chunk_start[c + 1];
  for (int s = s0 + lane; s < s1; s += 32) {
    const int b = blk_of[s];
    if (b < 0 || b >= nb) {  // an injected update order that is not a permutation left this cell without a block
      atomicCAS(err_flag, 0, 3);  // an out-of-range index (flag 1) is the more specific report
      continue;
    }
    const int sub = (nsub > 1 && blk_next) ? blk_next[s] : 0;
    atomicAdd(cnt + b * nsub + ((sub >= 0 && sub < nsub) ? sub : 0), 1);
  }
  __syncwarp();
  for (int j = lane; j < nb * nsub; j += 32) H[plan_hidx(j / nsub, j % nsub, c, nchunks, nsub, cq0, cnq)] = cnt[j];
}
// Single-CTA exclusive scan of an int array (in place), total written to *total.  Every warp owns a contiguous
// range and walks it 32 consecutive elements at a time (coalesced): pass 1 sums, pass 2 scans with a carry.
__global__ void __launch_bounds__(1024) k_scan_exclusive(int* __restrict__ data, int64_t n, int* __restrict__ total) {
  data += (size_t)blockIdx.x * (size_t)n;  // blockIdx.x: independent arrays of n elements, back to back
  if (total) total += blockIdx.x;
  __shared__ int wsum[32];
  __shared__ int carry_all;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const int64_t per = ((n + nw - 1) / nw + 31) & ~(int64_t)31;
  const int64_t lo = (int64_t)warp * per, hi = (lo + per < n) ? lo + per : n;
  int s = 0;
  for (int64_t i = lo + lane; i < hi; i += 32) s += data[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) wsum[warp] = s;
  __syncthreads();
  if (warp == 0) {
    int v = (lane < nw) ? wsum[lane] : 0;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    wsum[lane] = inc - v;
    if (lane == 31) carry_all = inc;
  }
  __syncthreads();
  int carry = wsum[warp];
  for (int64_t i0 = lo; i0 < hi; i0 += 32) {
    const int64_t i = i0 + lane;
    const int v = (i < hi) ? data[i] : 0;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (i < hi) data[i] = carry + inc - v;
    carry += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (tid == 0 && total) *total = carry_all;
}
// Exclusive scan of `nseg` independent int arrays of n elements (back to back in `data`, in place) by many CTAs:
// chained scan with dynamic tile numbers.  A CTA draws the next tile (8192 elements) of its segment from a counter
// — so a tile's predecessor has always been drawn, i.e. runs or has run: no deadlock whatever the dispatch order —,
// scans it locally, waits for the inclusive prefix of the tile before it, publishes its own (value and flag in one
// 64-bit word) and writes the results.  state: [nseg][1 + tiles] words, zeroed by the caller (word 0: the counter).
constexpr int SCAN_TILE = 8192;  // 1024 threads x 8 elements
__global__ void __launch_bounds__(1024) k_scan_chained(int* __restrict__ data, int64_t n, unsigned long long* __restrict__ state,
                                                       int tiles_per_seg) {
  __shared__ int wsum[32];
  __shared__ int sh_tile, sh_carry;
  const int seg = blockIdx.y;
  data += (size_t)seg * (size_t)n;
  unsigned long long* st = state + (size_t)seg * (tiles_per_seg + 1);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) sh_tile = (int)atomicAdd(st, 1ull);
  __syncthreads();
  const int tile = sh_tile;
  if (tile >= tiles_per_seg) return;
  const int64_t base = (int64_t)tile * SCAN_TILE + (int64_t)tid * 8;
  int v[8];
  int s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    v[i] = (base + i < n) ? data[base + i] : 0;
    s += v[i];
  }
  // exclusive scan of the threads' sums within the CTA
  int inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int w = wsum[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    wsum[lane] = winc - w;  // exclusive prefix of the warps
    if (lane == 31) {
      // tile aggregate = winc; chain: inclusive prefix of this tile = prefix of the previous one + aggregate
      int carry = 0;
      if (tile > 0) {
        unsigned long long p;
        do {
          asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(p) : "l"(st + tile) : "memory");  // word 1 + (tile - 1)
        } while ((p >> 32) == 0ull);
        carry = (int)(unsigned)(p & 0xffffffffull);
      }
      const unsigned long long mine = (1ull << 32) | (unsigned)(carry + winc);
      asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(st + tile + 1), "l"(mine) : "memory");
      sh_carry = carry;
    }
  }
  __syncthreads();
  int run = sh_carry + wsum[warp] + (inc - s);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (base + i < n) data[base + i] = run;
    run += v[i];
  }
}
// Stable scatter: order[offset(key, chunk) + rank] = cell, cells of a chunk visited in ascending order;
// next_at[same position] = block of the cell in the next round.
__global__ void k_plan_scatter(const int* __restrict__ blk_of, const int* __restrict__ blk_next,
                               const int* __restrict__ chunk_start, const int* __restrict__ cq0, const int* __restrict__ cnq,
                               int nchunks, int nb, int nsub, const int* __restrict__ Hoff, int* __restrict__ order,
                               const int* __restrict__ blk_prev, int* __restrict__ prev_at, int* __restrict__ next_at,
                               int64_t n_local, int rounds_with_next, int first_has_prev) {
  extern __shared__ int sh[];
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* cur = sh + warp * nb * nsub;
  int c = blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= nchunks) return;
  {  // blockIdx.y: round of the batch
    const size_t ro = (size_t)blockIdx.y * (size_t)n_local;
    blk_of += ro;
    blk_next = ((int)blockIdx.y < rounds_with_next) ? blk_of + n_local : nullptr;
    blk_prev = (blockIdx.y > 0 || first_has_prev) ? blk_of - n_local : nullptr;
    Hoff += (size_t)blockIdx.y * (size_t)nb * nsub * nchunks;
    order += ro;
    if (prev_at) prev_at += ro;
    if (next_at) next_at += ro;
  }
  for (int j = lane; j < nb * nsub; j += 32) cur[j] = Hoff[plan_hidx(j / nsub, j % nsub, c, nchunks, nsub, cq0, cnq)];
  __syncwarp();
  int s0 = chunk_start[c], s1 = chunk_start[c + 1];
  for (int base = s0; base < s1; base += 32) {
    int s = base + lane;
    bool act = s < s1;
    int b = act ? blk_of[s] : -1;
    act = act && b >= 0 && b < nb;  // cells without a block were flagged by k_plan_hist
    int nx = (act && blk_next) ? blk_next[s] : 0;
    if (nx < 0 || nx >= nb) nx = 0;
    int key = act ? b * nsub + (nsub > 1 ? nx : 0) : -1 - lane;  // inactive lanes get unique keys
    unsigned m = __match_any_sync(0xffffffffu, key);
    int rank = __popc(m & ((1u << lane) - 1u));
    int leader = __ffs(m) - 1;
    int start = 0;
    if (act && lane == leader) {
      start = cur[key];
      cur[key] = start + __popc(m);
    }
    start = __shfl_sync(0xffffffffu, start, leader);
    if (act) {
      order[start + rank] = s;
      if (prev_at) prev_at[start + rank] = blk_prev ? blk_prev[s] : 0;
      if (next_at) next_at[start + rank] = nx;
    }
    __syncwarp();
  }
}
// Segment (block, tuple) boundaries: seg s = blk*J + q starts at the offset of (blk, first chunk of q, sub 0).
__global__ void k_plan_segments(const int* __restrict__ Hoff, const int* __restrict__ tuple_chunk0, int nchunks,
                                int nb, int nsub, int J, int n_local, int* __restrict__ seg_start,
                                int* __restrict__ tile_base) {
  int S = nb * J;
  Hoff += (size_t)blockIdx.y * (size_t)nb * nsub * nchunks;  // blockIdx.y: round of the batch
  seg_start += (size_t)blockIdx.y * (S + 1);
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s <= S; s += gridDim.x * blockDim.x) {
    int v;
    if (s == S) {
      v = n_local;
    } else {
      int blk = s / J, q = s - blk * J;
      int c = tuple_chunk0[q];  // first chunk of tuple q (tuples without local cells point at the first later chunk)
      v = Hoff[(size_t)blk * nsub * nchunks + (size_t)nsub * c];
    }
    seg_start[s] = v;
  }
}
// Tuple-aligned work split of every block for the persistent update kernel (G CTAs): each CTA gets a contiguous
// slice of ONE (block, tuple) segment.  The block step ends when its most loaded CTA does, so the CTAs are dealt out
// to minimise the largest slice: every non-empty segment starts with one CTA and the remaining ones go, one at a
// time, to the segment with the most rows per CTA (exact comparison L_a n_b > L_b n_a; ties to the lower tuple).
// One CTA (256 threads) per (block j = blockIdx.x, round = blockIdx.y); J <= 2 J <= G <= 1024.
constexpr int PLAN_MAXJ = 512;
__global__ void __launch_bounds__(256) k_plan_ranges(const int* __restrict__ seg_start, int nb, int J, int G,
                                                     int4* __restrict__ ranges) {
  __shared__ int L[PLAN_MAXJ], nq[PLAN_MAXJ], first[PLAN_MAXJ + 1];
  seg_start += (size_t)blockIdx.y * ((size_t)nb * J + 1);  // blockIdx.y: round of the batch
  ranges += (size_t)blockIdx.y * (size_t)nb * G;
  const int j = blockIdx.x;
  const int* segs = seg_start + (size_t)j * J;
  const int tid = threadIdx.x, lane = tid & 31;
  for (int q = tid; q < J; q += blockDim.x) {
    L[q] = segs[q + 1] - segs[q];
    nq[q] = L[q] > 0 ? 1 : 0;
  }
  __syncthreads();
  if (tid < 32) {
    int nonempty = 0;
    for (int q = lane; q < J; q += 32) nonempty += nq[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nonempty += __shfl_xor_sync(0xffffffffu, nonempty, o);
    for (int rem = (nonempty > 0) ? G - nonempty : 0; rem > 0; --rem) {
      long long bl = 0, bn = 1;  // best ratio bl / bn of this lane
      int bq = J;
      for (int q = lane; q < J; q += 32)
        if (nq[q] > 0 && (long long)L[q] * bn > bl * (long long)nq[q]) {
          bl = L[q];
          bn = nq[q];
          bq = q;
        }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const long long ol = __shfl_xor_sync(0xffffffffu, bl, o), on = __shfl_xor_sync(0xffffffffu, bn, o);
        const int oq = __shfl_xor_sync(0xffffffffu, bq, o);
        const long long lhs = ol * bn, rhs = bl * on;
        if (lhs > rhs || (lhs == rhs && oq < bq)) {
          bl = ol;
          bn = on;
          bq = oq;
        }
      }
      if (lane == 0 && bq < J) nq[bq]++;
      __syncwarp();
    }
    if (lane == 0) {
      int c = 0;
      for (int q = 0; q < J; ++q) {
        first[q] = c;
        c += nq[q];
      }
      first[J] = c;
    }
  }
  __syncthreads();
  const int b0 = segs[0];
  for (int c = tid; c < G; c += blockDim.x) {
    int4 out = make_int4(b0, b0, 0, 0);
    if (c < first[J]) {
      int q = 0;
      while (first[q + 1] <= c) ++q;  // J is small
      const int n = nq[q], me = c - first[q];
      out = make_int4(segs[q] + (int)(((long long)L[q] * me) / n), segs[q] + (int)(((long long)L[q] * (me + 1)) / n), q, 0);
    }
    ranges[(size_t)j * G + c] = out;
  }
}
// 128-row tiles of the (block, tuple) segments of a round (the assignment step in plan order)
__global__ void k_plan_tilecount128(const int* __restrict__ seg_start, int S, int* __restrict__ tile_base) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s <= S; s += gridDim.x * blockDim.x)
    tile_base[s] = (s < S) ? (seg_start[s + 1] - seg_start[s] + 127) / 128 : 0;
}
__global__ void k_plan_tilefill128(const int* __restrict__ seg_start, const int* __restrict__ tile_base, int S, int J,
                                   int* __restrict__ p0, int* __restrict__ len, int* __restrict__ tuple,
                                   int* __restrict__ blk) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += gridDim.x * blockDim.x) {
    const int a = seg_start[s], e = seg_start[s + 1];
    int i = tile_base[s];
    for (int p = a; p < e; p += 128, ++i) {
      p0[i] = p;
      len[i] = min(128, e - p);
      tuple[i] = s % J;
      blk[i] = s / J;
    }
  }
}
__global__ void k_plan_tilecount(const int* __restrict__ seg_start, int S, int* __restrict__ tile_base) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s <= S; s += gridDim.x * blockDim.x) {
    int len = (s < S) ? seg_start[s + 1] - seg_start[s] : 0;
    tile_base[s] = (len + TM - 1) / TM;
  }
}

// ------------------------------------------------------------------------------------------------
// update_R block step (harmony.cpp:293-332)
// ------------------------------------------------------------------------------------------------
struct StepArgs {
  const float* U;
  float* R;
  const int* order;         // [n] cells sorted by (block, tuple, cell)
  const int* seg_start;     // [nb*J + 1]
  const int* tile_base;     // [nb*J + 1] exclusive scan of tiles per segment
  const int* tuple_levels;  // [J][C]
  const float* sigma;
  const float* P;           // [B][K] penalty table of this step
  float* acc_O;             // [B][K] column sums per level (rem_j or add_j)
  float* acc_rs;            // [K]
  double* obj_acc;          // [2]
  int blk, J, K, C, KP, KS;
};

// tile -> (segment, first position, length)
__device__ __forceinline__ bool locate_tile(const StepArgs& a, int t, int* sh_info) {
  // sh_info: [0] seg, [1] p0, [2] len, [3] valid
  if (threadIdx.x == 0) {
    int s_lo = a.blk * a.J, s_hi = (a.blk + 1) * a.J;
    int t0 = a.tile_base[s_lo], t1 = a.tile_base[s_hi];
    int tt = t0 + t;
    if (tt >= t1) {
      sh_info[3] = 0;
    } else {
      int lo = s_lo, hi = s_hi;  // find the last seg with tile_base[seg] <= tt
      while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (a.tile_base[mid] <= tt) lo = mid; else hi = mid;
      }
      int p0 = a.seg_start[lo] + (tt - a.tile_base[lo]) * TM;
      int len = a.seg_start[lo + 1] - p0;
      sh_info[0] = lo;
      sh_info[1] = p0;
      sh_info[2] = len < TM ? len : TM;
      sh_info[3] = 1;
    }
  }
  __syncthreads();
  return sh_info[3] != 0;
}

// Step 1 (:312-313): column sums of the block's current R, per level  ->  acc_O / acc_rs
template <int KQ>
__global__ void __launch_bounds__(ROW_THREADS) k_block_colsum(StepArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ int info[4];
  const int K = a.K, KP = a.KP;
  float* part = smem;  // [NWARP][KP]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int t = blockIdx.x;; t += gridDim.x) {
    __syncthreads();
    if (!locate_tile(a, t, info)) break;
    const int seg = info[0], p0 = info[1], len = info[2];
    const int q = seg - a.blk * a.J;
    float cs[KQ];
#pragma unroll
    for (int qq = 0; qq < KQ; ++qq) cs[qq] = 0.f;
    for (int r = warp; r < len; r += NWARP) {
      const size_t row = (size_t)a.order[p0 + r];
#pragma unroll
      for (int qq = 0; qq < KQ; ++qq) {
        int k = lane + 32 * qq;
        if (k < K) cs[qq] += a.R[row * a.KS + k];
      }
    }
#pragma unroll
    for (int qq = 0; qq < KQ; ++qq) {
      int k = lane + 32 * qq;
      if (k < KP) part[warp * KP + k] = cs[qq];
    }
    __syncthreads();
    for (int k = tid; k < K; k += ROW_THREADS) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < NWARP; ++w) s += part[w * KP + k];
      atomicAdd(a.acc_rs + k, s);
      for (int c = 0; c < a.C; ++c) atomicAdd(a.acc_O + (size_t)a.tuple_levels[q * a.C + c] * a.KS + k, s);
    }
  }
}

// Finish step j-1 and start step j on the K x B tables:
//   O += add_prev; E += rs_add_prev*Pr_b        (:329-330 of the previous block)
//   O -= rem;      E -= rs_rem*Pr_b             (:312-313 of this block)
//   P = ((2E+1)/(O+E+1))^theta                  (:322, harmony_pow utils.cpp:84-90)
// add_prev / rem may be null (first step of a round / finalisation after the last step).
__global__ void k_step_prepare(float* __restrict__ O, float* __restrict__ E, const float* __restrict__ add_O,
                               const float* __restrict__ add_rs, const float* __restrict__ rem_O,
                               const float* __restrict__ rem_rs, const float* __restrict__ Pr_b,
                               const float* __restrict__ theta, float* __restrict__ P, int B, int K, int KS) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * KS) return;
  int b = idx / KS, k = idx - b * KS;
  if (k >= K) return;
  float o = O[idx], e = E[idx];
  if (add_O) {
    e += add_rs[k] * Pr_b[b];
    o += add_O[idx];
  }
  if (rem_O) {
    e -= rem_rs[k] * Pr_b[b];
    o -= rem_O[idx];
  }
  O[idx] = o;
  E[idx] = e;
  if (P) P[idx] = powf(((2.f * e) + 1.f) / (o + e + 1.f), theta[b]);
}

// Step 2+3 (:318-330): R = L1norm(exp(U) * sum_c P[level_c]), column sums of the new R -> acc_O/acc_rs,
// objective partials of the new R.
template <int KQ>
__global__ void __launch_bounds__(ROW_THREADS) k_block_update(StepArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ int info[4];
  const int K = a.K, KP = a.KP;
  float* part = smem;             // [NWARP][KP]
  float* Psum = part + NWARP * KP;  // [KP]
  float* lP = Psum + KP;          // [KP]
  float* sig = lP + KP;           // [KP]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int k = tid; k < KP; k += ROW_THREADS) sig[k] = (k < K) ? a.sigma[k] : 1.f;
  float okd = 0.f, oent = 0.f;
  for (int t = blockIdx.x;; t += gridDim.x) {
    __syncthreads();
    if (!locate_tile(a, t, info)) break;
    const int seg = info[0], p0 = info[1], len = info[2];
    const int q = seg - a.blk * a.J;
    for (int k = tid; k < K; k += ROW_THREADS) {
      float s = 0.f;
      for (int c = 0; c < a.C; ++c) s += a.P[(size_t)a.tuple_levels[q * a.C + c] * a.KS + k];
      Psum[k] = s;
      lP[k] = logf(s);
    }
    __syncthreads();
    float cs[KQ];
#pragma unroll
    for (int qq = 0; qq < KQ; ++qq) cs[qq] = 0.f;
    for (int r = warp; r < len; r += NWARP) {
      const size_t row = (size_t)a.order[p0 + r];
      float u[KQ], e[KQ];
      float s = 0.f;
#pragma unroll
      for (int qq = 0; qq < KQ; ++qq) {
        int k = lane + 32 * qq;
        if (k < K) {
          u[qq] = ld_stream(a.U + row * a.KS + k);
          e[qq] = expf(u[qq]) * Psum[k];
        } else {
          u[qq] = 0.f;
          e[qq] = 0.f;
        }
        s += fabsf(e[qq]);
      }
      s = warp_sum(s);
      const float sdiv = (s == 0.f) ? 1.f : s;  // arma::normalise(.., 1, 0): zero norm divides by 1
      const float ls = logf(sdiv);
#pragma unroll
      for (int qq = 0; qq < KQ; ++qq) {
        int k = lane + 32 * qq;
        if (k < K) {
          float rv = e[qq] / sdiv;
          st_stream(a.R + row * a.KS + k, rv);
          cs[qq] += rv;
          okd += rv * (-sig[k] * u[qq]);
          if (rv > 0.f) oent += sig[k] * rv * (u[qq] + lP[k] - ls);
        }
      }
    }
#pragma unroll
    for (int qq = 0; qq < KQ; ++qq) {
      int k = lane + 32 * qq;
      if (k < KP) part[warp * KP + k] = cs[qq];
    }
    __syncthreads();
    for (int k = tid; k < K; k += ROW_THREADS) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < NWARP; ++w) s += part[w * KP + k];
      atomicAdd(a.acc_rs + k, s);
      for (int c = 0; c < a.C; ++c) atomicAdd(a.acc_O + (size_t)a.tuple_levels[q * a.C + c] * a.KS + k, s);
    }
  }
  okd = warp_sum(okd);
  oent = warp_sum(oent);
  if (lane == 0) {
    atomicAdd(a.obj_acc + 0, (double)okd);
    atomicAdd(a.obj_acc + 1, (double)oent);
  }
}

// compute_objective (harmony.cpp:158-170) once the per-cell sums are known:
//   cross = sum_kb sigma_k theta_b log((O+E+1)/(2E+1)) O_kb   (== the reference's N-pass, SURVEY §8a')
// Appends (total, dist, entropy, cross) * 2000/N to the device trace at slot `slot` and clears obj_acc.
__global__ void __launch_bounds__(256) k_objective_finalize(const float* __restrict__ O, const float* __restrict__ E,
                                                            const float* __restrict__ theta,
                                                            const float* __restrict__ sigma, double* obj_acc,
                                                            float* __restrict__ trace, int slot, int B, int K,
                                                            int KS, double N_global, double cross_scale) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int idx = threadIdx.x; idx < B * KS; idx += blockDim.x) {
    int b = idx / KS, k = idx - b * KS;
    if (k >= K) continue;
    float o = O[idx], e = E[idx];
    float l = theta[b] * logf((o + e + 1.f) / ((2.f * e) + 1.f));
    acc += (double)(sigma[k] * l) * (double)o;
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double cross = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) cross += red[w];
    cross *= cross_scale;  // 1 normally; the cross term is replicated, not sharded
    const float norm_const = 2000.f / (float)N_global;
    float kd = (float)obj_acc[0], ent = (float)obj_acc[1], cr = (float)cross;
    trace[4 * slot + 0] = (kd + ent + cr) * norm_const;
    trace[4 * slot + 1] = kd * norm_const;
    trace[4 * slot + 2] = ent * norm_const;
    trace[4 * slot + 3] = cr * norm_const;
    obj_acc[0] = 0.0;
    obj_acc[1] = 0.0;
  }
}

// Standalone per-cell objective sums from the stored R and U (for hb_compute_objective).
__global__ void __launch_bounds__(ROW_THREADS) k_objective_cells(const float* __restrict__ R, const float* __restrict__ U,
                                                                const float* __restrict__ sigma, int64_t n, int K,
                                                                int KS, double* obj_acc) {
  const int lane = threadIdx.x & 31;
  int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float okd = 0.f, oent = 0.f;
  for (int64_t r = w; r < n; r += nw) {
    for (int k = lane; k < K; k += 32) {
      float rv = R[r * KS + k], u = U[r * KS + k], sg = sigma[k];
      okd += rv * (-sg * u);
      if (rv > 0.f) oent += sg * rv * logf(rv);
    }
  }
  okd = warp_sum(okd);
  oent = warp_sum(oent);
  if (lane == 0) {
    atomicAdd(obj_acc + 0, (double)okd);
    atomicAdd(obj_acc + 1, (double)oent);
  }
}

// ------------------------------------------------------------------------------------------------
// K3: ridge sufficient statistics (harmony.cpp:561-567, 592-609 for all clusters at once)
//   S[q][k][0..d-1] = sum_{i in tuple q} R_ik * Zo_i      S[q][k][d] = sum_{i in tuple q} R_ik
// Output-stationary fp32 register tiling: thread (ty, tx) owns clusters ty*8..+7 x columns tx*4..+3.
// ------------------------------------------------------------------------------------------------
struct StatsArgs {
  const float* R;
  const float* Zo;
  const int* tile_cell0;
  const int* tile_len;
  const int* tile_tuple;
  float* S;  // [J][K][d+1]
  int ntiles, d, K, KS;  // KS = clusters per K-slice (blockIdx.y)
  int tiles_per_cta;
  int ldR, ldZ;          // row strides of R and Zo
};

__global__ void k_ridge_stats(StatsArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int d = a.d, K = a.K, D1 = d + 1;
  const int k0 = blockIdx.y * a.KS;
  const int ks = (K - k0 < a.KS) ? K - k0 : a.KS;  // clusters in this slice
  const int KSP = (a.KS + 7) & ~7;                   // padded slice width (multiple of 8)
  const int DP = (D1 + 3) & ~3;
  float* Rs = smem;                      // [TM][KSP]
  float* Zs = Rs + (size_t)TM * KSP;     // [TM][DP]
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int tid = ty * blockDim.x + tx, nthr = blockDim.x * blockDim.y;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  int cur_q = -1;
  const int t_begin = blockIdx.x * a.tiles_per_cta;
  const int t_end = (t_begin + a.tiles_per_cta < a.ntiles) ? t_begin + a.tiles_per_cta : a.ntiles;

  auto flush = [&](int q) {
    if (q < 0) return;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int k = ty * 8 + i;
      if (k < ks) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int c = tx * 4 + j;
          if (c < D1) atomicAdd(a.S + ((size_t)q * K + k0 + k) * D1 + c, acc[i][j]);
          acc[i][j] = 0.f;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
      }
    }
  };

  for (int tile = t_begin; tile < t_end; ++tile) {
    const int cell0 = a.tile_cell0[tile], len = a.tile_len[tile], q = a.tile_tuple[tile];
    if (q != cur_q) {
      flush(cur_q);
      cur_q = q;
    }
    __syncthreads();
    for (int idx = tid; idx < TM * KSP; idx += nthr) {
      int r = idx / KSP, k = idx - r * KSP;
      Rs[idx] = (r < len && k < ks) ? ld_stream(a.R + (size_t)(cell0 + r) * a.ldR + k0 + k) : 0.f;
    }
    for (int idx = tid; idx < TM * DP; idx += nthr) {
      int r = idx / DP, c = idx - r * DP;
      float v = 0.f;
      if (r < len) v = (c < d) ? ld_stream(a.Zo + (size_t)(cell0 + r) * a.ldZ + c) : ((c == d) ? 1.f : 0.f);
      Zs[idx] = v;
    }
    __syncthreads();
#pragma unroll 2
    for (int r = 0; r < TM; ++r) {
      float4 r0 = *reinterpret_cast<const float4*>(Rs + (size_t)r * KSP + ty * 8);
      float4 r1 = *reinterpret_cast<const float4*>(Rs + (size_t)r * KSP + ty * 8 + 4);
      float4 z = *reinterpret_cast<const float4*>(Zs + (size_t)r * DP + tx * 4);
      float rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
      float zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(rr[i], zz[j], acc[i][j]);
    }
  }
  flush(cur_q);
}

// ------------------------------------------------------------------------------------------------
// K4: per-cluster level filter + ridge solve (harmony.cpp:358-410, 561-611, 633); one CTA per cluster.
// Produces the per-tuple correction matrices V[q][k][:] = sum over the tuple's kept levels of W_k[level],
// the new centroid Y[k] (L2-normalised) and Wfull[k] = W_k expanded to B+1 rows (row 0 zeroed).
// ------------------------------------------------------------------------------------------------
struct SolveArgs {
  const float* S;             // [J][K][d+1]
  const float* O;             // [B][K]
  const float* E;             // [B][K]
  const float* N_b;           // [B]
  const float* lambda;        // [B+1] or null (estimation)
  const int* tuple_levels;    // [J][C]
  const int* cov_of;          // [B]
  float* Y;                   // [K][d]
  float* V;                   // [J][K][d]
  float* Wfull;               // [K][B+1][d]
  int* skipped;               // [K]
  float* scratch;             // [K][ 2*M*M + M*d ]  (G | inv | s),  M = B+1
  int* iscratch;              // [K][ 2*B + J ]      (pos | keep | part)
  int* err_flag;
  int J, K, B, C, d, KS;  // KS = row stride of O and E
  float alpha, cutoff;
};

__global__ void __launch_bounds__(256) k_ridge_solve(SolveArgs a) {
  const int k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const int J = a.J, K = a.K, B = a.B, C = a.C, d = a.d, D1 = d + 1, M = B + 1;
  __shared__ int sh_m;       // kept levels + 1
  __shared__ float sh_f[4];
  __shared__ int sh_piv;
  float* G = a.scratch + (size_t)k * (2 * (size_t)M * M + (size_t)M * d);
  float* inv = G + (size_t)M * M;
  float* sv = inv + (size_t)M * M;  // [m][d]
  int* pos = a.iscratch + (size_t)k * (2 * B + J);  // level -> kept index (or -1)
  int* keep = pos + B;                              // kept index -> level
  int* part = keep + B;                             // tuple participates?

  // ---- level filter (:358-410)
  extern __shared__ int sh_i[];  // [B] over-cutoff flags, [C] levels above the cutoff per covariate
  int* over = sh_i;
  int* cov_levels = sh_i + B;
  for (int c = tid; c < C; c += nt) cov_levels[c] = 0;
  __syncthreads();
  for (int b = tid; b < B; b += nt) {
    int ov = ((a.O[(size_t)b * a.KS + k] / a.N_b[b]) > a.cutoff) ? 1 : 0;
    over[b] = ov;
    if (ov) atomicAdd(&cov_levels[a.cov_of[b]], 1);
  }
  __syncthreads();
  if (tid == 0) {
    int nkeep = 0;
    for (int b = 0; b < B; ++b) {
      if (over[b] && cov_levels[a.cov_of[b]] > 1) {
        pos[b] = nkeep;
        keep[nkeep] = b;
        nkeep++;
      } else {
        pos[b] = -1;
      }
    }
    sh_m = nkeep + 1;
    a.skipped[k] = (nkeep == 0) ? 1 : 0;
  }
  __syncthreads();
  const int m = sh_m;
  float* Wk = a.Wfull + (size_t)k * M * d;
  if (m == 1) {  // no active covariate (:449-452): cluster untouched, Y[k] keeps its value
    for (int idx = tid; idx < J * d; idx += nt) {
      int q = idx / d, c = idx - q * d;
      a.V[((size_t)q * K + k) * d + c] = 0.f;
    }
    for (int idx = tid; idx < M * d; idx += nt) Wk[idx] = 0.f;
    return;
  }
  // ---- participating tuples, zero G and s
  for (int q = tid; q < J; q += nt) {
    int p = 0;
    for (int c = 0; c < C; ++c) p |= (pos[a.tuple_levels[q * C + c]] >= 0);
    part[q] = p;
  }
  for (int idx = tid; idx < m * m; idx += nt) G[idx] = 0.f;
  __syncthreads();
  // ---- G = Phi* diag(R_k) Phi*^T (:561-567) folded from the per-tuple sums n_kq = S[q][k][d]
  for (int q = tid; q < J; q += nt) {
    if (!part[q]) continue;
    float nq = a.S[((size_t)q * K + k) * D1 + d];
    atomicAdd(&G[0], nq);
    for (int c1 = 0; c1 < C; ++c1) {
      int p1 = pos[a.tuple_levels[q * C + c1]];
      if (p1 < 0) continue;
      atomicAdd(&G[(size_t)(p1 + 1) * m], nq);  // row 0
      atomicAdd(&G[(size_t)(p1 + 1)], nq);      // col 0
      for (int c2 = 0; c2 < C; ++c2) {
        int p2 = pos[a.tuple_levels[q * C + c2]];
        if (p2 < 0) continue;
        atomicAdd(&G[(size_t)(p2 + 1) * m + (p1 + 1)], nq);
      }
    }
  }
  // ---- s = Phi* diag(R_k) Zo^T: thread per embedding column, serial over tuples (no atomics)
  for (int c = tid; c < d; c += nt) {
    for (int r = 0; r < m; ++r) sv[(size_t)r * d + c] = 0.f;
    for (int q = 0; q < J; ++q) {
      if (!part[q]) continue;
      float v = a.S[((size_t)q * K + k) * D1 + c];
      sv[c] += v;
      for (int c1 = 0; c1 < C; ++c1) {
        int p1 = pos[a.tuple_levels[q * C + c1]];
        if (p1 >= 0) sv[(size_t)(p1 + 1) * d + c] += v;
      }
    }
  }
  __syncthreads();
  // ---- + diag(lambda): lambda_0 = 0, lambda_b = alpha*E_kb (find_lambda_cpp) or the fixed vector
  for (int j = tid; j < m - 1; j += nt) {
    int b = keep[j];
    float lam = a.lambda ? a.lambda[b + 1] : a.E[(size_t)b * a.KS + k] * a.alpha;
    G[(size_t)(j + 1) * m + (j + 1)] += lam;
  }
  if (tid == 0 && a.lambda) G[0] += a.lambda[0];
  __syncthreads();
  // ---- inverse
  if (C == 1) {
    // arrowhead closed form (:575-586)
    if (tid == 0) {
      float accum = 0.f;
      for (int j = 1; j < m; ++j) {
        float ac = -G[(size_t)j * m];
        float bj = 1.f / G[(size_t)j * m + j];
        accum += (ac * ac) * bj;
      }
      sh_f[0] = G[0] - accum;  // u
    }
    __syncthreads();
    const float u = sh_f[0];
    for (int idx = tid; idx < m * m; idx += nt) {
      int r = idx % m, c = idx / m;
      float acr = (r == 0) ? 1.f : (-G[(size_t)r * m]) * (1.f / G[(size_t)r * m + r]);
      float acc_ = (c == 0) ? 1.f : (-G[(size_t)c * m]) * (1.f / G[(size_t)c * m + c]);
      float v = (1.f / u) * (acr * acc_);
      if (r == c && r > 0) v += 1.f / G[(size_t)r * m + r];
      inv[idx] = v;
    }
    __syncthreads();
  } else {
    // Gauss-Jordan with partial pivoting (arma::inv -> getrf/getri, :573); column-major m x m
    for (int idx = tid; idx < m * m; idx += nt) inv[idx] = ((idx % m) == (idx / m)) ? 1.f : 0.f;
    __syncthreads();
    for (int c = 0; c < m; ++c) {
      if (tid == 0) {
        int piv = c;
        float best = fabsf(G[c + (size_t)c * m]);
        for (int r = c + 1; r < m; ++r) {
          float v = fabsf(G[r + (size_t)c * m]);
          if (v > best) {
            best = v;
            piv = r;
          }
        }
        sh_piv = piv;
        if (!(best > 0.f) || !isfinite(best)) atomicExch(a.err_flag, 2);
      }
      __syncthreads();
      const int piv = sh_piv;
      if (piv != c) {
        for (int j = tid; j < m; j += nt) {
          float t = G[c + (size_t)j * m];
          G[c + (size_t)j * m] = G[piv + (size_t)j * m];
          G[piv + (size_t)j * m] = t;
          t = inv[c + (size_t)j * m];
          inv[c + (size_t)j * m] = inv[piv + (size_t)j * m];
          inv[piv + (size_t)j * m] = t;
        }
        __syncthreads();
      }
      if (tid == 0) sh_f[1] = G[c + (size_t)c * m];
      __syncthreads();
      const float p = sh_f[1];
      for (int j = tid; j < m; j += nt) {
        G[c + (size_t)j * m] /= p;
        inv[c + (size_t)j * m] /= p;
      }
      __syncthreads();
      // eliminate column c from every other row: thread per (row, col) pair
      // first snapshot the factors (column c of G) into sv's tail? use registers per row instead:
      for (int idx = tid; idx < m * m; idx += nt) {
        int r = idx % m, j = idx / m;
        if (r == c) continue;
        float f = G[r + (size_t)c * m];
        if (j == c) continue;  // column c itself is cleared afterwards
        G[r + (size_t)j * m] -= f * G[c + (size_t)j * m];
      }
      for (int idx = tid; idx < m * m; idx += nt) {
        int r = idx % m, j = idx / m;
        if (r == c) continue;
        float f = G[r + (size_t)c * m];
        inv[r + (size_t)j * m] -= f * inv[c + (size_t)j * m];
      }
      __syncthreads();
      for (int r = tid; r < m; r += nt)
        if (r != c) G[r + (size_t)c * m] = 0.f;
      __syncthreads();
    }
  }
  // ---- W = inv * s  (:599-609), Y[k] = W[0] (:610), W[0] = 0 (:611)
  for (int idx = tid; idx < M * d; idx += nt) Wk[idx] = 0.f;
  __syncthreads();
  for (int idx = tid; idx < m * d; idx += nt) {
    int r = idx / d, c = idx - r * d;
    float w = 0.f;
    for (int j = 0; j < m; ++j) w += inv[r + (size_t)j * m] * sv[(size_t)j * d + c];
    if (r == 0)
      a.Y[(size_t)k * d + c] = w;
    else
      Wk[(size_t)(keep[r - 1] + 1) * d + c] = w;
  }
  __syncthreads();
  // ---- Y = normalise(Y, 2, 0) (:633) for this column
  if (tid < 32) {
    float s = 0.f;
    for (int c = tid; c < d; c += 32) {
      float v = a.Y[(size_t)k * d + c];
      s += v * v;
    }
    s = warp_sum(s);
    float nrm = sqrtf(s);
    if (nrm == 0.f) nrm = 1.f;
    for (int c = tid; c < d; c += 32) a.Y[(size_t)k * d + c] /= nrm;
  }
  // ---- V[q][k] = sum of the kept levels' betas of tuple q (0 for tuples that do not take part)
  for (int idx = tid; idx < J * d; idx += nt) {
    int q = idx / d, c = idx - q * d;
    float v = 0.f;
    if (part[q])
      for (int c1 = 0; c1 < C; ++c1) {
        int b = a.tuple_levels[q * C + c1];
        if (pos[b] >= 0) v += Wk[(size_t)(b + 1) * d + c];
      }
    a.V[((size_t)q * K + k) * d + c] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// K5: apply (harmony.cpp:347 + :615 for all clusters): Zc_i = Zo_i - sum_k R_ik V[q(i)][k][:]
// thread (ty, tx) owns cells ty*4..+3 x columns tx*4..+3 of a TM-cell tile.
// ------------------------------------------------------------------------------------------------
struct ApplyArgs {
  const float* R;
  const float* Zo;
  const float* V;  // [J][K][d]
  float* Zc;
  const int* tile_cell0;
  const int* tile_len;
  const int* tile_tuple;
  int ntiles, d, K, tiles_per_cta;
  int ldR, ldZ;
};

__global__ void k_ridge_apply(ApplyArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int d = a.d, K = a.K;
  const int DP = (d + 3) & ~3, KP4 = (K + 3) & ~3;
  float* Vs = smem;                      // [KP4][DP]  (rows >= K and columns >= d are zero)
  float* Rs = Vs + (size_t)KP4 * DP;     // [TM][KP4]
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int tid = ty * blockDim.x + tx, nthr = blockDim.x * blockDim.y;
  int cur_q = -1;
  const int t_begin = blockIdx.x * a.tiles_per_cta;
  const int t_end = (t_begin + a.tiles_per_cta < a.ntiles) ? t_begin + a.tiles_per_cta : a.ntiles;
  for (int tile = t_begin; tile < t_end; ++tile) {
    const int cell0 = a.tile_cell0[tile], len = a.tile_len[tile], q = a.tile_tuple[tile];
    __syncthreads();
    if (q != cur_q) {
      for (int idx = tid; idx < KP4 * DP; idx += nthr) {
        int k = idx / DP, c = idx - k * DP;
        Vs[idx] = (c < d && k < K) ? a.V[((size_t)q * K + k) * d + c] : 0.f;
      }
      cur_q = q;
    }
    for (int idx = tid; idx < TM * KP4; idx += nthr) {
      int r = idx / KP4, k = idx - r * KP4;
      Rs[idx] = (r < len && k < K) ? ld_stream(a.R + (size_t)(cell0 + r) * a.ldR + k) : 0.f;
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const float* rp = Rs + (size_t)(ty * 4) * KP4;
    const float* vp = Vs + tx * 4;
    for (int k = 0; k < KP4; k += 4) {
      float4 r4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) r4[i] = *reinterpret_cast<const float4*>(rp + (size_t)i * KP4 + k);
#pragma unroll
      for (int jk = 0; jk < 4; ++jk) {
        float4 v4 = *reinterpret_cast<const float4*>(vp + (size_t)(k + jk) * DP);
        float vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float rr = (jk == 0) ? r4[i].x : (jk == 1) ? r4[i].y : (jk == 2) ? r4[i].z : r4[i].w;
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(rr, vv[j], acc[i][j]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int r = ty * 4 + i;
      if (r < len) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int c = tx * 4 + j;
          if (c < d) {
            size_t g = (size_t)(cell0 + r) * a.ldZ + c;
            a.Zc[g] = a.Zo[g] - acc[i][j];
          }
        }
      }
    }
  }
}

}  // namespace hb
