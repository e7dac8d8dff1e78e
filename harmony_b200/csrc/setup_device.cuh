// setup_device.cuh — the covariate tuple dictionary of hb_setup built on the device (hb_setup_device, inputs already in
// device memory).  It produces what the host dictionary produces, bit for bit: tuple ids in ascending key order and a
// STABLE sort of the cells by tuple.  The sort is the plan builder's counting sort (k_plan_hist / k_scan_chained /
// k_plan_scatter) with the tuple id as the key: chunks of consecutive cells, chunk_q0 = 0 and nsub = 1 lay the
// histogram out as H[tuple][chunk], whose exclusive scan is the first position of every (tuple, chunk).
#pragma once
#include "kernels.cuh"

namespace hb {

// Per cell: mixed-radix key of its levels and presence of the key.  lv = [C][3] ints (first global row, number of
// levels, radix) of every covariate; the key space is at most 2^22, so keys and radices fit an int.  A level outside
// its covariate's rows records the lowest (cell * C + covariate) in *bad (atomicMin; the host path reports the first
// bad level it meets, i.e. that one) and leaves the cell out of the table, so nothing is indexed out of range.
__global__ void k_dict_keys(const int32_t* __restrict__ phi_i, int64_t n, int C, const int* __restrict__ lv,
                            int* __restrict__ key, int* __restrict__ present, unsigned long long* __restrict__ bad) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int kk = 0;
    bool ok = true;
    for (int c = 0; c < C; ++c) {
      const int b = phi_i[i * C + c], b0 = lv[3 * c];
      if (b < b0 || b >= b0 + lv[3 * c + 1]) {
        atomicMin(bad, (unsigned long long)(i * C + c));
        ok = false;
        break;
      }
      kk += (b - b0) * lv[3 * c + 2];
    }
    key[i] = ok ? kk : 0;
    if (ok) present[kk] = 1;
  }
}

// After the exclusive scan of the presence table (ids[k] = tuple id of key k, ids[key_space] = J): the unique keys in
// ascending order (uniq[ids[k]] = k for every present k) and every cell's tuple id in place of its key.
__global__ void k_dict_tuples(const int* __restrict__ ids, int64_t key_space, int* __restrict__ uniq,
                              int* __restrict__ key, int64_t n) {
  const int64_t m = key_space > n ? key_space : n;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < key_space && ids[i + 1] != ids[i]) uniq[ids[i]] = (int)i;
    if (i < n) key[i] = ids[key[i]];
  }
}

// Chunk tables of the counting sort: chunk c holds cells [c * CH, (c + 1) * CH).
__global__ void k_dict_chunks(int nchunks, int CH, int64_t n, int* __restrict__ chunk_start, int* __restrict__ cq0,
                              int* __restrict__ cnq) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c <= nchunks; c += gridDim.x * blockDim.x) {
    chunk_start[c] = (int)((int64_t)c * CH < n ? (int64_t)c * CH : n);
    if (c < nchunks) {
      cq0[c] = 0;
      cnq[c] = 1;
    }
  }
}

// inv_sort[sort_perm[s]] = s; tstart[q] = first position of tuple q (H scanned, [J][nchunks]), tstart[J] = n.
__global__ void k_dict_finish(const int* __restrict__ sort_perm, int* __restrict__ inv_sort, int64_t n,
                              const int* __restrict__ H, int nchunks, int J, int* __restrict__ tstart) {
  const int64_t m = n > (int64_t)J + 1 ? n : (int64_t)J + 1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < n) inv_sort[sort_perm[i]] = (int)i;
    if (i < J) tstart[i] = H[i * nchunks];
    if (i == J) tstart[i] = (int)n;
  }
}

}  // namespace hb
