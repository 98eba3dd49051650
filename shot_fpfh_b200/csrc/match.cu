// Kernel group M (everything except the tcgen05 GEMM, which lives in match_tc.cu):
//   M0 nonempty_kernel / sf_nonempty_rows <- np.any(desc, axis=1).nonzero()[0], matching.py:43-44, :162-163
//   M0 pack_kernel    : float64 rows -> float16 GEMM operands + float32 squared norms of the rounded rows
//   M1 topk_simt_kernel: CUDA-core shortlist kernel (cross-check of the tensor-core kernel, small problems)
//   M2 rerank_kernel  <- cdist(...).argmin(axis=1) and the nearest / second-nearest distances,
//                        matching.py:47-52, :164-168, :197-211: exact float64, sequential accumulation like SciPy
//   topk_merge_kernel : k-way merge of per-shard shortlists (after the all-gather when targets are sharded)
#include <cub/cub.cuh>
#include <cuda_fp16.h>

#include "sf_common.cuh"

namespace sf {

int launch_topk_tc(const __half* a, int64_t qa, const __half* b, const float* bnorm, int64_t qb, int width_padded,
                   int k, int index_offset, float* score, int32_t* idx, cudaStream_t stream);  // match_tc.cu

// absmax (optional): bit pattern of the largest |x| of the array, raised with an integer atomicMax (non-negative
// doubles order like their bit patterns; a NaN's pattern is above infinity's, so one NaN or infinity anywhere shows)
__global__ void __launch_bounds__(256)
    nonempty_kernel(const double* __restrict__ desc, int64_t n, int width, uint8_t* __restrict__ flags,
                    unsigned long long* __restrict__ absmax) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (row >= n) return;
  bool any = false;
  unsigned long long top = 0ull;
  for (int c = lane; c < width; c += 32) {
    const double v = desc[row * width + c];
    any |= v != 0.0;  // NaN counts as non-zero, like np.any
    const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(fabs(v)));
    top = bits > top ? bits : top;
  }
  any = __any_sync(kFull, any);
  if (lane == 0) flags[row] = any;
  if (absmax != nullptr) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(kFull, top, o);
      top = other > top ? other : top;
    }
    if (lane == 0 && top != 0ull) atomicMax(absmax, top);
  }
}

__global__ void __launch_bounds__(256)
    pack_kernel(const double* __restrict__ desc, int width, const int64_t* __restrict__ rows, int64_t count,
                double scale, __half* __restrict__ packed, int width_padded, float* __restrict__ sqnorm) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (r >= count) return;
  const double* src = desc + rows[r] * width;
  float acc = 0.0f;
  for (int c = lane; c < width_padded; c += 32) {
    const __half h = c < width ? __double2half(src[c] * scale) : __float2half(0.0f);
    packed[r * width_padded + c] = h;
    const float f = __half2float(h);
    acc += f * f;
  }
  acc = warp_sum(acc);
  if (lane == 0) sqnorm[r] = acc;
}

// ---- running top-k of (score, index), ascending, ties broken by the lower index ----------------------------
template <int K>
struct TopK {
  float s[K];
  int i[K];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int k = 0; k < K; ++k) { s[k] = INFINITY; i[k] = -1; }
  }
  __device__ __forceinline__ bool before(float sa, int ia, float sb, int ib) const {
    return sa < sb || (sa == sb && unsigned(ia) < unsigned(ib));
  }
  __device__ __forceinline__ void push(float score, int index) {
    if (!before(score, index, s[K - 1], i[K - 1])) return;
    s[K - 1] = score; i[K - 1] = index;
#pragma unroll
    for (int k = K - 1; k > 0; --k) {
      if (before(s[k], i[k], s[k - 1], i[k - 1])) {
        const float ts = s[k]; s[k] = s[k - 1]; s[k - 1] = ts;
        const int ti = i[k]; i[k] = i[k - 1]; i[k - 1] = ti;
      }
    }
  }
};

// ---- M1 (CUDA cores): 64 queries x 64 targets per tile, 4x4 micro-tiles, float32 accumulation ---------------
template <int K>
__global__ void __launch_bounds__(256)
    topk_simt_kernel(const __half* __restrict__ a, int64_t qa, const __half* __restrict__ b,
                     const float* __restrict__ bnorm, int64_t qb, int wp, int index_offset,
                     float* __restrict__ score, int32_t* __restrict__ idx) {
  __shared__ float sa[32][64 + 1];
  __shared__ float sb[32][64 + 1];
  __shared__ float sc[64][64 + 1];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // micro-tile: rows ty*4.., cols tx*4..
  const int64_t row0 = blockIdx.x * int64_t(64);
  TopK<K> top;
  top.init();
  for (int64_t col0 = 0; col0 < qb; col0 += 64) {
    float acc[4][4] = {};
    for (int k0 = 0; k0 < wp; k0 += 32) {
      for (int e = tid; e < 64 * 32; e += 256) {
        const int r = e >> 5, c = e & 31;
        sa[c][r] = row0 + r < qa ? __half2float(a[(row0 + r) * wp + k0 + c]) : 0.0f;
        sb[c][r] = col0 + r < qb ? __half2float(b[(col0 + r) * wp + k0 + c]) : 0.0f;
      }
      __syncthreads();
#pragma unroll 8
      for (int c = 0; c < 32; ++c) {
        float av[4], bv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { av[u] = sa[c][ty * 4 + u]; bv[u] = sb[c][tx * 4 + u]; }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(av[u], bv[v], acc[u][v]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int64_t col = col0 + tx * 4 + v;
        sc[ty * 4 + u][tx * 4 + v] = col < qb ? fmaf(-2.0f, acc[u][v], bnorm[col]) : INFINITY;
      }
    __syncthreads();
    if (tid < 64) {
      const int ncols = int(qb - col0 < 64 ? qb - col0 : 64);
      for (int c = 0; c < ncols; ++c) top.push(sc[tid][c], int(col0 + c) + index_offset);
    }
    __syncthreads();
  }
  if (tid < 64 && row0 + tid < qa) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      score[(row0 + tid) * K + k] = top.s[k];
      idx[(row0 + tid) * K + k] = top.i[k];
    }
  }
}

template <int K>
__global__ void __launch_bounds__(128)
    topk_merge_kernel(const float* __restrict__ score, const int32_t* __restrict__ idx, int parts, int64_t qa,
                      float* __restrict__ score_out, int32_t* __restrict__ idx_out) {
  const int64_t q = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (q >= qa) return;
  TopK<K> top;
  top.init();
  for (int p = 0; p < parts; ++p)
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int64_t o = (int64_t(p) * qa + q) * K + k;
      const int id = idx[o];
      if (id >= 0) top.push(score[o], id);
    }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    score_out[q * K + k] = top.s[k];
    idx_out[q * K + k] = top.i[k];
  }
}

// ---- M2: exact float64 re-rank, one warp per query row -----------------------------------------------------
// SciPy's cdist accumulates s += (u[e] - v[e])^2 sequentially in e, without FMA; the argmin (and the distances the
// filters see) are only bit-identical if the sums are formed in that order. The squares are order-independent, so
// the 32 lanes compute them for 32 columns at a time with coalesced row loads and park them in shared memory;
// lane c then folds the 32 squares of candidate c in ascending column order. Columns past the width contribute
// exact zeros (s + 0.0 == s).
constexpr int kRerankWarps = 8;
constexpr int kRerankMaxK = 16;

__global__ void __launch_bounds__(kRerankWarps * 32)
    rerank_kernel(const double* __restrict__ a, const int64_t* __restrict__ rows_a, int64_t qa,
                  const double* __restrict__ b, const int64_t* __restrict__ rows_b, int width,
                  const int32_t* __restrict__ cand, int k, int32_t* __restrict__ nn, double* __restrict__ d1,
                  double* __restrict__ d2) {
  __shared__ double squares[kRerankWarps][kRerankMaxK][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t q = blockIdx.x * int64_t(kRerankWarps) + warp;
  if (q >= qa) return;
  const double* ra = a + (rows_a ? rows_a[q] : q) * width;
  int my_id = -1;
  int64_t my_row = 0;
  if (lane < k) {
    my_id = cand[q * k + lane];
    if (my_id >= 0) my_row = rows_b ? rows_b[my_id] : int64_t(my_id);
  }
  double s = 0.0;
  for (int e0 = 0; e0 < width; e0 += 32) {
    const int e = e0 + lane;
    const double av = e < width ? ra[e] : 0.0;
    for (int c = 0; c < k; ++c) {
      const int id = __shfl_sync(kFull, my_id, c);
      const int64_t row = __shfl_sync(kFull, my_row, c);
      double sq = 0.0;
      if (id >= 0 && e < width) {
        const double d = av - b[row * width + e];
        sq = mul_rn(d, d);
      }
      squares[warp][c][lane] = sq;
    }
    __syncwarp();
    if (lane < k) {
#pragma unroll 8
      for (int t = 0; t < 32; ++t) s = add_rn(s, squares[warp][lane][t]);
    }
    __syncwarp();
  }
  const double my_dist = my_id >= 0 ? sqrt(s) : INFINITY;
  double best = INFINITY, second = INFINITY;
  int best_idx = -1;
  for (int c = 0; c < k; ++c) {  // every lane runs the same selection on the broadcast results
    const double dist = __shfl_sync(kFull, my_dist, c);
    const int id = __shfl_sync(kFull, my_id, c);
    if (id < 0) continue;
    if (dist < best || (dist == best && id < best_idx)) {
      second = best;
      best = dist;
      best_idx = id;
    } else if (dist < second) {
      second = dist;
    }
  }
  if (lane == 0) {
    nn[q] = best_idx;
    if (d1) d1[q] = best;
    if (d2) d2[q] = second;
  }
}

// ---- certificate of the float16 shortlist ------------------------------------------------------------------------
// The shortlist kernel ranks targets by score(b) = |b~|^2 - 2 a~.b~ on the float16-rounded, scaled rows a~ = fl16(s a),
// b~ = fl16(s b), so |a~ - b~|^2 = score + |a~|^2, and every target OUTSIDE a query's k-entry shortlist has
// score >= score_k. Bounds (u16 = 2^-11 relative rounding of a normal half, 2^-25 absolute below 2^-14; float32
// accumulation of `width` products, allowed twice the rounding-to-nearest bound for the tensor core's accumulator):
//   |a~ - b~| >= sqrt(max(0, score_k + |a~|^2 - 1e-4 (|a~| B + B^2))),   B = max |b~|
//   s |a - b| >= |a~ - b~| - 2^-11 (1 + 2^-10) (|a~| + B) - 2 sqrt(width) 2^-25
// A query is certified when its exact nearest (and, when asked, second-nearest) distance from the re-rank is strictly
// below that bound on everything outside the shortlist: the re-rank then saw the true nearest neighbours. The others
// (adversarial near-ties, rows that quantise to 0, ...) are flagged and redone exhaustively in float64.
__global__ void __launch_bounds__(256)
    certify_kernel(const float* __restrict__ score, int k, const float* __restrict__ a_sqnorm, const double* __restrict__ d1,
                   const double* __restrict__ d2, int64_t qa, double scale, double b_norm_max, int width, int64_t qb,
                   int want_second, uint8_t* __restrict__ flags) {
  const int64_t q = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (q >= qa) return;
  bool ok;
  if (qb <= k) {
    ok = true;  // every target is in the shortlist
  } else {
    const double sk = double(score[q * k + (k - 1)]), a2 = double(a_sqnorm[q]), an = sqrt(a2);
    const double lower2 = sk + a2 - 1e-4 * (an * b_norm_max + b_norm_max * b_norm_max);
    const double eps = 4.8828125e-4 * 1.001 * (an + b_norm_max) + 2.0 * sqrt(double(width)) * 2.98e-8;
    const double outside = sqrt(fmax(lower2, 0.0)) - eps;  // scaled distance to anything outside the shortlist
    const double need = want_second ? d2[q] : d1[q];
    ok = isfinite(sk) ? (scale * need < outside) : true;  // (infinite score_k: fewer than k finite scores)
    ok = ok && !(need != need) && !(sk != sk);
  }
  flags[q] = ok ? 0 : 1;
}

// Exhaustive float64 shortlist for the flagged queries: block per query, warps over the targets, lanes over the
// columns; the k smallest squared distances (any summation order: the exact re-rank decides among them, and exact
// ties carry identical values here) with the lowest index on ties.
template <int K>
__global__ void __launch_bounds__(256)
    exhaustive_topk_kernel(const double* __restrict__ a, const int64_t* __restrict__ rows_a,
                           const int64_t* __restrict__ which, int64_t n_which, const double* __restrict__ b,
                           const int64_t* __restrict__ rows_b, int64_t qb, int width, int32_t* __restrict__ cand) {
  __shared__ float ws[8][K];
  __shared__ int wi[8][K];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t item = blockIdx.x;
  if (item >= n_which) return;
  const int64_t q = which[item];
  const double* ra = a + (rows_a ? rows_a[q] : q) * width;
  // float32 images only ORDER the candidates of a warp before the merge; the distances themselves are float64 below
  double best_d[K];
  int best_i[K];
#pragma unroll
  for (int t = 0; t < K; ++t) { best_d[t] = INFINITY; best_i[t] = -1; }
  for (int64_t j = warp; j < qb; j += 8) {
    const double* rb = b + (rows_b ? rows_b[j] : j) * width;
    double s = 0.0;
    for (int e = lane; e < width; e += 32) {
      const double d = ra[e] - rb[e];
      s = fma(d, d, s);
    }
    s = warp_sum(s);
    // every lane keeps the same sorted list (ascending distance, then index)
    if (s < best_d[K - 1] || (s == best_d[K - 1] && int(j) < best_i[K - 1]) || best_i[K - 1] < 0) {
      if (!(s != s)) {
        best_d[K - 1] = s; best_i[K - 1] = int(j);
#pragma unroll
        for (int t = K - 1; t > 0; --t) {
          const bool swap = best_i[t - 1] < 0 || best_d[t] < best_d[t - 1] || (best_d[t] == best_d[t - 1] && best_i[t] < best_i[t - 1]);
          if (swap) {
            const double td = best_d[t]; best_d[t] = best_d[t - 1]; best_d[t - 1] = td;
            const int ti = best_i[t]; best_i[t] = best_i[t - 1]; best_i[t - 1] = ti;
          }
        }
      }
    }
  }
  __shared__ double wd[8][K];
  if (lane == 0) {
#pragma unroll
    for (int t = 0; t < K; ++t) { wd[warp][t] = best_d[t]; wi[warp][t] = best_i[t]; }
  }
  (void)ws;
  __syncthreads();
  if (threadIdx.x == 0) {  // merge the eight sorted lists
    int head[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int t = 0; t < K; ++t) {
      int pick = -1;
      for (int w = 0; w < 8; ++w) {
        if (head[w] >= K || wi[w][head[w]] < 0) continue;
        if (pick < 0 || wd[w][head[w]] < wd[pick][head[pick]] ||
            (wd[w][head[w]] == wd[pick][head[pick]] && wi[w][head[w]] < wi[pick][head[pick]]))
          pick = w;
      }
      cand[q * K + t] = pick >= 0 ? wi[pick][head[pick]] : -1;
      if (pick >= 0) ++head[pick];
    }
  }
}

// The exhaustive redo as ONE pass over the targets for all the flagged queries together. Only targets at most `limit[q]`
// away matter — the exact nearest (second-nearest) distance the re-rank already found bounds the true one from above —
// and the float64 re-rank decides among them afterwards, so this pass only has to FIND them: it runs in float32 on the
// CUDA cores with a proven slack (first form: float64, a warp per query against 32 staged target rows, one broadcast
// load per element: 21 ms for 514 flagged queries x 200k targets, as long as the tensor-core shortlist of all 200k).
//   * distances are accumulated as sum (a_i - b_i)^2 on the float32 images of the rows — not as |a|^2 + |b|^2 - 2 a.b,
//     whose error scales with the norms and not with the distance (the flagged queries ARE the near-duplicates);
//   * |fl32(a) - a| <= u |a| element-wise (u = 2^-24), so the distance of the images differs from the true one by at
//     most u (|a| + |b|) <= u * norm_bound; a sum of n squares accumulated in float32 is within (n + 2) u of itself,
//     relatively. A target is listed when   s <= (limit + 2 u norm_bound)^2 * (1 + (n + 8) 2^-23):   never misses one
//     that is within `limit`, lists a few more than the float64 test would;
//   * a block computes 64 flagged queries x 64 targets, 4 x 4 per thread, from shared-memory tiles of 32 columns.
// The list is capped at kExhaustiveCap; the selection below keeps at most 16 and marks longer lists for the
// block-per-query float64 kernel above.
constexpr int kExhaustiveCap = 64;
constexpr int kEx32Rows = 64, kEx32Cols = 32;

__global__ void __launch_bounds__(256)
    exhaustive_tile32_kernel(const double* __restrict__ a, const int64_t* __restrict__ rows_a,
                             const int64_t* __restrict__ which, int64_t n_which, const double* __restrict__ limit,
                             const double* __restrict__ b, const int64_t* __restrict__ rows_b, int64_t qb, int width,
                             double scale, double norm_bound, int32_t* __restrict__ counts,
                             double* __restrict__ list_d, int32_t* __restrict__ list_i) {
  // scale: the power of two that brings the largest |entry| of both sets just below 1 (the float16 operands' scale):
  // the rows are multiplied by it (exactly) before they are narrowed, so no square can overflow float32 whatever the
  // caller's units; limit and norm_bound (given in scaled units) follow.
  __shared__ __align__(16) float as[kEx32Cols][kEx32Rows + 4];  // [column][query of the tile]
  __shared__ __align__(16) float bs[kEx32Cols][kEx32Rows + 4];  // [column][target of the tile]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;  // 4 targets 4 tx.., 4 queries 4 ty..
  const int64_t j0 = blockIdx.x * int64_t(kEx32Rows), i0 = blockIdx.y * int64_t(kEx32Rows);
  // the rows this thread stages: row (tid >> 2) of both tiles, 8 of the 32 columns of a chunk (coalesced 64-byte pieces)
  const int load_row = tid >> 2, load_col = (tid & 3) * 8;
  const int64_t item_l = i0 + load_row, j_l = j0 + load_row;
  const double* src_a = item_l < n_which ? a + (rows_a ? rows_a[which[item_l]] : which[item_l]) * width : nullptr;
  const double* src_b = j_l < qb ? b + (rows_b ? rows_b[j_l] : j_l) * width : nullptr;
  float acc[4][4] = {};
  for (int c0 = 0; c0 < width; c0 += kEx32Cols) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int c = c0 + load_col + e;
      as[load_col + e][load_row] = (src_a != nullptr && c < width) ? float(__ldg(src_a + c) * scale) : 0.0f;
      bs[load_col + e][load_row] = (src_b != nullptr && c < width) ? float(__ldg(src_b + c) * scale) : 0.0f;
    }
    __syncthreads();
#pragma unroll 8
    for (int c = 0; c < kEx32Cols; ++c) {
      const float4 av = *reinterpret_cast<const float4*>(&as[c][4 * ty]);
      const float4 bv = *reinterpret_cast<const float4*>(&bs[c][4 * tx]);
      const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const float d = a4[u] - b4[v];
          acc[u][v] = fmaf(d, d, acc[u][v]);
        }
    }
    __syncthreads();
  }
  // (+ 1e-30: entries that underflow float32 after the scaling are off by at most 2^-150 each)
  const double slack = 2.0 * 5.9604644775390625e-8 * norm_bound + 1e-30, grow = 1.0 + double(width + 8) * 1.1920928955078125e-7;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t item = i0 + 4 * ty + u;
    if (item >= n_which) continue;
    const double lim = limit[item] * scale + slack, bound = lim * lim * grow;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int64_t j = j0 + 4 * tx + v;
      if (j < qb && double(acc[u][v]) <= bound) {
        const int slot = atomicAdd(counts + item, 1);
        if (slot < kExhaustiveCap) {
          list_d[item * kExhaustiveCap + slot] = double(acc[u][v]);
          list_i[item * kExhaustiveCap + slot] = int32_t(j);
        }
      }
    }
  }
}

// The listed targets of each flagged query in (float32 distance, index) order, -1 padded — all of them go to the float64
// re-rank, so the order only matters to nobody; cand[item][0] = -2 marks a list longer than the 16 the re-rank takes.
__global__ void exhaustive_select_kernel(int64_t n_which, const int32_t* __restrict__ counts,
                                         const double* __restrict__ list_d, const int32_t* __restrict__ list_i,
                                         int32_t* __restrict__ cand) {
  const int64_t item = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (item >= n_which) return;
  const int n = counts[item];
  int32_t* out = cand + item * 16;
  if (n > 16) {
    for (int t = 0; t < 16; ++t) out[t] = t == 0 ? -2 : -1;
    return;
  }
  const double* d = list_d + item * kExhaustiveCap;
  const int32_t* id = list_i + item * kExhaustiveCap;
  double last_d = -1.0;
  int last_i = -1;
  for (int t = 0; t < 16; ++t) {  // selection in (distance, index) order: the list is short
    int pick = -1;
    for (int e = 0; e < n; ++e) {
      const bool after = d[e] > last_d || (d[e] == last_d && id[e] > last_i);
      if (!after) continue;
      if (pick < 0 || d[e] < d[pick] || (d[e] == d[pick] && id[e] < id[pick])) pick = e;
    }
    out[t] = pick >= 0 ? id[pick] : -1;
    if (pick >= 0) { last_d = d[pick]; last_i = id[pick]; }
    else { last_d = INFINITY; }
  }
}

struct IsSet {
  const uint8_t* flags;
  __host__ __device__ bool operator()(int64_t i) const { return flags[i] != 0; }
};

}  // namespace sf

using namespace sf;

extern "C" int sf_nonempty_rows(const double* desc, int64_t n, int32_t width, int64_t* rows, int64_t* count_host,
                                double* absmax_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(desc && rows && count_host && n >= 0 && width > 0, SF_ERR_ARG, "sf_nonempty_rows: bad arguments");
  *count_host = 0;
  if (absmax_host) *absmax_host = 0.0;
  if (n == 0) return SF_OK;
  SF_REQUIRE(n < (int64_t(1) << 31), SF_ERR_ARG, "sf_nonempty_rows: too many rows");
  uint8_t* flags = nullptr;
  int64_t* count_dev = nullptr;
  void* temp = nullptr;
  size_t temp_bytes = 0;
  cub::CountingInputIterator<int64_t> ids(0);
  cub::DeviceSelect::Flagged(nullptr, temp_bytes, ids, flags, rows, count_dev, int(n), stream);
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&flags, size_t(n)));
  SF_CUDA(scratch.alloc(&count_dev, 2 * sizeof(int64_t)));
  SF_CUDA(scratch.alloc(&temp, temp_bytes + 16));
  unsigned long long* absmax_dev = reinterpret_cast<unsigned long long*>(count_dev + 1);
  SF_CUDA(cudaMemsetAsync(absmax_dev, 0, sizeof(unsigned long long), stream));
  nonempty_kernel<<<unsigned((n * 32 + 255) / 256), 256, 0, stream>>>(desc, n, width, flags,
                                                                     absmax_host ? absmax_dev : nullptr);
  SF_CUDA(cub::DeviceSelect::Flagged(temp, temp_bytes, ids, flags, rows, count_dev, int(n), stream));
  SF_CUDA(cudaMemcpyAsync(count_host, count_dev, sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
  if (absmax_host) SF_CUDA(cudaMemcpyAsync(absmax_host, absmax_dev, sizeof(double), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  return SF_OK;
}

extern "C" int sf_match_pack(const double* desc, int32_t width, const int64_t* rows, int64_t count, double scale,
                             void* packed, int32_t width_padded, float* sqnorm, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(desc && rows && packed && sqnorm, SF_ERR_ARG, "sf_match_pack: null argument");
  SF_REQUIRE(width > 0 && width_padded >= width && width_padded % 64 == 0, SF_ERR_ARG,
             "sf_match_pack: width_padded must be a multiple of 64 that is >= width");
  if (count == 0) return SF_OK;
  pack_kernel<<<unsigned((count * 32 + 255) / 256), 256, 0, stream>>>(desc, width, rows, count, scale,
                                                                     static_cast<__half*>(packed), width_padded, sqnorm);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

template <int K>
static int launch_simt(const __half* a, int64_t qa, const __half* b, const float* bnorm, int64_t qb, int wp, int off,
                       float* score, int32_t* idx, cudaStream_t stream) {
  topk_simt_kernel<K><<<unsigned((qa + 63) / 64), 256, 0, stream>>>(a, qa, b, bnorm, qb, wp, off, score, idx);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_match_topk(const void* a, int64_t qa, const void* b, const float* bnorm, int64_t qb,
                             int32_t width_padded, int32_t k, int32_t index_offset, float* score, int32_t* idx,
                             int32_t use_tensor_cores, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(a && b && bnorm && score && idx, SF_ERR_ARG, "sf_match_topk: null argument");
  SF_REQUIRE(width_padded > 0 && width_padded % 64 == 0, SF_ERR_ARG, "sf_match_topk: width_padded %% 64 != 0");
  SF_REQUIRE(k == 1 || k == 2 || k == 4 || k == 8 || k == 16, SF_ERR_CAPACITY, "sf_match_topk: k must be 1,2,4,8,16");
  SF_REQUIRE(qb + int64_t(index_offset) < (int64_t(1) << 31), SF_ERR_ARG, "sf_match_topk: target index overflow");
  if (qa == 0) return SF_OK;
  const __half* ha = static_cast<const __half*>(a);
  const __half* hb = static_cast<const __half*>(b);
  if (use_tensor_cores)
    return launch_topk_tc(ha, qa, hb, bnorm, qb, width_padded, k, index_offset, score, idx, stream);
  switch (k) {
    case 1: return launch_simt<1>(ha, qa, hb, bnorm, qb, width_padded, index_offset, score, idx, stream);
    case 2: return launch_simt<2>(ha, qa, hb, bnorm, qb, width_padded, index_offset, score, idx, stream);
    case 4: return launch_simt<4>(ha, qa, hb, bnorm, qb, width_padded, index_offset, score, idx, stream);
    case 8: return launch_simt<8>(ha, qa, hb, bnorm, qb, width_padded, index_offset, score, idx, stream);
    default: return launch_simt<16>(ha, qa, hb, bnorm, qb, width_padded, index_offset, score, idx, stream);
  }
}

template <int K>
static int launch_merge(const float* score, const int32_t* idx, int parts, int64_t qa, float* so, int32_t* io,
                        cudaStream_t stream) {
  topk_merge_kernel<K><<<unsigned((qa + 127) / 128), 128, 0, stream>>>(score, idx, parts, qa, so, io);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

namespace sf {
int launch_merge_partials(const float* score, const int32_t* idx, int parts, int64_t qa, int k, float* score_out,
                          int32_t* idx_out, cudaStream_t stream) {
  switch (k) {
    case 1: return launch_merge<1>(score, idx, parts, qa, score_out, idx_out, stream);
    case 2: return launch_merge<2>(score, idx, parts, qa, score_out, idx_out, stream);
    case 4: return launch_merge<4>(score, idx, parts, qa, score_out, idx_out, stream);
    case 8: return launch_merge<8>(score, idx, parts, qa, score_out, idx_out, stream);
    default: return launch_merge<16>(score, idx, parts, qa, score_out, idx_out, stream);
  }
}
// ---- merge of the exact (nearest, d1, d2) triples of target shards (the step after the all-gather) ----------------
// packed: (parts, q, 3) float64 = (d1, global index of the nearest, d2) per shard, shard p holding smaller target
// indices than shard p + 1. nearest = smallest d1, first shard among equals (= lowest index, what argmin returns);
// second = second smallest of the multiset of every shard's d1 and d2.
__global__ void __launch_bounds__(256)
    nearest_merge_kernel(const double* __restrict__ packed, int32_t parts, int64_t q, int64_t* __restrict__ nn,
                         double* __restrict__ d1, double* __restrict__ d2) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= q) return;
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  double best = inf, second = inf, index = -1.0;
  for (int p = 0; p < parts; ++p) {
    const double* t = packed + (int64_t(p) * q + i) * 3;
    const double a = t[0], b = t[2];
    if (p == 0 || a < best) {  // strict: the first shard keeps a tie
      second = fmin(second, best);
      best = a;
      index = t[1];
    } else {
      second = fmin(second, a);
    }
    second = fmin(second, b);
  }
  nn[i] = static_cast<int64_t>(index);
  d1[i] = best;
  d2[i] = second;
}
}  // namespace sf

extern "C" int sf_nearest_merge(const double* packed, int32_t parts, int64_t q, int64_t* nn, double* d1, double* d2,
                                void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(packed && nn && d1 && d2 && parts >= 1 && q >= 0, SF_ERR_ARG, "sf_nearest_merge: bad arguments");
  if (q == 0) return SF_OK;
  nearest_merge_kernel<<<unsigned((q + 255) / 256), 256, 0, stream>>>(packed, parts, q, nn, d1, d2);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_topk_merge(const float* score, const int32_t* idx, int32_t parts, int64_t qa, int32_t k,
                             float* score_out, int32_t* idx_out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(score && idx && score_out && idx_out && parts >= 1, SF_ERR_ARG, "sf_topk_merge: bad arguments");
  SF_REQUIRE(k == 1 || k == 2 || k == 4 || k == 8 || k == 16, SF_ERR_CAPACITY, "sf_topk_merge: k must be 1,2,4,8,16");
  if (qa == 0) return SF_OK;
  switch (k) {
    case 1: return launch_merge<1>(score, idx, parts, qa, score_out, idx_out, stream);
    case 2: return launch_merge<2>(score, idx, parts, qa, score_out, idx_out, stream);
    case 4: return launch_merge<4>(score, idx, parts, qa, score_out, idx_out, stream);
    case 8: return launch_merge<8>(score, idx, parts, qa, score_out, idx_out, stream);
    default: return launch_merge<16>(score, idx, parts, qa, score_out, idx_out, stream);
  }
}

extern "C" int sf_match_certify(const float* score, int32_t k, const float* a_sqnorm, const double* d1, const double* d2,
                                int64_t qa, double scale, double b_norm_max, int32_t width, int64_t qb,
                                int32_t want_second, uint8_t* flags, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(score && a_sqnorm && d1 && d2 && flags && k >= 1, SF_ERR_ARG, "sf_match_certify: bad arguments");
  if (qa == 0) return SF_OK;
  certify_kernel<<<unsigned((qa + 255) / 256), 256, 0, stream>>>(score, k, a_sqnorm, d1, d2, qa, scale, b_norm_max, width, qb,
                                                                want_second, flags);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_match_exhaustive_topk(const double* a, const int64_t* rows_a, const int64_t* which, int64_t n_which,
                                         const double* b, const int64_t* rows_b, int64_t qb, int32_t width, int32_t k,
                                         int32_t* cand, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(a && which && b && cand && width > 0, SF_ERR_ARG, "sf_match_exhaustive_topk: bad arguments");
  SF_REQUIRE(k == 8 || k == 16, SF_ERR_CAPACITY, "sf_match_exhaustive_topk: k must be 8 or 16");
  SF_REQUIRE(qb < (int64_t(1) << 31), SF_ERR_ARG, "sf_match_exhaustive_topk: too many targets");
  if (n_which == 0) return SF_OK;
  if (k == 8)
    exhaustive_topk_kernel<8><<<unsigned(n_which), 256, 0, stream>>>(a, rows_a, which, n_which, b, rows_b, qb, width, cand);
  else
    exhaustive_topk_kernel<16><<<unsigned(n_which), 256, 0, stream>>>(a, rows_a, which, n_which, b, rows_b, qb, width, cand);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_match_exhaustive(const double* a, const int64_t* rows_a, const int64_t* which, int64_t n_which,
                                   const double* limit, const double* b, const int64_t* rows_b, int64_t qb, int32_t width,
                                   double scale, double norm_bound, int32_t* cand16, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(a && which && limit && b && cand16 && width > 0, SF_ERR_ARG, "sf_match_exhaustive: bad arguments");
  SF_REQUIRE(norm_bound >= 0.0 && std::isfinite(norm_bound) && scale > 0.0 && std::isfinite(scale), SF_ERR_ARG,
             "sf_match_exhaustive: scale and norm_bound must be finite");
  SF_REQUIRE(qb < (int64_t(1) << 31), SF_ERR_ARG, "sf_match_exhaustive: too many targets");
  if (n_which == 0) return SF_OK;
  const int64_t query_tiles = (n_which + kEx32Rows - 1) / kEx32Rows;
  SF_REQUIRE(query_tiles <= 65535, SF_ERR_CAPACITY, "sf_match_exhaustive: %lld flagged queries", (long long)n_which);
  int32_t* counts = nullptr;
  double* list_d = nullptr;
  int32_t* list_i = nullptr;
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&counts, size_t(n_which) * 4));
  SF_CUDA(scratch.alloc(&list_d, size_t(n_which) * kExhaustiveCap * 8));
  SF_CUDA(scratch.alloc(&list_i, size_t(n_which) * kExhaustiveCap * 4));
  SF_CUDA(cudaMemsetAsync(counts, 0, size_t(n_which) * 4, stream));
  const dim3 grid(unsigned((qb + kEx32Rows - 1) / kEx32Rows), unsigned(query_tiles));
  exhaustive_tile32_kernel<<<grid, 256, 0, stream>>>(a, rows_a, which, n_which, limit, b, rows_b, qb, width, scale, norm_bound,
                                                     counts, list_d, list_i);
  exhaustive_select_kernel<<<unsigned((n_which + 127) / 128), 128, 0, stream>>>(n_which, counts, list_d, list_i, cand16);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_match_rerank(const double* a, const int64_t* rows_a, int64_t qa, const double* b,
                               const int64_t* rows_b, int32_t width, const int32_t* cand, int32_t k, int32_t* nn,
                               double* d1, double* d2, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(a && b && cand && nn && width > 0 && k >= 1, SF_ERR_ARG, "sf_match_rerank: bad arguments");
  if (qa == 0) return SF_OK;
  SF_REQUIRE(k <= kRerankMaxK, SF_ERR_CAPACITY, "sf_match_rerank: k must be <= %d", kRerankMaxK);
  rerank_kernel<<<unsigned((qa + kRerankWarps - 1) / kRerankWarps), kRerankWarps * 32, 0, stream>>>(
      a, rows_a, qa, b, rows_b, width, cand, k, nn, d1, d2);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}
