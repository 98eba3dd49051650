// Kernel group S: SHOT local reference frames and 352-bin descriptors.
//   S1 shot_lrf_kernel <- get_local_rf, shot.py:16-48 (fan-out shot_parallelization.py:46-84)
//   S2 shot_fast_kernel, shot_descriptor_block_kernel <- compute_single_shot_descriptor, shot.py:175-306 (fan-out :86-133)
//
// S2 implements the reference's actual semantics (SURVEY.md F1 / Appendix A): its ten `descriptor[idx] += v`
// statements are buffered NumPy fancy-index updates, so per statement and per bin only the neighbour with the
// largest distance that addresses the bin contributes (even with value 0). The float64 kernel keeps compact winner
// tables in shared memory (sf_math.cuh: three uint64 key tables raised with the native 64-bit atomicMax, five float
// value tables written by the threads that still hold a slot's key after a barrier); bins then sum their statements.
#include <cub/cub.cuh>

#include "sf_common.cuh"

namespace sf {

// ---- S1 ----------------------------------------------------------------------------------------------------
// Three launches; the (nq, 3, 3) output buffer doubles as scratch between them (9 float64 per query):
//   lrf_moments_kernel  warp per query   : 6 weighted second moments by warp reduction          -> out[0..5], K -> out[6]
//   lrf_eigen_kernel    THREAD per query : LAPACK-path 3x3 eigensolver (a long serial chain: run 32 independent
//                                          ones per warp instead of one per warp)               -> x, z axes in out[0..5]
//   lrf_votes_kernel    warp per query   : sign votes, y = z cross x, final row-major frame      -> out[0..8]
// (Round 1 history: one warp doing all three for one query took 690 us at C2, a warp per batch of 32 queries 240 us
// but with only 3 200 warps in flight for the two gather passes; this split keeps 100k warps available for them.)
__global__ void __launch_bounds__(256)
    lrf_moments_kernel(GridView g, const double* __restrict__ queries, int64_t nq, double radius,
                       const int64_t* __restrict__ offsets, const int32_t* __restrict__ nbr, double* __restrict__ lrf) {
  const int lane = threadIdx.x & 31;
  const int64_t q = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (q >= nq) return;
  const double qx = __ldg(queries + 3 * q), qy = __ldg(queries + 3 * q + 1), qz = __ldg(queries + 3 * q + 2);
  const int64_t begin = offsets[q], end = offsets[q + 1];
  // weighted covariance, weights (radius - distance), over ALL neighbours incl. the query itself (F5)
  double sw = 0, m[6] = {0, 0, 0, 0, 0, 0};
  for (int64_t i = begin + lane; i < end; i += 32) {
    const double4 p = load_pt(g.pts + __ldg(nbr + i));
    const double cx = p.x - qx, cy = p.y - qy, cz = p.z - qz;
    const double w = radius - sqrt(rdist3(cx, cy, cz));
    sw += w;
    m[0] += w * cx * cx; m[1] += w * cx * cy; m[2] += w * cx * cz;
    m[3] += w * cy * cy; m[4] += w * cy * cz; m[5] += w * cz * cz;
  }
  sw = warp_sum(sw);
#pragma unroll
  for (int k = 0; k < 6; ++k) m[k] = warp_sum(m[k]);
  if (lane < 7) {  // raw sums, the sum of the weights at [6]: lrf_eigen_kernel divides
    double v = m[0];
#pragma unroll
    for (int k = 1; k < 6; ++k) v = lane == k ? m[k] : v;
    lrf[9 * q + lane] = lane == 6 ? sw : v;
  }
}

// The solver's branches are data-dependent (QL or QR iteration, two to four sweeps, the 2x2 ending): with one query
// per thread in query order only 12 of a warp's 32 threads were active per instruction. The problems of a block are
// therefore regrouped between the two halves of the decomposition: every thread reduces ITS query to tridiagonal form,
// the block sorts the 128 tridiagonal problems by the direction dsteqr is about to take (through shared memory), and
// every thread finishes the problem it picked up and writes the axes of that problem's query.
constexpr int kEigenThreads = 128;

__global__ void __launch_bounds__(kEigenThreads)
    lrf_eigen_kernel(int64_t nq, const int64_t* __restrict__ offsets, const int32_t* __restrict__ counts,
                     double* __restrict__ lrf, float* __restrict__ frame32, const int32_t* __restrict__ status = nullptr) {
  __shared__ double rec[8][kEigenThreads];  // d[3], e[2], tau, v2, scale of the problem in each slot
  __shared__ int32_t owner[kEigenThreads];  // its query (offset inside the block), -1 = empty slot
  __shared__ int32_t warp_count[2][kEigenThreads / 32];
  if (status != nullptr && *status != 0) return;
  // frame32 (optional, 12 floats per query, 9 used): float32 images of the raw x, y = z cross x, z for shot_fast_kernel
  const int64_t q = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // empty neighbourhoods take no part: the votes step writes the identity
  const bool live = q < nq && !(counts ? counts[q] == 0 : offsets[q + 1] == offsets[q]);
  Tridiagonal3 t;
  bool up = false;
  if (live) {
    double m[6];
    const double sw = lrf[9 * q + 6];  // weighted covariance = sums / sum of the weights (shot.py:31-34)
#pragma unroll
    for (int k = 0; k < 6; ++k) m[k] = lrf[9 * q + k] / sw;
    eigh3_tridiagonal(m, t);
    up = eigh3_bottom_up(t);
  }
  owner[threadIdx.x] = -1;
  const unsigned down_mask = __ballot_sync(kFull, live && !up), up_mask = __ballot_sync(kFull, live && up);
  if (lane == 0) {
    warp_count[0][warp] = __popc(down_mask);
    warp_count[1][warp] = __popc(up_mask);
  }
  __syncthreads();
  if (live) {  // top-down problems fill the slots from the front, bottom-up ones from the back
    int before = __popc((up ? up_mask : down_mask) & lanemask_lt());
    for (int w = 0; w < warp; ++w) before += warp_count[up ? 1 : 0][w];
    const int slot = up ? kEigenThreads - 1 - before : before;
    rec[0][slot] = t.d[0]; rec[1][slot] = t.d[1]; rec[2][slot] = t.d[2]; rec[3][slot] = t.e[0]; rec[4][slot] = t.e[1];
    rec[5][slot] = t.tau; rec[6][slot] = t.v2; rec[7][slot] = t.scale;
    owner[slot] = threadIdx.x;
  }
  __syncthreads();
  const int mine = owner[threadIdx.x];
  if (mine < 0) return;
  t.d[0] = rec[0][threadIdx.x]; t.d[1] = rec[1][threadIdx.x]; t.d[2] = rec[2][threadIdx.x];
  t.e[0] = rec[3][threadIdx.x]; t.e[1] = rec[4][threadIdx.x];
  t.tau = rec[5][threadIdx.x]; t.v2 = rec[6][threadIdx.x]; t.scale = rec[7][threadIdx.x];
  const int64_t qo = blockIdx.x * int64_t(blockDim.x) + mine;
  double eval[3], evec[3][3];
  eigh3_finish(t, eval, evec);
  lrf[9 * qo + 0] = evec[2][0]; lrf[9 * qo + 1] = evec[2][1]; lrf[9 * qo + 2] = evec[2][2];  // x: largest eigenvalue
  lrf[9 * qo + 3] = evec[0][0]; lrf[9 * qo + 4] = evec[0][1]; lrf[9 * qo + 5] = evec[0][2];  // z: smallest eigenvalue
  if (frame32 != nullptr) {
    const double* x = evec[2];
    const double* z = evec[0];
    float* f = frame32 + 12 * qo;  // (kFrame32Stride: 48 bytes, one bulk copy)
    f[0] = float(x[0]); f[1] = float(x[1]); f[2] = float(x[2]);
    f[3] = float(z[1] * x[2] - z[2] * x[1]); f[4] = float(z[2] * x[0] - z[0] * x[2]); f[5] = float(z[0] * x[1] - z[1] * x[0]);
    f[6] = float(z[0]); f[7] = float(z[1]); f[8] = float(z[2]);
  }
}

__global__ void __launch_bounds__(256)
    lrf_votes_kernel(GridView g, const double* __restrict__ queries, int64_t nq, const int64_t* __restrict__ offsets,
                     const int32_t* __restrict__ nbr, double* __restrict__ lrf) {
  const int lane = threadIdx.x & 31;
  const int64_t q = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (q >= nq) return;
  const int64_t begin = offsets[q], end = offsets[q + 1];
  double* out = lrf + 9 * q;
  if (end == begin) {  // shot.py:24-25
    if (lane < 9) out[lane] = (lane % 4 == 0) ? 1.0 : 0.0;
    return;
  }
  const double qx = __ldg(queries + 3 * q), qy = __ldg(queries + 3 * q + 1), qz = __ldg(queries + 3 * q + 2);
  const double x[3] = {out[0], out[1], out[2]}, z[3] = {out[3], out[4], out[5]};
  // sign votes (shot.py:40-45)
  int neg_x = 0, neg_z = 0;
  for (int64_t i = begin + lane; i < end; i += 32) {
    const double4 p = load_pt(g.pts + __ldg(nbr + i));
    const double cx = p.x - qx, cy = p.y - qy, cz = p.z - qz;
    neg_x += (cx * x[0] + cy * x[1] + cz * x[2]) < 0.0;
    neg_z += (cx * z[0] + cy * z[1] + cz * z[2]) < 0.0;
  }
  neg_x = warp_sum(neg_x);
  neg_z = warp_sum(neg_z);
  const int k_all = int(end - begin);
  double f[9];
  shot_frame(x, z, neg_x > k_all - neg_x, neg_z > k_all - neg_z, f);
  __syncwarp();  // every lane has read the axes before the frame overwrites them
  if (lane < 3) {  // row `lane` of the frame (selects, not indexing: stays in registers)
#pragma unroll
    for (int c = 0; c < 3; ++c) out[3 * lane + c] = lane == 0 ? f[c] : (lane == 1 ? f[3 + c] : f[6 + c]);
  }
}

// ---- fused single-scale driver: search + moments in ONE pass over the candidates ----------------------------------
// The generic path scans the 27 cells twice (count, fill) and gathers the neighbours twice more for the frame
// (moments, votes). For the single-scale driver (shot_parallelization.py:135-183, the pipeline's default and the
// benchmark's headline) the neighbour list is an internal temporary, so it can be PADDED: query q owns the slots
// [cand_offsets[q], cand_offsets[q+1]) sized by its candidate count (a cell_start lookup, no distance test), the
// one scan writes the hits there, counts them and accumulates the frame's weighted moments while the points are
// in registers. The votes then run inside the descriptor kernel.
// One THREAD per query works out the query's cell, the gaps to its faces and its nine culled runs — the part of the
// search every lane of a warp would otherwise repeat (a third of search_moments_kernel's instructions in its first
// form) — and leaves them as a table of five int4: delta[0..8] = start - pref (candidate v of run j sits at
// v + delta[j]), pref[1..9] (running totals), two unused words.
// The query's slots in the padded list are handed out here as well: a block adds up its queries' candidate counts and
// takes its share of the list with ONE atomicAdd on a cursor (round 2; a device-wide prefix sum did this before: two
// more kernels and their launch gaps, 25 us of a 0.57 ms step). Where a query's slots lie is internal — the order of
// the neighbours inside them is what results depend on — so the arrival order of the blocks does not matter.
// status (speculative calls): raised to 2 when the list, sized from a previous call, cannot hold the candidates.
__global__ void __launch_bounds__(256)
    candidate_count_kernel(GridView g, const double* __restrict__ queries, int64_t nq, double r2,
                           int64_t* __restrict__ cand_offsets, int4* __restrict__ runs_table,
                           unsigned long long* __restrict__ cursor, int64_t capacity, int32_t* __restrict__ status,
                           unsigned long long* __restrict__ next_counters, int32_t* __restrict__ work_count) {
  __shared__ int warp_total[8];
  __shared__ unsigned long long block_base;
  // first kernel of the call: the counters of the NEXT call (the other set) and this call's work list are reset here
  // rather than by three memsets between the kernels
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    next_counters[0] = 0;
    next_counters[1] = 0;
    *work_count = 0;
  }
  const int64_t q = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int total = 0;
  if (q < nq) {
    const CellGaps cg = cell_gaps(g, queries[3 * q], queries[3 * q + 1], queries[3 * q + 2]);
    int start[9], pref[9];
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      int len;
      culled_run(g, cg, j, r2, start[j], len);
      start[j] -= total;  // (delta)
      total += len;
      pref[j] = total;
    }
    int4* t = runs_table + 5 * q;
    t[0] = make_int4(start[0], start[1], start[2], start[3]);
    t[1] = make_int4(start[4], start[5], start[6], start[7]);
    t[2] = make_int4(start[8], pref[0], pref[1], pref[2]);
    t[3] = make_int4(pref[3], pref[4], pref[5], pref[6]);
    t[4] = make_int4(pref[7], pref[8], 0, 0);
  }
  int incl = total;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_total[warp] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    int run = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const int t = warp_total[w];
      warp_total[w] = run;
      run += t;
    }
    block_base = atomicAdd(cursor, static_cast<unsigned long long>(run));
    if (status != nullptr && int64_t(block_base) + run > capacity) *status = 2;
  }
  __syncthreads();
  if (q < nq) cand_offsets[q] = int64_t(block_base) + warp_total[warp] + (incl - total);
}

__global__ void __launch_bounds__(256)
    search_moments_kernel(GridView g, const double* __restrict__ queries, int64_t nq, double radius, double r2,
                          const int64_t* __restrict__ cand_offsets, const int4* __restrict__ runs_table,
                          float4* __restrict__ nbr, int32_t* __restrict__ counts, double* __restrict__ lrf,
                          unsigned long long* __restrict__ pair_counter, const int32_t* __restrict__ status) {
  if (status != nullptr && *status != 0) return;  // a speculative call whose assumption failed: nothing is written
  const int lane = threadIdx.x & 31;
  const int64_t q = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (q >= nq) return;
  const double qx = __ldg(queries + 3 * q), qy = __ldg(queries + 3 * q + 1), qz = __ldg(queries + 3 * q + 2);
  // candidate_count_kernel's table (five broadcast loads; cells out of reach already dropped): candidate v of the
  // concatenated runs sits at v + delta[j] for the last run j with pref[j] <= v. The offset is SELECTED and added once
  // (written as start[j] + v - pref[j] per run, the compiler keeps nine running sums per lane and bumps them each round)
  int delta[9], pref[9];
  int total;
  {
    const int4* t = runs_table + 5 * q;
    const int4 t0 = __ldg(t), t1 = __ldg(t + 1), t2 = __ldg(t + 2), t3 = __ldg(t + 3), t4 = __ldg(t + 4);
    delta[0] = t0.x; delta[1] = t0.y; delta[2] = t0.z; delta[3] = t0.w;
    delta[4] = t1.x; delta[5] = t1.y; delta[6] = t1.z; delta[7] = t1.w; delta[8] = t2.x;
    pref[0] = 0; pref[1] = t2.y; pref[2] = t2.z; pref[3] = t2.w;
    pref[4] = t3.x; pref[5] = t3.y; pref[6] = t3.z; pref[7] = t3.w; pref[8] = t4.x;
    total = t4.y;
  }
  auto position = [&](int v) {
    int d = delta[0];
#pragma unroll
    for (int j = 1; j < 9; ++j) d = v >= pref[j] ? delta[j] : d;
    return v + d;
  };
  int64_t out = cand_offsets[q];
  int count = 0;
  double sw = 0, m[6] = {0, 0, 0, 0, 0, 0};
  // software pipeline: the candidate of the lane's NEXT round is requested before the current one is processed (the
  // kernel waits on these loads: 0.196 -> 0.173 ms; two rounds ahead spills and is slower, 0.182 ms)
  int pos_next = 0;
  double4 p_next = make_double4(0, 0, 0, 0);
  if (lane < total) {
    pos_next = position(lane);
    p_next = load_pt(g.pts + pos_next);
  }
  for (int base = 0; base < total; base += 32) {
    const int v = base + lane;
    bool hit = false, zero = false;
    float off[3] = {0.0f, 0.0f, 0.0f};
    const int pos = pos_next;
    const double4 p = p_next;
    if (v + 32 < total) {
      pos_next = position(v + 32);
      p_next = load_pt(g.pts + pos_next);
    }
    if (v < total) {
      const double cx = qx - p.x, cy = qy - p.y, cz = qz - p.z;  // second moments do not see the sign
      const double d2 = rdist3(cx, cy, cz);
      hit = d2 <= r2;
      zero = !(d2 > 0.0);
      off[0] = float(-cx); off[1] = float(-cy); off[2] = float(-cz);
      if (hit) {
        // (distance 0 — the query itself — would send the whole warp through sqrt's slow path once per query: the
        // argument is replaced for that lane, behind a barrier the compiler cannot fold the select through)
        double arg = zero ? 1.0 : d2;
        asm volatile("" : "+d"(arg));
        const double root = sqrt(arg);
        const double w = radius - (zero ? 0.0 : root);
        sw += w;
        m[0] += w * cx * cx; m[1] += w * cx * cy; m[2] += w * cx * cz;
        m[3] += w * cy * cy; m[4] += w * cy * cz; m[5] += w * cz * cz;
      }
    }
    const unsigned mask = __ballot_sync(kFull, hit);
    // list entry: the float32 image of the exact offset p - q (what shot_fast_kernel decides from) and the position;
    // bit 31 flags a neighbour at distance exactly 0 (the query itself, duplicates): shot.py:213 drops those from
    // the descriptor, and float32 cannot tell 0 from tiny
    if (hit)
      nbr[out + __popc(mask & lanemask_lt())] =
          make_float4(off[0], off[1], off[2], __uint_as_float(uint32_t(pos) | (zero ? 0x80000000u : 0u)));
    out += __popc(mask);
    count += __popc(mask);
  }
  // transposing butterfly over (sw, m0..m5, 0): after the exchange at distance 16 a lane carries four of the eight sums,
  // then two, then one (9 double-word exchanges instead of 35); the lanes whose bits 4..2 spell k end with value k
  {
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
    double a0 = h16 ? m[3] : sw, a1 = h16 ? m[4] : m[0], a2 = h16 ? m[5] : m[1], a3 = h16 ? 0.0 : m[2];
    a0 += __shfl_xor_sync(kFull, h16 ? sw : m[3], 16);
    a1 += __shfl_xor_sync(kFull, h16 ? m[0] : m[4], 16);
    a2 += __shfl_xor_sync(kFull, h16 ? m[1] : m[5], 16);
    a3 += __shfl_xor_sync(kFull, h16 ? m[2] : 0.0, 16);
    double b0 = h8 ? a2 : a0, b1 = h8 ? a3 : a1;
    b0 += __shfl_xor_sync(kFull, h8 ? a0 : a2, 8);
    b1 += __shfl_xor_sync(kFull, h8 ? a1 : a3, 8);
    double c0 = h4 ? b1 : b0;
    c0 += __shfl_xor_sync(kFull, h4 ? b0 : b1, 4);
    c0 += __shfl_xor_sync(kFull, c0, 2);
    c0 += __shfl_xor_sync(kFull, c0, 1);
    const int k = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);  // 0: sw, 1..6: m0..m5
    // raw sums: m0..m5 at [0..5], the sum of the weights at [6] (lrf_eigen_kernel divides)
    if ((lane & 3) == 0 && k <= 6) lrf[9 * q + (k == 0 ? 6 : k - 1)] = c0;
  }
  if (lane == 0) {
    counts[q] = count;
    atomicAdd(pair_counter, static_cast<unsigned long long>(count));
  }
}

// ---- S2, float64: a BLOCK per query -----------------------------------------------------------------------------------
// For the queries the fast kernel below hands over (a few hundred: 603 of 102 336 at C2; one warp per query walking its
// neighbours 32 at a time was 15-17 us of latency at the end of the step) and for every query under SF_SHOT_EXACT=1.
// uint64 keys[3][352] + float vals[5][352] = 15 488 B of shared memory per block (sf_math.cuh, "winner tables, compact
// form"). The four warps take the batches of 32 neighbours in turn (the sign votes as well). Per 128 neighbours:
// (a) float64 decisions, (b) three native 64-bit atomicMax on the key tables, (c) block barrier, (d) the threads that
// hold a slot's key compute the transcendental weights they need (only winners pay for acosf / atan2f) and store their
// values. After the last neighbour warp 0 assembles the 352 bins.
constexpr int kBlockQueryWarps = 4;

// Four consecutive 64-bit keys (32-byte aligned) as two 16-byte shared-memory reads.
__device__ __forceinline__ void load_keys4(const unsigned long long* k, unsigned long long out[4]) {
  const ulonglong2 a = reinterpret_cast<const ulonglong2*>(k)[0], b = reinterpret_cast<const ulonglong2*>(k)[1];
  out[0] = a.x; out[1] = a.y; out[2] = b.x; out[3] = b.y;
}

// 352 * sizeof(OutT) is a multiple of 16, so every row and every group of four bins is 16-byte aligned
__device__ __forceinline__ void store_group(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void store_group(double* p, float a, float b, float c, float d) {
  reinterpret_cast<double2*>(p)[0] = make_double2(a, b);
  reinterpret_cast<double2*>(p)[1] = make_double2(c, d);
}

template <typename OutT>
__global__ void __launch_bounds__(kBlockQueryWarps * 32)
    shot_descriptor_block_kernel(GridView g, const double* __restrict__ queries, int64_t nq, double radius,
                                 const int64_t* __restrict__ offsets, const int32_t* __restrict__ counts,
                                 const int32_t* __restrict__ nbr, double* __restrict__ lrf, int fuse_votes, int min_nb,
                                 int normalize, OutT* __restrict__ out, const int32_t* __restrict__ worklist,
                                 const int32_t* __restrict__ work_count, int nbr_stride,
                                 const int32_t* __restrict__ status) {
  if (status != nullptr && *status != 0) return;
  // counts == nullptr: classic CSR, neighbours of q are nbr[offsets[q] .. offsets[q+1]). Otherwise a padded list:
  // nbr[offsets[q] .. offsets[q] + counts[q]) (the fused single-scale driver).
  // fuse_votes: lrf[9q + 0..5] holds the RAW eigenvectors (x, z) from lrf_eigen_kernel; the sign votes of
  // shot.py:40-45 run here (the second pass over the same neighbours then hits L1) and the final frame is written
  // back to lrf[9q + 0..8].
  // worklist != nullptr: only the queries worklist[0 .. *work_count) (the ones shot_fast_kernel handed over); otherwise
  // all nq of them.
  // nbr_stride = 4: `nbr` is the fused driver's list of 16-byte entries (float32 offset, position | flag << 31), the
  // position is word 3 of an entry and offsets / counts are in entries; the flag (neighbour at distance 0) is masked:
  // this kernel decides that in float64 itself. nbr_stride = 1: plain int32 positions.
  __shared__ __align__(16) unsigned long long keys[kKeyCount];
  __shared__ __align__(16) float vals[kValCount];
  __shared__ int part[3][kBlockQueryWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double inv_radius = 1.0 / radius;
  const int nbr_word = nbr_stride - 1;
  const int n_items = worklist != nullptr ? *work_count : int(nq);
  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int64_t q = worklist != nullptr ? worklist[item] : item;
    // values are gated by their keys: only the keys are cleared (16 bytes per thread and store)
    for (int j = tid; j < kKeyCount / 2; j += kBlockQueryWarps * 32) reinterpret_cast<uint4*>(keys)[j] = make_uint4(0u, 0u, 0u, 0u);
    const double qx = __ldg(queries + 3 * q), qy = __ldg(queries + 3 * q + 1), qz = __ldg(queries + 3 * q + 2);
    const int64_t begin = offsets[q], end = counts ? begin + counts[q] : offsets[q + 1];
    double f[9];
    if (!fuse_votes) {
#pragma unroll
      for (int k = 0; k < 9; ++k) f[k] = lrf[9 * q + k];
    } else if (end == begin) {
#pragma unroll
      for (int k = 0; k < 9; ++k) f[k] = (k % 4 == 0) ? 1.0 : 0.0;  // shot.py:24-25
      if (tid < 9) lrf[9 * q + tid] = (tid % 4 == 0) ? 1.0 : 0.0;
    } else {
      const double x[3] = {lrf[9 * q], lrf[9 * q + 1], lrf[9 * q + 2]}, z[3] = {lrf[9 * q + 3], lrf[9 * q + 4], lrf[9 * q + 5]};
      int neg_x = 0, neg_z = 0;
      for (int64_t i = begin + tid; i < end; i += kBlockQueryWarps * 32) {
        const double4 p = load_pt(g.pts + (__ldg(nbr + i * nbr_stride + nbr_word) & 0x7fffffff));
        const double cx = p.x - qx, cy = p.y - qy, cz = p.z - qz;
        neg_x += (cx * x[0] + cy * x[1] + cz * x[2]) < 0.0;
        neg_z += (cx * z[0] + cy * z[1] + cz * z[2]) < 0.0;
      }
      neg_x = warp_sum(neg_x);
      neg_z = warp_sum(neg_z);
      if (lane == 0) { part[0][warp] = neg_x; part[1][warp] = neg_z; }
      __syncthreads();  // (also: every thread has read the raw axes before the frame overwrites them)
      neg_x = neg_z = 0;
#pragma unroll
      for (int w = 0; w < kBlockQueryWarps; ++w) { neg_x += part[0][w]; neg_z += part[1][w]; }
      const int k_all = int(end - begin);
      shot_frame(x, z, neg_x > k_all - neg_x, neg_z > k_all - neg_z, f);
      if (tid == 0) {
#pragma unroll
        for (int k = 0; k < 9; ++k) lrf[9 * q + k] = f[k];
      }
    }
    __syncthreads();  // the keys are cleared
    int positive = 0;
    for (int64_t base = begin; base < end; base += kBlockQueryWarps * 32) {  // block-uniform trip count (barriers inside)
      const int64_t i = base + tid;
      ShotDecision d;
      unsigned long long key = 0;
      bool active = false;
      if (i < end) {
        const int s = __ldg(nbr + i * nbr_stride + nbr_word) & 0x7fffffff;
        const double4 p = load_pt(g.pts + s), n = load_pt(g.nrm + s);
        const double cx = p.x - qx, cy = p.y - qy, cz = p.z - qz;
        const double d2 = rdist3(cx, cy, cz);
        if (d2 > 0.0) {  // shot.py:213: neighbours at distance 0 (the query itself, duplicates) are dropped
          active = true;
          ++positive;
          d = shot_decide_in_frame(cx, cy, cz, n.x, n.y, n.z, f, sqrt(d2), radius, inv_radius);
          key = shot_order_key(d.key, uint32_t(i - begin));
          atomicMax(keys + kKeyOwn + d.own, key);
          atomicMax(keys + kKeyCos + d.cos_nb, key);
          atomicMax(keys + kKeyAz + d.az_nb, key);
        }
      }
      __syncthreads();
      if (active)
        shot_store_winner(d, keys[kKeyOwn + d.own] == key, keys[kKeyCos + d.cos_nb] == key, keys[kKeyAz + d.az_nb] == key,
                          vals);
      __syncthreads();  // the stores above are ordered before the next round's key updates
    }
    positive = warp_sum(positive);
    if (lane == 0) part[2][warp] = positive;
    __syncthreads();
    if (warp == 0) {
      // assembly: lane handles the groups {lane, lane + 32, lane + 64} of four consecutive bins (one (cosine, azimuth)
      // cell: the radial / elevation partners are inside the group) -> eight 16-byte table reads and one 16-byte
      // store per group
      positive = 0;
#pragma unroll
      for (int w = 0; w < kBlockQueryWarps; ++w) positive += part[2][w];
      constexpr int kGroups = kShotLen / 4, kGroupRounds = (kGroups + 31) / 32;
      float v[kGroupRounds][4];
      double sq = 0.0;
#pragma unroll
      for (int j = 0; j < kGroupRounds; ++j) {
        const int grp = lane + 32 * j;
        if (grp < kGroups) {
          unsigned long long ko_[4], kc_[4], ka_[4];
          load_keys4(keys + kKeyOwn + 4 * grp, ko_);
          load_keys4(keys + kKeyCos + 4 * grp, kc_);
          load_keys4(keys + kKeyAz + 4 * grp, ka_);
          const float4 vo = *reinterpret_cast<const float4*>(vals + kValOwn + 4 * grp);
          const float4 vr = *reinterpret_cast<const float4*>(vals + kValRad + 4 * grp);
          const float4 ve = *reinterpret_cast<const float4*>(vals + kValEl + 4 * grp);
          const float4 vc = *reinterpret_cast<const float4*>(vals + kValCos + 4 * grp);
          const float4 va = *reinterpret_cast<const float4*>(vals + kValAz + 4 * grp);
          const float vo_[4] = {vo.x, vo.y, vo.z, vo.w}, vr_[4] = {vr.x, vr.y, vr.z, vr.w},
                      ve_[4] = {ve.x, ve.y, ve.z, ve.w}, vc_[4] = {vc.x, vc.y, vc.z, vc.w},
                      va_[4] = {va.x, va.y, va.z, va.w};
          shot_bin_group_compact(ko_, kc_, ka_, vo_, vr_, ve_, vc_, va_, v[j]);
#pragma unroll
          for (int t = 0; t < 4; ++t) sq += double(v[j][t]) * double(v[j][t]);
        }
      }
      sq = warp_sum(sq);
      const double norm = sqrt(sq);
      const bool keep = positive > min_nb && norm > 0.0;  // shot.py:212, :301-306
      const float inv = keep ? (normalize ? float(1.0 / norm) : 1.0f) : 0.0f;
      OutT* row = out + q * kShotLen;
#pragma unroll
      for (int j = 0; j < kGroupRounds; ++j) {
        const int grp = lane + 32 * j;
        if (grp < kGroups) store_group(row + 4 * grp, v[j][0] * inv, v[j][1] * inv, v[j][2] * inv, v[j][3] * inv);
      }
    }
    __syncthreads();  // the tables are read before the next query clears the keys
  }
}

// ---- S2, fast path: float32-filtered decisions -----------------------------------------------------------------------
// One warp per query with at most 128 neighbours (four slots of 32 per lane; a slot's code is skipped when the query
// has no neighbour for it). Slots 0-2 keep their state in registers; slot 3, which only the 6 % of the C2 queries with
// more than 96 neighbours use, keeps it in shared memory between the phases: the registers it would hold cost 20 -> 16
// warps per SM on every query. Round 1's float64 kernel, a warp per query, issued ~1650 warp instructions per query,
// half of them float64, re-gathered the neighbours for the frame's sign votes and kept 11 KB of tables per warp (20
// warps per SM). Here:
//   * in the fused driver the neighbour arrives as the float32 image of the EXACT float64 offset p - q that the search
//     kernel had in registers (16-byte list entries: offset + position), so nothing is gathered but the float32
//     normal and all margins are relative (8 u rho); caller-provided lists gather the grid's cell-relative float32
//     coordinates instead. All decisions come from float32 with proven margins (sf_math.cuh::shot_decide_fast);
//   * the sign votes need no second pass: the neighbours are projected on the RAW eigenvectors once, and flipping
//     an axis afterwards only negates coordinates (x -> -x negates X and Y = (z cross x) . c exactly);
//   * keys are unique inside a query (23 bits of distance + 7 bits of list position): one fire-and-forget shared
//     atomicMax per (neighbour, statement group), and a single re-read tells every lane whether it is THE winner;
//   * values are accumulated directly into the 352 output bins in five sub-phases (own-bin statements, radial
//     partner, elevation partner, statement 1, statement 9), each with at most one writer per bin: a fixed order
//     of float additions, bit-reproducible, no value tables and no assembly pass: 5.6 KB of shared memory per warp.
// A query goes to the exact kernel above (through `worklist`) when it has more than 128 neighbours, when a decision
// of one of its neighbours sits inside its float32 margin, or when two neighbours that compete for a bin are closer
// in distance than float32 can order (`amb_margin`).
constexpr int kFastSlots = 4;
constexpr int kFastRegSlots = 3;  // slots whose state stays in registers from the decisions to the value phases
constexpr int kFastMaxK = 32 * kFastSlots;
constexpr int kFastTableWords = kKeyCount + kShotLen;  // three key tables + the output bins
constexpr int kFrame32Stride = 12;                          // floats per query of lrf_eigen_kernel's float32 frame (x, y, z, pad)
// + the trash word losers write to (16-byte padding) + two staging buffers for the coming queries' inputs: 128 list
// entries, 12 floats of frame, an mbarrier each
constexpr int kFastWordsPerWarp = kFastTableWords + 4 + 2 * (kFastMaxK * 4 + kFrame32Stride + 4);
constexpr float kFastN2 = 1.001f;                        // unit normals up to rounding
static_assert(kFastMaxK <= (1 << kFastIndexBits), "a neighbour's list position must fit the key's index bits");
// The per-lane record of the last slot: its three addresses, its key and its five values, word f of lane l at word
// 32 f + l of the staging buffer the query's entries came from (read into registers before the record is written;
// the TMA unit refills that buffer only for the query after the next).
enum { kRecAddr = 0, kRecKey = 3, kRecOwn, kRecCos, kRecAz, kRecRad, kRecEl, kRecWords };
static_assert(kFastSlots == kFastRegSlots + 1, "one slot outside the registers");
static_assert(kRecWords * 32 <= kFastRegSlots * 32 * 4, "the record overlays the entries of the register slots only");

struct FastParams {
  float radius, inv_radius, edge32;
  float e_rel;          // records: bound on the error of rho, X, Y, Z relative to rho (8 u)
  float e_abs;          // gathered coordinates: absolute bound (24 u edge)
  float w_min;          // gathered coordinates: weights are left to float64 below this rho / hypot(X, Y)
  uint32_t amb_margin;  // in units of the 23-bit distance part of a key
  int fuse_votes, write_frame, min_nb, normalize;
};

// Shared-memory accesses by 32-bit address (the kernel keeps addresses, not bins, per neighbour).
__device__ __forceinline__ uint32_t smem_ld_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float smem_ld_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void smem_st_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void smem_st_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void smem_red_max(uint32_t addr, uint32_t v) {
  asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// kRecords: `list` holds the fused driver's float4 entries (float32 offset, position | zero-distance flag << 31);
// otherwise int32 cell-sorted positions of a caller's CSR (then `frame32` is null and lrf holds the FINAL frames).
template <typename OutT, bool kRecords, int kFastWarpsPerBlock, int kMinBlocks>
__global__ void __launch_bounds__(kFastWarpsPerBlock * 32, kMinBlocks)
    shot_fast_kernel(GridView g, const double* __restrict__ queries, int64_t nq, const int64_t* __restrict__ offsets,
                     const int32_t* __restrict__ counts, const void* __restrict__ list, double* __restrict__ lrf,
                     const float* __restrict__ frame32, FastParams fp, OutT* __restrict__ out,
                     int32_t* __restrict__ worklist, int32_t* __restrict__ work_count,
                     const int32_t* __restrict__ status) {
  if (status != nullptr && *status != 0) return;
  extern __shared__ __align__(16) uint32_t table_mem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  uint32_t* keys = table_mem + warp * kFastWordsPerWarp;
  float* desc = reinterpret_cast<float*>(keys + kKeyCount);
  const uint32_t keys_addr = uint32_t(__cvta_generic_to_shared(keys));
  const uint32_t trash = keys_addr + uint32_t(kFastTableWords) * 4u;
  const int64_t warps_total = int64_t(gridDim.x) * kFastWarpsPerBlock;
  constexpr int kGroups = kShotLen / 4, kGroupRounds = (kGroups + 31) / 32;
  const uint32_t amb_span = (fp.amb_margin << kFastIndexBits) | ((1u << kFastIndexBits) - 1u);

  // Software pipeline over the warp's queries, two deep: in an iteration the header (list position, neighbour count)
  // of the query after the next is requested, and at its top one lane asks the TMA unit for the NEXT query's list
  // entries and frame (two bulk copies into one of the warp's two staging buffers, completion on that buffer's
  // mbarrier): a whole iteration hides the copy (the 117 MB list comes from DRAM), and no register is carried for it.
  constexpr int kStageBytes = kFastMaxK * 16 + kFrame32Stride * 4 + 16;  // entries, frame, mbarrier (+ padding)
  const uint32_t stage_base = keys_addr + uint32_t(kFastTableWords + 4) * 4u;
  const char* stage_ptr = reinterpret_cast<const char*>(keys + kFastTableWords + 4);
  uint32_t phase_bits = 0;  // bit b: the parity buffer b's mbarrier completes next
  if (kRecords) {
    if (lane == 0) {
#pragma unroll
      for (int b = 0; b < 2; ++b)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(stage_base + b * kStageBytes + kFastMaxK * 16 + 48), "r"(1));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
  }
  auto header = [&](int64_t query, int64_t& first, int& count) {
    first = 0;
    count = 0;
    if (query < nq) {
      first = offsets[query];
      count = counts ? counts[query] : int(offsets[query + 1] - first);
    }
  };
  auto stage = [&](int64_t query, int64_t first, int count, int buffer) {
    if (kRecords && count > 0 && count <= kFastMaxK && lane == 0) {
      const uint32_t dst = stage_base + buffer * kStageBytes, bar = dst + kFastMaxK * 16 + 48;
      const uint32_t bytes = uint32_t(count) * 16u;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes + 48u) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                   "l"(static_cast<const float4*>(list) + first), "r"(bytes), "r"(bar)
                   : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       dst + uint32_t(kFastMaxK) * 16u),
                   "l"(frame32 + kFrame32Stride * query), "r"(48u), "r"(bar)
                   : "memory");
    }
  };
  int64_t q = blockIdx.x * int64_t(kFastWarpsPerBlock) + warp;
  int64_t begin, begin_next;
  int K, K_next, buffer = 0;
  header(q, begin, K);
  stage(q, begin, K, 0);
  header(q + warps_total, begin_next, K_next);
  for (; q < nq;) {
    const int64_t q_next = q + warps_total;
    stage(q_next, begin_next, K_next, buffer ^ 1);  // (its header was requested an iteration ago)
    bool defer = K > kFastMaxK;  // too many for four per lane: the exact kernel takes it
    const bool work = K > 0 && !defer;
    uint32_t addr[kFastRegSlots][3], key[kFastRegSlots];
    float v_own[kFastRegSlots], v_cos[kFastRegSlots], v_az[kFastRegSlots], v_rad[kFastRegSlots], v_el[kFastRegSlots];
    // the last slot's record (warp-uniform: only when K > 96)
    const bool last_slot = K > kFastRegSlots * 32;
    const uint32_t rec = stage_base + buffer * kStageBytes + 4u * lane;
    auto rec_ld = [&](int f) { return smem_ld_u32(rec + 128u * f); };
    auto rec_ldf = [&](int f) { return smem_ld_f32(rec + 128u * f); };
    auto rec_st = [&](int f, uint32_t v) { smem_st_u32(rec + 128u * f, v); };
    float fsx = 1.0f, fsz = 1.0f;
    int positive = 0;
    if (work) {
      for (int j = lane; j < kFastTableWords / 4; j += 32) reinterpret_cast<uint4*>(keys)[j] = make_uint4(0u, 0u, 0u, 0u);
      if (lane == 0) keys[kFastTableWords] = 0xffffffffu;  // the trash word: never below a key, never equal to one
      // ---- the frame's axes in float32 (raw eigenvectors when the votes are fused) ----
      float ax[3], ay[3], az[3];
      const float4* stage_entries = reinterpret_cast<const float4*>(stage_ptr + buffer * kStageBytes);
      if (kRecords) {  // staged by the TMA unit: the entries and x, y = z cross x, z of lrf_eigen_kernel
        const float* stage_axes = reinterpret_cast<const float*>(stage_entries + kFastMaxK);
        const uint32_t bar = stage_base + buffer * kStageBytes + kFastMaxK * 16 + 48, phase = (phase_bits >> buffer) & 1u;
        uint32_t done;
        do {
          asm volatile(
              "{\n\t"
              ".reg .pred p;\n\t"
              "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
              "selp.u32 %0, 1, 0, p;\n\t"
              "}"
              : "=r"(done)
              : "r"(bar), "r"(phase)
              : "memory");
        } while (!done);
        phase_bits ^= 1u << buffer;
#pragma unroll
        for (int a = 0; a < 3; ++a) { ax[a] = stage_axes[a]; ay[a] = stage_axes[3 + a]; az[a] = stage_axes[6 + a]; }
      } else {  // final frame, row-major, columns [x y z]
        const double* frame = lrf + 9 * q;
#pragma unroll
        for (int a = 0; a < 3; ++a) { ax[a] = float(frame[3 * a]); ay[a] = float(frame[3 * a + 1]); az[a] = float(frame[3 * a + 2]); }
      }
      // ---- neighbours: offsets, projection on the axes, request of the normals ----
      float X0[kFastSlots], Y0[kFastSlots], Z0[kFastSlots], R2[kFastSlots];
      float4 pb[kFastSlots];
      unsigned valid = 0, zero_bits = 0;
      bool unsure = false;  // a decision of this lane is inside its float32 margin: the exact kernel takes the query
      if (kRecords) {
#pragma unroll
        for (int s = 0; s < kFastSlots; ++s) {
          X0[s] = Y0[s] = Z0[s] = R2[s] = 0.0f;
          if (s * 32 < K) {  // (warp-uniform; inside, every lane computes: a lane past the end re-reads the last entry
                             // and is masked out where its results would land)
            const float4 entry = stage_entries[min(s * 32 + lane, K - 1)];
            const uint32_t w = __float_as_uint(entry.w);
            pb[s] = __ldg(g.nrm32 + (w & 0x7fffffffu));
            const float c[3] = {entry.x, entry.y, entry.z};
            R2[s] = dot3f(c, c);
            X0[s] = dot3f(c, ax);
            Y0[s] = dot3f(c, ay);
            Z0[s] = dot3f(c, az);
            if (s * 32 + lane < K) valid |= 1u << s;
            zero_bits |= (w >> 31) << s;
          }
        }
      } else {
        const int32_t* nbr = static_cast<const int32_t*>(list) + begin;
        const double* query = queries + 3 * q;
        const double qd[3] = {__ldg(query), __ldg(query + 1), __ldg(query + 2)};
        int cq[3];
        float lq[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) cq[a] = cell_coord(qd[a], g.origin[a], g.inv_cell, g.dims[a]);
        shot_cell_local(qd, g.origin, g.cell, cq, lq);
        const uint32_t cq_bits = shot_cellbits(cq);
#pragma unroll
        for (int s = 0; s < kFastSlots; ++s) {
          X0[s] = Y0[s] = Z0[s] = R2[s] = 0.0f;
          if (s * 32 < K) {
            if (s * 32 + lane < K) {
              const int pos = __ldg(nbr + s * 32 + lane);
              const float4 e = __ldg(g.xyzc + pos);
              pb[s] = __ldg(g.nrm32 + pos);
              const float lp[3] = {e.x, e.y, e.z};
              float c[3];
              shot_rel32(lp, __float_as_uint(e.w), lq, cq_bits, fp.edge32, c);
              R2[s] = dot3f(c, c);
              X0[s] = dot3f(c, ax);
              Y0[s] = dot3f(c, ay);
              Z0[s] = dot3f(c, az);
              valid |= 1u << s;
              if (R2[s] == 0.0f) {
                // no flags in a caller's list: a float32 offset of exactly 0 is the query itself or a duplicate when
                // the float64 coordinates agree exactly — anything else this close is left to the exact kernel
                const double4 p = load_pt(g.pts + pos);
                if (p.x == qd[0] && p.y == qd[1] && p.z == qd[2]) zero_bits |= 1u << s;
                else unsure = true;
              }
            }
          }
        }
      }
      const unsigned act = valid & ~zero_bits;
      if (fp.fuse_votes) {  // shot.py:40-45: flip when strictly more neighbours project negatively (distance 0: not negative)
        // (a projection inside its float32 margin makes the vote unsure: the decisions below test exactly that,
        // |X| and |Z| against e_loc, on every neighbour that votes)
        int neg_x = 0, neg_z = 0;
#pragma unroll
        for (int s = 0; s < kFastSlots; ++s) {
          if (s * 32 < K) {
            const bool on = (act >> s) & 1u;
            neg_x += __popc(__ballot_sync(kFull, on && X0[s] < 0.0f));
            neg_z += __popc(__ballot_sync(kFull, on && Z0[s] < 0.0f));
          }
        }
        if (neg_x > K - neg_x) fsx = -1.0f;
        if (neg_z > K - neg_z) fsz = -1.0f;
      }
      __syncwarp();  // the tables are cleared
      // ---- decisions; one fire-and-forget shared max per (neighbour, statement group) ----
      // Per neighbour: the shared-memory byte addresses of its three key slots, its key and its five values. The
      // bins sit kKeyCount words above the key tables: a value goes to (slot of group t) + (kKeyCount - 352 t) words.
      auto decide = [&](int s, uint32_t(&a)[3], uint32_t& k) {
        const bool on = (act >> s) & 1u;
        const float nv[3] = {pb[s].x, pb[s].y, pb[s].z};
        const float inv_rho = sf_rsqrtf(fmaxf(R2[s], 1e-37f)), rho = R2[s] * inv_rho;
        ShotFastMargins m;
        m.e_loc = kRecords ? fp.e_rel * rho : fp.e_abs;
        m.e_rho = m.e_loc;
        m.w_rho_min = kRecords ? 0.0f : fp.w_min;
        m.w_xy_min = kRecords ? 0.01f * rho : fp.w_min;
        m.n2 = kFastN2;
        ShotDecision d;
        // (the cosine margin assumes |n|^2 <= kFastN2: longer normals are left to the exact kernel)
        const bool sure = shot_decide_fast(fsx * X0[s], fsx * fsz * Y0[s], fsz * Z0[s], fsz * dot3f(nv, az), rho, inv_rho,
                                           fp.radius, fp.inv_radius, m, d) &&
                          dot3f(nv, nv) <= kFastN2;
        unsure = unsure || (on && !sure);
        const bool use = on && sure;
        const ShotFastRecord r = shot_fast_record(d, uint32_t(s * 32 + lane));
        k = use ? r.key : 0u;
        // (an unsure decision may hold any bin: its addresses are never formed)
        a[0] = use ? keys_addr + 4u * uint32_t(kKeyOwn + d.own) : trash;
        a[1] = use ? keys_addr + 4u * uint32_t(kKeyCos + d.cos_nb) : trash;
        a[2] = use ? keys_addr + 4u * uint32_t(kKeyAz + d.az_nb) : trash;
#pragma unroll
        for (int t = 0; t < 3; ++t) smem_red_max(a[t], k);  // (0 on the trash word: no effect)
        positive += __popc(__ballot_sync(kFull, on));
        return r;
      };
      // the last slot first: decided after the others, it needs four registers more than there are at 20 warps per SM
      // (the keys do not depend on the order of the maxima)
      if (last_slot) {  // (every lane has read the staged entries: the __syncwarp above)
        uint32_t a[3], k;
        const ShotFastRecord r = decide(kFastRegSlots, a, k);
#pragma unroll
        for (int t = 0; t < 3; ++t) rec_st(kRecAddr + t, a[t]);
        rec_st(kRecKey, k);
        rec_st(kRecOwn, __float_as_uint(r.v_own));
        rec_st(kRecCos, __float_as_uint(r.v_cos));
        rec_st(kRecAz, __float_as_uint(r.v_az));
        rec_st(kRecRad, __float_as_uint(r.v_rad));
        rec_st(kRecEl, __float_as_uint(r.v_el));
      }
#pragma unroll
      for (int s = 0; s < kFastRegSlots; ++s) {
        if (s * 32 < K) {
          const ShotFastRecord r = decide(s, addr[s], key[s]);
          v_own[s] = r.v_own; v_cos[s] = r.v_cos; v_az[s] = r.v_az; v_rad[s] = r.v_rad; v_el[s] = r.v_el;
        }
      }
      __syncwarp();  // the shared maxima are ordered before the reads below
      defer = __any_sync(kFull, unsure);
    }
    // the header of the query after the next (requested here rather than at the top: the decisions above need the
    // registers more, and the rest of the iteration still hides the load)
    int64_t begin_after;
    int K_after;
    header(q_next + warps_total, begin_after, K_after);
    if (work && !defer) {
      // ---- winners (keys are unique: equality = THE winner) and competitors float32 cannot order ----
      // A slot that did not win (or holds no neighbour) is redirected to the warp's trash word, so that the value
      // phases below run without branches: every lane does load - add - store, losers on the trash word.
      // The last slot re-reads its state from the record in every phase (a bin has one writer per sub-phase, so where
      // in a sub-phase that slot's load - add - store runs does not change any sum).
      uint32_t closest = 0xffffffffu;  // smallest (winner key - own key - 1) over this lane's losing slots
      auto winner = [&](uint32_t(&a)[3], uint32_t k) {
        uint32_t seen[3];
#pragma unroll
        for (int t = 0; t < 3; ++t) seen[t] = smem_ld_u32(a[t]);  // >= k (trash: 0xffffffff; no key is 0)
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          closest = min(closest, seen[t] - k - 1u);  // (a winner wraps to 0xffffffff)
          a[t] = seen[t] == k ? a[t] + uint32_t(kKeyCount - t * kShotLen) * 4u : trash;
        }
      };
#pragma unroll
      for (int s = 0; s < kFastRegSlots; ++s)
        if (s * 32 < K) winner(addr[s], key[s]);
      if (last_slot) {
        uint32_t a[3] = {rec_ld(kRecAddr), rec_ld(kRecAddr + 1), rec_ld(kRecAddr + 2)};
        winner(a, rec_ld(kRecKey));
#pragma unroll
        for (int t = 0; t < 3; ++t) rec_st(kRecAddr + t, a[t]);
      }
      bool amb = closest < amb_span;  // a winner at most amb_span above one of this lane's keys: unordered
      // ---- values, one writer per bin and sub-phase (loads of a sub-phase first, then its stores) ----
#pragma unroll
      for (int s = 0; s < kFastRegSlots; ++s)
        if (s * 32 < K) smem_st_f32(addr[s][0], v_own[s]);  // statements 2 + 5 + 8 + 10
      if (last_slot) smem_st_f32(rec_ld(kRecAddr), rec_ldf(kRecOwn));
      __syncwarp();
#pragma unroll
      for (int t = 0; t < 2; ++t) {  // radial partner (statement 3 or 4), then elevation partner (6 or 7)
        // the own-bin winner's partner bin: its value slot is the own value slot's address with bit 2 (3) flipped,
        // its own-group key sits kKeyCount words below
        auto partner = [&](uint32_t own) { return own != trash ? own ^ (4u << t) : trash; };
        auto partner_key = [&](uint32_t dst) { return smem_ld_u32(dst != trash ? dst - uint32_t(kKeyCount) * 4u : trash); };
        auto settle = [&](uint32_t dst, uint32_t pk, uint32_t k) {
          amb = amb || (dst != trash && max(pk, k) - min(pk, k) <= amb_span);
          return k > pk ? dst : trash;  // (pk of a non-winner: the trash word, above every key)
        };
        uint32_t dst[kFastRegSlots], pk[kFastRegSlots];
        float cur[kFastRegSlots];
#pragma unroll
        for (int s = 0; s < kFastRegSlots; ++s)
          if (s * 32 < K) {
            dst[s] = partner(addr[s][0]);
            pk[s] = partner_key(dst[s]);
          }
#pragma unroll
        for (int s = 0; s < kFastRegSlots; ++s)
          if (s * 32 < K) {
            dst[s] = settle(dst[s], pk[s], key[s]);
            cur[s] = smem_ld_f32(dst[s]);
          }
#pragma unroll
        for (int s = 0; s < kFastRegSlots; ++s)
          if (s * 32 < K) smem_st_f32(dst[s], cur[s] + (t == 0 ? v_rad[s] : v_el[s]));
        if (last_slot) {
          const uint32_t d = partner(rec_ld(kRecAddr));
          const uint32_t w = settle(d, partner_key(d), rec_ld(kRecKey));
          smem_st_f32(w, smem_ld_f32(w) + rec_ldf(t == 0 ? kRecRad : kRecEl));
        }
        __syncwarp();
      }
#pragma unroll
      for (int t = 1; t < 3; ++t) {  // statement 1, then statement 9
        float cur[kFastRegSlots];
#pragma unroll
        for (int s = 0; s < kFastRegSlots; ++s)
          if (s * 32 < K) cur[s] = smem_ld_f32(addr[s][t]);
#pragma unroll
        for (int s = 0; s < kFastRegSlots; ++s)
          if (s * 32 < K) smem_st_f32(addr[s][t], cur[s] + (t == 1 ? v_cos[s] : v_az[s]));
        if (last_slot) {
          const uint32_t a = rec_ld(kRecAddr + t);
          smem_st_f32(a, smem_ld_f32(a) + rec_ldf(t == 1 ? kRecCos : kRecAz));
        }
        __syncwarp();
      }
      defer = __any_sync(kFull, amb);  // float32 cannot order two competitors: the exact kernel redoes the query
    }
    if (defer) {
      if (lane == 0) worklist[atomicAdd(work_count, 1)] = int32_t(q);
    } else {
      // ---- norm + row (K == 0: shot.py:24-25 identity frame, :306 zero row) ----
      float4 v[kGroupRounds];
      float sq = 0.0f;
#pragma unroll
      for (int j = 0; j < kGroupRounds; ++j) {
        v[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (work && lane + 32 * j < kGroups) v[j] = reinterpret_cast<const float4*>(desc)[lane + 32 * j];
        sq = fmaf(v[j].x, v[j].x, fmaf(v[j].y, v[j].y, fmaf(v[j].z, v[j].z, fmaf(v[j].w, v[j].w, sq))));
      }
      sq = warp_sum(sq);
      const bool keep = positive > fp.min_nb && sq > 0.0f;  // shot.py:212, :301-306
      const float inv = keep ? (fp.normalize ? rsqrtf(sq) : 1.0f) : 0.0f;
      OutT* row = out + q * kShotLen;
#pragma unroll
      for (int j = 0; j < kGroupRounds; ++j)
        if (lane + 32 * j < kGroups)
          store_group(row + 4 * (lane + 32 * j), v[j].x * inv, v[j].y * inv, v[j].z * inv, v[j].w * inv);
      if (fp.fuse_votes && fp.write_frame) {  // the final frame replaces the raw eigenvectors (every lane has read them)
        if (!work) {
          if (lane < 9) lrf[9 * q + lane] = (lane % 4 == 0) ? 1.0 : 0.0;
        } else {
          const double* frame = lrf + 9 * q;
          double f[9];
          shot_frame(frame, frame + 3, fsx < 0.0f, fsz < 0.0f, f);
          __syncwarp();
          if (lane < 3) {
#pragma unroll
            for (int c = 0; c < 3; ++c) lrf[9 * q + 3 * lane + c] = lane == 0 ? f[c] : (lane == 1 ? f[3 + c] : f[6 + c]);
          }
        }
      }
    }
    // the record's stores and loads are ordered before the TMA unit refills its buffer
    if (kRecords && last_slot) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();  // all lanes have read the tables before the next query clears them
    q = q_next;
    begin = begin_next;
    K = K_next;
    begin_next = begin_after;
    K_next = K_after;
    buffer ^= 1;
  }
}

}  // namespace sf

using namespace sf;

extern "C" int sf_shot_lrf(sf_grid* g, const double* queries, int64_t nq, double radius, const int64_t* offsets,
                           const int32_t* nbr, double* lrf, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_shot_lrf: grid not built");
  if (nq == 0) return SF_OK;  // (an empty query block has null pointers: zero-row tensors)
  SF_REQUIRE(queries && offsets && lrf && nq > 0, SF_ERR_ARG, "sf_shot_lrf: bad arguments");
  const unsigned warp_blocks = unsigned((nq * 32 + 255) / 256);
  lrf_moments_kernel<<<warp_blocks, 256, 0, stream>>>(g->view(), queries, nq, radius, offsets, nbr, lrf);
  lrf_eigen_kernel<<<unsigned((nq + 127) / 128), 128, 0, stream>>>(nq, offsets, nullptr, lrf, nullptr);
  lrf_votes_kernel<<<warp_blocks, 256, 0, stream>>>(g->view(), queries, nq, offsets, nbr, lrf);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

// Optional per-kernel timing of the fused drivers (bench.py's roofline needs the dominant kernel's own duration and
// a driver is a single C call): CUDA events recorded on the launching stream around its three stages.
static bool g_profile = false;
static cudaEvent_t g_events[4] = {nullptr, nullptr, nullptr, nullptr};

namespace sf {
void profile_mark(int i, cudaStream_t stream) {
  if (g_profile) cudaEventRecord(g_events[i], stream);
}
}  // namespace sf

extern "C" int sf_profile_enable(int32_t enable) {
  if (enable && g_events[0] == nullptr)
    for (auto& e : g_events) SF_CUDA(cudaEventCreate(&e));
  g_profile = enable != 0;
  return SF_OK;
}

// ms_out[0..2] = the three stages of the LAST fused driver call (sf_shot_single_scale: search+moments, eigen,
// votes+descriptor; sf_fpfh_cloud: search+weights, SPFH, FPFH). Synchronises.
extern "C" int sf_profile_read(float* ms_out) {
  SF_REQUIRE(g_profile && g_events[0] != nullptr && ms_out != nullptr, SF_ERR_ARG, "sf_profile_read: profiling is off");
  SF_CUDA(cudaEventSynchronize(g_events[3]));
  for (int i = 0; i < 3; ++i) SF_CUDA(cudaEventElapsedTime(ms_out + i, g_events[i], g_events[i + 1]));
  return SF_OK;
}

static int64_t g_last_deferred = 0;

// Queries the fast kernel handed to the exact kernel in the last sf_shot_single_scale call that asked for `pairs_host`.
extern "C" int sf_shot_last_deferred(int64_t* deferred) {
  SF_REQUIRE(deferred != nullptr, SF_ERR_ARG, "sf_shot_last_deferred: null output");
  *deferred = g_last_deferred;
  return SF_OK;
}

static bool env_flag(const char* name) {
  const char* v = getenv(name);
  return v != nullptr && v[0] == '1';
}

// Descriptors of nq queries: shot_fast_kernel on everything, then the exact kernel on the queries the fast one handed
// over (more than 128 neighbours, a decision inside its float32 margin, or two competitors float32 cannot order).
// SF_SHOT_EXACT=1 sends every query to the exact kernel (the tests' reference for the fast one).
//   records == false : `list` = int32 positions of a CSR (offsets[nq + 1]), lrf = the final frames
//   records == true  : the fused driver's padded list of float4 entries (offsets + counts), lrf = raw eigenvectors,
//                      frame32 = their float32 images (lrf_eigen_kernel)
//   worklist / work_count : nq int32 + one int32 of scratch (work_count zeroed here)
static int launch_descriptor(sf_grid* g, const double* queries, int64_t nq, double radius, const int64_t* offsets,
                             const int32_t* counts, const void* list, bool records, double* lrf, const float* frame32,
                             int write_frame, int min_nb, int normalize, void* out, int out_is_f64, int32_t* worklist,
                             int32_t* work_count, const int32_t* status, cudaStream_t stream,
                             bool work_count_is_reset = false) {
  SF_REQUIRE(reinterpret_cast<uintptr_t>(out) % 16 == 0, SF_ERR_ARG, "SHOT output rows must be 16-byte aligned");
  SF_REQUIRE(nq < (int64_t(1) << 31), SF_ERR_ARG, "SHOT: %lld queries in one call", (long long)nq);
  const bool exact_only = env_flag("SF_SHOT_EXACT");
  const int fuse_votes = records ? 1 : 0;
  const GridView view = g->view();
  if (!exact_only) {
    FastParams fp;
    const double u = 5.9604645e-8;  // 2^-24; the bounds below are sf_math.cuh's, rounded up
    fp.radius = float(radius);
    fp.inv_radius = float(1.0 / radius);
    fp.edge32 = float(g->cell);
    fp.e_rel = float(8.0 * u * 1.0001);
    fp.e_abs = float(24.0 * u * g->cell * 1.0001);
    fp.w_min = float(0.01 * radius);
    // two keys, each within (bound on rho) / radius of the exact 23-bit distance part, + the roundings of the scaling
    const double rho_err_units = (records ? 8.0 * u : 24.0 * u * g->cell / radius) * 8388608.0 + 1.5;
    fp.amb_margin = uint32_t(2.0 * rho_err_units + 1.0);
    fp.fuse_votes = fuse_votes;
    fp.write_frame = write_frame;
    fp.min_nb = min_nb;
    fp.normalize = normalize;
    if (!work_count_is_reset) SF_CUDA(cudaMemsetAsync(work_count, 0, sizeof(int32_t), stream));
    // persistent: 148 SMs x 2 resident blocks, capped by the work. The fused driver's lists: blocks of 10 warps, 20 per
    // SM (96 registers without spills; 9.6 KB of tables + staging per warp, 195 KB per SM with the per-block reserve).
    // Caller-provided lists: blocks of 8 warps (128 registers; at 96 that instantiation spills).
    auto launch = [&](auto kernel, auto* typed_out, int warps, int per_sm) -> cudaError_t {
      const size_t fast_smem = size_t(warps) * kFastWordsPerWarp * 4;
      cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(fast_smem));
      // (no shared-memory carveout preference: the L1 that is left serves the normals' gather — neighbouring queries
      // run on the same SM — and forcing the maximum carveout cost 10-25 %)
      if (err != cudaSuccess) return err;
      const int64_t needed = (nq + warps - 1) / warps;
      const unsigned blocks = unsigned(needed < 148 * per_sm ? needed : 148 * per_sm);
      kernel<<<blocks, warps * 32, fast_smem, stream>>>(view, queries, nq, offsets, counts, list, lrf, frame32, fp, typed_out,
                                                        worklist, work_count, status);
      return cudaGetLastError();
    };
    float* fo = static_cast<float*>(out);
    double* dout = static_cast<double*>(out);
    if (out_is_f64) {
      if (records) SF_CUDA(launch(shot_fast_kernel<double, true, 10, 2>, dout, 10, 2));
      else SF_CUDA(launch(shot_fast_kernel<double, false, 8, 2>, dout, 8, 2));
    } else {
      if (records) SF_CUDA(launch(shot_fast_kernel<float, true, 10, 2>, fo, 10, 2));
      else SF_CUDA(launch(shot_fast_kernel<float, false, 8, 2>, fo, 8, 2));
    }
  }
  // the exact kernel, a block per query, on the work list of the fast kernel or on every query (as many blocks as the
  // device holds at once; each strides over the list, whose length only the device knows)
  const unsigned blocks = unsigned(std::min<int64_t>(nq, 148 * 8));
  const int32_t* wl = exact_only ? nullptr : worklist;
  const int32_t* nbr = static_cast<const int32_t*>(list);
  const int stride = records ? 4 : 1;
  if (out_is_f64)
    shot_descriptor_block_kernel<double><<<blocks, kBlockQueryWarps * 32, 0, stream>>>(
        view, queries, nq, radius, offsets, counts, nbr, lrf, fuse_votes, min_nb, normalize, static_cast<double*>(out), wl,
        work_count, stride, status);
  else
    shot_descriptor_block_kernel<float><<<blocks, kBlockQueryWarps * 32, 0, stream>>>(
        view, queries, nq, radius, offsets, counts, nbr, lrf, fuse_votes, min_nb, normalize, static_cast<float*>(out), wl,
        work_count, stride, status);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_shot_descriptor(sf_grid* g, const double* queries, int64_t nq, double radius,
                                  const int64_t* offsets, const int32_t* nbr, const double* lrf, int32_t min_nb,
                                  int32_t normalize, void* out, int32_t out_is_f64, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0 && g->has_normals, SF_ERR_ARG, "sf_shot_descriptor: grid built without normals");
  if (nq == 0) return SF_OK;  // (an empty query block has null pointers: zero-row tensors)
  SF_REQUIRE(queries && offsets && lrf && out && nq > 0, SF_ERR_ARG, "sf_shot_descriptor: bad arguments");
  int32_t* worklist = nullptr;
  Scratch scratch(stream);
  SF_CUDA(scratch.alloc(&worklist, size_t(nq + 1) * 4));
  return launch_descriptor(g, queries, nq, radius, offsets, nullptr, nbr, false, const_cast<double*>(lrf), nullptr, 0,
                           min_nb, normalize, out, out_is_f64, worklist + 1, worklist, nullptr, stream);
}

// Scratch of the fused driver, kept by the grid handle between calls (the stream-ordered pool cost a dozen
// allocations per call).
static int shot_reserve_queries(sf_grid* g, int64_t nq) {
  if (nq <= g->shot_q_capacity) return SF_OK;
  cudaFree(g->shot_cand_offsets); cudaFree(g->shot_counts); cudaFree(g->shot_lrf);
  cudaFree(g->shot_runs); cudaFree(g->shot_frame32); cudaFree(g->shot_worklist);
  g->shot_q_capacity = 0;
  const int64_t cap = nq + nq / 8 + 64;
  SF_CUDA(cudaMalloc(&g->shot_cand_offsets, size_t(cap + 1) * 8));
  SF_CUDA(cudaMalloc(&g->shot_counts, size_t(cap) * 4));
  SF_CUDA(cudaMalloc(&g->shot_runs, size_t(cap) * 5 * sizeof(int4)));
  SF_CUDA(cudaMalloc(&g->shot_lrf, size_t(cap) * 9 * 8));
  SF_CUDA(cudaMalloc(&g->shot_frame32, size_t(cap) * kFrame32Stride * 4));
  SF_CUDA(cudaMalloc(&g->shot_worklist, size_t(cap + 1) * 4));
  if (g->shot_pairs == nullptr) {  // two sets of (pairs found, list cursor): a call resets the set of the next one
    SF_CUDA(cudaMalloc(&g->shot_pairs, 32));
    SF_CUDA(cudaMemset(g->shot_pairs, 0, 32));
    g->shot_call_parity = 0;
  }
  g->shot_q_capacity = cap;
  return SF_OK;
}

static int shot_reserve_entries(sf_grid* g, int64_t entries) {
  if (entries <= g->shot_nbr_capacity) return SF_OK;
  cudaFree(g->shot_nbr);
  g->shot_nbr_capacity = 0;
  SF_CUDA(cudaMalloc(&g->shot_nbr, size_t(entries) * sizeof(float4)));
  g->shot_nbr_capacity = entries;
  return SF_OK;
}

extern "C" int sf_shot_single_scale(sf_grid* g, const double* queries, int64_t nq, double radius, int32_t min_nb,
                                    int32_t normalize, void* out, int32_t out_is_f64, double* lrf_out,
                                    int64_t* pairs_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0 && g->has_normals, SF_ERR_ARG, "sf_shot_single_scale: grid built without normals");
  if (pairs_host) *pairs_host = 0;
  if (nq == 0) return SF_OK;  // (an empty query block has null pointers: zero-row tensors)
  SF_REQUIRE(queries && out && nq > 0, SF_ERR_ARG, "sf_shot_single_scale: bad arguments");
  SF_REQUIRE(radius_fits(g, radius), SF_ERR_ARG,
             "sf_shot_single_scale: radius %g exceeds the cell edge %g the grid was built for", radius, g->cell);
  if (int rc = shot_reserve_queries(g, nq)) return rc;
  int64_t* cand_offsets = g->shot_cand_offsets;
  int32_t* counts = g->shot_counts;
  float* frame32 = g->shot_frame32;
  double* lrf = lrf_out != nullptr ? lrf_out : g->shot_lrf;
  // [0] neighbour pairs found, [1] cursor of the padded list — of this call's set of counters
  unsigned long long* pair_counter = g->shot_pairs + 2 * g->shot_call_parity;
  unsigned long long* next_counters = g->shot_pairs + 2 * (g->shot_call_parity ^ 1);
  int32_t* worklist = g->shot_worklist;  // [0] = number of queries handed to the exact kernel, then their indices
  const GridView view = g->view();
  // The padded list holds one 16-byte entry per CANDIDATE; its size is read back (the one synchronisation of the
  // call) unless the handle is in speculative mode and a previous call left an estimate: then the list is sized
  // from that estimate, the device checks it (status 2) and every kernel below returns at once when it does not fit.
  const bool assume_size = (g->speculative & 2) && g->shot_entries_per_query > 0.0 && pairs_host == nullptr;
  const int32_t* status = nullptr;
  if (assume_size) {
    if (int rc = shot_reserve_entries(g, int64_t(g->shot_entries_per_query * 1.25 * double(nq)) + 4096)) return rc;
    status = g->status_dev;
  }
  candidate_count_kernel<<<unsigned((nq + 255) / 256), 256, 0, stream>>>(
      view, queries, nq, radius * radius, cand_offsets, g->shot_runs, pair_counter + 1,
      assume_size ? g->shot_nbr_capacity : INT64_MAX, assume_size ? g->status_dev : nullptr, next_counters, worklist);
  SF_CUDA(cudaGetLastError());
  g->shot_call_parity ^= 1;  // (only once the kernel that resets the other set is in the stream)
  if (!assume_size) {
    int64_t total = 0;
    SF_CUDA(cudaMemcpyAsync(&total, pair_counter + 1, 8, cudaMemcpyDeviceToHost, stream));
    SF_CUDA(cudaStreamSynchronize(stream));
    if (int rc = shot_reserve_entries(g, total + total / 16 + 4096)) return rc;
    g->shot_entries_per_query = double(total) / double(nq);
  }
  float4* nbr = g->shot_nbr;  // padded list of 16-byte entries: float32 offset, position | zero-distance flag << 31
  const unsigned warp_blocks = unsigned((nq * 32 + 255) / 256);
  profile_mark(0, stream);
  search_moments_kernel<<<warp_blocks, 256, 0, stream>>>(view, queries, nq, radius, radius * radius, cand_offsets,
                                                        g->shot_runs, nbr, counts, lrf, pair_counter, status);
  profile_mark(1, stream);
  lrf_eigen_kernel<<<unsigned((nq + 127) / 128), 128, 0, stream>>>(nq, cand_offsets, counts, lrf, frame32, status);
  profile_mark(2, stream);
  int rc = launch_descriptor(g, queries, nq, radius, cand_offsets, counts, nbr, true, lrf, frame32, lrf_out != nullptr, min_nb,
                             normalize, out, out_is_f64, worklist + 1, worklist, status, stream, true);
  profile_mark(3, stream);
  if (rc == SF_OK && pairs_host != nullptr) {  // neighbour pairs found (logging / algorithmic-byte accounting)
    unsigned long long pairs = 0;
    int32_t deferred = 0;
    SF_CUDA(cudaMemcpyAsync(&pairs, pair_counter, 8, cudaMemcpyDeviceToHost, stream));
    SF_CUDA(cudaMemcpyAsync(&deferred, worklist, 4, cudaMemcpyDeviceToHost, stream));
    SF_CUDA(cudaStreamSynchronize(stream));
    *pairs_host = int64_t(pairs);
    g_last_deferred = env_flag("SF_SHOT_EXACT") ? nq : int64_t(deferred);
  }
  return rc;
}
