// Kernel group P: FPFH (compute_fpfh_descriptor, fpfh.py:16-117).
//   P1 SPFH <- fpfh.py:38-90: Darboux-frame features (alpha, phi, theta) of every neighbour at distance > 0, binned
//      with NumPy's histogram semantics (float64 edges from np.linspace handed in by the host), integer counts in
//      shared memory (order-independent, hence exact), divided by the neighbourhood size INCLUDING the point itself.
//      Rows are written in cell-sorted order so that stage 2 gathers them with good locality.
//        spfh_tile_kernel  warp per tile of 32 points, pairs flattened over the lanes (rows of up to 128 bins)
//        spfh_kernel       warp per point (wider rows; reference of the tile kernel in the tests)
//      Both take the three bins of a pair from sf_math.cuh::fpfh_pair_bins (float32-filtered, float64 where unsure).
//   P2 FPFH <- fpfh.py:97-116: spfh[i] + (sum_{j, d_j > 0} spfh[j] / d_j) / K_i on the keypoints.
//        fpfh_rows4_kernel the fused drivers' padded rows: one load instruction fetches the rows of 32 / L neighbours
//        fpfh_kernel       the piecewise sf_fpfh (caller's CSR, float64 distances) and rows wider than 128 bins
//   Fused drivers: sf_fpfh_cloud (one GPU) and sf_fpfh_block_begin / _spfh / _rows (one block of the cell-sorted cloud
//   per GPU, the all-gather of the SPFH rows between the last two): search_weights_kernel writes the padded neighbour
//   lists and the float32 weights 1 / d in ONE scan of the candidate cells.
#include <cub/cub.cuh>

#include "sf_common.cuh"

namespace sf {

constexpr int kMaxBins = 64;
__constant__ double c_edges[3][kMaxBins + 1];
__constant__ double c_scale[3];  // n_bins / (last edge - first edge), per feature
__constant__ float c_lo32[3], c_scale32[3];  // float32 roundings of the first edges and of the scales (filtered bins)

__global__ void __launch_bounds__(256, 4)
    spfh_kernel(GridView g, int64_t first, int64_t count, const int64_t* __restrict__ offsets,
                const int32_t* __restrict__ counts, const int32_t* __restrict__ nbr, int n_bins, int decorrelated,
                int width, int stride, int allow_fast, float* __restrict__ spfh) {
  // stride >= width: floats between consecutive rows (the fused driver pads rows to 16 bytes; the pad holds zeros)
  // allow_fast: bins from the float32-filtered features (sf_math.cuh::fpfh_bins_fast), float64 where unsure
  // counts == nullptr: CSR rows [offsets[s], offsets[s+1]); otherwise padded rows [offsets[s], offsets[s] + counts[s])
  extern __shared__ int hist_mem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int warps_per_block = blockDim.x >> 5;
  int* hist = hist_mem + warp * width;
  const int64_t warps_total = int64_t(gridDim.x) * warps_per_block;
  for (int64_t s = blockIdx.x * int64_t(warps_per_block) + warp; s < count; s += warps_total) {
    for (int b = lane; b < width; b += 32) hist[b] = 0;
    __syncwarp();
    const double4 p = load_pt(g.pts + first + s);
    const double4 un = load_pt(g.nrm + first + s);
    const double u[3] = {un.x, un.y, un.z};
    const float u32[3] = {float(un.x), float(un.y), float(un.z)};
    const float u_norm = sqrtf(u32[0] * u32[0] + u32[1] * u32[1] + u32[2] * u32[2]);
    const int64_t begin = offsets[s], end = counts ? begin + counts[s] : offsets[s + 1];
    for (int64_t i = begin + lane; i < end; i += 32) {
      const int j = __ldg(nbr + i);
      const double4 pj = load_pt(g.pts + j);
      const double4 nj4 = load_pt(g.nrm + j);
      const double rel[3] = {pj.x - p.x, pj.y - p.y, pj.z - p.z};
      const double nj[3] = {nj4.x, nj4.y, nj4.z};
      int ia, ip, it;
      if (fpfh_pair_bins(rel, u, u32, u_norm, nj, n_bins, &c_edges[0][0], kMaxBins + 1, c_scale, c_lo32, c_scale32,
                         allow_fast != 0, ia, ip, it)) {
        if (decorrelated) {  // three independent np.histogram calls: each feature dropped on its own
          if (ia >= 0) atomicAdd(hist + ia, 1);
          if (ip >= 0) atomicAdd(hist + n_bins + ip, 1);
          if (it >= 0) atomicAdd(hist + 2 * n_bins + it, 1);
        } else if (ia >= 0 && ip >= 0 && it >= 0) {  // np.histogramdd: dropped when any coordinate is outside
          atomicAdd(hist + (ia * n_bins + ip) * n_bins + it, 1);
        }
      }
    }
    __syncwarp();
    // hist / K (fpfh.py:79: K counts the point itself and duplicates). The rows are float32 values: the quotient
    // is formed in float32 (two roundings, 1.2e-7 relative, against the 1e-4 bar) instead of a float64 division
    // per bin.
    const float inv_k = end > begin ? 1.0f / float(end - begin) : 0.0f;
    float* row = spfh + s * int64_t(stride);
    for (int b = lane; b < stride; b += 32) row[b] = b < width ? float(hist[b]) * inv_k : 0.0f;
    __syncwarp();
  }
}

// SPFH by TILES of 32 consecutive cell-sorted points, one warp per tile: the tile's neighbour pairs (about 2 400 at
// C3) are flattened and dealt to the lanes 32 at a time, whatever point they belong to. Against one warp per point
// (spfh_kernel: K = 74 pairs in three rounds of 32 lanes, i.e. 77 % of the lanes busy, plus a prologue / epilogue of
// ~360 instructions per point for 780 of pair arithmetic) every round but the tile's last is full and the per-point
// work (coordinates, normal, clearing and writing the histogram) is done once per tile with all lanes. The owners'
// data and the 32 integer histograms live in shared memory. Rows of up to 128 bins; wider rows use spfh_kernel.
constexpr int kSpfhTileWarps = 4;
struct SpfhTile {  // per warp
  double px[32], py[32], pz[32], ux[32], uy[32], uz[32];
  float4 u32[32];  // float32 rounding of the normal, .w = its norm
  int64_t cursor[32];
  int prefix[33];
  float inv_k[32];
};

__global__ void __launch_bounds__(kSpfhTileWarps * 32, 8)
    spfh_tile_kernel(GridView g, int64_t first, int64_t count, const int64_t* __restrict__ offsets,
                     const int32_t* __restrict__ counts, const int32_t* __restrict__ nbr, int n_bins, int decorrelated,
                     int width, int stride, int allow_fast, float* __restrict__ spfh) {
  extern __shared__ unsigned char tile_mem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const size_t per_warp = sizeof(SpfhTile) + size_t(32) * width * sizeof(int);
  SpfhTile& st = *reinterpret_cast<SpfhTile*>(tile_mem + warp * per_warp);
  int* hist = reinterpret_cast<int*>(tile_mem + warp * per_warp + sizeof(SpfhTile));
  const int64_t tiles = (count + 31) / 32;
  const int64_t warps_total = int64_t(gridDim.x) * kSpfhTileWarps;
  for (int64_t tile = blockIdx.x * int64_t(kSpfhTileWarps) + warp; tile < tiles; tile += warps_total) {
    const int64_t s0 = tile * 32;
    const int in_tile = int(count - s0 < 32 ? count - s0 : 32);
    int cnt = 0;
    if (lane < in_tile) {
      const double4 p = load_pt(g.pts + first + s0 + lane);
      const double4 un = load_pt(g.nrm + first + s0 + lane);
      st.px[lane] = p.x; st.py[lane] = p.y; st.pz[lane] = p.z;
      st.ux[lane] = un.x; st.uy[lane] = un.y; st.uz[lane] = un.z;
      const float fx = float(un.x), fy = float(un.y), fz = float(un.z);
      st.u32[lane] = make_float4(fx, fy, fz, sqrtf(fx * fx + fy * fy + fz * fz));
      const int64_t begin = offsets[s0 + lane];
      cnt = counts ? counts[s0 + lane] : int(offsets[s0 + lane + 1] - begin);
      st.cursor[lane] = begin;
      // hist / K (fpfh.py:79: K counts the point itself and duplicates); float32 quotient, see spfh_kernel
      st.inv_k[lane] = cnt > 0 ? 1.0f / float(cnt) : 0.0f;
    }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(kFull, incl, o);
      if (lane >= o) incl += t;
    }
    st.prefix[lane + 1] = incl;
    if (lane == 0) st.prefix[0] = 0;
    const int total = __shfl_sync(kFull, incl, 31);
    for (int b = lane; b < in_tile * width; b += 32) hist[b] = 0;
    __syncwarp();
    int owner = 0;
    for (int idx = lane; idx < total; idx += 32) {
      while (idx >= st.prefix[owner + 1]) ++owner;  // idx < total = prefix[32]: stops at an owner with pairs
      const int j = __ldg(nbr + st.cursor[owner] + (idx - st.prefix[owner]));
      const double4 pj = load_pt(g.pts + j);
      const double4 nj4 = load_pt(g.nrm + j);
      const double rel[3] = {pj.x - st.px[owner], pj.y - st.py[owner], pj.z - st.pz[owner]};
      const double u[3] = {st.ux[owner], st.uy[owner], st.uz[owner]};
      const double nj[3] = {nj4.x, nj4.y, nj4.z};
      const float4 uf = st.u32[owner];
      const float u32[3] = {uf.x, uf.y, uf.z};
      int ia, ip, it;
      if (fpfh_pair_bins(rel, u, u32, uf.w, nj, n_bins, &c_edges[0][0], kMaxBins + 1, c_scale, c_lo32, c_scale32,
                         allow_fast != 0, ia, ip, it)) {
        int* h = hist + owner * width;
        if (decorrelated) {  // three independent np.histogram calls: each feature dropped on its own
          if (ia >= 0) atomicAdd(h + ia, 1);
          if (ip >= 0) atomicAdd(h + n_bins + ip, 1);
          if (it >= 0) atomicAdd(h + 2 * n_bins + it, 1);
        } else if (ia >= 0 && ip >= 0 && it >= 0) {  // np.histogramdd: dropped when any coordinate is outside
          atomicAdd(h + (ia * n_bins + ip) * n_bins + it, 1);
        }
      }
    }
    __syncwarp();
    for (int r = 0; r < in_tile; ++r) {
      float* row = spfh + (s0 + r) * int64_t(stride);
      const float inv_k = st.inv_k[r];
      for (int b = lane; b < stride; b += 32) row[b] = b < width ? float(hist[r * width + b]) * inv_k : 0.0f;
    }
    __syncwarp();  // the tables are rewritten by the next tile
  }
}

// Fused driver, stage 0: ONE scan of the candidate cells of every cloud point (cell-sorted order) writes the
// neighbours into a PADDED list (slots sized by the candidate count, a cell_start lookup — no counting pass over
// the candidates), the float32 weights 1/d that stage 2 needs (fpfh.py:112-114; 0 where d == 0) and the counts.
//
// Work unit: a TILE of 32 consecutive cell-sorted points, one warp. The points of a tile lie in a handful of cells
// (7.6 points per occupied cell at C3: the cloud is a surface), and all the points of a cell share their candidate set (the 9 runs around the cell): per distinct cell of the
// tile the warp stages the candidates in shared memory once (chunks of kSearchChunk), then each of the cell's
// points in the tile scans them from there with all 32 lanes. Against one warp per point walking the runs in
// global memory this removes the per-point run setup, the run lookup per candidate and the L1 traffic
// (measured at C3: 1.28 -> 0.93 ms), and the neighbour order is the same (run order, ascending position).
constexpr int kSearchChunk = 256;
constexpr int kSearchWarps = 8;

struct SearchStage {  // per warp, in shared memory
  double x[kSearchChunk], y[kSearchChunk], z[kSearchChunk];
  int pos[kSearchChunk];
  // ring of hits waiting for their weight: the float64 sqrt and reciprocal are evaluated 32 hits at a time with
  // every lane busy (about a third of the candidates are hits) and the list is written with full-warp stores
  double hit_d2[64];
  int hit_pos[64];
};

__global__ void __launch_bounds__(kSearchWarps * 32)
    search_weights_kernel(GridView g, int64_t block_first, int64_t n, double r2,
                          const int64_t* __restrict__ cand_offsets,
                          int32_t* __restrict__ nbr, float* __restrict__ weights, int32_t* __restrict__ counts,
                          unsigned long long* __restrict__ pair_counter) {
  extern __shared__ unsigned char stage_mem[];
  const int lane = threadIdx.x & 31;
  SearchStage& st = reinterpret_cast<SearchStage*>(stage_mem)[threadIdx.x >> 5];
  const int64_t tile = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  const int64_t s0 = tile * 32;
  if (s0 >= n) return;
  const int in_tile = int(n - s0 < 32 ? n - s0 : 32);
  // lane l owns point s0 + l: its coordinates, its cell, its running count and output cursor
  double4 me = make_double4(0, 0, 0, 0);
  int cx = 0, cy = 0, cz = 0;
  int64_t cursor = 0;
  if (lane < in_tile) {  // the cell-sorted points [block_first, block_first + n); offsets / counts relative to it
    me = load_pt(g.pts + block_first + s0 + lane);
    cx = cell_coord(me.x, g.origin[0], g.inv_cell, g.dims[0]);
    cy = cell_coord(me.y, g.origin[1], g.inv_cell, g.dims[1]);
    cz = cell_coord(me.z, g.origin[2], g.inv_cell, g.dims[2]);
    cursor = cand_offsets[s0 + lane];
  }
  int my_count = 0;
  int first = 0;  // first lane of the current group (lanes of one cell are consecutive: the points are cell-sorted)
  while (first < in_tile) {
    const int gx = __shfl_sync(kFull, cx, first), gy = __shfl_sync(kFull, cy, first), gz = __shfl_sync(kFull, cz, first);
    const unsigned same = __ballot_sync(kFull, lane >= first && lane < in_tile && cx == gx && cy == gy && cz == gz);
    const int last = 32 - __clz(same);  // one past the group's last lane
    const Runs runs = build_runs_cell(g, gx, gy, gz, lane);
    const int total = runs.pref[9];
    for (int chunk = 0; chunk < total; chunk += kSearchChunk) {
      const int len = total - chunk < kSearchChunk ? total - chunk : kSearchChunk;
      __syncwarp();  // the previous chunk has been consumed
      for (int v = lane; v < len; v += 32) {
        const int pos = run_position(runs, chunk + v);
        const double4 p = load_pt(g.pts + pos);
        st.x[v] = p.x; st.y[v] = p.y; st.z[v] = p.z;
        st.pos[v] = pos;
      }
      __syncwarp();
      for (int owner = first; owner < last; ++owner) {
        const double qx = __shfl_sync(kFull, me.x, owner), qy = __shfl_sync(kFull, me.y, owner),
                     qz = __shfl_sync(kFull, me.z, owner);
        int64_t out = __shfl_sync(kFull, cursor, owner);
        int found = 0, head = 0, tail = 0;  // found = hits written out; ring entries [head, tail)
        for (int base = 0; base < len; base += 32) {
          const int v = base + lane;
          bool hit = false;
          double d2 = 0.0;
          if (v < len) {
            d2 = rdist3(qx - st.x[v], qy - st.y[v], qz - st.z[v]);
            hit = d2 <= r2;
          }
          const unsigned mask = __ballot_sync(kFull, hit);
          if (hit) {
            const int slot = (tail + __popc(mask & lanemask_lt())) & 63;
            st.hit_d2[slot] = d2;
            st.hit_pos[slot] = st.pos[v];
          }
          tail += __popc(mask);
          __syncwarp();
          if (tail - head >= 32) {
            const int slot = (head + lane) & 63;
            const double h2 = st.hit_d2[slot];
            nbr[out + found + lane] = st.hit_pos[slot];
            weights[out + found + lane] = h2 > 0.0 ? float(1.0 / sqrt(h2)) : 0.0f;
            head += 32;
            found += 32;
            __syncwarp();
          }
        }
        if (lane < tail - head) {  // what is left in the ring
          const int slot = (head + lane) & 63;
          const double h2 = st.hit_d2[slot];
          nbr[out + found + lane] = st.hit_pos[slot];
          weights[out + found + lane] = h2 > 0.0 ? float(1.0 / sqrt(h2)) : 0.0f;
        }
        found += tail - head;
        __syncwarp();
        if (lane == owner) {
          cursor += found;
          my_count += found;
        }
      }
    }
    first = last;
  }
  if (lane < in_tile) counts[s0 + lane] = my_count;
  const int tile_pairs = warp_sum(my_count);
  if (lane == 0) atomicAdd(pair_counter, static_cast<unsigned long long>(tile_pairs));
}

__global__ void __launch_bounds__(256)
    self_candidate_count_kernel(GridView g, int64_t first, int64_t n, int64_t* __restrict__ cand) {
  const int64_t s = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (s >= n) return;
  const double4 me = load_pt(g.pts + first + s);
  const int cx = cell_coord(me.x, g.origin[0], g.inv_cell, g.dims[0]);
  const int cy = cell_coord(me.y, g.origin[1], g.inv_cell, g.dims[1]);
  const int cz = cell_coord(me.z, g.origin[2], g.inv_cell, g.dims[2]);
  const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dims[0] - 1);
  int total = 0;
  for (int dz = -1; dz <= 1; ++dz)
    for (int dy = -1; dy <= 1; ++dy) {
      const int yy = cy + dy, zz = cz + dz;
      if (yy < 0 || yy >= g.dims[1] || zz < 0 || zz >= g.dims[2]) continue;
      const int64_t base = (int64_t(zz) * g.dims[1] + yy) * g.dims[0];
      total += __ldg(g.cell_start + base + x1 + 1) - __ldg(g.cell_start + base + x0);
    }
  cand[s] = total;
}

__global__ void __launch_bounds__(256)
    keypoint_position_kernel(const int32_t* __restrict__ inv_perm, const int64_t* __restrict__ keypoints, int64_t nq,
                             int32_t* __restrict__ pos, int32_t* __restrict__ ids) {
  const int64_t q = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (q >= nq) return;
  pos[q] = inv_perm[keypoints[q]];
  ids[q] = int32_t(q);
}

// One warp per keypoint. The neighbour list is consumed in chunks of 32: each lane loads one (index, 1/d) pair,
// then the pairs are broadcast by shuffle and every lane accumulates its own bins — the row loads of consecutive
// neighbours are independent, so several are in flight at once. Column blocks of 32 bins are register tiles;
// a remainder of at most 4 columns (e.g. bin 32 of the 33-bin layout) is handled lane-per-neighbour and reduced.
template <int kBlocks, typename OutT>
__global__ void __launch_bounds__(256)
    fpfh_kernel(const int32_t* __restrict__ inv_perm, const int64_t* __restrict__ offsets,
                const int32_t* __restrict__ counts, const int32_t* __restrict__ nbr, const double* __restrict__ dist,
                const float* __restrict__ weights, int csr_by_keypoint,
                const float* __restrict__ spfh, int width, int bin_base, int rem,
                const int64_t* __restrict__ keypoints, const int32_t* __restrict__ order, int64_t nq,
                int64_t first, OutT* __restrict__ out) {
  // first: the CSR rows cover the cell-sorted points [first, ...) (a block of the cloud, multi-GPU)
  const int lane = threadIdx.x & 31;
  const int64_t slot = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (slot >= nq) return;
  // `order`: the keypoints sorted by their cell-sorted position, so that the warps in flight gather SPFH rows of the
  // same neighbourhood of the cloud (L1/L2 hits instead of DRAM: callers pass keypoints in arbitrary order)
  const int64_t q = order ? order[slot] : slot;
  const int64_t s = inv_perm[keypoints[q]];
  const int64_t row_id = csr_by_keypoint ? q : s - first;  // CSR rows follow the keypoints, or the cell-sorted points
  // counts: padded rows (fused driver); weights: float32 1/d precomputed by the search (0 where d == 0)
  const int64_t begin = offsets[row_id], end = counts ? begin + counts[row_id] : offsets[row_id + 1];
  float acc[kBlocks];
#pragma unroll
  for (int r = 0; r < kBlocks; ++r) acc[r] = 0.0f;
  float tail[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  const int rem_base = bin_base + 32 * kBlocks;
  const bool last_ok = bin_base + lane + 32 * (kBlocks - 1) < width;
  for (int64_t base = begin; base < end; base += 32) {
    const int64_t i = base + lane;
    int my_j = 0;
    float my_w = 0.0f;
    if (i < end) {
      my_j = __ldg(nbr + i);
      if (weights != nullptr) {
        my_w = __ldg(weights + i);
      } else {
        const double d = __ldg(dist + i);
        my_w = d > 0.0 ? float(1.0 / d) : 0.0f;  // fpfh.py:112-114: the tree's own distances decide
      }
    }
    const int cnt = int(end - base < 32 ? end - base : 32);
    if (rem > 0 && my_w != 0.0f) {
      const float* row = spfh + int64_t(my_j) * width + rem_base;
      for (int c = 0; c < rem; ++c) tail[c] += __ldg(row + c) * my_w;
    }
#pragma unroll 8
    for (int t = 0; t < cnt; ++t) {
      const int j = __shfl_sync(kFull, my_j, t);
      const float w = __shfl_sync(kFull, my_w, t);
      const float* row = spfh + int64_t(j) * width + bin_base + lane;
#pragma unroll
      for (int r = 0; r < kBlocks; ++r)  // w == 0 contributes 0; the last block may be partially masked
        if (r < kBlocks - 1 || last_ok) acc[r] = fmaf(__ldg(row + 32 * r), w, acc[r]);
    }
  }
  const float k_all = float(end - begin);
  const float* own = spfh + s * width;
  OutT* dst = out + q * int64_t(width);
#pragma unroll
  for (int r = 0; r < kBlocks; ++r) {
    const int b = bin_base + lane + 32 * r;
    if (b < width) dst[b] = OutT(end > begin ? own[b] + acc[r] / k_all : 0.0f);
  }
  for (int c = 0; c < rem; ++c) {
    const float total = warp_sum(tail[c]);
    if (lane == 0) dst[rem_base + c] = OutT(end > begin ? own[rem_base + c] + total / k_all : 0.0f);
  }
}



// The fused driver's FPFH stage: SPFH rows padded to a multiple of four floats (16-byte aligned), L = stride / 4
// lanes per row, each loading one float4, so that ONE load instruction of the warp fetches the rows of
// G = 32 / L neighbours (33 bins: L = 9, three neighbours per instruction; fpfh_kernel spends a load, two shuffles
// and the address arithmetic on every single neighbour and was issue-bound). Lane l serves neighbour slot l / L and
// columns 4 (l % L) .. 4 (l % L) + 3; the G partial sums of a column are added at the end. Rows of up to 128 bins.
template <int L, typename OutT>
__global__ void __launch_bounds__(256)
    fpfh_rows4_kernel(const int32_t* __restrict__ inv_perm, const int64_t* __restrict__ offsets,
                      const int32_t* __restrict__ counts, const int32_t* __restrict__ nbr,
                      const float* __restrict__ weights, const float4* __restrict__ spfh4, int width,
                      const int64_t* __restrict__ keypoints, const int32_t* __restrict__ order, int64_t nq,
                      int64_t first, OutT* __restrict__ out) {
  constexpr int G = 32 / L, kSteps = (32 + G - 1) / G;
  const int lane = threadIdx.x & 31;
  const int64_t slot = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (slot >= nq) return;
  const int64_t q = order ? order[slot] : slot;
  const int64_t s = inv_perm[keypoints[q]];
  const int64_t begin = offsets[s - first];  // the lists cover the cell-sorted points [first, ...)
  const int cnt = counts[s - first];
  // lanes beyond G * L ride along with the last slot (their loads hit sectors that slot fetches anyway) and their
  // sums are never read: no predication inside the loop
  const int grp = lane / L < G ? lane / L : G - 1;
  const int sub = lane - (lane / L) * L;
  const float4* col = spfh4 + sub;
  float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  // one step: the G slots fetch the rows of neighbours src = t * G + slot of this batch of 32 list entries
#define SF_ROWS4_STEP(t, guard)                                             \
  {                                                                         \
    const int src = (t) * G + grp;                                          \
    const int j = __shfl_sync(kFull, my_j, src);                            \
    float w = __shfl_sync(kFull, my_w, src);                                \
    if (guard) w = src < 32 ? w : 0.0f; /* the shuffle wraps beyond 31 */   \
    const float4 x = __ldg(col + int64_t(j) * L);                           \
    acc.x = fmaf(x.x, w, acc.x);                                            \
    acc.y = fmaf(x.y, w, acc.y);                                            \
    acc.z = fmaf(x.z, w, acc.z);                                            \
    acc.w = fmaf(x.w, w, acc.w);                                            \
  }
  for (int base = 0; base < cnt; base += 32) {
    const int i = base + lane;
    int my_j = 0;
    float my_w = 0.0f;  // 0 beyond the list and for the point itself (d == 0): contributes nothing
    if (i < cnt) {
      my_j = __ldg(nbr + begin + i);
      my_w = __ldg(weights + begin + i);
    }
    const int left = cnt - base;
    if (left >= 32) {
#pragma unroll
      for (int t = 0; t < kSteps; ++t) SF_ROWS4_STEP(t, G * kSteps > 32 && t == kSteps - 1)
    } else {
      const int steps = (left + G - 1) / G;  // entries beyond `left` carry weight 0
#pragma unroll 2
      for (int t = 0; t < steps; ++t) SF_ROWS4_STEP(t, G * kSteps > 32)
    }
  }
#undef SF_ROWS4_STEP
  const float4 part = acc;  // lanes sub + gi * L hold the other partial sums of column block `sub` (read unmodified:
                            // a shuffle from beyond lane 31 returns the caller's own value)
#pragma unroll
  for (int gi = 1; gi < G; ++gi) {
    acc.x += __shfl_down_sync(kFull, part.x, gi * L);
    acc.y += __shfl_down_sync(kFull, part.y, gi * L);
    acc.z += __shfl_down_sync(kFull, part.z, gi * L);
    acc.w += __shfl_down_sync(kFull, part.w, gi * L);
  }
  if (lane < L) {  // fpfh.py:115: spfh[i] + sum / K, K counting the point itself
    const float k_all = float(cnt);
    const float4 own = __ldg(spfh4 + s * L + lane);
    const float v[4] = {own.x + acc.x / k_all, own.y + acc.y / k_all, own.z + acc.z / k_all, own.w + acc.w / k_all};
    OutT* dst = out + q * int64_t(width) + 4 * lane;
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (4 * lane + c < width) dst[c] = OutT(cnt > 0 ? v[c] : 0.0f);
  }
}

}  // namespace sf

using namespace sf;

// Floats per SPFH row: 3 n_bins (decorrelated) or n_bins^3, with n_bins in [1, kMaxBins] and at most 8192 bins.
static int histogram_width(const char* who, int32_t n_bins, int32_t decorrelated, int* width) {
  SF_REQUIRE(n_bins >= 1 && n_bins <= kMaxBins, SF_ERR_CAPACITY, "%s: n_bins must be in [1, %d]", who, kMaxBins);
  const int64_t width64 = decorrelated ? 3 * int64_t(n_bins) : int64_t(n_bins) * n_bins * n_bins;
  SF_REQUIRE(width64 <= 8192, SF_ERR_CAPACITY, "%s: histogram width %lld exceeds 8192", who, (long long)width64);
  *width = int(width64);
  return SF_OK;
}

static int launch_spfh(sf_grid* g, int64_t first, int64_t count, const int64_t* offsets, const int32_t* counts,
                       const int32_t* nbr, int32_t n_bins, int32_t decorrelated, const double* edges_host, float* spfh,
                       int stride, cudaStream_t stream) {
  SF_REQUIRE(g != nullptr && g->n > 0 && g->has_normals, SF_ERR_ARG, "sf_spfh: grid built without normals");
  SF_REQUIRE(offsets && nbr && edges_host && spfh, SF_ERR_ARG, "sf_spfh: null argument");
  SF_REQUIRE(first >= 0 && count >= 0 && first + count <= g->n, SF_ERR_ARG, "sf_spfh: point range outside the cloud");
  if (count == 0) return SF_OK;
  int width = 0;
  if (int rc = histogram_width("sf_spfh", n_bins, decorrelated, &width)) return rc;
  double edges[3][kMaxBins + 1] = {};
  for (int f = 0; f < 3; ++f)
    for (int b = 0; b <= n_bins; ++b) edges[f][b] = edges_host[f * (n_bins + 1) + b];
  double scale[3];
  for (int f = 0; f < 3; ++f) scale[f] = double(n_bins) / (edges[f][n_bins] - edges[f][0]);
  SF_CUDA(cudaMemcpyToSymbolAsync(c_edges, edges, sizeof(edges), 0, cudaMemcpyHostToDevice, stream));
  SF_CUDA(cudaMemcpyToSymbolAsync(c_scale, scale, sizeof(scale), 0, cudaMemcpyHostToDevice, stream));
  float lo32[3], scale32[3];
  for (int f = 0; f < 3; ++f) {
    lo32[f] = float(edges[f][0]);
    scale32[f] = float(scale[f]);
  }
  SF_CUDA(cudaMemcpyToSymbolAsync(c_lo32, lo32, sizeof(lo32), 0, cudaMemcpyHostToDevice, stream));
  SF_CUDA(cudaMemcpyToSymbolAsync(c_scale32, scale32, sizeof(scale32), 0, cudaMemcpyHostToDevice, stream));
  // SF_SPFH_EXACT=1 (tests, measurements): every pair through the float64 path
  const char* exact_env = getenv("SF_SPFH_EXACT");
  const int allow_fast = (exact_env != nullptr && exact_env[0] == '1') ? 0 : 1;
  SF_CUDA(cudaStreamSynchronize(stream));  // `edges` is a stack buffer
  const int row_stride = stride > 0 ? stride : width;
  const char* no_tiles = getenv("SF_SPFH_NO_TILES");  // measurement / test switch
  if (width <= 128 && !(no_tiles != nullptr && no_tiles[0] == '1')) {
    const size_t smem = size_t(kSpfhTileWarps) * (sizeof(SpfhTile) + size_t(32) * width * sizeof(int));
    if (smem > 48 * 1024)
      SF_CUDA(cudaFuncSetAttribute(spfh_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    const int64_t blocks_needed = ((count + 31) / 32 + kSpfhTileWarps - 1) / kSpfhTileWarps;
    const unsigned blocks = unsigned(blocks_needed < 148 * 16 ? blocks_needed : 148 * 16);
    spfh_tile_kernel<<<blocks, kSpfhTileWarps * 32, smem, stream>>>(g->view(), first, count, offsets, counts, nbr, n_bins,
                                                                    decorrelated, width, row_stride, allow_fast, spfh);
  } else {
    int warps = 8;
    while (warps > 1 && size_t(warps) * width * sizeof(int) > 64 * 1024) warps >>= 1;
    const size_t smem = size_t(warps) * width * sizeof(int);
    if (smem > 48 * 1024)
      SF_CUDA(cudaFuncSetAttribute(spfh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    const int64_t blocks_needed = (count + warps - 1) / warps;
    const unsigned blocks = unsigned(blocks_needed < 148 * 8 ? blocks_needed : 148 * 8);
    spfh_kernel<<<blocks, warps * 32, smem, stream>>>(g->view(), first, count, offsets, counts, nbr, n_bins, decorrelated,
                                                      width, row_stride, allow_fast, spfh);
  }
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_spfh(sf_grid* g, int64_t first, int64_t count, const int64_t* offsets, const int32_t* nbr,
                       int32_t n_bins, int32_t decorrelated, const double* edges_host, float* spfh, void* stream_) {
  return launch_spfh(g, first, count, offsets, nullptr, nbr, n_bins, decorrelated, edges_host, spfh, 0,
                     static_cast<cudaStream_t>(stream_));
}

template <typename OutT>
static int launch_fpfh(sf_grid* g, const int64_t* offsets, const int32_t* counts, const int32_t* nbr, const double* dist,
                       const float* weights, int by_kp, const float* spfh, int width, int stride, int rows4,
                       const int64_t* keypoints, int64_t nq, int64_t first, OutT* out, cudaStream_t stream) {
  // rows4: the fused driver's rows, `stride` a multiple of four floats (at most 128) -> fpfh_rows4_kernel
  const int64_t threads = nq * 32;
  const unsigned blocks = unsigned((threads + 255) / 256);
  // processing order: keypoints by cell-sorted position (see fpfh_kernel); not worth a sort for a handful
  int32_t *pos = nullptr, *ids = nullptr, *pos_sorted = nullptr, *order = nullptr;
  void* sort_temp = nullptr;
  Scratch scratch(stream);
  if (nq >= 4096 && nq < (int64_t(1) << 31)) {
    size_t sort_bytes = 0;
    int end_bit = 1;
    while ((int64_t(1) << end_bit) < g->n) ++end_bit;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, pos, pos_sorted, ids, order, int(nq), 0, end_bit, stream);
    SF_CUDA(scratch.alloc(&pos, size_t(nq) * 4));
    SF_CUDA(scratch.alloc(&ids, size_t(nq) * 4));
    SF_CUDA(scratch.alloc(&pos_sorted, size_t(nq) * 4));
    SF_CUDA(scratch.alloc(&order, size_t(nq) * 4));
    SF_CUDA(scratch.alloc(&sort_temp, sort_bytes + 16));
    keypoint_position_kernel<<<unsigned((nq + 255) / 256), 256, 0, stream>>>(g->inv_perm, keypoints, nq, pos, ids);
    SF_CUDA(cub::DeviceRadixSort::SortPairs(sort_temp, sort_bytes, pos, pos_sorted, ids, order, int(nq), 0, end_bit,
                                            stream));
  }
  if (rows4) {
    const float4* spfh4 = reinterpret_cast<const float4*>(spfh);
#define SF_LAUNCH_ROWS4(LL) \
  case LL: fpfh_rows4_kernel<LL, OutT><<<blocks, 256, 0, stream>>>(g->inv_perm, offsets, counts, nbr, weights, spfh4, width, keypoints, order, nq, first, out); break;
    switch (stride / 4) {
      SF_LAUNCH_ROWS4(1) SF_LAUNCH_ROWS4(2) SF_LAUNCH_ROWS4(3) SF_LAUNCH_ROWS4(4) SF_LAUNCH_ROWS4(5) SF_LAUNCH_ROWS4(6)
      SF_LAUNCH_ROWS4(7) SF_LAUNCH_ROWS4(8) SF_LAUNCH_ROWS4(9) SF_LAUNCH_ROWS4(10) SF_LAUNCH_ROWS4(11) SF_LAUNCH_ROWS4(12)
      SF_LAUNCH_ROWS4(13) SF_LAUNCH_ROWS4(14) SF_LAUNCH_ROWS4(15) SF_LAUNCH_ROWS4(16) SF_LAUNCH_ROWS4(17) SF_LAUNCH_ROWS4(18)
      SF_LAUNCH_ROWS4(19) SF_LAUNCH_ROWS4(20) SF_LAUNCH_ROWS4(21) SF_LAUNCH_ROWS4(22) SF_LAUNCH_ROWS4(23) SF_LAUNCH_ROWS4(24)
      SF_LAUNCH_ROWS4(25) SF_LAUNCH_ROWS4(26) SF_LAUNCH_ROWS4(27) SF_LAUNCH_ROWS4(28) SF_LAUNCH_ROWS4(29) SF_LAUNCH_ROWS4(30)
      SF_LAUNCH_ROWS4(31) SF_LAUNCH_ROWS4(32)
      default: set_error("fpfh: padded stride %d unsupported", stride); return SF_ERR_ARG;
    }
#undef SF_LAUNCH_ROWS4
    SF_CUDA(cudaGetLastError());
    return SF_OK;
  }
  // Passes of up to 4 column blocks of 32 bins (register tiles). A final partial block is masked, except when it
  // is at most 4 columns wide and follows a full block (the 33-bin layout): then it rides along as the "tail".
  int base = 0;
  while (base < width) {
    const int left = width - base;
    int blocks_n = left / 32 < 4 ? left / 32 : 4;
    int rem = 0;
    if (blocks_n < 4) {
      const int r = left - blocks_n * 32;
      if (r > 0 && r <= 4 && blocks_n >= 1) rem = r;
      else if (r > 0) blocks_n += 1;
    }
#define SF_LAUNCH_FPFH(B) \
  fpfh_kernel<B, OutT><<<blocks, 256, 0, stream>>>(g->inv_perm, offsets, counts, nbr, dist, weights, by_kp, spfh, width, base, rem, keypoints, order, nq, first, out)
    switch (blocks_n) {
      case 1: SF_LAUNCH_FPFH(1); break;
      case 2: SF_LAUNCH_FPFH(2); break;
      case 3: SF_LAUNCH_FPFH(3); break;
      default: SF_LAUNCH_FPFH(4); break;
    }
#undef SF_LAUNCH_FPFH
    base += blocks_n * 32 + rem;
  }
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

extern "C" int sf_fpfh(sf_grid* g, const int64_t* offsets, const int32_t* nbr, const double* dist,
                       int32_t csr_by_keypoint, const float* spfh, int32_t width, const int64_t* keypoints, int64_t nq, void* out, int32_t out_is_f64,
                       void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_fpfh: grid not built");
  SF_REQUIRE(offsets && nbr && dist && spfh && keypoints && out && width > 0, SF_ERR_ARG, "sf_fpfh: null argument");
  if (nq == 0) return SF_OK;
  return out_is_f64 ? launch_fpfh(g, offsets, nullptr, nbr, dist, nullptr, csr_by_keypoint, spfh, width, width, 0, keypoints,
                                  nq, 0, static_cast<double*>(out), stream)
                    : launch_fpfh(g, offsets, nullptr, nbr, dist, nullptr, csr_by_keypoint, spfh, width, width, 0, keypoints,
                                  nq, 0, static_cast<float*>(out), stream);
}

// ---- the fused drivers: four stages on the cell-sorted points [first, first + count) ----------------------------------
//   candidates  padded list offsets (fpfh_candidates)                             sf_fpfh_block_begin
//   search      padded neighbour lists, weights 1 / d, counts (fpfh_search)       sf_fpfh_block_spfh
//   SPFH        rows of `stride` floats (launch_spfh)                             sf_fpfh_block_spfh
//   (multi-GPU caller: all-gather of the blocks' SPFH rows)
//   rows        FPFH rows of the keypoints in the block (launch_fpfh)             sf_fpfh_block_rows
// sf_fpfh_cloud runs the four on the whole cloud with its own temporaries; the block entry points run them on one block
// per GPU, and the temporaries between them belong to the caller.

// SPFH rows of up to 128 bins are padded to a multiple of four floats for fpfh_rows4_kernel (SF_FPFH_NO_ROWS4=1:
// measurement / test switch back to the per-neighbour gather of fpfh_kernel, on unpadded rows).
static void fpfh_row_layout(int width, int* stride, int* rows4) {
  const char* no_rows4 = getenv("SF_FPFH_NO_ROWS4");
  *rows4 = (width <= 128 && !(no_rows4 != nullptr && no_rows4[0] == '1')) ? 1 : 0;
  *stride = *rows4 ? (width + 3) / 4 * 4 : width;
}

// count > 0; reads *total = cand_offsets[count] back (synchronises the stream)
static int fpfh_candidates(sf_grid* g, int64_t first, int64_t count, int64_t* cand_offsets, int64_t* total,
                           Scratch& scratch, cudaStream_t stream) {
  int64_t* cand = nullptr;
  void* scan_temp = nullptr;
  size_t scan_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, cand, cand_offsets, int(count + 1), stream);
  SF_CUDA(scratch.alloc(&cand, size_t(count + 1) * 8));
  SF_CUDA(scratch.alloc(&scan_temp, scan_bytes + 16));
  SF_CUDA(cudaMemsetAsync(cand + count, 0, 8, stream));
  self_candidate_count_kernel<<<unsigned((count + 255) / 256), 256, 0, stream>>>(g->view(), first, count, cand);
  SF_CUDA(cub::DeviceScan::ExclusiveSum(scan_temp, scan_bytes, cand, cand_offsets, int(count + 1), stream));
  SF_CUDA(cudaMemcpyAsync(total, cand_offsets + count, 8, cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  return SF_OK;
}

// adds the number of neighbour pairs to *pair_counter (zeroed by the caller)
static int fpfh_search(sf_grid* g, double radius, int64_t first, int64_t count, const int64_t* cand_offsets,
                       int32_t* nbr, float* weights, int32_t* counts, unsigned long long* pair_counter,
                       cudaStream_t stream) {
  const size_t smem = size_t(kSearchWarps) * sizeof(SearchStage);
  static bool configured = false;
  if (!configured) {
    SF_CUDA(cudaFuncSetAttribute(search_weights_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    configured = true;
  }
  const int64_t tiles = (count + 31) / 32;
  search_weights_kernel<<<unsigned((tiles + kSearchWarps - 1) / kSearchWarps), kSearchWarps * 32, smem, stream>>>(
      g->view(), first, count, radius * radius, cand_offsets, nbr, weights, counts, pair_counter);
  SF_CUDA(cudaGetLastError());
  return SF_OK;
}

// synchronises the stream
static int read_pairs(const unsigned long long* pair_counter, int64_t* pairs_host, cudaStream_t stream) {
  unsigned long long pairs = 0;
  SF_CUDA(cudaMemcpyAsync(&pairs, pair_counter, 8, cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  *pairs_host = int64_t(pairs);
  return SF_OK;
}

// What compute_fpfh_descriptor (fpfh.py:16-117) does for one cloud — search around EVERY cloud point, SPFH of every
// point, FPFH of the keypoints — with the neighbour list as an internal, padded temporary.
extern "C" int sf_fpfh_cloud(sf_grid* g, double radius, int32_t n_bins, int32_t decorrelated, const double* edges_host,
                             const int64_t* keypoints, int64_t nq, void* out, int32_t out_is_f64, int64_t* pairs_host,
                             void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0 && g->has_normals, SF_ERR_ARG, "sf_fpfh_cloud: grid built without normals");
  SF_REQUIRE(edges_host && (nq == 0 || (keypoints && out)) && nq >= 0, SF_ERR_ARG, "sf_fpfh_cloud: bad arguments");
  SF_REQUIRE(radius_fits(g, radius), SF_ERR_ARG,
             "sf_fpfh_cloud: radius %g exceeds the cell edge %g the grid was built for", radius, g->cell);
  int width = 0, stride = 0, rows4 = 0;
  if (int rc = histogram_width("sf_fpfh_cloud", n_bins, decorrelated, &width)) return rc;
  fpfh_row_layout(width, &stride, &rows4);
  const int64_t n = g->n;
  if (pairs_host) *pairs_host = 0;
  Scratch scratch(stream);
  int64_t* cand_offsets = nullptr;
  int64_t total = 0;
  SF_CUDA(scratch.alloc(&cand_offsets, size_t(n + 1) * 8));
  if (int rc = fpfh_candidates(g, 0, n, cand_offsets, &total, scratch, stream)) return rc;
  int32_t *counts = nullptr, *nbr = nullptr;
  float *weights = nullptr, *spfh = nullptr;
  unsigned long long* pair_counter = nullptr;
  SF_CUDA(scratch.alloc(&counts, size_t(n) * 4));
  SF_CUDA(scratch.alloc(&pair_counter, 8));
  SF_CUDA(scratch.alloc(&spfh, size_t(n) * stride * sizeof(float)));
  SF_CUDA(scratch.alloc(&nbr, size_t(total > 0 ? total : 1) * 4));
  SF_CUDA(scratch.alloc(&weights, size_t(total > 0 ? total : 1) * 4));
  SF_CUDA(cudaMemsetAsync(pair_counter, 0, 8, stream));
  profile_mark(0, stream);
  if (int rc = fpfh_search(g, radius, 0, n, cand_offsets, nbr, weights, counts, pair_counter, stream)) return rc;
  profile_mark(1, stream);
  if (int rc = launch_spfh(g, 0, n, cand_offsets, counts, nbr, n_bins, decorrelated, edges_host, spfh, stride, stream))
    return rc;
  profile_mark(2, stream);
  if (int rc = sf_fpfh_block_rows(g, 0, n, cand_offsets, counts, nbr, weights, spfh, width, keypoints, nq, out, out_is_f64,
                                  stream))
    return rc;
  profile_mark(3, stream);
  return pairs_host != nullptr ? read_pairs(pair_counter, pairs_host, stream) : SF_OK;
}

extern "C" int sf_fpfh_row_stride(int32_t width, int32_t* stride_out) {
  SF_REQUIRE(width > 0 && stride_out != nullptr, SF_ERR_ARG, "sf_fpfh_row_stride: bad arguments");
  int stride = 0, rows4 = 0;
  fpfh_row_layout(width, &stride, &rows4);
  *stride_out = stride;
  return SF_OK;
}

extern "C" int sf_fpfh_block_begin(sf_grid* g, double radius, int64_t first, int64_t count, int64_t* cand_offsets,
                                   int64_t* total_host, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_fpfh_block_begin: grid not built");
  SF_REQUIRE(first >= 0 && count >= 0 && first + count <= g->n && cand_offsets && total_host, SF_ERR_ARG,
             "sf_fpfh_block_begin: bad arguments");
  SF_REQUIRE(radius_fits(g, radius), SF_ERR_ARG,
             "sf_fpfh_block_begin: radius %g exceeds the cell edge %g the grid was built for", radius, g->cell);
  *total_host = 0;
  if (count == 0) {
    SF_CUDA(cudaMemsetAsync(cand_offsets, 0, 8, stream));
    return SF_OK;
  }
  Scratch scratch(stream);
  return fpfh_candidates(g, first, count, cand_offsets, total_host, scratch, stream);
}

extern "C" int sf_fpfh_block_spfh(sf_grid* g, double radius, int32_t n_bins, int32_t decorrelated,
                                  const double* edges_host, int64_t first, int64_t count, const int64_t* cand_offsets,
                                  int32_t* nbr, float* weights, int32_t* counts, float* spfh_block, int64_t* pairs_host,
                                  void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0 && g->has_normals, SF_ERR_ARG, "sf_fpfh_block_spfh: grid built without normals");
  SF_REQUIRE(first >= 0 && count >= 0 && first + count <= g->n && edges_host, SF_ERR_ARG, "sf_fpfh_block_spfh: bad arguments");
  if (pairs_host) *pairs_host = 0;
  if (count == 0) return SF_OK;
  SF_REQUIRE(cand_offsets && nbr && weights && counts && spfh_block, SF_ERR_ARG, "sf_fpfh_block_spfh: null argument");
  int width = 0, stride = 0, rows4 = 0;
  if (int rc = histogram_width("sf_fpfh_block_spfh", n_bins, decorrelated, &width)) return rc;
  fpfh_row_layout(width, &stride, &rows4);
  Scratch scratch(stream);
  unsigned long long* pair_counter = nullptr;
  SF_CUDA(scratch.alloc(&pair_counter, 8));
  SF_CUDA(cudaMemsetAsync(pair_counter, 0, 8, stream));
  if (int rc = fpfh_search(g, radius, first, count, cand_offsets, nbr, weights, counts, pair_counter, stream)) return rc;
  if (int rc = launch_spfh(g, first, count, cand_offsets, counts, nbr, n_bins, decorrelated, edges_host, spfh_block,
                           stride, stream))
    return rc;
  return pairs_host != nullptr ? read_pairs(pair_counter, pairs_host, stream) : SF_OK;
}

extern "C" int sf_fpfh_block_rows(sf_grid* g, int64_t first, int64_t count, const int64_t* cand_offsets,
                                  const int32_t* counts, const int32_t* nbr, const float* weights, const float* spfh_all,
                                  int32_t width, const int64_t* keypoints, int64_t nq, void* out, int32_t out_is_f64,
                                  void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(g != nullptr && g->n > 0, SF_ERR_ARG, "sf_fpfh_block_rows: grid not built");
  SF_REQUIRE(first >= 0 && count >= 0 && first + count <= g->n && width > 0 && nq >= 0, SF_ERR_ARG,
             "sf_fpfh_block_rows: bad arguments");
  if (nq == 0) return SF_OK;
  SF_REQUIRE(cand_offsets && counts && nbr && weights && spfh_all && keypoints && out, SF_ERR_ARG,
             "sf_fpfh_block_rows: null argument");
  int stride = 0, rows4 = 0;
  fpfh_row_layout(width, &stride, &rows4);
  return out_is_f64 ? launch_fpfh(g, cand_offsets, counts, nbr, nullptr, weights, 0, spfh_all, width, stride, rows4, keypoints,
                                  nq, first, static_cast<double*>(out), stream)
                    : launch_fpfh(g, cand_offsets, counts, nbr, nullptr, weights, 0, spfh_all, width, stride, rows4, keypoints,
                                  nq, first, static_cast<float*>(out), stream);
}
