// Shared declarations of the sm_100a library behind include/shotfpfh_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <cmath>

#include "../../include/shotfpfh_b200.h"
#include "sf_math.cuh"

namespace sf {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// Last error text, readable through sf_last_error(). No exceptions cross the C ABI.
void set_error(const char* fmt, ...);
// Measurement hook (shot.cu): records event `i` (0..3) on `stream` when sf_profile_enable(1) is in effect.
void profile_mark(int i, cudaStream_t stream);

#define SF_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t err__ = (call);                                                                    \
    if (err__ != cudaSuccess) {                                                                    \
      sf::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(err__));      \
      return SF_ERR_CUDA;                                                                          \
    }                                                                                              \
  } while (0)

#define SF_REQUIRE(cond, code, ...)      \
  do {                                   \
    if (!(cond)) {                       \
      sf::set_error(__VA_ARGS__);        \
      return code;                       \
    }                                    \
  } while (0)

// Stream-ordered scratch memory of one call: every buffer alloc() hands out is freed on the stream when the Scratch
// goes out of scope, whichever way the call returns. The status of the free is ignored: an error that matters surfaces
// at the call's synchronisation or at the next call.
class Scratch {
 public:
  explicit Scratch(cudaStream_t stream) : stream_(stream) {}
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  ~Scratch() {
    for (int i = 0; i < count_; ++i) cudaFreeAsync(ptrs_[i], stream_);
  }

  template <typename T>
  cudaError_t alloc(T** p, size_t bytes) {
    if (count_ == kMaxBuffers) return cudaErrorMemoryAllocation;  // more buffers than one call is written for
    keep_freed_memory();
    const cudaError_t err = cudaMallocAsync(p, bytes, stream_);
    if (err == cudaSuccess) ptrs_[count_++] = *p;
    return err;
  }

 private:
  // The default memory pool returns freed memory to the OS at every synchronisation (release threshold 0), which made
  // each call re-pay a cudaMalloc (measured: 21 ms per matching step for 0.4 ms of kernels); the threshold is raised
  // once so that the pool keeps what it has been given.
  static void keep_freed_memory() {
    static bool configured = false;
    if (configured) return;
    configured = true;
    int device = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&device) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      uint64_t keep = ~uint64_t(0);
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }

  static constexpr int kMaxBuffers = 16;
  cudaStream_t stream_;
  void* ptrs_[kMaxBuffers];
  int count_ = 0;
};

// Device-side view of a built grid (passed by value to kernels).
struct GridView {
  const double4* pts;       // cell-sorted coordinates; .w carries the original index (bit pattern of an int64)
  const double4* nrm;       // cell-sorted normals (may be null)
  const int32_t* cell_start;  // [ncells + 1], exclusive prefix of the per-cell counts
  const float4* xyzc;       // cell-sorted float32 side copy: coordinates relative to the point's cell corner, .w = the
                            // cell coordinates modulo 4 (sf_math.cuh::shot_cellbits) — 16 B per candidate test
  const float4* nrm32;      // cell-sorted float32 normals (may be null)
  int64_t n;
  double origin[3];
  double inv_cell;
  double cell;
  int dims[3];
};

}  // namespace sf

// The opaque handle of the C ABI.
struct sf_grid {
  int64_t n = 0;
  int64_t capacity = 0;
  double cell = 0.0;
  double origin[3] = {0, 0, 0};
  int dims[3] = {0, 0, 0};
  int64_t ncells = 0;
  int64_t cells_capacity = 0;
  bool has_normals = false;
  int device = 0;
  double4* pts = nullptr;
  double4* nrm = nullptr;
  float4* xyzc = nullptr;
  float4* nrm32 = nullptr;
  int32_t* perm = nullptr;      // sorted position -> original index
  int32_t* inv_perm = nullptr;  // original index -> sorted position
  int32_t* cell_start = nullptr;
  int32_t* cell_count = nullptr;
  uint32_t* keys_in = nullptr;
  uint32_t* keys_out = nullptr;
  int32_t* vals_in = nullptr;
  double* bbox = nullptr;  // 6 doubles, device
  void* cub_temp = nullptr;
  size_t cub_bytes = 0;
  // ---- calls without host synchronisation (sf_grid_set_speculative, include/shotfpfh_b200.h) ----
  // A repeated call on the same handle reuses what the previous one learned on the host (the grid's box, the size of
  // the neighbour list) instead of reading it back; the kernels check the assumption on the device and, when it
  // fails, raise status_dev and do nothing. The caller reads the verdict with sf_grid_poll after synchronising.
  int speculative = 0;         // bit 0: builds, bit 1: the fused SHOT driver's list
  bool sized = false;          // origin / dims / cell below come from a synchronising build of ...
  int64_t sized_n = 0;         // ... this many points
  double sized_radius = 0.0;   // ... for this radius
  int32_t* status_dev = nullptr;   // 0 = fine; 1 = a point outside the assumed box; 2 = neighbour list too small
  // scratch of sf_shot_single_scale, kept between calls
  int64_t shot_q_capacity = 0;
  int64_t* shot_cand_offsets = nullptr;
  int32_t* shot_counts = nullptr;
  int shot_call_parity = 0;          // which of the two sets of shot_pairs counters the next call uses
  int4* shot_runs = nullptr;         // 5 x int4 per query: start[9], pref[1..9] of its culled runs (candidate_count_kernel)
  double* shot_lrf = nullptr;
  float* shot_frame32 = nullptr;
  int32_t* shot_worklist = nullptr;
  unsigned long long* shot_pairs = nullptr;
  float4* shot_nbr = nullptr;
  int64_t shot_nbr_capacity = 0;     // entries
  double shot_entries_per_query = 0; // from the last call that read the total back
  sf::GridView view() const {
    sf::GridView v;
    v.pts = pts;
    v.nrm = has_normals ? nrm : nullptr;
    v.cell_start = cell_start;
    v.xyzc = xyzc;
    v.nrm32 = has_normals ? nrm32 : nullptr;
    v.n = n;
    for (int i = 0; i < 3; ++i) {
      v.origin[i] = origin[i];
      v.dims[i] = dims[i];
    }
    v.inv_cell = 1.0 / cell;
    v.cell = cell;
    return v;
  }
};

namespace sf {

// A fixed-radius search on the grid looks at the 27 cells around a query: the radius must not exceed the cell edge
// (with margin for the rounding of the cell coordinates).
inline bool radius_fits(const sf_grid* g, double radius) {
  return radius > 0.0 && std::isfinite(radius) && radius * 1.0005 <= g->cell;
}

// ---- warp helpers -----------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
  return v;
}
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// 16-byte-pair load of one cell-sorted record through the read-only path.
__device__ __forceinline__ double4 load_pt(const double4* p) {
  const double2* q = reinterpret_cast<const double2*>(p);
  const double2 a = __ldg(q), b = __ldg(q + 1);
  return make_double4(a.x, a.y, b.x, b.y);
}

// ---- the candidate set of one query: 9 contiguous runs of the cell-sorted array ----------------------------
// Cells are keyed (z * ny + y) * nx + x, so the three x-adjacent cells of a row are one contiguous run.
// Each warp builds the runs once (lane j < 9 owns run j) and then walks the concatenation of the runs with all
// 32 lanes busy: lane l visits virtual positions l, l + 32, ... and maps each to (run, offset).
struct Runs {
  int start[9];
  int pref[10];  // pref[j] = number of candidates before run j; pref[9] = total
};

__device__ __forceinline__ int cell_coord(double q, double origin, double inv_cell, int dim) {
  double c = floor((q - origin) * inv_cell);
  c = fmax(-2.0, fmin(c, double(dim) + 1.0));
  return int(c);
}

// Lane j < 9 owns run j of the cell (cx, cy, cz) — coordinates may lie outside the grid (queries off the cloud):
// its start in the cell-sorted array and its length (0 for the other lanes and for rows outside the grid).
__device__ __forceinline__ void run_of_lane(const GridView& g, int cx, int cy, int cz, int lane, int& s, int& len) {
  s = 0;
  len = 0;
  if (lane < 9) {
    const int yy = cy + (lane % 3) - 1, zz = cz + (lane / 3) - 1;
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dims[0] - 1);
    if (yy >= 0 && yy < g.dims[1] && zz >= 0 && zz < g.dims[2] && x0 <= x1) {
      const int64_t base = (int64_t(zz) * g.dims[1] + yy) * g.dims[0];
      s = __ldg(g.cell_start + base + x0);
      len = __ldg(g.cell_start + base + x1 + 1) - s;
    }
  }
}

// The table of runs from the (start, length) lanes 0..8 hold.
__device__ __forceinline__ Runs runs_from_lanes(int s, int len, int lane) {
  int incl = len;
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) {
    const int t = __shfl_up_sync(kFull, incl, o);
    if (lane >= o) incl += t;
  }
  Runs r;
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    r.start[j] = __shfl_sync(kFull, s, j);
    r.pref[j + 1] = __shfl_sync(kFull, incl, j);
  }
  r.pref[0] = 0;
  return r;
}

// The runs around cell (cx, cy, cz).
__device__ __forceinline__ Runs build_runs_cell(const GridView& g, int cx, int cy, int cz, int lane) {
  int s, len;
  run_of_lane(g, cx, cy, cz, lane, s, len);
  return runs_from_lanes(s, len, lane);
}

__device__ __forceinline__ Runs build_runs(const GridView& g, double qx, double qy, double qz, int lane) {
  return build_runs_cell(g, cell_coord(qx, g.origin[0], g.inv_cell, g.dims[0]),
                         cell_coord(qy, g.origin[1], g.inv_cell, g.dims[1]),
                         cell_coord(qz, g.origin[2], g.inv_cell, g.dims[2]), lane);
}

// ---- culled candidate set of a fixed-radius query ---------------------------------------------------------------
// A neighbouring cell whose nearest face lies farther than the radius from the query cannot hold a neighbour: with a
// cell edge just above the radius that removes about half of the 8 corner cells and a fifth of the 12 edge cells (a
// quarter of the candidates the exact test then rejects one by one). The gaps are LOWER bounds of the distance from the
// query to the faces of its own cell (shrunk by more than the rounding of cell_coord on either side of a face), so a
// cell is dropped only when every point that key_kernel can have put in it is out of reach.
struct CellGaps {
  int c[3];
  double lo[3], hi[3];
};

__device__ __forceinline__ CellGaps cell_gaps(const GridView& g, double qx, double qy, double qz) {
  const double q[3] = {qx, qy, qz};
  CellGaps r;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    r.c[a] = cell_coord(q[a], g.origin[a], g.inv_cell, g.dims[a]);
    const double face = g.origin[a] + double(r.c[a]) * g.cell;
    const double slack = 1e-9 * g.cell + 1e-14 * (fabs(q[a]) + fabs(g.origin[a]) + double(g.dims[a]) * g.cell);
    r.lo[a] = fmax(0.0, (q[a] - face) - slack);
    r.hi[a] = fmax(0.0, ((face + g.cell) - q[a]) - slack);
  }
  return r;
}

// Run j (0..8: row cy + j % 3 - 1, slab cz + j / 3 - 1) of the query's neighbourhood without the cells out of reach.
__device__ __forceinline__ void culled_run(const GridView& g, const CellGaps& cg, int j, double r2, int& s, int& len) {
  s = 0;
  len = 0;
  const int dy = j % 3 - 1, dz = j / 3 - 1;
  const int yy = cg.c[1] + dy, zz = cg.c[2] + dz;
  const double gy = dy < 0 ? cg.lo[1] : (dy > 0 ? cg.hi[1] : 0.0);
  const double gz = dz < 0 ? cg.lo[2] : (dz > 0 ? cg.hi[2] : 0.0);
  const double reach = r2 * (1.0 + 1e-9);
  const double yz2 = gy * gy + gz * gz;
  if (yz2 > reach) return;
  int x0 = cg.c[0] - 1, x1 = cg.c[0] + 1;
  if (yz2 + cg.lo[0] * cg.lo[0] > reach) x0 = cg.c[0];
  if (yz2 + cg.hi[0] * cg.hi[0] > reach) x1 = cg.c[0];
  x0 = max(x0, 0);
  x1 = min(x1, g.dims[0] - 1);
  if (yy >= 0 && yy < g.dims[1] && zz >= 0 && zz < g.dims[2] && x0 <= x1) {
    const int64_t base = (int64_t(zz) * g.dims[1] + yy) * g.dims[0];
    s = __ldg(g.cell_start + base + x0);
    len = __ldg(g.cell_start + base + x1 + 1) - s;
  }
}

// The runs of a query that looks for neighbours within sqrt(r2) (r2 must not exceed the square of the cell edge).
__device__ __forceinline__ Runs build_runs(const GridView& g, double qx, double qy, double qz, int lane, double r2) {
  const CellGaps cg = cell_gaps(g, qx, qy, qz);
  int s = 0, len = 0;
  if (lane < 9) culled_run(g, cg, lane, r2, s, len);
  return runs_from_lanes(s, len, lane);
}

// Position in the cell-sorted array of virtual candidate v (0 <= v < pref[9]).
__device__ __forceinline__ int run_position(const Runs& r, int v) {
  int pos = r.start[0] + v;
#pragma unroll
  for (int j = 1; j < 9; ++j)
    if (v >= r.pref[j]) pos = r.start[j] + (v - r.pref[j]);
  return pos;
}

}  // namespace sf
