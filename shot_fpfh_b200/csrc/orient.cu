// Kernel group O: consistent normal orientation (Hoppe et al. 1992), no counterpart in the reference; the specification
// is the restatement in oracle/orientation_oracle.py. The signs are propagated along the minimum spanning forest of the
// k-NN graph under the unique key (w = 1 - |n_i . n_j|, min(i, j), max(i, j)), found by Borůvka rounds with parity
// labels: every step is data-parallel, no tree is rooted or walked.
//   orient_edges_kernel   one thread per list entry: the undirected edge {i, j} once, with its key and flip bit
//   per round, over the live edges and the components' representatives:
//     min_weight_kernel   atomicMin of the weight's ordered bits into both endpoints' components
//     min_key_kernel      atomicMin of the packed (lo, hi, flip) among the edges that reached that weight
//     hook_kernel         component C hooks onto D along its chosen edge (mutual choice: the higher id hooks), with
//                         hpar = C's parity relative to D
//     jump_kernel         pointer jumping (double-buffered), until every hook points at a root
//     relabel_kernel      par ^= hpar[comp], comp = hook[comp]
//   then CUB DeviceSelect keeps the roots and the edges between two components.
//   tree_members_kernel   lowest member of each tree (and the `towards` votes); orient_final_kernel negates.
#include <cub/cub.cuh>

#include <climits>
#include <cmath>

#include "sf_common.cuh"

namespace sf {

// One undirected edge: `w` = the weight's bits mapped so that unsigned order is the order of the values;
// `key` = lo << 33 | hi << 1 | flip (indices < 2^31), whose unsigned order is the order of (lo, hi).
struct OrientEdge {
  unsigned long long w;
  unsigned long long key;
};

constexpr unsigned long long kNoKey = ~0ull;

// (a.x*b.x + a.y*b.y) + a.z*b.z, every product and sum rounded: NumPy's value, bit for bit.
__device__ __forceinline__ double dot3_rn(double ax, double ay, double az, double bx, double by, double bz) {
  return __dadd_rn(__dadd_rn(__dmul_rn(ax, bx), __dmul_rn(ay, by)), __dmul_rn(az, bz));
}

// float64 -> uint64 with the same order (negative weights come from normals longer than 1).
__device__ __forceinline__ unsigned long long ordered_bits(double v) {
  const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ void edge_ends(unsigned long long key, int32_t& lo, int32_t& hi, int& flip) {
  lo = int32_t(key >> 33);
  hi = int32_t((key >> 1) & 0xffffffffull);
  flip = int(key & 1ull);
}

// Entry s of point i's list names j. The edge {i, j} is kept from the list of min(i, j) when it appears there, else
// from the other one: each undirected edge once. Entries j == i are not edges; an entry outside [0, n) raises *bad.
__global__ void __launch_bounds__(256)
    orient_edges_kernel(const double* __restrict__ normals, const int32_t* __restrict__ nbr, int64_t n, int K,
                        OrientEdge* __restrict__ edges, uint8_t* __restrict__ keep, int32_t* __restrict__ bad) {
  const int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (e >= n * K) return;
  const int64_t i = e / K;
  const int32_t j = __ldg(nbr + e);
  bool ok = false;
  if (j < 0 || j >= n) {
    *bad = 1;
  } else if (j != i) {
    ok = true;
    if (j < i)
      for (int t = 0; t < K; ++t)
        if (__ldg(nbr + int64_t(j) * K + t) == i) ok = false;
  }
  keep[e] = ok;
  if (!ok) return;
  const double* a = normals + 3 * i;
  const double* b = normals + 3 * int64_t(j);
  const double d = dot3_rn(__ldg(a), __ldg(a + 1), __ldg(a + 2), __ldg(b), __ldg(b + 1), __ldg(b + 2));
  const unsigned long long lo = i < j ? i : j, hi = i < j ? j : i;
  edges[e] = OrientEdge{ordered_bits(__dsub_rn(1.0, fabs(d))), (lo << 33) | (hi << 1) | (d < 0.0 ? 1ull : 0ull)};
}

__global__ void reset_best_kernel(const int32_t* __restrict__ reps, int64_t nr, unsigned long long* __restrict__ best_w,
                                  unsigned long long* __restrict__ best_key) {
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (r >= nr) return;
  const int32_t c = reps[r];
  best_w[c] = kNoKey;
  best_key[c] = kNoKey;
}

// Every live edge joins two components; it is offered to both. The plain read skips most atomics once a component's
// minimum has settled (a stale read only costs an atomic).
__global__ void __launch_bounds__(256)
    min_weight_kernel(const OrientEdge* __restrict__ edges, int64_t m, const int32_t* __restrict__ comp,
                      unsigned long long* best_w) {
  const int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (e >= m) return;
  const OrientEdge ed = edges[e];
  int32_t lo, hi;
  int flip;
  edge_ends(ed.key, lo, hi, flip);
  const int32_t cu = __ldg(comp + lo), cv = __ldg(comp + hi);
  if (ed.w < best_w[cu]) atomicMin(best_w + cu, ed.w);
  if (ed.w < best_w[cv]) atomicMin(best_w + cv, ed.w);
}

__global__ void __launch_bounds__(256)
    min_key_kernel(const OrientEdge* __restrict__ edges, int64_t m, const int32_t* __restrict__ comp,
                   const unsigned long long* __restrict__ best_w, unsigned long long* best_key) {
  const int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (e >= m) return;
  const OrientEdge ed = edges[e];
  int32_t lo, hi;
  int flip;
  edge_ends(ed.key, lo, hi, flip);
  const int32_t cu = __ldg(comp + lo), cv = __ldg(comp + hi);
  if (ed.w == best_w[cu]) atomicMin(best_key + cu, ed.key);
  if (ed.w == best_w[cv]) atomicMin(best_key + cv, ed.key);
}

// Component C with chosen edge (u in C, v in D): hook[C] = D and hpar[C] = par[u] ^ flip ^ par[v] (C's sign relative
// to D's). When D chose the same key (the same undirected edge: compared by key, not by slot) only the higher id hooks.
__global__ void hook_kernel(const int32_t* __restrict__ reps, int64_t nr, const int32_t* __restrict__ comp,
                            const uint8_t* __restrict__ par, const unsigned long long* __restrict__ best_w,
                            const unsigned long long* __restrict__ best_key, int32_t* __restrict__ hook,
                            uint8_t* __restrict__ hpar) {
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (r >= nr) return;
  const int32_t c = reps[r];
  const unsigned long long key = best_key[c];
  int32_t to = c;
  uint8_t p = 0;
  if (key != kNoKey) {
    int32_t lo, hi;
    int flip;
    edge_ends(key, lo, hi, flip);
    const bool lo_in_c = comp[lo] == c;
    const int32_t u = lo_in_c ? lo : hi, v = lo_in_c ? hi : lo;
    const int32_t d = comp[v];
    if (!(best_key[d] == key && best_w[d] == best_w[c] && c < d)) {
      to = d;
      p = uint8_t(par[u] ^ flip ^ par[v]);
    }
  }
  hook[c] = to;
  hpar[c] = p;
}

__global__ void jump_kernel(const int32_t* __restrict__ reps, int64_t nr, const int32_t* __restrict__ hook_in,
                            const uint8_t* __restrict__ hpar_in, int32_t* __restrict__ hook_out,
                            uint8_t* __restrict__ hpar_out, int32_t* __restrict__ changed) {
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (r >= nr) return;
  const int32_t c = reps[r];
  const int32_t h = hook_in[c], hh = hook_in[h];
  hook_out[c] = hh;
  hpar_out[c] = uint8_t(hpar_in[c] ^ hpar_in[h]);
  if (hh != h) *changed = 1;
}

__global__ void __launch_bounds__(256)
    relabel_kernel(int64_t n, const int32_t* __restrict__ hook, const uint8_t* __restrict__ hpar,
                   int32_t* __restrict__ comp, uint8_t* __restrict__ par) {
  const int64_t x = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (x >= n) return;
  const int32_t c = comp[x];
  par[x] ^= hpar[c];
  comp[x] = hook[c];
}

struct IsRoot {
  const int32_t* hook;
  __device__ __forceinline__ bool operator()(int32_t c) const { return hook[c] == c; }
};

struct CrossesComponents {
  const int32_t* comp;
  __device__ __forceinline__ bool operator()(const OrientEdge& e) const {
    int32_t lo, hi;
    int flip;
    edge_ends(e.key, lo, hi, flip);
    return comp[lo] != comp[hi];
  }
};

__global__ void reset_tree_kernel(const int32_t* __restrict__ reps, int64_t nr, int32_t* __restrict__ low,
                                  int32_t* __restrict__ votes) {
  const int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (r >= nr) return;
  const int32_t c = reps[r];
  low[c] = INT_MAX;
  votes[2 * int64_t(c)] = 0;
  votes[2 * int64_t(c) + 1] = 0;
}

// Lowest member of each tree; with `towards` also the votes n . (t - p) > 0 / < 0 under the parity relative to the
// representative (a negation flips the sign of the dot exactly). Lanes of one tree add their votes once per warp.
__global__ void __launch_bounds__(256)
    tree_members_kernel(int64_t n, const int32_t* __restrict__ comp, const uint8_t* __restrict__ par,
                        const double* __restrict__ xyz, const double* __restrict__ normals, int has_towards, double tx,
                        double ty, double tz, int32_t* low, int32_t* votes) {
  const int64_t x = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const bool in = x < n;
  const int32_t c = in ? comp[x] : -1;
  if (in && int32_t(x) < low[c]) atomicMin(low + c, int32_t(x));
  if (!has_towards) return;
  int vote = 0;
  if (in) {
    const double* p = xyz + 3 * x;
    const double* nx = normals + 3 * x;
    const double s = dot3_rn(__ldg(nx), __ldg(nx + 1), __ldg(nx + 2), __dsub_rn(tx, __ldg(p)),
                             __dsub_rn(ty, __ldg(p + 1)), __dsub_rn(tz, __ldg(p + 2)));
    vote = s > 0.0 ? 1 : (s < 0.0 ? -1 : 0);
    if (par[x]) vote = -vote;
  }
  const unsigned active = __activemask();
  const unsigned same = __match_any_sync(active, c);
  const int plus = __popc(__ballot_sync(active, vote > 0) & same), minus = __popc(__ballot_sync(active, vote < 0) & same);
  const int lane = threadIdx.x & 31;
  if (in && lane == __ffs(same) - 1) {
    if (plus) atomicAdd(votes + 2 * int64_t(c), plus);
    if (minus) atomicAdd(votes + 2 * int64_t(c) + 1, minus);
  }
}

__global__ void __launch_bounds__(256)
    orient_final_kernel(int64_t n, const int32_t* __restrict__ comp, const uint8_t* __restrict__ par,
                        const int32_t* __restrict__ low, const int32_t* __restrict__ votes, int has_towards,
                        const double* __restrict__ normals, double* __restrict__ out) {
  const int64_t x = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (x >= n) return;
  const int32_t c = comp[x];
  int b = par[low[c]];  // the lowest member keeps its input sign
  if (has_towards) {
    const int plus = votes[2 * int64_t(c)], minus = votes[2 * int64_t(c) + 1];
    if (plus != minus) b = minus > plus;
  }
  const bool neg = (par[x] ^ b) != 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double v = __ldg(normals + 3 * x + a);
    out[3 * x + a] = neg ? -v : v;
  }
}

__global__ void __launch_bounds__(256)
    init_kernel(int64_t n, int32_t* __restrict__ comp, uint8_t* __restrict__ par, int32_t* __restrict__ reps) {
  const int64_t x = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (x >= n) return;
  comp[x] = int32_t(x);
  par[x] = 0;
  reps[x] = int32_t(x);
}

inline unsigned blocks_for(int64_t threads, int per_block) { return unsigned((threads + per_block - 1) / per_block); }

}  // namespace sf

using namespace sf;

extern "C" int sf_orient_normals(const double* xyz, const double* normals, int64_t n, const int32_t* nbr_index,
                                 int32_t k_stride, const double* towards, double* out, int64_t* n_trees,
                                 void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  SF_REQUIRE(n_trees != nullptr, SF_ERR_ARG, "sf_orient_normals: null tree count");
  *n_trees = 0;
  SF_REQUIRE(n >= 0 && n <= INT_MAX, SF_ERR_ARG, "sf_orient_normals: n = %lld not in [0, 2^31)", (long long)n);
  if (n == 0) return SF_OK;
  SF_REQUIRE(xyz && normals && nbr_index && out && k_stride >= 1, SF_ERR_ARG, "sf_orient_normals: bad arguments");
  SF_REQUIRE(towards == nullptr || (std::isfinite(towards[0]) && std::isfinite(towards[1]) && std::isfinite(towards[2])),
             SF_ERR_ARG, "sf_orient_normals: non-finite viewpoint");
  const int64_t slots = n * k_stride;

  // CUB temporary storage, sized for the largest of the three selections
  size_t b_flag = 0, b_edges = 0, b_reps = 0;
  SF_CUDA(cub::DeviceSelect::Flagged(nullptr, b_flag, static_cast<OrientEdge*>(nullptr), static_cast<uint8_t*>(nullptr),
                                     static_cast<OrientEdge*>(nullptr), static_cast<int64_t*>(nullptr), slots, stream));
  SF_CUDA(cub::DeviceSelect::If(nullptr, b_edges, static_cast<OrientEdge*>(nullptr), static_cast<OrientEdge*>(nullptr),
                                static_cast<int64_t*>(nullptr), slots, CrossesComponents{nullptr}, stream));
  SF_CUDA(cub::DeviceSelect::If(nullptr, b_reps, static_cast<int32_t*>(nullptr), static_cast<int32_t*>(nullptr),
                                static_cast<int64_t*>(nullptr), n, IsRoot{nullptr}, stream));
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t temp_bytes = up(std::max(b_flag, std::max(b_edges, b_reps)));

  // scratch: two edge buffers (ping-pong), the entry flags, and per point: comp, par, best weight / key, two hook and
  // two hpar buffers (pointer jumping reads one, writes the other), two representative lists, low, votes; counters
  Scratch scratch(stream);
  OrientEdge *edges_a = nullptr, *edges_b = nullptr;
  SF_CUDA(scratch.alloc(&edges_a, size_t(slots) * sizeof(OrientEdge)));
  SF_CUDA(scratch.alloc(&edges_b, size_t(slots) * sizeof(OrientEdge)));
  const size_t n4 = up(size_t(n) * 4), n8 = up(size_t(n) * 8), n1 = up(size_t(n));
  const size_t point_bytes = up(size_t(slots)) + 2 * n8 + 6 * n4 + 3 * n1 + n8 + 256 + temp_bytes;
  char* base = nullptr;
  SF_CUDA(scratch.alloc(&base, point_bytes));
  char* at = base;
  auto take = [&at](size_t bytes) {
    char* p = at;
    at += bytes;
    return p;
  };
  uint8_t* keep = reinterpret_cast<uint8_t*>(take(up(size_t(slots))));
  unsigned long long* best_w = reinterpret_cast<unsigned long long*>(take(n8));
  unsigned long long* best_key = reinterpret_cast<unsigned long long*>(take(n8));
  int32_t* comp = reinterpret_cast<int32_t*>(take(n4));
  int32_t* hook[2] = {reinterpret_cast<int32_t*>(take(n4)), reinterpret_cast<int32_t*>(take(n4))};
  int32_t* reps[2] = {reinterpret_cast<int32_t*>(take(n4)), reinterpret_cast<int32_t*>(take(n4))};
  int32_t* low = reinterpret_cast<int32_t*>(take(n4));
  uint8_t* par = reinterpret_cast<uint8_t*>(take(n1));
  uint8_t* hpar[2] = {reinterpret_cast<uint8_t*>(take(n1)), reinterpret_cast<uint8_t*>(take(n1))};
  int32_t* votes = reinterpret_cast<int32_t*>(take(n8));
  int64_t* counts = reinterpret_cast<int64_t*>(take(256));  // [0] edges, [1] representatives, [2] flag words
  int32_t* flags = reinterpret_cast<int32_t*>(counts + 2);   // [0] bad entry, [1] pointer jumping changed something
  void* temp = take(temp_bytes);

  const unsigned pb = blocks_for(n, 256);
  init_kernel<<<pb, 256, 0, stream>>>(n, comp, par, reps[0]);
  SF_CUDA(cudaGetLastError());
  SF_CUDA(cudaMemsetAsync(counts, 0, 256, stream));
  orient_edges_kernel<<<blocks_for(slots, 256), 256, 0, stream>>>(normals, nbr_index, n, k_stride, edges_a, keep,
                                                                   flags);
  SF_CUDA(cudaGetLastError());
  size_t bytes = temp_bytes;
  SF_CUDA(cub::DeviceSelect::Flagged(temp, bytes, edges_a, keep, edges_b, counts, slots, stream));
  int64_t host[3] = {0, 0, 0};  // live edges, representatives, the two flag words
  SF_CUDA(cudaMemcpyAsync(host, counts, sizeof(host), cudaMemcpyDeviceToHost, stream));
  SF_CUDA(cudaStreamSynchronize(stream));
  SF_REQUIRE(reinterpret_cast<int32_t*>(host + 2)[0] == 0, SF_ERR_ARG,
             "sf_orient_normals: a neighbour index lies outside [0, %lld)", (long long)n);
  int64_t m = host[0], nr = n;
  OrientEdge* live = edges_b;
  OrientEdge* spare = edges_a;
  int r = 0;  // which of reps[] holds the current representatives
  while (m > 0) {
    reset_best_kernel<<<blocks_for(nr, 256), 256, 0, stream>>>(reps[r], nr, best_w, best_key);
    min_weight_kernel<<<blocks_for(m, 256), 256, 0, stream>>>(live, m, comp, best_w);
    min_key_kernel<<<blocks_for(m, 256), 256, 0, stream>>>(live, m, comp, best_w, best_key);
    hook_kernel<<<blocks_for(nr, 256), 256, 0, stream>>>(reps[r], nr, comp, par, best_w, best_key, hook[0], hpar[0]);
    SF_CUDA(cudaGetLastError());
    int h = 0;  // which of hook[] / hpar[] holds the current pointers
    for (;;) {
      SF_CUDA(cudaMemsetAsync(flags + 1, 0, sizeof(int32_t), stream));
      jump_kernel<<<blocks_for(nr, 256), 256, 0, stream>>>(reps[r], nr, hook[h], hpar[h], hook[h ^ 1], hpar[h ^ 1],
                                                           flags + 1);
      SF_CUDA(cudaGetLastError());
      h ^= 1;
      int32_t changed = 0;
      SF_CUDA(cudaMemcpyAsync(&changed, flags + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
      SF_CUDA(cudaStreamSynchronize(stream));
      if (!changed) break;
    }
    relabel_kernel<<<pb, 256, 0, stream>>>(n, hook[h], hpar[h], comp, par);
    SF_CUDA(cudaGetLastError());
    bytes = temp_bytes;
    SF_CUDA(cub::DeviceSelect::If(temp, bytes, reps[r], reps[r ^ 1], counts + 1, nr, IsRoot{hook[h]}, stream));
    r ^= 1;
    bytes = temp_bytes;
    SF_CUDA(cub::DeviceSelect::If(temp, bytes, live, spare, counts, m, CrossesComponents{comp}, stream));
    std::swap(live, spare);
    SF_CUDA(cudaMemcpyAsync(host, counts, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    SF_CUDA(cudaStreamSynchronize(stream));
    m = host[0];
    nr = host[1];
  }

  reset_tree_kernel<<<blocks_for(nr, 256), 256, 0, stream>>>(reps[r], nr, low, votes);
  const double t[3] = {towards ? towards[0] : 0.0, towards ? towards[1] : 0.0, towards ? towards[2] : 0.0};
  tree_members_kernel<<<pb, 256, 0, stream>>>(n, comp, par, xyz, normals, towards != nullptr, t[0], t[1], t[2], low,
                                               votes);
  orient_final_kernel<<<pb, 256, 0, stream>>>(n, comp, par, low, votes, towards != nullptr, normals, out);
  SF_CUDA(cudaGetLastError());
  *n_trees = nr;
  return SF_OK;
}
