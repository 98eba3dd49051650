// TEST INFRASTRUCTURE ONLY. g++ host instantiation of shot_fpfh_b200/csrc/sf_math.cuh, the header the sm_100a
// kernels inline, so that the per-neighbour arithmetic (bin decisions, interpolation weights, winner tables, 3x3
// eigen-solver, FPFH features and NumPy-compatible binning) is checked against the oracle on machines without
// a GPU (tests/test_host_math.py). The loops below mirror the kernels' control flow sequentially; the product
// never loads this library.
#include <cstring>
#include <vector>

#include "../../shot_fpfh_b200/csrc/sf_math.cuh"

using namespace sf;

extern "C" {

double hm_rdist3(double dx, double dy, double dz) { return rdist3(dx, dy, dz); }

void hm_eigh3(const double* m, double* eval, double* evec9) {
  double e[3], v[3][3];
  eigh3(m, e, v);
  for (int c = 0; c < 3; ++c) {
    eval[c] = e[c];
    for (int k = 0; k < 3; ++k) evec9[3 * c + k] = v[c][k];
  }
}

// The statically-indexed dsteqr3 (what the kernels run) against the loop-for-loop transcription of LAPACK's dsteqr, on n
// tridiagonal problems (d3, e2 per problem): the number of problems on which any of the 14 outputs differs in any BIT.
long hm_dsteqr3_static_vs_generic(const double* d3, const double* e2, long n) {
  long differ = 0;
  for (long i = 0; i < n; ++i) {
    double da[3] = {d3[3 * i], d3[3 * i + 1], d3[3 * i + 2]}, ea[2] = {e2[2 * i], e2[2 * i + 1]}, za[3][3];
    double db[3] = {da[0], da[1], da[2]}, eb[2] = {ea[0], ea[1]}, zb[3][3];
    lapack3::dsteqr3(da, ea, za);
    lapack3::dsteqr3_generic(db, eb, zb);
    differ += memcmp(da, db, sizeof(da)) != 0 || memcmp(ea, eb, sizeof(ea)) != 0 || memcmp(za, zb, sizeof(za)) != 0;
  }
  return differ;
}

int hm_azimuth_octant(double x, double y) { return azimuth_octant(x, y); }

double hm_acos_half_pi_max() { return kAcosHalfPiMax; }

// local = rel @ lrf for k offsets (rel: k x 3, lrf9 row-major, columns [x y z]) as the float64 kernels round it
void hm_frame_local(const double* rel, long k, const double* f, double* local) {
  for (long i = 0; i < k; ++i)
    for (int j = 0; j < 3; ++j) local[3 * i + j] = frame_dot(rel[3 * i], rel[3 * i + 1], rel[3 * i + 2], f[j], f[3 + j], f[6 + j]);
}

// Mirrors shot_lrf_kernel: lrf9 row-major, columns [x y z].
void hm_lrf(const double* point, const double* nbrs, int k, double radius, double* lrf9) {
  if (k == 0) {
    for (int i = 0; i < 9; ++i) lrf9[i] = (i % 4 == 0) ? 1.0 : 0.0;
    return;
  }
  double sw = 0, m[6] = {0, 0, 0, 0, 0, 0};
  for (int i = 0; i < k; ++i) {
    const double cx = nbrs[3 * i] - point[0], cy = nbrs[3 * i + 1] - point[1], cz = nbrs[3 * i + 2] - point[2];
    const double w = radius - sqrt(rdist3(cx, cy, cz));
    sw += w;
    m[0] += w * cx * cx; m[1] += w * cx * cy; m[2] += w * cx * cz;
    m[3] += w * cy * cy; m[4] += w * cy * cz; m[5] += w * cz * cz;
  }
  for (int j = 0; j < 6; ++j) m[j] /= sw;
  double eval[3], evec[3][3];
  eigh3(m, eval, evec);
  const double* x = evec[2];
  const double* z = evec[0];
  int neg_x = 0, neg_z = 0;
  for (int i = 0; i < k; ++i) {
    const double cx = nbrs[3 * i] - point[0], cy = nbrs[3 * i + 1] - point[1], cz = nbrs[3 * i + 2] - point[2];
    neg_x += (cx * x[0] + cy * x[1] + cz * x[2]) < 0.0;
    neg_z += (cx * z[0] + cy * z[1] + cz * z[2]) < 0.0;
  }
  shot_frame(x, z, neg_x > k - neg_x, neg_z > k - neg_z, lrf9);
}

// Mirrors shot_descriptor_block_kernel for one query: compact winner tables, neighbours taken 32 at a time (key pass,
// then value pass; the kernel takes 128, which changes nothing since keys are unique), atomicMax replaced by a
// sequential max.
void hm_shot_descriptor(const double* point, const double* nbrs, const double* normals, int k, double radius,
                        const double* f, int normalize, int min_nb, float* out352) {
  std::vector<uint64_t> keys(kKeyCount, 0u);
  std::vector<float> vals(kValCount, 0.0f);
  int positive = 0;
  const double inv_radius = 1.0 / radius;
  for (int base = 0; base < k; base += 32) {
    ShotDecision d[32];
    uint64_t key[32];
    bool active[32];
    for (int lane = 0; lane < 32; ++lane) {
      active[lane] = false;
      const int i = base + lane;
      if (i >= k) continue;
      const double cx = nbrs[3 * i] - point[0], cy = nbrs[3 * i + 1] - point[1], cz = nbrs[3 * i + 2] - point[2];
      const double d2 = rdist3(cx, cy, cz);
      if (!(d2 > 0.0)) continue;
      active[lane] = true;
      ++positive;
      d[lane] = shot_decide_in_frame(cx, cy, cz, normals[3 * i], normals[3 * i + 1], normals[3 * i + 2], f, sqrt(d2),
                                     radius, inv_radius);
      key[lane] = shot_order_key(d[lane].key, uint32_t(i));
      if (key[lane] > keys[kKeyOwn + d[lane].own]) keys[kKeyOwn + d[lane].own] = key[lane];
      if (key[lane] > keys[kKeyCos + d[lane].cos_nb]) keys[kKeyCos + d[lane].cos_nb] = key[lane];
      if (key[lane] > keys[kKeyAz + d[lane].az_nb]) keys[kKeyAz + d[lane].az_nb] = key[lane];
    }
    for (int lane = 0; lane < 32; ++lane) {
      if (!active[lane]) continue;
      const ShotDecision& e = d[lane];
      shot_store_winner(e, keys[kKeyOwn + e.own] == key[lane], keys[kKeyCos + e.cos_nb] == key[lane],
                        keys[kKeyAz + e.az_nb] == key[lane], vals.data());
    }
  }
  double sq = 0.0;
  float v[kShotLen];
  for (int g = 0; g < kShotLen / 4; ++g) {  // four bins of one (cosine, azimuth) cell at a time, as the kernel does
    const uint64_t* k = keys.data() + 4 * g;
    const float* x = vals.data() + 4 * g;
    shot_bin_group_compact(k + kKeyOwn, k + kKeyCos, k + kKeyAz, x + kValOwn, x + kValRad, x + kValEl, x + kValCos,
                           x + kValAz, v + 4 * g);
    for (int t = 0; t < 4; ++t) {
      if (v[4 * g + t] != shot_bin_value_compact(keys.data(), vals.data(), 4 * g + t)) v[4 * g + t] = NAN;  // must agree
      sq += double(v[4 * g + t]) * double(v[4 * g + t]);
    }
  }
  const double norm = sqrt(sq);
  const bool keep = positive > min_nb && norm > 0.0;
  const float inv = keep ? (normalize ? float(1.0 / norm) : 1.0f) : 0.0f;
  for (int b = 0; b < kShotLen; ++b) out352[b] = v[b] * inv;
}

// Mirrors spfh_kernel for one point: integer histogram of width 3n or n^3.
void hm_spfh_counts(const double* point, const double* normal, const double* nbrs, const double* nbr_normals, int k,
                    int n_bins, int decorrelated, const double* edges, int* hist) {
  const int width = decorrelated ? 3 * n_bins : n_bins * n_bins * n_bins;
  std::memset(hist, 0, sizeof(int) * width);
  for (int i = 0; i < k; ++i) {
    const double rel[3] = {nbrs[3 * i] - point[0], nbrs[3 * i + 1] - point[1], nbrs[3 * i + 2] - point[2]};
    const double d2 = rdist3(rel[0], rel[1], rel[2]);
    const double* e[3] = {edges, edges + (n_bins + 1), edges + 2 * (n_bins + 1)};
    double scale[3];
    float lo32[3], scale32[3];
    for (int f = 0; f < 3; ++f) {
      scale[f] = double(n_bins) / (e[f][n_bins] - e[f][0]);
      lo32[f] = float(e[f][0]);
      scale32[f] = float(scale[f]);
    }
    // as the kernel: float32-filtered bins, float64 (reciprocal first guess, filtered theta) where unsure
    const float u32[3] = {float(normal[0]), float(normal[1]), float(normal[2])};
    const float u_norm = sqrtf(u32[0] * u32[0] + u32[1] * u32[1] + u32[2] * u32[2]);
    int ia, ip, it;
    const bool counted = fpfh_pair_bins(rel, normal, u32, u_norm, nbr_normals + 3 * i, n_bins, edges, n_bins + 1, scale,
                                        lo32, scale32, true, ia, ip, it);
    if (counted != (d2 > 0.0)) {
      hist[0] = -2000000;
      return;
    }
    if (!counted) continue;
    {  // the filtered path must give the bins of the plain float64 path
      double a2, p2, theta;
      fpfh_features(rel, sqrt(d2), normal, nbr_normals + 3 * i, a2, p2, theta);
      if (ia != histogram_bin(a2, e[0], n_bins) || ip != histogram_bin(p2, e[1], n_bins) ||
          it != histogram_bin(theta, e[2], n_bins)) {
        hist[0] = -1000000;
        return;
      }
    }
    if (decorrelated) {
      if (ia >= 0) ++hist[ia];
      if (ip >= 0) ++hist[n_bins + ip];
      if (it >= 0) ++hist[2 * n_bins + it];
    } else if (ia >= 0 && ip >= 0 && it >= 0) {
      ++hist[(ia * n_bins + ip) * n_bins + it];
    }
  }
}

// One pair through the float32 filter alone: returns 1 and the three bins when the filter is sure, 0 otherwise.
int hm_fpfh_bins_fast(const double* rel, const double* u, const double* nj, int n_bins, const double* edges, int* bins) {
  float lo32[3], scale32[3];
  for (int f = 0; f < 3; ++f) {
    const double* e = edges + f * (n_bins + 1);
    lo32[f] = float(e[0]);
    scale32[f] = float(double(n_bins) / (e[n_bins] - e[0]));
  }
  const float rel32[3] = {float(rel[0]), float(rel[1]), float(rel[2])};
  const float u32[3] = {float(u[0]), float(u[1]), float(u[2])};
  const float nj32[3] = {float(nj[0]), float(nj[1]), float(nj[2])};
  const float u_norm = sqrtf(u32[0] * u32[0] + u32[1] * u32[1] + u32[2] * u32[2]);
  return fpfh_bins_fast(rel32, u32, u_norm, nj32, n_bins, lo32, scale32, bins[0], bins[1], bins[2]) ? 1 : 0;
}
// The same pair through the plain float64 path (np.histogram semantics): bins, or returns 0 when d == 0.
int hm_fpfh_bins_float64(const double* rel, const double* u, const double* nj, int n_bins, const double* edges, int* bins) {
  const double d2 = rdist3(rel[0], rel[1], rel[2]);
  if (!(d2 > 0.0)) return 0;
  double a, p, theta;
  fpfh_features(rel, sqrt(d2), u, nj, a, p, theta);
  bins[0] = histogram_bin(a, edges, n_bins);
  bins[1] = histogram_bin(p, edges + (n_bins + 1), n_bins);
  bins[2] = histogram_bin(theta, edges + 2 * (n_bins + 1), n_bins);
  return 1;
}

// Batch of pairs: stats[0] = pairs the filter was sure about, stats[1] = of those, pairs whose bins differ from the
// float64 path's (or that the float64 path drops) — must be 0; first_bad = index of the first such pair or -1.
void hm_fpfh_fast_check(long n_pairs, const double* rel, const double* u, const double* nj, int n_bins,
                        const double* edges, long* stats, long* first_bad) {
  stats[0] = stats[1] = 0;
  *first_bad = -1;
  for (long i = 0; i < n_pairs; ++i) {
    int fast[3], exact[3];
    if (!hm_fpfh_bins_fast(rel + 3 * i, u + 3 * i, nj + 3 * i, n_bins, edges, fast)) continue;
    ++stats[0];
    const int counted = hm_fpfh_bins_float64(rel + 3 * i, u + 3 * i, nj + 3 * i, n_bins, edges, exact);
    if (!counted || fast[0] != exact[0] || fast[1] != exact[1] || fast[2] != exact[2]) {
      ++stats[1];
      if (*first_bad < 0) *first_bad = i;
    }
  }
}

int hm_histogram_bin(double x, const double* edges, int n) { return histogram_bin(x, edges, n); }
int hm_histogram_bin_scaled(double x, const double* edges, int n) {
  return histogram_bin_scaled(x, edges, n, double(n) / (edges[n] - edges[0]));
}
int hm_theta_bin_float64(double ny, double nx, const double* edges, int n) {  // the unfiltered path
  return histogram_bin(atan2(ny, nx), edges, n);
}
int hm_theta_bin(double ny, double nx, const double* edges, int n) {
  return fpfh_theta_bin(ny, nx, edges, n, double(n) / (edges[n] - edges[0]));
}

// ---- the fast descriptor kernel (shot.cu::shot_fast_kernel), mirrored for one query ------------------------------
// records != 0: the fused driver's mode — float32 images of the exact float64 offsets (what search_moments_kernel
// stores), votes on the RAW eigenvectors (`frame` = raw x, raw z: 6 doubles). records == 0: a caller's list — the
// grid's cell-relative float32 coordinates, `frame` = the final 3x3 frame (row-major, columns x y z).
// Then as the kernel: float32-filtered decisions, unique keys, winners by maximum, values added in five sub-phases.
// Returns 0 and the row when the kernel would keep the query, 1 when it would hand it to the exact kernel
// (more than 128 neighbours, a decision inside its float32 margin, or two competitors float32 cannot order).
// stats[0] += neighbours decided, stats[1] += neighbours whose float32 decision was unsure.
int hm_shot_descriptor_fast(const double* point, const double* nbrs, const double* normals, int k, double radius,
                            const double* origin, double edge, const double* frame, int records, int normalize,
                            int min_nb, float* out352, double* frame_out9, long* stats) {
  if (k > 128) return 1;
  if (k == 0) {
    for (int b = 0; b < kShotLen; ++b) out352[b] = 0.0f;
    return 0;
  }
  const double inv_cell = 1.0 / edge;
  auto cell_of = [&](const double p[3], int c[3]) {
    for (int a = 0; a < 3; ++a) c[a] = int(floor((p[a] - origin[a]) * inv_cell));
  };
  const double u = 5.9604645e-8;
  const float e_rel = float(8.0 * u * 1.0001), e_abs = float(24.0 * u * edge * 1.0001), w_min = float(0.01 * radius);
  const float edge32 = float(edge), radius32 = float(radius), inv_radius32 = float(1.0 / radius);
  const uint32_t amb_margin = uint32_t(2.0 * ((records ? 8.0 * u : 24.0 * u * edge / radius) * 8388608.0 + 1.5) + 1.0);
  const int fuse_votes = records;
  float ax[3], ay[3], az[3];
  if (fuse_votes) {
    const double* x = frame;
    const double* z = frame + 3;
    ay[0] = float(z[1] * x[2] - z[2] * x[1]);
    ay[1] = float(z[2] * x[0] - z[0] * x[2]);
    ay[2] = float(z[0] * x[1] - z[1] * x[0]);
    for (int a = 0; a < 3; ++a) { ax[a] = float(x[a]); az[a] = float(z[a]); }
  } else {
    for (int a = 0; a < 3; ++a) { ax[a] = float(frame[3 * a]); ay[a] = float(frame[3 * a + 1]); az[a] = float(frame[3 * a + 2]); }
  }
  int cq[3];
  float lq[3];
  cell_of(point, cq);
  shot_cell_local(point, origin, edge, cq, lq);
  const uint32_t cq_bits = shot_cellbits(cq);
  std::vector<float> X0(k), Y0(k), Z0(k), C0(k), R2(k), NN(k);
  std::vector<char> zero(k, 0);
  bool unsure = false;
  int neg_x = 0, neg_z = 0;
  for (int i = 0; i < k; ++i) {
    float c[3];
    if (records) {
      for (int a = 0; a < 3; ++a) c[a] = float(nbrs[3 * i + a] - point[a]);
      zero[i] = nbrs[3 * i] == point[0] && nbrs[3 * i + 1] == point[1] && nbrs[3 * i + 2] == point[2];
    } else {
      int cp[3];
      float lp[3];
      cell_of(nbrs + 3 * i, cp);
      shot_cell_local(nbrs + 3 * i, origin, edge, cp, lp);
      shot_rel32(lp, shot_cellbits(cp), lq, cq_bits, edge32, c);
    }
    R2[i] = dot3f(c, c);
    X0[i] = dot3f(c, ax); Y0[i] = dot3f(c, ay); Z0[i] = dot3f(c, az);
    const float nv[3] = {float(normals[3 * i]), float(normals[3 * i + 1]), float(normals[3 * i + 2])};
    C0[i] = dot3f(nv, az);
    NN[i] = dot3f(nv, nv);
    if (!records && R2[i] == 0.0f) {
      if (nbrs[3 * i] == point[0] && nbrs[3 * i + 1] == point[1] && nbrs[3 * i + 2] == point[2]) zero[i] = 1;
      else unsure = true;
    }
    if (fuse_votes && !zero[i]) {
      const float e = e_rel * sqrtf(R2[i]);
      neg_x += X0[i] < 0.0f;
      neg_z += Z0[i] < 0.0f;
      unsure = unsure || !(fabsf(X0[i]) > e && fabsf(Z0[i]) > e);
    }
  }
  float fsx = 1.0f, fsz = 1.0f;
  if (fuse_votes) {
    if (neg_x > k - neg_x) fsx = -1.0f;
    if (neg_z > k - neg_z) fsz = -1.0f;
  }
  if (frame_out9 != nullptr && fuse_votes) shot_frame(frame, frame + 3, fsx < 0.0f, fsz < 0.0f, frame_out9);
  std::vector<ShotFastRecord> rec(k);
  std::vector<char> act(k, 0);
  int positive = 0;
  for (int i = 0; i < k; ++i) {
    if (zero[i]) continue;
    ++positive;
    const float inv_rho = 1.0f / sqrtf(fmaxf(R2[i], 1e-37f)), rho = R2[i] * inv_rho;
    ShotFastMargins m;
    m.e_loc = records ? e_rel * rho : e_abs;
    m.e_rho = m.e_loc;
    m.w_rho_min = records ? 0.0f : w_min;
    m.w_xy_min = records ? 0.01f * rho : w_min;
    m.n2 = 1.001f;
    ShotDecision d;
    const bool sure = shot_decide_fast(fsx * X0[i], fsx * fsz * Y0[i], fsz * Z0[i], fsz * C0[i], rho, inv_rho, radius32,
                                       inv_radius32, m, d) && NN[i] <= 1.001f;
    if (stats) { stats[0] += 1; stats[1] += !sure; }
    unsure = unsure || !sure;
    if (!sure) continue;
    rec[i] = shot_fast_record(d, uint32_t(i));
    act[i] = 1;
  }
  if (unsure) return 1;
  std::vector<uint32_t> keys(kKeyCount, 0u);
  std::vector<float> desc(kShotLen, 0.0f);
  for (int i = 0; i < k; ++i)
    if (act[i])
      for (int t = 0; t < 3; ++t) {
        uint32_t& slot = keys[t * kShotLen + ((rec[i].bins >> (9 * t)) & 511u)];
        if (rec[i].key > slot) slot = rec[i].key;
      }
  bool amb = false;
  std::vector<char> win(3 * k, 0);
  for (int i = 0; i < k; ++i)
    if (act[i])
      for (int t = 0; t < 3; ++t) {
        const uint32_t o = keys[t * kShotLen + ((rec[i].bins >> (9 * t)) & 511u)];
        if (o == rec[i].key) win[3 * i + t] = 1;
        else amb = amb || shot_keys_ambiguous(o, rec[i].key, amb_margin);
      }
  for (int i = 0; i < k; ++i)
    if (win[3 * i]) desc[rec[i].bins & 511u] = rec[i].v_own;
  for (int t = 0; t < 2; ++t)
    for (int i = 0; i < k; ++i)
      if (win[3 * i]) {
        const uint32_t partner = (rec[i].bins & 511u) ^ uint32_t(1 + t);
        const uint32_t pk = keys[kKeyOwn + partner], key = rec[i].key;
        amb = amb || (pk != 0u && shot_keys_ambiguous(pk, key, amb_margin));
        const float v = t == 0 ? rec[i].v_rad : rec[i].v_el;
        if (key > pk && v != 0.0f) desc[partner] += v;
      }
  for (int i = 0; i < k; ++i)
    if (win[3 * i + 1]) desc[(rec[i].bins >> 9) & 511u] += rec[i].v_cos;
  for (int i = 0; i < k; ++i)
    if (win[3 * i + 2]) desc[(rec[i].bins >> 18) & 511u] += rec[i].v_az;
  if (amb) return 1;
  float sq = 0.0f;
  for (int b = 0; b < kShotLen; ++b) sq += desc[b] * desc[b];
  const bool keep = positive > min_nb && sq > 0.0f;
  const float inv = keep ? (normalize ? 1.0f / sqrtf(sq) : 1.0f) : 0.0f;
  for (int b = 0; b < kShotLen; ++b) out352[b] = desc[b] * inv;
  return 0;
}

// shot_decide_fast against shot_decide on n inputs: rows of (X, Y, Z, cosine, rho) in float64 (the exact values) and
// their float32 images with errors inside the documented bounds; relative != 0: the fused driver's margins (8 u rho),
// else the gathered coordinates' (24 u edge, weights guarded at 1 % of the radius).
// stats[0] = sure, stats[1] = sure but a bin / sign differs from the float64 decision (must be 0),
// stats[2] = largest |weight difference| among the sure ones, in 1e-9 units.
void hm_shot_decide_fast_check(long n, const double* exact5, const float* approx5, double radius, double edge,
                               int relative, long* stats) {
  const double u = 5.9604645e-8;
  stats[0] = stats[1] = stats[2] = 0;
  for (long i = 0; i < n; ++i) {
    const double* x = exact5 + 5 * i;
    const float* f = approx5 + 5 * i;
    ShotDecision df;
    ShotFastMargins m;
    m.e_loc = m.e_rho = relative ? float(8.0 * u * 1.0001) * f[4] : float(24.0 * u * edge * 1.0001);
    m.w_rho_min = relative ? 0.0f : float(0.01 * radius);
    m.w_xy_min = relative ? 0.01f * f[4] : float(0.01 * radius);
    m.n2 = 1.001f;
    if (!shot_decide_fast(f[0], f[1], f[2], f[3], f[4], 1.0f / f[4], float(radius), float(1.0 / radius), m, df)) continue;
    ++stats[0];
    const ShotDecision de = shot_decide(x[0], x[1], x[2], fmin(1.0, fmax(-1.0, x[3])), x[4], radius, 1.0 / radius);
    if (df.own != de.own || df.cos_nb != de.cos_nb || df.az_nb != de.az_nb || df.ti != de.ti || df.ei != de.ei ||
        df.saz != de.saz)
      ++stats[1];
    float ov_f, ot_f, ov_e, ot_e;
    shot_elevation_fast(df, ov_f, ot_f);
    shot_elevation(de, ov_e, ot_e);
    const double w = fmax(fmax(fabs(double(df.a_cos) - de.a_cos), fabs(double(df.own_shell) - de.own_shell)),
                          fmax(fmax(fabs(double(df.other_shell) - de.other_shell), fabs(double(shot_azimuth_fast(df)) - shot_azimuth(de))),
                               fmax(fabs(double(ov_f) - ov_e), fabs(double(ot_f) - ot_e))));
    if (long(w * 1e9) > stats[2]) stats[2] = long(w * 1e9);
  }
}

// the two polynomial weights against libm on float32 inputs: max |difference| over n samples
double hm_shot_trig_check(long n, const float* fx, const float* fy, const float* ratio) {
  double worst = 0.0;
  for (long i = 0; i < n; ++i) {
    ShotDecision d;
    d.fx = fx[i]; d.fy = fy[i]; d.ratio = ratio[i];
    d.ti = azimuth_octant(fx[i], fy[i]);
    d.ei = ratio[i] > 0.0f;
    d.saz = 1;
    float a, b, c, e;
    shot_elevation_fast(d, a, b);
    shot_elevation(d, c, e);
    worst = fmax(worst, fmax(fabs(double(a) - c), fabs(double(b) - e)));
    worst = fmax(worst, fabs(double(shot_azimuth_fast(d)) - shot_azimuth(d)));
  }
  return worst;
}

}  // extern "C"
