// Per-neighbour / per-query arithmetic of the SHOT and FPFH kernels, written as __host__ __device__ inline
// functions so that the exact same code is (a) inlined into the sm_100a kernels and (b) compiled by g++ into the
// CPU-only unit test tests/host_math (which checks it against the oracle without a GPU). It is NOT a CPU
// fallback: nothing in the product calls the host instantiation.
//
// Precision policy (DESIGN.md "Precision"): everything that DECIDES something (neighbour predicate, bin indices,
// interpolation signs, LRF sign votes, distance ordering) is evaluated in float64 from the float64 inputs, with
// explicit non-fused operations where the reference's result depends on the rounding of individual operations.
// Only the interpolation WEIGHTS (continuous in their inputs) go through float32 transcendental functions.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define SF_HD __host__ __device__ __forceinline__
#else
#define SF_HD inline
#endif

#include "sf_eigh3.cuh"  // eigh3(): LAPACK-path 3x3 eigen-solver (replaces np.linalg.eigh at shot.py:36)

namespace sf {

constexpr int kShotCos = 11, kShotAz = 8, kShotEl = 2, kShotRad = 2;
constexpr int kShotLen = kShotCos * kShotAz * kShotEl * kShotRad;  // 352

// a*b and a+b rounded separately (never contracted into an FMA), as NumPy / scikit-learn / SciPy compute them.
SF_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  volatile double p = a * b;
  return p;
#endif
}
SF_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  volatile double s = a + b;
  return s;
#endif
}

// Reduced squared distance exactly as sklearn's euclidean rdist accumulates it: ((dx*dx + dy*dy) + dz*dz).
// (sklearn/metrics/_dist_metrics: `for j: tmp = x1[j] - x2[j]; d += tmp * tmp`, d starting at 0.)
SF_HD double rdist3(double dx, double dy, double dz) {
  return add_rn(add_rn(mul_rn(dx, dx), mul_rn(dy, dy)), mul_rn(dz, dz));
}

// One coordinate in the local frame, c . (column of the frame), rounded as the oracle's `rel @ lrf` rounds it: NumPy's
// float64 matmul (OpenBLAS dgemm) accumulates k = 0, 1, 2 with fused multiply-adds. On a plane Z is rounding noise of
// either sign and its sign picks the elevation bin, so the order of the roundings is part of the result there.
SF_HD double frame_dot(double cx, double cy, double cz, double f0, double f1, double f2) {
  return fma(cz, f2, fma(cy, f1, mul_rn(cx, f0)));
}

// ----------------------------------------------------------------------------------------------------------
// SHOT: one neighbour -> its own bin, the five "other" targets and the six values (SURVEY.md Appendix A).
// ----------------------------------------------------------------------------------------------------------
// Azimuth octant by comparisons only (shot.py:60-70); octant 0 starts at -pi.
SF_HD int azimuth_octant(double x, double y) {
  const bool upper = (y > 0.0) || (y == 0.0 && x < 0.0);
  const bool right = (x > 0.0) || (x == 0.0 && y > 0.0);
  const bool second = ((x * y > 0.0) || (x == 0.0)) ? (fabs(x) < fabs(y)) : (fabs(x) > fabs(y));
  return 4 * int(upper) + 2 * int(right != upper) + int(second);
}

struct ShotRecord {
  int own;        // flat bin ((ci*8 + ti)*2 + ei)*2 + ri
  int cos_nb;     // statement 1 target (cosine neighbour bin, or `own` when the cosine sits on a bin centre)
  int az_nb;      // statement 9 target (azimuth neighbour bin, or `own`)
  float v_own;    // statements 2 + 5 + 8 + 10 (all address `own`, hence share one winner)
  float v_cos;    // statement 1
  float v_az;     // statement 9
  float v_rad;    // statement 3 or 4, whichever targets the OTHER radial shell (the one targeting `own` writes 0)
  float v_el;     // statement 6 or 7, whichever targets the OTHER elevation half
  uint32_t key;   // distance order: larger = later in the reference's ascending-rho order = wins
};

SF_HD int shot_flat(int ci, int ti, int ei, int ri) { return ((ci * kShotAz + ti) * kShotEl + ei) * kShotRad + ri; }

// Unit vectors of the octant centre directions, angle = -pi + (t + 0.5) * pi/4.
SF_HD void octant_centre(int t, double& cx, double& cy) {
  const double c = 0.92387953251128673848;  // cos(pi/8)
  const double s = 0.38268343236508978178;  // sin(pi/8)
  switch (t) {
    case 0: cx = -c; cy = -s; break;
    case 1: cx = -s; cy = -c; break;
    case 2: cx = s; cy = -c; break;
    case 3: cx = c; cy = -s; break;
    case 4: cx = c; cy = s; break;
    case 5: cx = s; cy = c; break;
    case 6: cx = -s; cy = c; break;
    default: cx = -c; cy = s; break;
  }
}

// ---- step 1: everything that DECIDES, float64 (bins, interpolation signs, distance key) + the cheap weights --------
// local = (X, Y, Z) coordinates in the LRF (float64), cosine = clip(n . z_axis) (float64), rho > 0, radius and its
// reciprocal (computed once per launch: the weights are continuous, so multiplying by 1/radius instead of
// dividing moves them by an ulp at most, and it removes four float64 divisions per neighbour).
struct ShotDecision {
  int own, cos_nb, az_nb;  // flat bins: own, statement-1 target, statement-9 target
  uint32_t key;            // distance order (see ShotRecord::key)
  int ti, ei, saz;         // azimuth octant, elevation bit, sign of the azimuth offset from the octant centre
  bool equator;            // Z > 0 but the reference's float64 phi = arccos(Z / rho) is exactly pi / 2 (see below)
  float a_cos;             // |cosine offset| (statement 1 value; 1 - a_cos goes to the own bin)
  float own_shell;         // radial weight of the own bin (statement 5)
  float other_shell;       // radial weight sent to the OTHER shell (statement 3 or 4)
  float fx, fy, ratio;     // float32 inputs of the two transcendental weights: atan2f(fy, fx), acosf(ratio)
};

// Largest Z / rho > 0 whose float64 arccos is exactly pi / 2 (np.arccos, glibc's correctly rounded acos): the double
// pi / 2 lies 6.1e-17 below the true value, so arccos(t) = pi/2 - t rounds to it up to t = half an ulp + 6.1e-17.
// On a plane that is not axis-aligned, Z of an in-plane neighbour is rounding noise of either sign (|Z| ~ 1e-17 rho),
// so about half of the neighbours land in this window. tests/test_host_math.py pins the value against np.arccos.
constexpr double kAcosHalfPiMax = 1.7225464241988333e-16;

SF_HD ShotDecision shot_decide(double X, double Y, double Z, double cosine, double rho, double radius, double inv_radius) {
  ShotDecision d;
  const double pos = (cosine + 1.0) * double(kShotCos) / 2.0 - 0.5;  // shot.py:228
  const double ci_f = rint(pos);                                      // round-half-even like np.rint
  const int ci = int(ci_f);
  const double dcos = pos - ci_f;
  const int scos = (dcos > 0.0) - (dcos < 0.0);
  d.ti = azimuth_octant(X, Y);
  d.ei = Z > 0.0;
  // the reference bins by Z > 0 but interpolates by phi: with phi == pi/2 its statement 7 (`lower`, phi < pi/2)
  // writes 0 although the neighbour sits in the upper half (the division only runs for |Z| below 1e-15 rho)
  d.equator = Z > 0.0 && Z < 1e-15 * rho && Z / rho <= kAcosHalfPiMax;
  const int ri = rho > radius / 2;
  d.own = shot_flat(ci, d.ti, d.ei, ri);
  int cnb = ci + scos;
  cnb = cnb < 0 ? cnb + kShotCos : (cnb >= kShotCos ? cnb - kShotCos : cnb);
  d.cos_nb = shot_flat(cnb, d.ti, d.ei, ri);
  // sign of the azimuth offset from the octant centre: cross(centre, (X, Y)) instead of a float64 atan2
  double cx, cy;
  octant_centre(d.ti, cx, cy);
  const double cr = cx * Y - cy * X;
  // on the LRF's z axis (X == Y == 0) the reference gets theta = atan2(0, 0) = 0 in octant 0: offset clipped to +0.5
  d.saz = (X == 0.0 && Y == 0.0) ? 1 : (cr > 0.0) - (cr < 0.0);
  d.az_nb = shot_flat(ci, (d.ti + d.saz + kShotAz) & (kShotAz - 1), d.ei, ri);
  d.a_cos = float(fabs(dcos));
  // radial (shot.py:95-118); rho == radius/2 exactly gives 0 everywhere, as in the reference
  const double half = radius / 2, quarter = radius / 4, three_q = radius * 3 / 4, inv_half = 2.0 * inv_radius;
  if (ri) {  // rho > r/2: statement 4 carries `inner`, statement 3 writes 0 to `own`
    d.own_shell = float(1.0 - fabs(rho - three_q) * inv_half);
    d.other_shell = rho < three_q ? float((three_q - rho) * inv_half) : 0.0f;
  } else {
    d.own_shell = rho < half ? float(1.0 - fabs(rho - quarter) * inv_half) : 0.0f;
    d.other_shell = (rho < half && rho > quarter) ? float((rho - quarter) * inv_half) : 0.0f;
  }
  d.fx = float(X);
  d.fy = float(Y);
  d.ratio = fminf(1.0f, fmaxf(-1.0f, float(Z) / float(rho)));
  // order key: rho / radius in 32-bit fixed point (monotone in rho; resolution radius * 2^-32)
  const double scaled = rho * inv_radius * 4294967296.0;
  d.key = scaled >= 4294967295.0 ? 0xFFFFFFFFu : (scaled < 1.0 ? 1u : uint32_t(scaled));
  return d;
}

// The float64 step of one neighbour: offset c = p - q and normal n in the frame f (row-major, columns [x y z]).
SF_HD ShotDecision shot_decide_in_frame(double cx, double cy, double cz, double nx, double ny, double nz,
                                        const double f[9], double rho, double radius, double inv_radius) {
  const double X = frame_dot(cx, cy, cz, f[0], f[3], f[6]);
  const double Y = frame_dot(cx, cy, cz, f[1], f[4], f[7]);
  const double Z = frame_dot(cx, cy, cz, f[2], f[5], f[8]);
  double cosine = nx * f[2] + ny * f[5] + nz * f[8];
  cosine = fmin(1.0, fmax(-1.0, cosine));
  return shot_decide(X, Y, Z, cosine, rho, radius, inv_radius);
}

// The local reference frame from the raw eigenvectors x, z and the sign votes of shot.py:40-45 (an axis is negated when
// strictly more neighbours project negatively on it than not), y = z cross x in float64. f: row-major, columns [x y z].
SF_HD void shot_frame(const double x_raw[3], const double z_raw[3], bool flip_x, bool flip_z, double f[9]) {
  const double sx = flip_x ? -1.0 : 1.0, sz = flip_z ? -1.0 : 1.0;  // (exact negation)
  const double x[3] = {sx * x_raw[0], sx * x_raw[1], sx * x_raw[2]}, z[3] = {sz * z_raw[0], sz * z_raw[1], sz * z_raw[2]};
  const double y[3] = {z[1] * x[2] - z[2] * x[1], z[2] * x[0] - z[0] * x[2], z[0] * x[1] - z[1] * x[0]};
  f[0] = x[0]; f[1] = y[0]; f[2] = z[0];
  f[3] = x[1]; f[4] = y[1]; f[5] = z[1];
  f[6] = x[2]; f[7] = y[2]; f[8] = z[2];
}

// ---- step 2: the two transcendental weights, float32 (continuous in their inputs) ---------------------------------
// elevation (shot.py:142-171): phi < pi/2 <=> Z > 0 (see DESIGN.md), except in the window of kAcosHalfPiMax
SF_HD void shot_elevation(const ShotDecision& d, float& own_vol, float& other_vol) {
  const float kPi = 3.14159265358979323846f, inv_h = 0.63661977236758134308f;  // 1 / (pi / 2)
  const float phi = acosf(d.ratio);
  if (d.ei) {  // upper half-space, elevation bin 1, centre pi/4; statement 7 carries `lower`
    own_vol = 1.0f - fabsf(phi - 0.25f * kPi) * inv_h;
    other_vol = phi >= 0.25f * kPi && !d.equator ? (phi - 0.25f * kPi) * inv_h : 0.0f;
  } else {     // Z <= 0, elevation bin 0, centre 3pi/4; statement 6 carries `upper`
    own_vol = 1.0f - fabsf(phi - 0.75f * kPi) * inv_h;
    other_vol = phi <= 0.75f * kPi ? (0.75f * kPi - phi) * inv_h : 0.0f;
  }
  other_vol = fmaxf(other_vol, 0.0f);
}
// azimuth (shot.py:282-298): |offset from the octant centre| in octant widths, clipped to 0.5
SF_HD float shot_azimuth(const ShotDecision& d) {
  const float kPi = 3.14159265358979323846f, q = 0.25f * kPi, inv_q = 1.27323954473516268615f;  // 1 / (pi / 4)
  const float theta = atan2f(d.fy, d.fx);
  float daz = (theta - (-kPi + float(d.ti) * q)) * inv_q - 0.5f;
  daz = fminf(0.5f, fmaxf(-0.5f, daz));
  return d.saz == 0 ? 0.0f : fabsf(daz);
}

SF_HD ShotRecord shot_record(double X, double Y, double Z, double cosine, double rho, double radius, double inv_radius) {
  const ShotDecision d = shot_decide(X, Y, Z, cosine, rho, radius, inv_radius);
  float own_vol, other_vol;
  shot_elevation(d, own_vol, other_vol);
  const float a_az = shot_azimuth(d);
  ShotRecord r;
  r.own = d.own; r.cos_nb = d.cos_nb; r.az_nb = d.az_nb; r.key = d.key;
  r.v_cos = d.a_cos;
  r.v_rad = d.other_shell;
  r.v_el = other_vol;
  r.v_az = a_az;
  r.v_own = (1.0f - d.a_cos) + d.own_shell + own_vol + (1.0f - a_az);
  return r;
}

// ----------------------------------------------------------------------------------------------------------
// SHOT, float32-filtered decisions (the fast descriptor kernel, shot.cu::shot_fast_kernel).
//
// Every decision of shot_decide is a comparison of a quantity that is continuous in the inputs against a fixed
// boundary, so it can be taken from a float32 evaluation whenever the float32 value keeps a proven distance from
// the boundary; a query with any neighbour inside a margin is handed to the float64 kernel (1-3 % of the queries on
// a surface scan, where Z clusters around 0).
//
// Two sources of float32 offsets c = p - q, u = 2^-24:
//  (a) the fused driver: its search kernel has the exact float64 offset in registers and stores its float32 image
//      in the neighbour list: each component within u |c_a| of the float64 value, so with rho = |c|
//        rho      : 1.7 u rho (c) + 1.5 u rho (sum of squares) + 3.5 u rho (rsqrt, product)      <= 8 u rho
//        X, Y, Z  : 1.7 u rho (c) + 1.7 u rho (axis rounded to float32) + 3 u rho (dot product)  <= 8 u rho
//  (b) caller-provided lists: the grid's cell-relative float32 coordinates (grid.cu: lp = float((p - origin) -
//      cell * edge), |lp| <= edge, plus the cell coordinates modulo 4): c = lp - lq + (cell_p - cell_q) * edge with
//      cell_p - cell_q in {-1, 0, 1}, each component within 7 u edge wherever the cloud sits (roundings of lp, lq,
//      lp - lq, edge, the fma: 5 u edge; float64 roundings of (p - origin) - cell * edge: below u edge because
//      extent / edge < 2^25):  rho, X, Y, Z <= 24 u edge.
//  cosine = n . z : 7 u |n|, |n|^2 <= n2;  pos = (cosine + 1) * 5.5 - 0.5  <= (44 n2 + 40) u
// A decision is accepted when the value is farther than its bound from the boundary (the float64 reference carries
// its own rounding, 1e-16 relative: far below). The continuous WEIGHTS follow the inputs, except where they are badly
// conditioned: the elevation weight moves by (error of c) / rho and the azimuth weight by (error of c) / hypot(X, Y);
// neighbours below `w_rho_min` / `w_xy_min` are left to float64 ((a): none / hypot below 1 % of rho; (b): 1 % of
// the radius each — a per-weight error below 2e-4 in the worst case of the bounds, ~1e-5 in practice).
// Checked on the host against shot_decide on millions of perturbed inputs (tests/test_host_math.py) and on the GPU
// against the goldens and against the float64 kernel.
// ----------------------------------------------------------------------------------------------------------
constexpr float kEps32 = 5.9604645e-8f;  // 2^-24

// a / b for weights (continuous in their inputs): the device's approximate division (2 ulp, no slow-path call)
SF_HD float sf_divf(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fdividef(a, b);
#else
  return a / b;
#endif
}
SF_HD float sf_rsqrtf(float x);  // (defined with the FPFH helpers below)

// cell-relative float32 coordinates of p in cell c (grid.cu writes them; the kernels compute the query's)
SF_HD void shot_cell_local(const double p[3], const double origin[3], double edge, const int c[3], float out[3]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int a = 0; a < 3; ++a) out[a] = float((p[a] - origin[a]) - double(c[a]) * edge);
}
SF_HD uint32_t shot_cellbits(const int c[3]) {
  return uint32_t(c[0] & 3) | (uint32_t(c[1] & 3) << 2) | (uint32_t(c[2] & 3) << 4);
}
// p - q from the cell-relative coordinates; bits_p / bits_q = the cells' coordinates modulo 4 (2 bits per axis)
SF_HD void shot_rel32(const float lp[3], uint32_t bits_p, const float lq[3], uint32_t bits_q, float edge32, float c[3]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int a = 0; a < 3; ++a) {
    const uint32_t code = ((bits_p >> (2 * a)) - (bits_q >> (2 * a)) + 1u) & 3u;  // cell_p - cell_q + 1
    const float shift = code == 0u ? -edge32 : (code == 2u ? edge32 : (code == 1u ? 0.0f : 2.0f * edge32));
    c[a] = (lp[a] - lq[a]) + shift;
  }
}
SF_HD float dot3f(const float a[3], const float b[3]) { return fmaf(a[2], b[2], fmaf(a[1], b[1], a[0] * b[0])); }

struct ShotFastMargins {
  float e_loc;     // bound on the error of X, Y, Z
  float e_rho;     // bound on the error of rho
  float w_rho_min, w_xy_min;  // weights are left to float64 below these (see above)
  float n2;        // the cosine margin assumes |n|^2 <= n2
};

// shot_decide from float32 inputs. Returns false when any decision is within its margin of a boundary; the decision
// is only meaningful when true is returned. cosine = n . z, not yet clipped; rho = |c| > 0.
// d.key = rho / radius in 23-bit fixed point (taken from the mantissa of 1 + rho / radius: no conversion).
SF_HD bool shot_decide_fast(float X, float Y, float Z, float cosine, float rho, float inv_rho, float radius,
                            float inv_radius, const ShotFastMargins& m, ShotDecision& d) {
  const float cosc = fminf(1.0f, fmaxf(-1.0f, cosine));
  const float pos = fmaf(cosc + 1.0f, 0.5f * float(kShotCos), -0.5f);  // shot.py:228
  const float e_pos = (44.0f * m.n2 + 40.0f) * kEps32;
  // round-half-even by the float32 adder: pos in [-0.5, 10.5], 1.5 * 2^23 + pos keeps the integer in the mantissa
  const float magic = 12582912.0f;
  const float shifted = pos + magic;
#if defined(__CUDA_ARCH__)
  const int ci = __float_as_int(shifted) - 0x4B400000;
#else
  int ci;
  { float t = shifted; uint32_t bits; memcpy(&bits, &t, 4); ci = int(bits) - 0x4B400000; }
#endif
  const float dcos = pos - (shifted - magic);
  bool sure = (0.5f - fabsf(dcos) > e_pos) && (fabsf(dcos) > e_pos);
  const int scos = dcos > 0.0f ? 1 : -1;
  const float ax = fabsf(X), ay = fabsf(Y), hi = fmaxf(ax, ay);
  sure = sure && ax > m.e_loc && ay > m.e_loc && fabsf(ax - ay) > 2.0f * m.e_loc && fabsf(Z) > m.e_loc;
  const bool upper = Y > 0.0f, right = X > 0.0f;
  const bool wide = ax > ay;  // the octant hugs the x axis
  const bool second = (upper == right) ? !wide : wide;  // azimuth_octant with X, Y != 0
  d.ti = 4 * int(upper) + 2 * int(right != upper) + int(second);
  d.ei = Z > 0.0f;
  d.equator = false;  // a sure decision has |Z| > e_loc >= 8 u rho, far above the window of kAcosHalfPiMax
  const float half = 0.5f * radius;
  const int ri = rho > half;
  sure = sure && fabsf(rho - half) > m.e_rho && rho < radius * 1.001f && rho > m.w_rho_min && hi > m.w_xy_min;
  d.own = shot_flat(ci, d.ti, d.ei, ri);
  int cnb = ci + scos;
  cnb = cnb < 0 ? cnb + kShotCos : (cnb >= kShotCos ? cnb - kShotCos : cnb);
  d.cos_nb = shot_flat(cnb, d.ti, d.ei, ri);
  // sign of the offset from the octant centre: the centre has the signs of (X, Y) and its larger component along
  // the larger of |X|, |Y|, so cross(centre, (X, Y)) = sign(X) sign(Y) (m1 |Y| - m2 |X|), (m1, m2) = (cos, sin)(pi/8)
  // when |X| > |Y|, swapped otherwise
  const float kc = 0.92387953251128673848f, ks = 0.38268343236508978178f;
  const float cr = wide ? fmaf(kc, ay, -ks * ax) : fmaf(ks, ay, -kc * ax);
  sure = sure && fabsf(cr) > 2.0f * m.e_loc;
  d.saz = ((cr > 0.0f) == (upper == right)) ? 1 : -1;
  d.az_nb = shot_flat(ci, (d.ti + d.saz + kShotAz) & (kShotAz - 1), d.ei, ri);
  d.a_cos = fabsf(dcos);
  const float quarter = 0.25f * radius, three_q = 0.75f * radius, inv_half = 2.0f * inv_radius;
  if (ri) {
    d.own_shell = 1.0f - fabsf(rho - three_q) * inv_half;
    d.other_shell = fmaxf(0.0f, (three_q - rho) * inv_half);
  } else {
    d.own_shell = 1.0f - fabsf(rho - quarter) * inv_half;
    d.other_shell = fmaxf(0.0f, (rho - quarter) * inv_half);
  }
  d.fx = X;
  d.fy = Y;
  d.ratio = fminf(1.0f, fmaxf(-1.0f, Z * inv_rho));
  const float one_plus = fminf(fmaf(rho, inv_radius, 1.0f), 1.99999988f);  // [1, 2): mantissa = rho / radius * 2^23
#if defined(__CUDA_ARCH__)
  d.key = __float_as_uint(one_plus) & 0x7FFFFFu;
#else
  { uint32_t bits; memcpy(&bits, &one_plus, 4); d.key = bits & 0x7FFFFFu; }
#endif
  return sure;
}

// The two transcendental weights without atan2f / acosf: the octant and the half-space are already decided, only
// the angle INSIDE them is needed.
//   azimuth  : |offset from the octant centre| in octant widths = |atan(min(|X|,|Y|) / max(|X|,|Y|)) * 4/pi - 0.5|
//              in every octant (the angle from the nearest axis runs 0 .. pi/4 across the octant, up or down)
//   elevation: with g = asin(|Z| / rho) * 2/pi (elevation above the tangent plane, in quarter turns):
//              own half-space volume 1 - |0.5 - g|, other one max(0, 0.5 - g) (shot_elevation with phi = pi/2 -+ asin)
// Polynomials: atan(t) / t in t^2 on [0, 1] (degree 7) and (asin(w) - w) / w^3 in w^2 on [0, 0.5] (degree 4, the
// upper half through asin(w) = pi/2 - 2 asin(sqrt((1 - w) / 2))); max error 1.8e-7 / 1.6e-7 rad in float32
// arithmetic (tests/test_host_math.py), i.e. the same 1e-7 level as atan2f / acosf on float32 inputs.
SF_HD float shot_azimuth_fast(const ShotDecision& d) {
  const float ax = fabsf(d.fx), ay = fabsf(d.fy);
  const float hi = fmaxf(ax, ay), lo = fminf(ax, ay);
  if (d.saz == 0) return 0.0f;
  if (!(hi > 0.0f)) return 0.5f;  // on the frame's z axis: theta = atan2(0, 0) = 0 in octant 0, offset clipped to 0.5
  const float t = sf_divf(lo, hi), s = t * t;
  float p = -0.004668773151934147f;
  p = fmaf(p, s, 0.02416618913412094f);
  p = fmaf(p, s, -0.0593671016395092f);
  p = fmaf(p, s, 0.09906096756458282f);
  p = fmaf(p, s, -0.14016585052013397f);
  p = fmaf(p, s, 0.19969235360622406f);
  p = fmaf(p, s, -0.33331960439682007f);
  p = fmaf(p, s, 0.9999998807907104f);
  return fabsf(fmaf(p * t, 1.27323954473516268615f, -0.5f));
}
SF_HD void shot_elevation_fast(const ShotDecision& d, float& own_vol, float& other_vol) {
  const float w = fabsf(d.ratio);
  const bool big = w > 0.5f;
  const float z = big ? (1.0f - w) * 0.5f : w * w;
  const float r = big ? z * sf_rsqrtf(fmaxf(z, 1e-37f)) : w;
  float p = 0.0382063128054142f;
  p = fmaf(p, z, 0.026494354009628296f);
  p = fmaf(p, z, 0.04501068592071533f);
  p = fmaf(p, z, 0.07498808950185776f);
  p = fmaf(p, z, 0.16666673123836517f);
  const float a = fmaf(r * z, p, r);                                        // asin(r)
  const float g = (big ? fmaf(-2.0f, a, 1.57079632679489661923f) : a) * 0.63661977236758134308f;
  own_vol = 1.0f - fabsf(0.5f - g);
  other_vol = fmaxf(0.0f, 0.5f - g);
}

// What a neighbour contributes, in the form the fast kernel keeps per neighbour: the three target bins, an order key
// that is UNIQUE inside the query (23 bits of rho / radius, then the neighbour's position in the list, < 128) and
// the five values. Two competitors whose distance parts are closer than the kernel's margin make the query
// ambiguous for float32; it is then redone by the float64 kernel.
struct ShotFastRecord {
  uint32_t bins;  // own | cos_nb << 9 | az_nb << 18
  uint32_t key;
  float v_own, v_cos, v_az, v_rad, v_el;
};
constexpr int kFastIndexBits = 7;

SF_HD ShotFastRecord shot_fast_record(const ShotDecision& d, uint32_t index_in_list) {
  ShotFastRecord r;
  r.bins = uint32_t(d.own) | (uint32_t(d.cos_nb) << 9) | (uint32_t(d.az_nb) << 18);
  r.key = 0x80000000u | (d.key << kFastIndexBits) | index_in_list;  // never 0 (0 = nobody)
  float own_vol, other_vol;
  shot_elevation_fast(d, own_vol, other_vol);
  const float a_az = shot_azimuth_fast(d);
  r.v_own = (1.0f - d.a_cos) + d.own_shell + own_vol + (1.0f - a_az);
  r.v_cos = d.a_cos;
  r.v_az = a_az;
  r.v_rad = d.other_shell;
  r.v_el = other_vol;
  return r;
}
// Two keys whose distance parts differ by at most `margin` (23-bit units) cannot be ordered by float32.
SF_HD bool shot_keys_ambiguous(uint32_t a, uint32_t b, uint32_t margin) {
  const uint32_t x = (a >> kFastIndexBits) & 0x7FFFFFu, y = (b >> kFastIndexBits) & 0x7FFFFFu;
  return (x > y ? x - y : y - x) <= margin;
}

// ---- winner tables, compact form (what the kernel uses) -----------------------------------------------------------
// The seven statement groups need only THREE winner decisions per neighbour: the four statements that address the
// neighbour's own bin share one winner, and so do the radial / elevation "other bin" statements, because every
// neighbour of own bin b addresses the same radial partner b^1 (and elevation partner b^2): the winner of the slot
// "radial statement, bins {b, b^1}" is whichever of the two own-bin winners is farther, and it contributes its
// `other_shell` weight to the bin it is NOT in (0 to its own). So per query:
//   keys  uint64 [3][352] : order key (shot_order_key) of the winner of {own-bin group, statement 1, statement 9},
//                           0 = nobody
//   vals  float  [5][352] : v_own, v_rad (other_shell), v_el (other_vol) of the own-bin winner; v_cos; v_az
// Keys are raised with a native 64-bit atomicMax; after a barrier the lane whose key is (still) the slot's key stores
// its values. The key is the 32-bit distance key, then the neighbour's position in the query's list: keys are unique
// inside a query, so two neighbours at the same distance (exact ties, or distances within radius * 2^-32) cannot both
// win a slot, and the later one in the list wins whatever the schedule — every run and every thread count gives the
// same row. (The reference breaks such ties by its unstable argsort: the tie itself stays an exemption, DESIGN.md §2.)
SF_HD uint64_t shot_order_key(uint32_t distance_key, uint32_t position) {
  return (uint64_t(distance_key) << 32) | position;
}
constexpr int kKeyOwn = 0, kKeyCos = kShotLen, kKeyAz = 2 * kShotLen, kKeyCount = 3 * kShotLen;
constexpr int kValOwn = 0, kValRad = kShotLen, kValEl = 2 * kShotLen, kValCos = 3 * kShotLen, kValAz = 4 * kShotLen,
              kValCount = 5 * kShotLen;

// The values of a neighbour that holds (still, after the barrier) the key of its own-bin, statement-1 and / or
// statement-9 slot; only a winner pays for the transcendental weights it needs.
SF_HD void shot_store_winner(const ShotDecision& d, bool win_own, bool win_cos, bool win_az, float* vals) {
  float a_az = 0.0f;
  if (win_own || win_az) a_az = shot_azimuth(d);
  if (win_own) {
    float own_vol, other_vol;
    shot_elevation(d, own_vol, other_vol);
    vals[kValOwn + d.own] = (1.0f - d.a_cos) + d.own_shell + own_vol + (1.0f - a_az);
    vals[kValRad + d.own] = d.other_shell;
    vals[kValEl + d.own] = other_vol;
  }
  if (win_cos) vals[kValCos + d.cos_nb] = d.a_cos;
  if (win_az) vals[kValAz + d.az_nb] = a_az;
}

template <typename Key>
SF_HD float shot_bin_value_compact(const Key* keys, const float* vals, int flat) {
  const Key k_own = keys[kKeyOwn + flat];
  float v = k_own ? vals[kValOwn + flat] : 0.0f;
  if (keys[kKeyCos + flat]) v += vals[kValCos + flat];
  if (keys[kKeyAz + flat]) v += vals[kValAz + flat];
  const int radial_partner = flat ^ 1, elevation_partner = flat ^ 2;
  // the partner bin's winner is farther than this bin's (or this bin is empty): it wrote its "other" weight here
  if (keys[kKeyOwn + radial_partner] > k_own) v += vals[kValRad + radial_partner];
  if (keys[kKeyOwn + elevation_partner] > k_own) v += vals[kValEl + elevation_partner];
  return v;
}

// The same assembly for the four bins {4g .. 4g+3} of one (cosine, azimuth) cell at once: their radial / elevation
// partners are inside the group, so a lane needs exactly eight 16-byte table reads (what the kernel does).
template <typename Key>
SF_HD void shot_bin_group_compact(const Key ko[4], const Key kc[4], const Key ka[4], const float vo[4],
                                  const float vr[4], const float ve[4], const float vc[4], const float va[4],
                                  float out[4]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int t = 0; t < 4; ++t) {
    float v = ko[t] ? vo[t] : 0.0f;
    if (kc[t]) v += vc[t];
    if (ka[t]) v += va[t];
    if (ko[t ^ 1] > ko[t]) v += vr[t ^ 1];
    if (ko[t ^ 2] > ko[t]) v += ve[t ^ 2];
    out[t] = v;
  }
}

// ----------------------------------------------------------------------------------------------------------
// FPFH pair features (fpfh.py:47-57), float64. rel = p_j - p_i (dist > 0), u = n_i, nj = n_j.
// ----------------------------------------------------------------------------------------------------------
// `ny`, `nx`: the arguments of theta = atan2(ny, nx); the caller bins theta with fpfh_theta_bin.
SF_HD void fpfh_features_raw(const double rel[3], double dist, const double u[3], const double nj[3], double& alpha,
                             double& phi, double& ny, double& nx) {
  // v = rel x u ; w = u x v   (np.cross: each component is a*b - c*d, products rounded separately)
  const double v0 = add_rn(mul_rn(rel[1], u[2]), -mul_rn(rel[2], u[1]));
  const double v1 = add_rn(mul_rn(rel[2], u[0]), -mul_rn(rel[0], u[2]));
  const double v2 = add_rn(mul_rn(rel[0], u[1]), -mul_rn(rel[1], u[0]));
  const double w0 = add_rn(mul_rn(u[1], v2), -mul_rn(u[2], v1));
  const double w1 = add_rn(mul_rn(u[2], v0), -mul_rn(u[0], v2));
  const double w2 = add_rn(mul_rn(u[0], v1), -mul_rn(u[1], v0));
  alpha = add_rn(add_rn(mul_rn(v0, nj[0]), mul_rn(v1, nj[1])), mul_rn(v2, nj[2]));
  phi = add_rn(add_rn(mul_rn(rel[0], u[0]), mul_rn(rel[1], u[1])), mul_rn(rel[2], u[2])) / dist;
  ny = add_rn(add_rn(mul_rn(nj[0], w0), mul_rn(nj[1], w1)), mul_rn(nj[2], w2));
  nx = add_rn(add_rn(mul_rn(nj[0], u[0]), mul_rn(nj[1], u[1])), mul_rn(nj[2], u[2]));
}

SF_HD void fpfh_features(const double rel[3], double dist, const double u[3], const double nj[3], double& alpha,
                         double& phi, double& theta) {
  double ny, nx;
  fpfh_features_raw(rel, dist, u, nj, alpha, phi, ny, nx);
  theta = atan2(ny, nx);
}

// NumPy histogram bin of `x` for n equal bins with float64 edges e[0..n] (= np.linspace(lo, hi, n + 1)):
// a value on an interior edge goes to the upper bin, e[n] belongs to the last bin, outside -> -1.
SF_HD int histogram_bin(double x, const double* e, int n) {
  if (!(x >= e[0]) || !(x <= e[n])) return -1;  // also drops NaN
  int idx = int((x - e[0]) / (e[n] - e[0]) * n);
  idx = idx < 0 ? 0 : (idx > n - 1 ? n - 1 : idx);
  while (idx > 0 && x < e[idx]) --idx;
  while (idx < n - 1 && x >= e[idx + 1]) ++idx;
  return idx;
}

// The same bin, the first guess taken with a multiplication by `scale` = n / (e[n] - e[0]) instead of a division:
// the two correction loops make the result independent of the guess.
SF_HD int histogram_bin_scaled(double x, const double* e, int n, double scale) {
  if (!(x >= e[0]) || !(x <= e[n])) return -1;
  int idx = int((x - e[0]) * scale);
  idx = idx < 0 ? 0 : (idx > n - 1 ? n - 1 : idx);
  while (idx > 0 && x < e[idx]) --idx;
  while (idx < n - 1 && x >= e[idx + 1]) ++idx;
  return idx;
}

// Bin of theta = atan2(ny, nx) (fpfh.py:57, :72-76 / :84-87). A float64 atan2 costs ~200 instructions per pair and
// only its BIN is used, so the angle is first taken in float32 (error < 1e-6 rad including the rounding of the
// arguments); when that lands at least 1e-5 rad away from every bin edge (and from the ends of the range) the bin
// is decided, otherwise — a few pairs in 100 000 — the float64 angle is computed and binned exactly.
SF_HD int fpfh_theta_bin(double ny, double nx, const double* e, int n, double scale) {
  const float fy = float(ny), fx = float(nx);
  if (fmaxf(fabsf(fy), fabsf(fx)) > 1e-30f) {
    const double pos = (double(atan2f(fy, fx)) - e[0]) * scale;  // in bin widths
    const double margin = 1e-5 * scale;
    if (pos < -margin || pos > double(n) + margin) return -1;  // safely outside [e[0], e[n]]
    const double cell = floor(pos);
    if (pos > margin && pos < double(n) - margin && pos - cell > margin && cell + 1.0 - pos > margin) return int(cell);
  }
  return histogram_bin_scaled(atan2(ny, nx), e, n, scale);
}

// ----------------------------------------------------------------------------------------------------------
// The three SPFH bins of one pair, float32-filtered. Only the BINS of (alpha, phi, theta) are used, and a bin is
// 1/n of the feature's range wide, so the features are first evaluated in float32 from the float32 roundings of
// rel = p_j - p_i (formed in float64), u and n_j, together with a bound on how far the float32 value can be from
// the reference's float64 value; a bin is accepted only when the value keeps that distance (times a safety factor
// of 4) from every edge and from the ends of the range. Otherwise — a few pairs in 100 000 on generic data, every
// pair on degenerate data such as alpha == 0 on an edge — the caller evaluates the exact float64 path.
//
// Error bounds, eps = 2^-24, C = |rel|, U = |u|, N = |n_j| (Euclidean norms), first order, worst case:
//   v = rel x u      each component  <= 4 eps C U   (two roundings of the inputs, product and sum roundings)
//   alpha = v . n_j  <= 7 eps CUN (from v) + eps CUN (n_j) + 3 eps CUN (sum)              <= 16 eps C U N
//   phi = rel.u / d  <= 5 eps U (dot) + 4 eps U (rsqrt, product)                           <= 16 eps U
//   w = u x v        <= 12 eps U^2 C ;  ny = n_j . w <= 16 eps N U^2 C ;  nx = n_j . u <= 5 eps N U
//   theta            <= (err ny + err nx) / hypot(ny, nx)  +  5e-7 (atan2f, 2 ulp at pi)
// The float64 reference carries its own rounding (1e-16 relative): far below these margins.
// ----------------------------------------------------------------------------------------------------------
constexpr int kBinUnsure = -2;

SF_HD float sf_rsqrtf(float x) {
#if defined(__CUDA_ARCH__)
  return rsqrtf(x);
#else
  return 1.0f / sqrtf(x);
#endif
}

// Bin of x in n equal bins over [lo, lo + n / scale] when x is known to `margin` (same units as x); -1 when x is
// safely outside the range; kBinUnsure when an edge or an end of the range is within the margin.
SF_HD int fpfh_bin_fast(float x, float lo, float scale, int n, float margin) {
  const float eps = 5.9604645e-8f;
  const float pos = (x - lo) * scale;                      // in bin widths
  const float mm = margin * scale + 8.0f * eps * float(n);  // + the roundings of lo, the difference and the product
  if (pos < -mm || pos > float(n) + mm) return -1;
  const float cell = floorf(pos), frac = pos - cell;
  if (pos > mm && pos < float(n) - mm && frac > mm && 1.0f - frac > mm) return int(cell);
  return kBinUnsure;  // also NaN
}

// rel, u, nj: float32 roundings; U = |u| in float32. Returns false when any of the three bins is unsure (or the
// pair is too short / too long for float32 — the caller's float64 path then also decides whether d > 0).
SF_HD bool fpfh_bins_fast(const float rel[3], const float u[3], float U, const float nj[3], int n, const float lo[3],
                          const float scale[3], int& ia, int& ip, int& it) {
  const float eps = 5.9604645e-8f;
  const float c2 = rel[0] * rel[0] + rel[1] * rel[1] + rel[2] * rel[2];
  if (!(c2 > 1e-30f && c2 < 1e30f)) return false;
  const float inv_c = sf_rsqrtf(c2), C = c2 * inv_c;
  // |n_j| enters the margins only: max(1, |n_j|^2) >= |n_j| saves the square root (unit normals: 1 + 1e-7)
  const float N = fmaxf(1.0f, nj[0] * nj[0] + nj[1] * nj[1] + nj[2] * nj[2]);
  const float v0 = rel[1] * u[2] - rel[2] * u[1], v1 = rel[2] * u[0] - rel[0] * u[2], v2 = rel[0] * u[1] - rel[1] * u[0];
  const float w0 = u[1] * v2 - u[2] * v1, w1 = u[2] * v0 - u[0] * v2, w2 = u[0] * v1 - u[1] * v0;
  const float alpha = v0 * nj[0] + v1 * nj[1] + v2 * nj[2];
  const float phi = (rel[0] * u[0] + rel[1] * u[1] + rel[2] * u[2]) * inv_c;
  const float ny = nj[0] * w0 + nj[1] * w1 + nj[2] * w2;
  const float nx = nj[0] * u[0] + nj[1] * u[1] + nj[2] * u[2];
  const float r2 = ny * ny + nx * nx;
  if (!(r2 > 1e-30f && r2 < 1e30f)) return false;
  const float NU = N * U, CU = C * U;
  const float m_alpha = 64.0f * eps * CU * N;
  const float m_phi = 64.0f * eps * U;
  const float m_theta = 4.0f * eps * NU * (16.0f * CU + 5.0f) * sf_rsqrtf(r2) + 2e-6f;
  ia = fpfh_bin_fast(alpha, lo[0], scale[0], n, m_alpha);
  ip = fpfh_bin_fast(phi, lo[1], scale[1], n, m_phi);
  it = fpfh_bin_fast(atan2f(ny, nx), lo[2], scale[2], n, m_theta);
  return ia != kBinUnsure && ip != kBinUnsure && it != kBinUnsure;
}

// One pair of the SPFH loop (fpfh.py:47-76): false when the pair is dropped (d == 0), else the three NumPy bins
// (-1 = outside the feature's range). `e` = float64 edges [3][stride], `scale` = n / (e[n] - e[0]) per feature,
// lo32 / scale32 their float32 roundings, u32 / U the float32 rounding of u and its norm (per point, by the caller).
SF_HD bool fpfh_pair_bins(const double rel[3], const double u[3], const float u32[3], float U, const double nj[3], int n,
                          const double* e, int stride, const double scale[3], const float lo32[3],
                          const float scale32[3], bool allow_fast, int& ia, int& ip, int& it) {
  if (allow_fast) {
    const float rel32[3] = {float(rel[0]), float(rel[1]), float(rel[2])};
    const float nj32[3] = {float(nj[0]), float(nj[1]), float(nj[2])};
    if (fpfh_bins_fast(rel32, u32, U, nj32, n, lo32, scale32, ia, ip, it)) return true;
  }
  const double d2 = rdist3(rel[0], rel[1], rel[2]);
  if (!(d2 > 0.0)) return false;
  double alpha, phi, ny, nx;
  fpfh_features_raw(rel, sqrt(d2), u, nj, alpha, phi, ny, nx);
  ia = histogram_bin_scaled(alpha, e, n, scale[0]);
  ip = histogram_bin_scaled(phi, e + stride, n, scale[1]);
  it = fpfh_theta_bin(ny, nx, e + 2 * stride, n, scale[2]);
  return true;
}

}  // namespace sf
