// DSAC* pose solver on sm_100a: RANSAC hypothesis sampling (P3P), soft-inlier scoring, argmax selection and
// iterative PnP refinement of the winner. Re-designed from the behaviour of the reference's CPU/OpenMP/OpenCV
// operator (dsacstar/dsacstar.cpp:66-186, dsacstar/dsacstar_util.h:59-76,135-221,316-446,522-597,684-770).
//
// Kernel 1 (dsac_sample_score_kernel): grid (hypothesis chunks, images); one warp per hypothesis.
//   - the 32 lanes evaluate 32 consecutive *tries* of that hypothesis in parallel (counter-based RNG keyed by
//     (seed, image, hypothesis, try)); the lowest passing try wins, which is exactly the sequential
//     "repeat until the 4 sampled points reproject within the threshold" rule of dsacstar_util.h:158-219;
//   - the warp then scores the hypothesis over all cells (lanes stride the cells, warp-shuffle reduction);
//   - scene coordinates of the image are staged once per CTA in shared memory.
// Kernel 2 (dsac_refine_kernel): one CTA per image: block argmax, then the refinement loop of
//   dsacstar_util.h:522-597 with an in-kernel Levenberg-Marquardt (the algorithm of OpenCV's CvLevMarq that
//   cv::solvePnP(SOLVEPNP_ITERATIVE, useExtrinsicGuess=true) runs: max 20 iterations, eps FLT_EPSILON),
//   block-wide reduction of the normal equations in double, accumulated in the rotation's tangent space and with ONE pass
//   over the inliers per LM iteration (dsac_refine_body.inc).
// Arithmetic: the soft-inlier SCORES are summed in FP32 (11 FFMA + 4 MUFU per hypothesis and cell); every hard decision - the
// 4-point acceptance test of a minimal set, inlier sets, the LM - is taken in double (OpenCV's projectPoints computes in
// double and stores float pixels); no cheirality test (z ? 1/z : 1), as in OpenCV. Not HBM-bound, no tensor cores.
#include <stdlib.h>

#include "common.cuh"

namespace acez {

struct HypRec {
  double R[9];
  double t[3];
  double score;
  int tries;
  int ok;
};

static constexpr int kDsacThreads = 256;
static constexpr int kRefineThreads = 128;   // refinement: one CTA per image, 3-4 CTAs per SM (60x80 maps: 62 KB of shared memory each)
static constexpr int kMaxSmemCells = 16000;  // 3 floats + 1 flag byte per cell must fit in ~200 KB

// ---------------------------------------------------------------- RNG
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// cell (x, y) of draw j for (seed, image, hypothesis, try); x in [0,w), y in [0,h)
__host__ __device__ __forceinline__ void draw_cell(uint64_t seed, int image, int hyp, int tr, int j, int w, int h, int& x,
                                          int& y) {
  uint64_t s = splitmix64(seed);
  s = splitmix64(s ^ (uint64_t)(uint32_t)image);
  s = splitmix64(s ^ (uint64_t)(uint32_t)hyp);
  s = splitmix64(s ^ (uint64_t)(uint32_t)tr);
  const uint64_t r = splitmix64(s + (uint64_t)j);
  x = (int)(((r & 0xffffffffull) * (uint64_t)w) >> 32);
  y = (int)(((r >> 32) * (uint64_t)h) >> 32);
}

// ---------------------------------------------------------------- small linear algebra (double)
__host__ __device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
__host__ __device__ __forceinline__ double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__host__ __device__ __forceinline__ double norm3(const double* a) { return sqrt(dot3(a, a)); }

// axis-angle -> rotation (cv::Rodrigues forward)
__host__ __device__ inline void rodrigues(const double r[3], double R[9]) {
  const double th = norm3(r);
  if (th < 2.220446049250313e-16) {  // DBL_EPSILON, as OpenCV
    R[0] = 1; R[1] = 0; R[2] = 0; R[3] = 0; R[4] = 1; R[5] = 0; R[6] = 0; R[7] = 0; R[8] = 1;
    return;
  }
  const double c = cos(th), s = sin(th), c1 = 1.0 - c, it = 1.0 / th;
  const double x = r[0] * it, y = r[1] * it, z = r[2] * it;
  R[0] = c + c1 * x * x;     R[1] = c1 * x * y - s * z; R[2] = c1 * x * z + s * y;
  R[3] = c1 * x * y + s * z; R[4] = c + c1 * y * y;     R[5] = c1 * y * z - s * x;
  R[6] = c1 * x * z - s * y; R[7] = c1 * y * z + s * x; R[8] = c + c1 * z * z;
}

// rotation -> axis-angle (cv::Rodrigues inverse for an orthonormal input)
__host__ __device__ inline void rodrigues_inv(const double R[9], double r[3]) {
  double rx = R[7] - R[5], ry = R[2] - R[6], rz = R[3] - R[1];
  const double s = sqrt((rx * rx + ry * ry + rz * rz) * 0.25);
  double c = (R[0] + R[4] + R[8] - 1.0) * 0.5;
  c = c > 1.0 ? 1.0 : (c < -1.0 ? -1.0 : c);
  const double th = acos(c);
  if (s < 1e-5) {
    if (c > 0) { r[0] = r[1] = r[2] = 0; return; }
    // theta ~ pi: recover the axis from the symmetric part
    double t0 = sqrt(fmax((R[0] + 1) * 0.5, 0.0));
    double t1 = sqrt(fmax((R[4] + 1) * 0.5, 0.0)) * (R[1] < 0 ? -1.0 : 1.0);
    double t2 = sqrt(fmax((R[8] + 1) * 0.5, 0.0)) * (R[2] < 0 ? -1.0 : 1.0);
    if (fabs(t0) < fabs(t1) && fabs(t0) < fabs(t2) && ((R[5] > 0) != (t1 * t2 > 0))) t2 = -t2;
    const double n = th / sqrt(t0 * t0 + t1 * t1 + t2 * t2);
    r[0] = t0 * n; r[1] = t1 * n; r[2] = t2 * n;
    return;
  }
  const double vth = 0.5 / s * th;
  r[0] = rx * vth; r[1] = ry * vth; r[2] = rz * vth;
}

// ---------------------------------------------------------------- quartic / P3P (Grunert, as in Haralick et al. 1994)
// real roots of x^4 + a x^3 + b x^2 + c x + d via Ferrari's resolvent cubic, polished with Newton steps
__host__ __device__ inline int solve_quartic(double a, double b, double c, double d, double roots[4]) {
  const double a2 = a * a;
  const double p = b - 0.375 * a2;
  const double q = c - 0.5 * a * b + 0.125 * a2 * a;
  const double r = d - 0.25 * a * c + 0.0625 * a2 * b - (3.0 / 256.0) * a2 * a2;
  int n = 0;
  double y[4];
  if (fabs(q) < 1e-14 * (1.0 + fabs(p) + fabs(r))) {
    // biquadratic y^4 + p y^2 + r
    const double disc = p * p - 4 * r;
    if (disc >= 0) {
      const double sd = sqrt(disc);
      const double z1 = 0.5 * (-p + sd), z2 = 0.5 * (-p - sd);
      if (z1 >= 0) { y[n++] = sqrt(z1); y[n++] = -sqrt(z1); }
      if (z2 >= 0) { y[n++] = sqrt(z2); y[n++] = -sqrt(z2); }
    }
  } else {
    // resolvent cubic z^3 + 2p z^2 + (p^2 - 4r) z - q^2 = 0 has a positive real root
    const double A = 2 * p, B = p * p - 4 * r, C = -q * q;
    const double Q = (3 * B - A * A) / 9.0, Rr = (9 * A * B - 27 * C - 2 * A * A * A) / 54.0;
    const double D = Q * Q * Q + Rr * Rr;
    double z0;
    if (D >= 0) {
      const double sD = sqrt(D);
      z0 = cbrt(Rr + sD) + cbrt(Rr - sD) - A / 3.0;
    } else {
      const double th = acos(fmax(-1.0, fmin(1.0, Rr / sqrt(-Q * Q * Q))));
      const double m = 2 * sqrt(-Q);
      const double z1 = m * cos(th / 3.0) - A / 3.0;
      const double z2 = m * cos((th + 2 * 3.14159265358979323846) / 3.0) - A / 3.0;
      const double z3 = m * cos((th + 4 * 3.14159265358979323846) / 3.0) - A / 3.0;
      z0 = fmax(z1, fmax(z2, z3));
    }
    // one Newton polish of the cubic root
    for (int it = 0; it < 2; ++it) {
      const double fz = ((z0 + A) * z0 + B) * z0 + C, dfz = (3 * z0 + 2 * A) * z0 + B;
      if (dfz != 0) z0 -= fz / dfz;
    }
    if (z0 > 0) {
      const double sz = sqrt(z0);
      // y^2 + sz y + (p + z0 - q/sz)/2 = 0  and  y^2 - sz y + (p + z0 + q/sz)/2 = 0
      const double e1 = 0.5 * (p + z0 - q / sz), e2 = 0.5 * (p + z0 + q / sz);
      const double d1 = z0 - 4 * e1, d2 = z0 - 4 * e2;
      if (d1 >= 0) { const double s1 = sqrt(d1); y[n++] = 0.5 * (-sz + s1); y[n++] = 0.5 * (-sz - s1); }
      if (d2 >= 0) { const double s2 = sqrt(d2); y[n++] = 0.5 * (sz + s2); y[n++] = 0.5 * (sz - s2); }
    }
  }
  for (int i = 0; i < n; ++i) {
    double x = y[i] - 0.25 * a;
    for (int it = 0; it < 3; ++it) {  // Newton on the original quartic
      const double f = (((x + a) * x + b) * x + c) * x + d;
      const double df = ((4 * x + 3 * a) * x + 2 * b) * x + c;
      if (df == 0) break;
      x -= f / df;
    }
    roots[i] = x;
  }
  return n;
}

// Up to 4 poses (R, t scene->camera) from 3 correspondences: Pw world points, fb unit bearing vectors.
__host__ __device__ inline int p3p_grunert(const double Pw[3][3], const double fb[3][3], double Rs[4][9], double ts[4][3]) {
  double d12[3], d13[3], d23[3];
  for (int i = 0; i < 3; ++i) { d12[i] = Pw[1][i] - Pw[0][i]; d13[i] = Pw[2][i] - Pw[0][i]; d23[i] = Pw[2][i] - Pw[1][i]; }
  const double a2 = dot3(d23, d23), b2 = dot3(d13, d13), c2 = dot3(d12, d12);
  if (!(a2 > 0) || !(b2 > 0) || !(c2 > 0)) return 0;  // repeated point
  const double ca = dot3(fb[1], fb[2]), cb = dot3(fb[0], fb[2]), cg = dot3(fb[0], fb[1]);
  const double q = (a2 - c2) / b2, ac = (a2 + c2) / b2;
  const double A4 = (q - 1) * (q - 1) - 4 * c2 / b2 * ca * ca;
  const double A3 = 4 * (q * (1 - q) * cb - (1 - ac) * ca * cg + 2 * c2 / b2 * ca * ca * cb);
  const double A2 = 2 * (q * q - 1 + 2 * q * q * cb * cb + 2 * (b2 - c2) / b2 * ca * ca - 4 * ac * ca * cb * cg +
                         2 * (b2 - a2) / b2 * cg * cg);
  const double A1 = 4 * (-q * (1 + q) * cb + 2 * a2 / b2 * cg * cg * cb - (1 - ac) * ca * cg);
  const double A0 = (1 + q) * (1 + q) - 4 * a2 / b2 * cg * cg;
  double v[4];
  int nr;
  if (fabs(A4) < 1e-14) return 0;
  nr = solve_quartic(A3 / A4, A2 / A4, A1 / A4, A0 / A4, v);
  // world-side orthonormal frame of the triangle
  double e1[3], e2[3], e3[3], tmp[3];
  const double n12 = sqrt(c2);
  for (int i = 0; i < 3; ++i) e1[i] = d12[i] / n12;
  cross3(e1, d13, tmp);
  const double nt = norm3(tmp);
  if (!(nt > 1e-12 * sqrt(b2))) return 0;  // collinear
  for (int i = 0; i < 3; ++i) e3[i] = tmp[i] / nt;
  cross3(e3, e1, e2);
  int ns = 0;
  for (int k = 0; k < nr; ++k) {
    const double vv = v[k];
    if (!(vv > 0) || !isfinite(vv)) continue;
    const double den = 2 * (cg - vv * ca);
    if (fabs(den) < 1e-14) continue;
    const double u = ((q - 1) * vv * vv - 2 * q * cb * vv + 1 + q) / den;
    if (!(u > 0)) continue;
    const double s1sq = c2 / (1 + u * u - 2 * u * cg);
    if (!(s1sq > 0)) continue;
    const double s1 = sqrt(s1sq), s2 = u * s1, s3 = vv * s1;
    double C1[3], C2[3], C3[3];
    for (int i = 0; i < 3; ++i) { C1[i] = s1 * fb[0][i]; C2[i] = s2 * fb[1][i]; C3[i] = s3 * fb[2][i]; }
    double g1[3], g2[3], g3[3], c12[3], c13[3];
    for (int i = 0; i < 3; ++i) { c12[i] = C2[i] - C1[i]; c13[i] = C3[i] - C1[i]; }
    const double m12 = norm3(c12);
    if (!(m12 > 0)) continue;
    for (int i = 0; i < 3; ++i) g1[i] = c12[i] / m12;
    cross3(g1, c13, tmp);
    const double mt = norm3(tmp);
    if (!(mt > 0)) continue;
    for (int i = 0; i < 3; ++i) g3[i] = tmp[i] / mt;
    cross3(g3, g1, g2);
    // R = [g1 g2 g3] [e1 e2 e3]^T
    double* R = Rs[ns];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) R[i * 3 + j] = g1[i] * e1[j] + g2[i] * e2[j] + g3[i] * e3[j];
    for (int i = 0; i < 3; ++i) ts[ns][i] = C1[i] - (R[i * 3] * Pw[0][0] + R[i * 3 + 1] * Pw[0][1] + R[i * 3 + 2] * Pw[0][2]);
    ++ns;
  }
  return ns;
}

// cv::projectPoints for one point: double arithmetic, float pixel out, no cheirality test
__device__ __forceinline__ void project_pt(const double R[9], const double t[3], double X, double Y, double Z, double f,
                                           double cx, double cy, float& u, float& v) {
  const double x = R[0] * X + R[1] * Y + R[2] * Z + t[0];
  const double y = R[3] * X + R[4] * Y + R[5] * Z + t[1];
  double z = R[6] * X + R[7] * Y + R[8] * Z + t[2];
  z = z ? 1.0 / z : 1.0;
  u = (float)(x * z * f + cx);
  v = (float)(y * z * f + cy);
}
// reprojection error as dsacstar_util.h:437-443: float pixel difference, double norm, float result
__device__ __forceinline__ float repro_err(float px, float py, float u, float v, float max_reproj) {
  const float dx = px - u, dy = py - v;
  const float e = (float)sqrt((double)dx * dx + (double)dy * dy);
  return fminf(e, max_reproj);  // non-finite -> max_reproj (documented divergence: the reference propagates NaN)
}

struct DsacArgs {
  const float* sc;
  int n, h, w;
  const float* focal; const float* ppx; const float* ppy;
  acez_dsac_params p;
  const int* injected;
  HypRec* ws;
  float* out_pose;
  int* out_inliers;
  acez_dsac_debug dbg;
  int stage_smem;
};

// stage the image's scene coordinates (3 planes) into shared memory. The kernels index the `extern __shared__` array itself
// afterwards (a pointer that may be global OR shared compiles to generic LD.E in the scoring loop)
__device__ __forceinline__ void stage_sc(const DsacArgs& a, int img, float* smem, int cells) {
  const float* g = a.sc + (size_t)img * 3 * cells;
  for (int i = threadIdx.x; i < 3 * cells; i += blockDim.x) smem[i] = __ldg(g + i);
  __syncthreads();
}

// ---------------------------------------------------------------- kernel 1: sample + score
__global__ void __launch_bounds__(kDsacThreads) dsac_sample_score_kernel(const DsacArgs a) {
#include "dsac_sample_body.inc"
}

// ---------------------------------------------------------------- kernel 2: select + refine
// dR/dr_i for the Rodrigues map (Gallego & Yezzi 2015): dR/dr_i = ([r]x r_i + [r x (I - R) e_i]x) R / |r|^2
__host__ __device__ inline void rodrigues_jac(const double r[3], const double R[9], double dR[3][9]) {
  const double th2 = dot3(r, r);
  if (th2 < 1e-24) {
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 9; ++k) dR[i][k] = 0;
    dR[0][5] = -1; dR[0][7] = 1;   // [e_x]x
    dR[1][2] = 1;  dR[1][6] = -1;  // [e_y]x
    dR[2][1] = -1; dR[2][3] = 1;   // [e_z]x
    return;
  }
  for (int i = 0; i < 3; ++i) {
    double ImR_e[3] = {(i == 0) - R[0 * 3 + i], (i == 1) - R[1 * 3 + i], (i == 2) - R[2 * 3 + i]};
    double w[3];
    cross3(r, ImR_e, w);
    // S = [r]x r_i + [w]x
    const double sx = r[0] * r[i] + w[0], sy = r[1] * r[i] + w[1], sz = r[2] * r[i] + w[2];
    const double S[9] = {0, -sz, sy, sz, 0, -sx, -sy, sx, 0};
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b)
        dR[i][a * 3 + b] = (S[a * 3] * R[b] + S[a * 3 + 1] * R[3 + b] + S[a * 3 + 2] * R[6 + b]) / th2;
  }
}

// 6x6 SPD solve with partial-pivot Gaussian elimination (double); returns false on a singular system
__host__ __device__ inline bool solve6(double A[6][6], double b[6], double x[6]) {
  for (int c = 0; c < 6; ++c) {
    int piv = c;
    double mx = fabs(A[c][c]);
    for (int r = c + 1; r < 6; ++r)
      if (fabs(A[r][c]) > mx) { mx = fabs(A[r][c]); piv = r; }
    if (!(mx > 0) || !isfinite(mx)) return false;
    if (piv != c) {
      for (int k = 0; k < 6; ++k) { const double tmp = A[c][k]; A[c][k] = A[piv][k]; A[piv][k] = tmp; }
      const double tb = b[c]; b[c] = b[piv]; b[piv] = tb;
    }
    for (int r = c + 1; r < 6; ++r) {
      const double m = A[r][c] / A[c][c];
      for (int k = c; k < 6; ++k) A[r][k] -= m * A[c][k];
      b[r] -= m * b[c];
    }
  }
  for (int r = 5; r >= 0; --r) {
    double s = b[r];
    for (int k = r + 1; k < 6; ++k) s -= A[r][k] * x[k];
    x[r] = s / A[r][r];
  }
  return true;
}

// block-wide sum of `cnt` doubles per thread into smem result (all threads get the totals through smem)
template <int CNT>
__device__ void block_sum(double (&v)[CNT], double* s_part /*[warps][CNT]*/, double* s_out /*[CNT]*/) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < CNT; ++k) v[k] = warp_sum(v[k]);
  __syncthreads();  // previous consumers of s_part / s_out are done
  if (lane == 0)
    for (int k = 0; k < CNT; ++k) s_part[warp * CNT + k] = v[k];
  __syncthreads();
  if (threadIdx.x < CNT) {
    double t = 0;
    for (int w = 0; w < warps; ++w) t += s_part[w * CNT + threadIdx.x];
    s_out[threadIdx.x] = t;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kRefineThreads, 3) dsac_refine_kernel(const DsacArgs a) {
#include "dsac_refine_body.inc"
}

}  // namespace acez

using namespace acez;

extern "C" size_t acez_dsac_workspace_bytes(int n, int h, int w, int hyps) {
  (void)h; (void)w;
  if (n < 0 || hyps < 0) return 0;
  return (size_t)n * (size_t)hyps * sizeof(HypRec) + 256;
}

extern "C" int acez_dsac_forward_rgb_batch(const float* sc, int n, int h, int w, const float* focal, const float* ppx,
                                           const float* ppy, const acez_dsac_params* p, const int* injected_idx,
                                           float* out_pose, int* out_inliers, const acez_dsac_debug* dbg,
                                           void* workspace, size_t workspace_bytes, acez_stream_t stream) {
  ACEZ_REQUIRE(sc && focal && ppx && ppy && p && out_pose && out_inliers && workspace, "dsac: null argument");
  ACEZ_REQUIRE(n >= 0 && h > 0 && w > 0, "dsac: bad shape n=%d h=%d w=%d", n, h, w);
  ACEZ_REQUIRE(p->hyps >= 1 && p->hyps <= (1 << 20), "dsac: hyps=%d out of range", p->hyps);
  ACEZ_REQUIRE(p->inlier_threshold > 0 && p->subsample >= 1, "dsac: bad threshold / subsample");
  ACEZ_REQUIRE(workspace_bytes >= acez_dsac_workspace_bytes(n, h, w, p->hyps), "dsac: workspace too small");
  int rc = acez_device_check();
  if (rc) return rc;
  if (n == 0) return ACEZ_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  DsacArgs a{};
  a.sc = sc; a.n = n; a.h = h; a.w = w;
  a.focal = focal; a.ppx = ppx; a.ppy = ppy;
  a.p = *p;
  a.injected = injected_idx;
  a.ws = reinterpret_cast<HypRec*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  a.out_pose = out_pose;
  a.out_inliers = out_inliers;
  if (dbg) a.dbg = *dbg;
  const int cells = h * w;
  ACEZ_REQUIRE(cells <= kMaxSmemCells, "dsac: %d cells exceed the shared-memory staging budget (%d)", cells, kMaxSmemCells);
  a.stage_smem = 1;
  const size_t smem1 = (size_t)cells * 12;
  const size_t smem2 = smem1 + (size_t)cells * 2;
  if ((rc = set_max_dynamic_smem<dsac_sample_score_kernel>(200 * 1024))) return rc;
  if ((rc = set_max_dynamic_smem<dsac_refine_kernel>(224 * 1024))) return rc;
  ACEZ_REQUIRE(smem2 <= 224 * 1024, "dsac: %d cells exceed the refinement kernel's shared-memory budget", cells);
  const int warps = kDsacThreads / 32;
  // enough CTAs per image to fill the GPU when n is small; one chunk of 8 hypotheses per CTA pass
  int chunks = (p->hyps + warps - 1) / warps;
  const int want = (2 * sm_count() + n - 1) / n;
  if (chunks > want) chunks = want < 1 ? 1 : want;
  dim3 grid1(chunks, n);
  dsac_sample_score_kernel<<<grid1, kDsacThreads, smem1, s>>>(a);
  ACEZ_CUDA(cudaGetLastError());
  dsac_refine_kernel<<<n, kRefineThreads, smem2, s>>>(a);
  ACEZ_CUDA(cudaGetLastError());
  return ACEZ_OK;
}

// ----------------------------------------------------------------------------------------------
// host-callable views of the solver's building blocks (CPU unit tests of the host-compilable math; not a product path)
// ----------------------------------------------------------------------------------------------
extern "C" int acez_host_p3p(const double* Pw9, const double* bearings9, double* Rs36, double* ts12) {
  double Pw[3][3], fb[3][3], Rs[4][9], ts[4][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { Pw[i][j] = Pw9[i * 3 + j]; fb[i][j] = bearings9[i * 3 + j]; }
  const int n = p3p_grunert(Pw, fb, Rs, ts);
  for (int s = 0; s < n; ++s) {
    for (int k = 0; k < 9; ++k) Rs36[s * 9 + k] = Rs[s][k];
    for (int k = 0; k < 3; ++k) ts12[s * 3 + k] = ts[s][k];
  }
  return n;
}
extern "C" void acez_host_draw_cell(uint64_t seed, int image, int hyp, int tr, int j, int w, int h, int* xy) {
  draw_cell(seed, image, hyp, tr, j, w, h, xy[0], xy[1]);
}
extern "C" int acez_host_solve_quartic(const double* abcd, double* roots) {
  return solve_quartic(abcd[0], abcd[1], abcd[2], abcd[3], roots);
}
extern "C" void acez_host_rodrigues(const double* r3, double* R9, double* dR27) {
  rodrigues(r3, R9);
  if (dR27) {
    double dR[3][9];
    rodrigues_jac(r3, R9, dR);
    for (int i = 0; i < 3; ++i)
      for (int k = 0; k < 9; ++k) dR27[i * 9 + k] = dR[i][k];
  }
}
extern "C" void acez_host_rodrigues_inv(const double* R9, double* r3) { rodrigues_inv(R9, r3); }
