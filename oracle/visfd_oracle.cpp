// oracle/visfd_oracle.cpp -- TEST INFRASTRUCTURE ONLY.
//
// CPU restatement (our own code, C-style, flat arrays, 64-bit indices) of the
// reference's algorithm for the filter_mrc membrane/blob hot path.  Each
// function cites the reference file:line whose arithmetic it follows, including
// the reference's mixed float/double/long double evaluation types, so that on
// the same compiler/libm the results are bit-identical to oracle/_ref (the
// reference itself); tests/test_oracle_golden.py pins that, and the committed
// fixtures under tests/golden/ (generated from oracle/_ref by
// tests/golden/make_golden.py) pin it where /root/reference is absent.
//
// It is C-style C++ rather than C for one reason: the only third-party
// arithmetic on the path, libstdc++'s std::cyl_bessel_i(long double,long double)
// (call site lib/visfd/filter1d.hpp:438), is reachable only from C++.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference
// arm may load this library.  The product (visfd_b200/, include/) never does.
//
// Build: oracle/Makefile (g++ -O2 -ffp-contract=off: no FMA contraction, like
// the reference's x86-64 baseline build).

#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <algorithm>
#include <array>
#include <functional>
#include <queue>
#include <tuple>
#include <vector>

typedef int64_t i64;

#define IDX(ix, iy, iz) ((i64(iz) * ny + (iy)) * i64(nx) + (ix))

extern "C" {

int vo_version() { return 1; }

// ---------------------------------------------------------------------------
// Gaussian taps: lib/visfd/filter1d.hpp:411-460 (GenFilterGauss1D<float>)
//   discrete Gaussian kernel exp(-s^2) I_|i|(s^2) when s<=10 and |i|<=20
//   (:436-440), sampled continuous Gaussian otherwise (:441-447), evaluated in
//   long double, stored as float, then divided by the long double sum of the
//   stored floats (:452-457).
// ---------------------------------------------------------------------------
void vo_gen_gauss1d(float sigma, int hw, float *taps /* 2*hw+1, index i+hw */) {
  long double sum = 0.0L;
  for (int i = -hw; i <= hw; i++) {
    float v;
    if (sigma == 0.0f) {
      v = (i == 0) ? 1.0f : 0.0f;
    } else {
      long double S = sigma;
      long double I = i;
      if ((S <= 10.0) && (fabsl(I) <= 20.0)) {
        long double h = expl(-S * S) * std::cyl_bessel_i(fabsl(I), S * S);
        v = (float)h;
      } else {
        v = (float)(expl(-(I * I) / (2.0 * S * S)) / sqrtl(2 * S * S * M_PI));
      }
    }
    taps[i + hw] = v;
    sum += v;
  }
  for (int i = -hw; i <= hw; i++) taps[i + hw] = (float)(taps[i + hw] / sum);
}

// ---------------------------------------------------------------------------
// 1-D convolution along one line: lib/visfd/filter1d.hpp:47-104 (plain) and
// :204-295 (mask + denominator).  g[i] = sum_{j=-hw..hw, 0<=i-j<n} h[j]*f[i-j],
// j ascending, float multiply then float add.  The reference's "sparse input"
// skip (:59-94, :219-256) only short-cuts windows whose data (or mask) are all
// zero, where the sum is 0 anyway, so it is not restated.
// ---------------------------------------------------------------------------
static void conv_line(const float *h /*centre*/, int hw, i64 n, const float *f,
                      i64 fstride, float *g) {
  for (i64 i = 0; i < n; i++) {
    float acc = 0.0f;
    for (int j = -hw; j <= hw; j++) {
      i64 k = i - j;
      if (k < 0 || k >= n) continue;
      acc += h[j] * f[k * fstride];
    }
    g[i] = acc;
  }
}
static void conv_line_masked(const float *h, int hw, i64 n, const float *f,
                             const float *m, i64 stride, float *g, float *d) {
  for (i64 i = 0; i < n; i++) {
    float acc = 0.0f, den = 0.0f;
    for (int j = -hw; j <= hw; j++) {
      i64 k = i - j;
      if (k < 0 || k >= n) continue;
      float fv = h[j];
      fv *= m[k * stride];           // filter1d.hpp:273-275
      float dg = fv * f[k * stride]; // :281
      acc += dg;
      den += fv;                     // :285-286
    }
    g[i] = acc;
    d[i] = den;
  }
}

// ---------------------------------------------------------------------------
// Separable filter: lib/visfd/filter3d.hpp:688-1050 (ApplySeparable<float>).
// Sweep order Z, Y, X (:741-981).  With a mask the Z sweep filters mask*src and
// the mask (:799-803); Y and X sweeps filter both volumes (:868-879, :948-959);
// normalisation divides by the 3-D denominator where it is >0 (:986-992).
// Without a mask normalisation divides by dx[ix]*dy[iy]*dz[iz], the 1-D
// responses to an all-ones line (:1004-1022).  Returns h_x[0]*h_y[0]*h_z[0].
// taps[d] points at 2*hw[d]+1 floats (index i+hw), d = 0:x 1:y 2:z.
// ---------------------------------------------------------------------------
float vo_apply_separable(i64 nx, i64 ny, i64 nz, const float *src, float *dst,
                         const float *mask, const float *const taps[3],
                         const int hw[3], int normalize) {
  i64 N = nx * ny * nz;
  memcpy(dst, src, N * sizeof(float));
  std::vector<float> denom;
  bool use_denom = normalize && mask;
  if (use_denom) denom.assign(N, 1.0f);
  const float *hx = taps[0] + hw[0], *hy = taps[1] + hw[1], *hz = taps[2] + hw[2];
  i64 sy = nx, sz = nx * ny;

  // Z sweep
#pragma omp parallel
  {
    std::vector<float> line(nz), out(nz), mline(mask ? nz : 0), dline(nz);
#pragma omp for collapse(2)
    for (i64 iy = 0; iy < ny; iy++)
      for (i64 ix = 0; ix < nx; ix++) {
        i64 o = iy * sy + ix;
        for (i64 iz = 0; iz < nz; iz++) line[iz] = dst[o + iz * sz];
        if (mask) {
          for (i64 iz = 0; iz < nz; iz++) mline[iz] = mask[o + iz * sz];
          conv_line_masked(hz, hw[2], nz, line.data(), mline.data(), 1,
                           out.data(), dline.data());
        } else {
          conv_line(hz, hw[2], nz, line.data(), 1, out.data());
        }
        for (i64 iz = 0; iz < nz; iz++) {
          dst[o + iz * sz] = out[iz];
          if (use_denom) denom[o + iz * sz] = dline[iz];
        }
      }
  }
  // Y sweep
#pragma omp parallel
  {
    std::vector<float> line(ny), out(ny);
#pragma omp for collapse(2)
    for (i64 iz = 0; iz < nz; iz++)
      for (i64 ix = 0; ix < nx; ix++) {
        i64 o = iz * sz + ix;
        for (i64 iy = 0; iy < ny; iy++) line[iy] = dst[o + iy * sy];
        conv_line(hy, hw[1], ny, line.data(), 1, out.data());
        for (i64 iy = 0; iy < ny; iy++) dst[o + iy * sy] = out[iy];
        if (use_denom) {
          for (i64 iy = 0; iy < ny; iy++) line[iy] = denom[o + iy * sy];
          conv_line(hy, hw[1], ny, line.data(), 1, out.data());
          for (i64 iy = 0; iy < ny; iy++) denom[o + iy * sy] = out[iy];
        }
      }
  }
  // X sweep
#pragma omp parallel
  {
    std::vector<float> line(nx), out(nx);
#pragma omp for collapse(2)
    for (i64 iz = 0; iz < nz; iz++)
      for (i64 iy = 0; iy < ny; iy++) {
        i64 o = iz * sz + iy * sy;
        for (i64 ix = 0; ix < nx; ix++) line[ix] = dst[o + ix];
        conv_line(hx, hw[0], nx, line.data(), 1, out.data());
        for (i64 ix = 0; ix < nx; ix++) dst[o + ix] = out[ix];
        if (use_denom) {
          for (i64 ix = 0; ix < nx; ix++) line[ix] = denom[o + ix];
          conv_line(hx, hw[0], nx, line.data(), 1, out.data());
          for (i64 ix = 0; ix < nx; ix++) denom[o + ix] = out[ix];
        }
      }
  }
  if (normalize) {
    if (mask) {
      for (i64 i = 0; i < N; i++)
        if (denom[i] > 0.0f) dst[i] /= denom[i];
    } else {
      std::vector<float> ones, d[3];
      i64 n[3] = {nx, ny, nz};
      const float *h[3] = {hx, hy, hz};
      for (int a = 0; a < 3; a++) {
        ones.assign(n[a], 1.0f);
        d[a].resize(n[a]);
        conv_line(h[a], hw[a], n[a], ones.data(), 1, d[a].data());
      }
      for (i64 iz = 0; iz < nz; iz++)
        for (i64 iy = 0; iy < ny; iy++)
          for (i64 ix = 0; ix < nx; ix++) {
            float den = d[0][ix] * d[1][iy] * d[2][iz]; // filter3d.hpp:1016-1018
            dst[IDX(ix, iy, iz)] /= den;
          }
    }
  }
  return hx[0] * hy[0] * hz[0]; // filter3d.hpp:1044-1046
}

// lib/visfd/filter3d.hpp:1088-1124 (ApplyGauss with explicit halfwidths)
float vo_apply_gauss(i64 nx, i64 ny, i64 nz, const float *src, float *dst,
                     const float *mask, const float sigma[3], const int hw[3],
                     int normalize) {
  std::vector<float> t[3];
  const float *tp[3];
  for (int d = 0; d < 3; d++) {
    t[d].resize(2 * hw[d] + 1);
    vo_gen_gauss1d(sigma[d], hw[d], t[d].data());
    tp[d] = t[d].data();
  }
  return vo_apply_separable(nx, ny, nz, src, dst, mask, tp, hw, normalize);
}

// halfwidth rule of lib/visfd/filter3d.hpp:1241-1246: max(1, floor(sigma*ratio))
// and of bin/filter_mrc/filter3d_variants.hpp:500-528: a non-positive ratio
// means ratio = sqrt(-2 ln threshold).
int vo_gauss_halfwidth(float sigma, float truncate_ratio,
                       float truncate_threshold) {
  if (truncate_ratio <= 0)
    truncate_ratio = sqrt(-2 * log(truncate_threshold)); // float <- double
  int hw = floor(sigma * truncate_ratio);
  if (hw < 1) hw = 1;
  return hw;
}

// lib/visfd/filter3d.hpp:1340-1402 (ApplyDog): G_a(src) - G_b(src), both
// normalised (:1373,:1383), same halfwidths.
void vo_apply_dog(i64 nx, i64 ny, i64 nz, const float *src, float *dst,
                  const float *mask, const float sigma_a[3],
                  const float sigma_b[3], const int hw[3], float *pA, float *pB) {
  i64 N = nx * ny * nz;
  std::vector<float> tmp(N);
  float A = vo_apply_gauss(nx, ny, nz, src, dst, mask, sigma_a, hw, 1);
  float B = vo_apply_gauss(nx, ny, nz, src, tmp.data(), mask, sigma_b, hw, 1);
  for (i64 i = 0; i < N; i++) dst[i] -= tmp[i];
  if (pA) *pA = A;
  if (pB) *pB = B;
}

// lib/visfd/filter3d.hpp:1430-1507 (ApplyLog): sigma(1 -/+ delta/2) evaluated
// in double and stored as float (:1453-1458), shared halfwidth
// floor(ratio*max(sigma_a,sigma_b)) (:1460-1464), result *= 1/delta^2 (:1493).
void vo_log_params(const float sigma[3], float delta, float truncate_ratio,
                   float sigma_a[3], float sigma_b[3], int hw[3], float *scale) {
  for (int d = 0; d < 3; d++) {
    sigma_a[d] = (float)(sigma[d] * (1.0 - 0.5 * delta));
    sigma_b[d] = (float)(sigma[d] * (1.0 + 0.5 * delta));
    hw[d] = floor(truncate_ratio * std::max(sigma_a[d], sigma_b[d]));
  }
  *scale = (float)(1.0 / (delta * delta)); // SQR(float) is float; 1.0/float -> double -> float
}
void vo_apply_log(i64 nx, i64 ny, i64 nz, const float *src, float *dst,
                  const float *mask, const float sigma[3], float delta,
                  float truncate_ratio, float *pA, float *pB) {
  float sa[3], sb[3], scale;
  int hw[3];
  vo_log_params(sigma, delta, truncate_ratio, sa, sb, hw, &scale);
  vo_apply_dog(nx, ny, nz, src, dst, mask, sa, sb, hw, pA, pB);
  i64 N = nx * ny * nz;
  for (i64 i = 0; i < N; i++) dst[i] *= scale;
  if (pA) *pA *= scale;
  if (pB) *pB *= scale;
}

// ---------------------------------------------------------------------------
// Finite differences on the smoothed image:
//   lib/visfd/visfd_utils.hpp:530-565 (19-point Hessian), :579-616 (stencil
//   centre clamped to [1,n-2]), :631-669 (central-difference gradient);
//   scaled by sigma / sigma^2 in lib/visfd/feature.hpp:1289-1291, :1331-1333.
// Outputs: grad[N][3], hess[N][6] in flat order xx,yy,zz,xy,yz,xz
//   (lib/visfd/lin3_utils.hpp:400-406).  Voxels with mask==0 are skipped.
// ---------------------------------------------------------------------------
void vo_hessian_fd(i64 nx, i64 ny, i64 nz, const float *sm, const float *mask,
                   float sigma, float *grad, float *hess) {
  float s2 = sigma * sigma;
#pragma omp parallel for collapse(2)
  for (i64 iz = 0; iz < nz; iz++)
    for (i64 iy = 0; iy < ny; iy++)
      for (i64 ix = 0; ix < nx; ix++) {
        i64 i = IDX(ix, iy, iz);
        if (mask && mask[i] == 0.0f) continue;
        i64 x = ix, y = iy, z = iz;
        if (x == 0) x++; else if (x == nx - 1) x--;
        if (y == 0) y++; else if (y == ny - 1) y--;
        if (z == 0) z++; else if (z == nz - 1) z--;
#define F(dx, dy, dz) sm[IDX(x + (dx), y + (dy), z + (dz))]
        float c = F(0, 0, 0);
        if (grad) {
          grad[3 * i + 0] = (0.5f * (F(1, 0, 0) - F(-1, 0, 0))) * sigma;
          grad[3 * i + 1] = (0.5f * (F(0, 1, 0) - F(0, -1, 0))) * sigma;
          grad[3 * i + 2] = (0.5f * (F(0, 0, 1) - F(0, 0, -1))) * sigma;
        }
        float hxx = F(1, 0, 0) + F(-1, 0, 0) - 2 * c;
        float hyy = F(0, 1, 0) + F(0, -1, 0) - 2 * c;
        float hzz = F(0, 0, 1) + F(0, 0, -1) - 2 * c;
        float hxy = 0.25f * (F(1, 1, 0) + F(-1, -1, 0) - F(1, -1, 0) - F(-1, 1, 0));
        float hyz = 0.25f * (F(0, 1, 1) + F(0, -1, -1) - F(0, 1, -1) - F(0, -1, 1));
        float hxz = 0.25f * (F(1, 0, 1) + F(-1, 0, -1) - F(-1, 0, 1) - F(1, 0, -1));
#undef F
        hess[6 * i + 0] = hxx * s2;
        hess[6 * i + 1] = hyy * s2;
        hess[6 * i + 2] = hzz * s2;
        hess[6 * i + 3] = hxy * s2;
        hess[6 * i + 4] = hyz * s2;
        hess[6 * i + 5] = hxz * s2;
      }
}

// lib/visfd/feature.hpp:1210-1348 (CalcHessian): normalised Gaussian with
// hw = floor(sigma*ratio) (:1223, :1248-1255), then the stencils above.
// Returns 1 if any dimension < 3 (the reference throws, :1260-1264).
int vo_calc_hessian(i64 nx, i64 ny, i64 nz, const float *src, const float *mask,
                    float sigma, float truncate_ratio, float *grad, float *hess,
                    float *smoothed_out /* optional */) {
  int h = floor(sigma * truncate_ratio);
  float sg[3] = {sigma, sigma, sigma};
  int hw[3] = {h, h, h};
  std::vector<float> sm(nx * ny * nz);
  vo_apply_gauss(nx, ny, nz, src, sm.data(), mask, sg, hw, 1);
  if (smoothed_out) memcpy(smoothed_out, sm.data(), sm.size() * sizeof(float));
  if (nx < 3 || ny < 3 || nz < 3) return 1;
  vo_hessian_fd(nx, ny, nz, sm.data(), mask, sigma, grad, hess);
  return 0;
}

// ---------------------------------------------------------------------------
// 3x3 symmetric eigensolver in double:
//   lib/visfd/eigen3_simple.hpp:49-82 (computeRoots3: trigonometric closed
//   form on the shifted+scaled matrix), :88-133 (extract_kernel3: eigenvector
//   as the larger cross product of columns of A - lambda I), :139-266
//   (DiagonalizeSym3: shift by trace/3, scale by max|a_ij|, most-distinct
//   eigenvalue first, degenerate branches, swap of first/last for the requested
//   order).  order: 0 = INCREASING_EIVALS, 1 = DECREASING_EIVALS.
// ---------------------------------------------------------------------------
static void cross3(const double a[3], const double b[3], double c[3]) {
  c[2] = a[0] * b[1] - a[1] * b[0];
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
}
static double dot3(const double a[3], const double b[3]) {
  return a[0] * b[0] + a[1] * b[1] + a[2] * b[2];
}
static void normalize3(double a[3]) { // lin3_utils.hpp:142-155
  double L = std::sqrt(dot3(a, a));
  if (L > 0.0) {
    L = 1.0 / L;
    for (int d = 0; d < 3; d++) a[d] *= L;
  } else {
    a[0] = 1.0; a[1] = 0.0; a[2] = 0.0;
  }
}
static void roots3(const double m[3][3], double roots[3]) {
  const double inv3 = 1.0 / 3.0;
  const double sqrt3 = std::sqrt(3.0);
  double c0 = m[0][0] * m[1][1] * m[2][2] + 2.0 * m[1][0] * m[2][0] * m[2][1] -
              m[0][0] * m[2][1] * m[2][1] - m[1][1] * m[2][0] * m[2][0] -
              m[2][2] * m[1][0] * m[1][0];
  double c1 = m[0][0] * m[1][1] - m[1][0] * m[1][0] + m[0][0] * m[2][2] -
              m[2][0] * m[2][0] + m[1][1] * m[2][2] - m[2][1] * m[2][1];
  double c2 = m[0][0] + m[1][1] + m[2][2];
  double c2_3 = c2 * inv3;
  double a_3 = (c2 * c2_3 - c1) * inv3;
  a_3 = std::max(a_3, 0.0);
  double half_b = 0.5 * (c0 + c2_3 * (2.0 * c2_3 * c2_3 - c1));
  double q = a_3 * a_3 * a_3 - half_b * half_b;
  q = std::max(q, 0.0);
  double rho = std::sqrt(a_3);
  double theta = std::atan2(std::sqrt(q), half_b) * inv3;
  double ct = std::cos(theta), st = std::sin(theta);
  roots[0] = c2_3 - rho * (ct + sqrt3 * st);
  roots[1] = c2_3 - rho * (ct - sqrt3 * st);
  roots[2] = c2_3 + 2.0 * rho * ct;
}
static void kernel3(const double mat[3][3], double res[3], double rep[3]) {
  int i0 = 0;
  double md = std::fabs(mat[0][0]);
  for (int d = 1; d < 3; d++)
    if (std::fabs(mat[d][d]) > md) { i0 = d; md = std::fabs(mat[d][d]); }
  double col[3][3]; // col[k] = k-th column of mat
  for (int k = 0; k < 3; k++)
    for (int d = 0; d < 3; d++) col[k][d] = mat[d][k];
  for (int d = 0; d < 3; d++) rep[d] = col[i0][d];
  double c0[3], c1[3];
  cross3(rep, col[(i0 + 1) % 3], c0);
  cross3(rep, col[(i0 + 2) % 3], c1);
  double n0 = dot3(c0, c0), n1 = dot3(c1, c1);
  if (n0 > n1) {
    double s = 1.0 / std::sqrt(n0);
    for (int d = 0; d < 3; d++) res[d] = c0[d] * s;
  } else {
    double s = 1.0 / std::sqrt(n1);
    for (int d = 0; d < 3; d++) res[d] = c1[d] * s;
  }
}
void vo_diagonalize_sym3(const double mat[3][3], double ev[3], double evec[3][3],
                         int order) {
  const double EPS = 2.220446049250313e-16;
  double shift = (mat[0][0] + mat[1][1] + mat[2][2]) / 3.0;
  double sm[3][3];
  memcpy(sm, mat, sizeof(sm));
  for (int d = 0; d < 3; d++) sm[d][d] -= shift;
  double scale = -1.0;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++)
      if (std::fabs(sm[i][j]) > scale) scale = std::fabs(sm[i][j]);
  if (scale > 0) {
    double si = 1.0 / scale;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) sm[i][j] *= si;
  }
  roots3(sm, ev);
  if ((ev[2] - ev[0]) <= EPS) {
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) evec[i][j] = (i == j) ? 1.0 : 0.0;
  } else {
    double d0 = ev[2] - ev[1], d1 = ev[1] - ev[0];
    int k = 0, l = 2;
    if (d0 > d1) { d0 = d1; std::swap(k, l); }
    double tmp[3][3];
    memcpy(tmp, sm, sizeof(tmp));
    for (int d = 0; d < 3; d++) tmp[d][d] -= ev[k];
    kernel3(tmp, evec[k], evec[l]);
    if (d0 <= 2 * EPS * d1) {
      // eigen3_simple.hpp:220-223 (sic: subtracts a multiple of itself)
      double kl = dot3(evec[k], evec[l]);
      for (int d = 0; d < 3; d++) evec[l][d] -= kl * evec[l][d];
      normalize3(evec[l]);
    } else {
      memcpy(tmp, sm, sizeof(tmp));
      for (int d = 0; d < 3; d++) tmp[d][d] -= ev[l];
      double dummy[3];
      kernel3(tmp, evec[l], dummy);
    }
    cross3(evec[2], evec[0], evec[1]);
    normalize3(evec[1]);
  }
  for (int d = 0; d < 3; d++) { ev[d] *= scale; ev[d] += shift; }
  if ((order == 0 && ev[0] > ev[2]) || (order == 1 && ev[0] < ev[2])) {
    std::swap(ev[0], ev[2]);
    for (int d = 0; d < 3; d++) std::swap(evec[0][d], evec[2][d]);
  }
}

// lib/visfd/eigen3_simple.hpp:273-342 (DiagonalizeFlatSym3): double solve,
// flip evec[0] if det<0 (:316-319), in-place Transpose3 which swaps every pair
// twice and therefore changes nothing (lin3_utils.hpp:199-203), rotation ->
// quaternion (lin3_utils.hpp:231-269) -> Shoemake coordinates (:344-375),
// stored as 3 floats after the 3 float eigenvalues.
void vo_diagonalize_flat_sym3(const float m6[6], float out6[6], int order) {
  static const int map[3][3] = {{0, 3, 5}, {3, 1, 4}, {5, 4, 2}};
  double M[3][3], ev[3], E[3][3];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) M[i][j] = m6[map[i][j]];
  vo_diagonalize_sym3(M, ev, E, order);
  double v12[3];
  cross3(E[0], E[1], v12);
  if (dot3(E[2], v12) < 0.0)
    for (int d = 0; d < 3; d++) E[0][d] *= -1.0;
  // Matrix2Quaternion
  double S, qw, qx, qy, qz;
  double tr = E[0][0] + E[1][1] + E[2][2];
  if (tr > 0) {
    S = std::sqrt(tr + 1.0) * 2;
    qw = 0.25 * S;
    qx = (E[2][1] - E[1][2]) / S;
    qy = (E[0][2] - E[2][0]) / S;
    qz = (E[1][0] - E[0][1]) / S;
  } else if ((E[0][0] > E[1][1]) && (E[0][0] > E[2][2])) {
    S = std::sqrt(1.0 + E[0][0] - E[1][1] - E[2][2]) * 2;
    qw = (E[2][1] - E[1][2]) / S;
    qx = 0.25 * S;
    qy = (E[0][1] + E[1][0]) / S;
    qz = (E[0][2] + E[2][0]) / S;
  } else if (E[1][1] > E[2][2]) {
    S = std::sqrt(1.0 + E[1][1] - E[0][0] - E[2][2]) * 2;
    qw = (E[0][2] - E[2][0]) / S;
    qx = (E[0][1] + E[1][0]) / S;
    qy = 0.25 * S;
    qz = (E[1][2] + E[2][1]) / S;
  } else {
    S = std::sqrt(1.0 + E[2][2] - E[0][0] - E[1][1]) * 2;
    qw = (E[1][0] - E[0][1]) / S;
    qx = (E[0][2] + E[2][0]) / S;
    qy = (E[1][2] + E[2][1]) / S;
    qz = 0.25 * S;
  }
  // Quaternion2Shoemake with q = {qw,qx,qy,qz}
  const double TWO_PI = 6.283185307179586;
  double r1 = std::sqrt(qw * qw + qx * qx);
  double r2 = std::sqrt(qy * qy + qz * qz);
  double X0 = r2 * r2;
  double th1 = 0.0, th2 = 0.0;
  if (r1 > 0) th1 = std::atan2(qw, qx);
  if (r2 > 0) th2 = std::atan2(qy, qz);
  out6[0] = (float)ev[0];
  out6[1] = (float)ev[1];
  out6[2] = (float)ev[2];
  out6[3] = (float)X0;
  out6[4] = (float)(th1 / TWO_PI);
  out6[5] = (float)(th2 / TWO_PI);
}

// lib/visfd/lin3_utils.hpp:567-584 (ConvertDiagFlatSym2Evects3<float>) ->
// Shoemake2Quaternion<float> (:311-337) -> Quaternion2Matrix<float> (:280-305),
// with the reference's float/double mix (literals 1.0 are double).
void vo_diag_flat_to_evects(const float m6[6], float ev[3], float E[3][3]) {
  ev[0] = m6[0]; ev[1] = m6[1]; ev[2] = m6[2];
  const float TWO_PI = 6.283185307179586;
  float X0 = m6[3], X1 = m6[4], X2 = m6[5];
  float th1 = TWO_PI * X1, th2 = TWO_PI * X2;
  float r1 = (float)std::sqrt(1.0 - X0);
  float r2 = std::sqrt(X0);
  float s1 = std::sin(th1), c1 = std::cos(th1);
  float s2 = std::sin(th2), c2 = std::cos(th2);
  float q[4] = {s1 * r1, c1 * r1, s2 * r2, c2 * r2};
  E[0][0] = (float)(1.0 - 2 * (q[2] * q[2]) - 2 * (q[3] * q[3]));
  E[1][1] = (float)(1.0 - 2 * (q[1] * q[1]) - 2 * (q[3] * q[3]));
  E[2][2] = (float)(1.0 - 2 * (q[1] * q[1]) - 2 * (q[2] * q[2]));
  E[0][1] = 2 * (q[1] * q[2] - q[3] * q[0]);
  E[1][0] = 2 * (q[1] * q[2] + q[3] * q[0]);
  E[1][2] = 2 * (q[2] * q[3] - q[1] * q[0]);
  E[2][1] = 2 * (q[2] * q[3] + q[1] * q[0]);
  E[0][2] = 2 * (q[1] * q[3] + q[2] * q[0]);
  E[2][0] = 2 * (q[1] * q[3] - q[2] * q[0]);
}

// Eigen + ridge score per voxel as in bin/filter_mrc/handlers.cpp:1645-1746:
// ConvertFlatSym2Evects3 (eigen3_simple.hpp:392-405), ScoreHessianPlanar
// (feature.hpp:1529-1561: (l1^2-l2^2)^2 in double from the float eigenvalues)
// or ScoreHessianLinear (:1572-1581: l1*l2-l3^2); direction = evects[0].
void vo_hessian_eigen_score(i64 N, const float *hess, const float *mask,
                            int order, int score_kind, float *sal, float *dir,
                            float *eivals_out) {
#pragma omp parallel for
  for (i64 i = 0; i < N; i++) {
    sal[i] = 0.0f;
    if (mask && mask[i] == 0.0f) continue;
    float d6[6], ev[3], E[3][3];
    vo_diagonalize_flat_sym3(hess + 6 * i, d6, order);
    vo_diag_flat_to_evects(d6, ev, E);
    double l1 = ev[0], l2 = ev[1], l3 = ev[2];
    double sc;
    if (score_kind == 1) {
      sc = l1 * l2 - l3 * l3;
    } else {
      sc = l1 * l1 - l2 * l2;
      sc *= sc;
    }
    float score = (float)sc;
    score *= 1.0f; // peak_height (no background subtraction)
    sal[i] = score;
    dir[3 * i + 0] = E[0][0];
    dir[3 * i + 1] = E[0][1];
    dir[3 * i + 2] = E[0][2];
    if (eivals_out) {
      eivals_out[3 * i + 0] = ev[0];
      eivals_out[3 * i + 1] = ev[1];
      eivals_out[3 * i + 2] = ev[2];
    }
  }
}

// Saliency cut: bin/filter_mrc/handlers.cpp:1751-1797.  Fraction f: copy the
// un-masked saliencies, sort descending, threshold = element floor(n*f) where
// n*f is a float product (:1779-1782); then every voxel (masked or not) with
// saliency < threshold becomes 0 (:1789-1796; ties survive).
float vo_saliency_cut(i64 N, float *sal, const float *mask, float cut,
                      int is_fraction) {
  float thr = cut;
  if (is_fraction) {
    std::vector<float> v;
    v.reserve(N);
    for (i64 i = 0; i < N; i++)
      if (!(mask && mask[i] == 0)) v.push_back(sal[i]);
    std::sort(v.begin(), v.end(), std::greater<float>());
    size_t n = v.size();
    // fraction >= 1 indexes past the end in the reference; clamped to the last element, as the library does
    size_t k = std::min((size_t)floorf((float)n * cut), n - 1);
    thr = v[k];
  }
  for (i64 i = 0; i < N; i++)
    if (sal[i] < thr) sal[i] = 0.0f;
  return thr;
}

// ---------------------------------------------------------------------------
// Tensor-voting tables: lib/visfd/feature.hpp:1669-1675 (hw = floor(sigma*ratio)),
// :2419-2432 -> lib/visfd/filter3d.hpp:546-601 GenFilterGenGauss3D(sigma,m=2,hw):
// h = exp(-pow(r,2)), r = sqrt((ix/s)^2+(iy/s)^2+(iz/s)^2) in float; entries
// below exp(-pow(hw/s,2)) are zeroed (:574-575); sum -> 1 (:585-589).
// Displacements: feature.hpp:2468-2482, j/|j| with |j| = float(sqrt(double(int))).
// ---------------------------------------------------------------------------
int vo_tv_halfwidth(float sigma, float cutoff_ratio) {
  return (int)floor(sigma * cutoff_ratio);
}
void vo_tv_tables(float sigma, int hw, float *decay, float *disp) {
  int w = 2 * hw + 1;
  float thr = 1.0f;
  {
    float h = (sigma > 0) ? expf(-powf(hw / sigma, 2.0f)) : 1.0f;
    if (h < thr) thr = h;
  }
  float total = 0;
  for (int iz = -hw; iz <= hw; iz++)
    for (int iy = -hw; iy <= hw; iy++)
      for (int ix = -hw; ix <= hw; ix++) {
        float x = (!((sigma == 0.0f) && (ix == 0))) ? ix / sigma : 0.0f;
        float y = (!((sigma == 0.0f) && (iy == 0))) ? iy / sigma : 0.0f;
        float z = (!((sigma == 0.0f) && (iz == 0))) ? iz / sigma : 0.0f;
        float r = sqrtf(x * x + y * y + z * z);
        float h = (r > 0) ? expf(-powf(r, 2.0f)) : 1.0f;
        if (fabsf(h) < thr) h = 0.0f;
        decay[(size_t(iz + hw) * w + (iy + hw)) * w + (ix + hw)] = h;
        total += h;
      }
  for (size_t i = 0; i < size_t(w) * w * w; i++) decay[i] /= total;
  if (disp)
    for (int iz = -hw; iz <= hw; iz++)
      for (int iy = -hw; iy <= hw; iy++)
        for (int ix = -hw; ix <= hw; ix++) {
          float len = (float)sqrt((double)(ix * ix + iy * iy + iz * iz));
          if (len == 0) len = 1.0f;
          size_t o = (size_t(iz + hw) * w + (iy + hw)) * w + (ix + hw);
          disp[3 * o + 0] = ix / len;
          disp[3 * o + 1] = iy / len;
          disp[3 * o + 2] = iz / len;
        }
}

// Dense stick voting, gather form: lib/visfd/feature.hpp:1915-2037 and
// :2218-2384 (TVReceiveStickVotes).  For receiver i and offset j (jz,jy,jx
// ascending), voter = i-j; skipped if outside the image, voter mask==0,
// saliency==0 or decay==0; a non-zero voter mask multiplies the decay
// (:2261-2265).  s = r.n; w = sal*decay*(1-s^2)^(e/2); v = 2 s r - n (surfaces)
// or n - 2 s r with (s^2)^(e/2) (curves); T += w v v^T (6 components, float,
// product evaluated left to right :2353-2356).  normalize is not restated
// (filter_mrc passes false, bin/filter_mrc/handlers.cpp:1834).
void vo_tv_dense_stick(i64 nx, i64 ny, i64 nz, const float *sal,
                       const float *dir, const float *mask_src,
                       const float *mask_dst, float sigma, int exponent,
                       float cutoff_ratio, int curves, float *tensor) {
  int hw = vo_tv_halfwidth(sigma, cutoff_ratio);
  int w = 2 * hw + 1;
  std::vector<float> decay(size_t(w) * w * w), disp(size_t(w) * w * w * 3);
  vo_tv_tables(sigma, hw, decay.data(), disp.data());
  i64 N = nx * ny * nz;
  memset(tensor, 0, N * 6 * sizeof(float));
#pragma omp parallel for collapse(2) schedule(dynamic, 4)
  for (i64 iz = 0; iz < nz; iz++)
    for (i64 iy = 0; iy < ny; iy++)
      for (i64 ix = 0; ix < nx; ix++) {
        i64 i = IDX(ix, iy, iz);
        if (mask_dst && mask_dst[i] == 0.0f) continue;
        float *T = tensor + 6 * i;
        for (int jz = -hw; jz <= hw; jz++) {
          i64 vz = iz - jz;
          if (vz < 0 || vz >= nz) continue;
          for (int jy = -hw; jy <= hw; jy++) {
            i64 vy = iy - jy;
            if (vy < 0 || vy >= ny) continue;
            for (int jx = -hw; jx <= hw; jx++) {
              i64 vx = ix - jx;
              if (vx < 0 || vx >= nx) continue;
              size_t o = (size_t(jz + hw) * w + (jy + hw)) * w + (jx + hw);
              float fv = decay[o];
              i64 v = IDX(vx, vy, vz);
              if (mask_src) {
                float mv = mask_src[v];
                if (mv == 0.0f) continue;
                fv *= mv;
              }
              float s = sal[v];
              if (s == 0.0f) continue;
              if (fv == 0.0f) continue;
              const float *r = &disp[3 * o];
              const float *n = &dir[3 * v];
              float st = r[0] * n[0] + r[1] * n[1] + r[2] * n[2];
              float sx2 = st * 2.0f;
              float sin2 = st * st;
              float cos2 = 1.0f - sin2;
              float ang2 = curves ? sin2 : cos2;
              float da;
              switch (exponent) {
              case 2: da = ang2; break;
              case 4: da = ang2 * ang2; break;
              default: da = (float)pow((double)ang2, 0.5 * exponent); break;
              }
              float nr[3];
              for (int d = 0; d < 3; d++)
                nr[d] = curves ? (n[d] - sx2 * r[d]) : (sx2 * r[d] - n[d]);
              T[0] += s * fv * da * nr[0] * nr[0];
              T[3] += s * fv * da * nr[0] * nr[1];
              T[5] += s * fv * da * nr[0] * nr[2];
              T[1] += s * fv * da * nr[1] * nr[1];
              T[4] += s * fv * da * nr[1] * nr[2];
              T[2] += s * fv * da * nr[2] * nr[2];
            }
          }
        }
      }
}

// Post-vote score: bin/filter_mrc/handlers.cpp:1870-1892; DiagonalizeFlatSym3
// then ScoreTensorPlanar = l1 - l2 in double (feature.hpp:1593-1598) or
// ScoreTensorLinear = l1*l2 - l3^2 (:1610-1612).  mask==0 voxels keep out[i].
void vo_tensor_score(i64 N, const float *tensor, const float *mask, int order,
                     int score_kind, float *out) {
#pragma omp parallel for
  for (i64 i = 0; i < N; i++) {
    if (mask && mask[i] == 0.0f) continue;
    float d6[6];
    vo_diagonalize_flat_sym3(tensor + 6 * i, d6, order);
    double l1 = d6[0], l2 = d6[1], l3 = d6[2];
    double sc = (score_kind == 1) ? (l1 * l2 - l3 * l3) : (l1 - l2);
    out[i] = (float)sc * 1.0f;
  }
}

// Whole membrane path of HandleTV (bin/filter_mrc/handlers.cpp:1618-1892, no
// background subtraction).  Optional outputs may be NULL.  Returns threshold.
float vo_membrane_background(i64 nx, i64 ny, i64 nz, const float *src, const float *mask,
                             float sigma, float truncate_ratio, int order, float cut,
                             int cut_is_fraction, float tv_sigma, int tv_exponent,
                             float tv_cutoff_ratio, float background_sigma, int normalize,
                             float *hess_sal_out, float *dir_out, float *tensor_out, float *out) {
  i64 N = nx * ny * nz;
  std::vector<float> grad(N * 3, 0.0f), hess(N * 6, 0.0f), sal(N, 0.0f);
  // handlers.cpp:1577-1592 (`-membrane-background`): peak_height = tomo_in - Gauss(tomo_in, width_b) multiplies the
  // ridge score (:1698-1702) and the post-vote score (:1883-1887).  (The second blur of that block, into tomo_out,
  // is overwritten before anyone reads it.)
  std::vector<float> peak;
  if (background_sigma > 0.0f) {
    std::vector<float> bg(src, src + N);               // tomo_background = tomo_in: masked voxels keep the source
    float sg[3] = {background_sigma, background_sigma, background_sigma};
    int h = (int)std::floor(background_sigma * truncate_ratio);
    int hw[3] = {h, h, h};
    vo_apply_gauss(nx, ny, nz, src, bg.data(), mask, sg, hw, normalize);
    peak.resize(N);
    for (i64 i = 0; i < N; i++) peak[i] = src[i] - bg[i];
  }
  vo_calc_hessian(nx, ny, nz, src, mask, sigma, truncate_ratio, grad.data(),
                  hess.data(), nullptr);
  std::vector<float> dir(grad); // direction aliases gradient storage (:1633)
  vo_hessian_eigen_score(N, hess.data(), mask, order, 0, sal.data(), dir.data(),
                         nullptr);
  if (!peak.empty())
    for (i64 i = 0; i < N; i++)
      if (!(mask && mask[i] == 0.0f)) sal[i] *= peak[i];
  float thr = vo_saliency_cut(N, sal.data(), mask, cut, cut_is_fraction);
  if (hess_sal_out) memcpy(hess_sal_out, sal.data(), N * sizeof(float));
  if (dir_out) memcpy(dir_out, dir.data(), 3 * N * sizeof(float));
  memcpy(out, sal.data(), N * sizeof(float));
  if (tv_sigma > 0.0f) {
    std::vector<float> tensor(N * 6);
    vo_tv_dense_stick(nx, ny, nz, sal.data(), dir.data(), mask, mask, tv_sigma,
                      tv_exponent, tv_cutoff_ratio, 0, tensor.data());
    vo_tensor_score(N, tensor.data(), mask, order, 0, out);
    if (!peak.empty())
      for (i64 i = 0; i < N; i++)
        if (!(mask && mask[i] == 0.0f)) out[i] *= peak[i];
    if (tensor_out) memcpy(tensor_out, tensor.data(), 6 * N * sizeof(float));
  }
  return thr;
}

float vo_membrane(i64 nx, i64 ny, i64 nz, const float *src, const float *mask,
                  float sigma, float truncate_ratio, int order, float cut,
                  int cut_is_fraction, float tv_sigma, int tv_exponent,
                  float tv_cutoff_ratio, float *hess_sal_out, float *dir_out,
                  float *tensor_out, float *out) {
  return vo_membrane_background(nx, ny, nz, src, mask, sigma, truncate_ratio, order, cut, cut_is_fraction, tv_sigma,
                                tv_exponent, tv_cutoff_ratio, 0.0f, 1, hess_sal_out, dir_out, tensor_out, out);
}

// ---------------------------------------------------------------------------
// Threshold maps: lib/threshold/threshold.hpp:10-12 (IsBetween), :52-77
// (Threshold2), :117-169 (Threshold4); single-threshold form and clipping as in
// bin/filter_mrc/handlers.cpp:1049-1064.
// ---------------------------------------------------------------------------
static bool is_between(float x, float a, float b) {
  return ((a <= x) && (x < b)) || ((b < x) && (x <= a));
}
static float thr2(float x, float a, float b, float outA, float outB) {
  float g;
  if (is_between(x, a, b))
    g = (x - a) / (b - a);
  else if ((x - a) * (b - a) > 0.0)
    g = 1.0;
  else
    g = 0.0;
  return outA + g * (outB - outA);
}
void vo_threshold1(i64 N, const float *in, float *out, float a, float outA,
                   float outB) {
  for (i64 i = 0; i < N; i++) out[i] = (in[i] > a) ? outB : outA;
}
void vo_threshold2(i64 N, const float *in, float *out, float a, float b,
                   float outA, float outB) {
  for (i64 i = 0; i < N; i++) out[i] = thr2(in[i], a, b, outA, outB);
}
void vo_threshold4(i64 N, const float *in, float *out, float a01, float b01,
                   float a10, float b10, float outA, float outB) {
  for (i64 i = 0; i < N; i++) {
    float x = in[i];
    float g = thr2(x, a01, b01, 0, 1);
    if ((b01 == a10) && (b01 == b10)) { out[i] = g; continue; } // :131-133 (sic: returns g unscaled)
    if (is_between(x, a01, b01))
      g = thr2(x, a01, b01, 0, 1);
    else if (is_between(x, a10, b10))
      g = thr2(x, a10, b10, 0, 1);
    else if (b01 <= a10)
      g = is_between(x, b01, a10) ? 1.0f : 0.0f;
    else if (b10 <= a01)
      g = is_between(x, b10, a01) ? 0.0f : 1.0f;
    out[i] = outA + g * (outB - outA);
  }
}
// lib/visfd/visfd_utils.hpp:685-708, 764-790: float accumulators, raster order
float vo_average(i64 N, const float *in, const float *w) {
  float total = 0.0f, denom = 0.0f;
  for (i64 i = 0; i < N; i++) {
    float h = in[i];
    if (w) { h *= w[i]; denom += w[i]; } else denom += 1.0f;
    total += h;
  }
  return total / denom;
}
float vo_stddev(i64 N, const float *in, const float *w) {
  float ave = vo_average(N, in, w);
  float total = 0.0f, denom = 0.0f;
  for (i64 i = 0; i < N; i++) {
    float h = in[i] - ave;
    h *= h;
    if (w) { h *= w[i]; denom += w[i]; } else denom += 1.0f;
    total += h;
  }
  return (float)sqrt(total / denom);
}

// ---------------------------------------------------------------------------
// Binning: lib/visfd/resample.hpp:53-104 (BinArray3D) and :106-166 (UnbinArray3D).
// size_* = {nx, ny, nz}; offset may be NULL.  Returns 0, or 1 for the arguments the
// reference rejects (offset out of range, :62-70 / :128-136).
// ---------------------------------------------------------------------------
int vo_bin3d(const i64 size_src[3], const i64 size_dst[3], const float *src, float *dst, const int *offset) {
  i64 b[3];
  for (int d = 0; d < 3; d++) {
    b[d] = size_src[d] / size_dst[d];
    if (offset && (offset[d] >= b[d] || offset[d] < 0)) return 1;
  }
  for (i64 Z = 0; Z < size_dst[2]; Z++)
    for (i64 Y = 0; Y < size_dst[1]; Y++)
      for (i64 X = 0; X < size_dst[0]; X++) {
        float sum = 0.0f;
        for (i64 dz = 0; dz < b[2]; dz++)
          for (i64 dy = 0; dy < b[1]; dy++)
            for (i64 dx = 0; dx < b[0]; dx++) {
              i64 ix = X * b[0] + dx, iy = Y * b[1] + dy, iz = Z * b[2] + dz;
              if (offset) { ix += offset[0]; iy += offset[1]; iz += offset[2]; }
              sum += src[(iz * size_src[1] + iy) * size_src[0] + ix];
            }
        dst[(Z * size_dst[1] + Y) * size_dst[0] + X] = sum / (float)(int)(b[0] * b[1] * b[2]);
      }
  return 0;
}
int vo_unbin3d(const i64 size_src[3], const i64 size_dst[3], const float *src, float *dst, const int *offset) {
  i64 b[3], o[3] = {0, 0, 0};
  for (int d = 0; d < 3; d++) {
    b[d] = size_dst[d] / size_src[d];
    if (offset && (offset[d] >= b[d] || offset[d] < 0)) return 1;
    if (offset) o[d] = offset[d];
  }
  for (i64 Z = 0; Z < size_dst[2]; Z++)
    for (i64 Y = 0; Y < size_dst[1]; Y++)
      for (i64 X = 0; X < size_dst[0]; X++) {
        i64 ix = (X - o[0]) / b[0], iy = (Y - o[1]) / b[1], iz = (Z - o[2]) / b[2];   // C division, :151-153
        if (ix < 0) ix = 0;
        if (iy < 0) iy = 0;
        if (iz < 0) iz = 0;
        if (ix >= size_src[0]) ix = size_src[0] - 1;
        if (iy >= size_src[1]) iy = size_src[1] - 1;
        if (iz >= size_src[2]) iz = size_src[2] - 1;
        dst[(Z * size_dst[1] + Y) * size_dst[0] + X] = src[(iz * size_src[1] + iy) * size_src[0] + ix];
      }
  return 0;
}

// ---------------------------------------------------------------------------
// Mask rasterisation: lib/visfd/draw.hpp:90-237 (DrawRegions).  Regions are painted in list
// order; a region of negative value clears positive voxels when negative_means_subtract is
// set (:162-166, :203-207), otherwise its value is stored (:168-170).  An all-zero image
// whose first region is negative is first filled with ones (:98-134).  Masked voxels
// (mask == 0) are skipped everywhere.
//   sphere (:139-172): Ri = ceil(R - 0.5); centre = floor(c + 0.5); for |jz|,|jy| <= Ri:
//                      descr = R*R - (jy*jy + jz*jz) in float, skipped if < 0;
//                      |jx| <= floor(sqrt(descr))
//   box    (:176-211): corners floor(v + 0.5) kept as floats, clipped to the image
// ---------------------------------------------------------------------------
struct vo_region { int32_t type; float p[6]; float value; };
static void vo_paint(float &v, float value, bool subtract) {
  if (value < 0) {
    if (subtract && v > 0) v = 0.0f;
  } else {
    v = value;
  }
}
int vo_draw_regions(int nx, int ny, int nz, float *image, const float *mask, const vo_region *regions, int n,
                    int negative_means_subtract) {
  const bool subtract = negative_means_subtract != 0;
  const i64 N = (i64)nx * ny * nz;
  if (subtract && n > 0 && regions[0].value < 0) {
    bool all_zero = true;
    for (i64 i = 0; i < N && all_zero; i++)
      if (!(mask && mask[i] == 0.0f) && image[i] != 0.0f) all_zero = false;
    if (all_zero)
      for (i64 i = 0; i < N; i++)
        if (!(mask && mask[i] == 0.0f)) image[i] = 1.0f;
  }
  const int size[3] = {nx, ny, nz};
  for (int k = 0; k < n; k++) {
    const vo_region &r = regions[k];
    if (r.type == 1) {
      const float R = r.p[3];
      const int Ri = (int)std::ceil(R - 0.5);
      const int cx = (int)std::floor(r.p[0] + 0.5), cy = (int)std::floor(r.p[1] + 0.5), cz = (int)std::floor(r.p[2] + 0.5);
      for (int jz = -Ri; jz <= Ri; jz++)
        for (int jy = -Ri; jy <= Ri; jy++) {
          const float descr = R * R - (jy * jy + jz * jz);
          if (descr < 0.0) continue;
          const int xr = (int)std::floor(std::sqrt(descr));
          for (int jx = -xr; jx <= xr; jx++) {
            const int x = cx + jx, y = cy + jy, z = cz + jz;
            if (x < 0 || x >= nx || y < 0 || y >= ny || z < 0 || z >= nz) continue;
            const i64 at = ((i64)z * ny + y) * nx + x;
            if (mask && mask[at] == 0.0f) continue;
            vo_paint(image[at], r.value, subtract);
          }
        }
    } else {
      float lo[3], hi[3];
      for (int d = 0; d < 3; d++) {
        lo[d] = std::max<float>((float)std::floor(r.p[2 * d] + 0.5), 0);
        hi[d] = std::min<float>((float)std::floor(r.p[2 * d + 1] + 0.5), size[d] - 1);
      }
      for (int z = (int)lo[2]; z <= hi[2]; z++)
        for (int y = (int)lo[1]; y <= hi[1]; y++)
          for (int x = (int)lo[0]; x <= hi[0]; x++) {
            const i64 at = ((i64)z * ny + y) * nx + x;
            if (mask && mask[at] == 0.0f) continue;
            vo_paint(image[at], r.value, subtract);
          }
    }
  }
  return 0;
}

// ---------------------------------------------------------------------------
// Scale-space blob detection: lib/visfd/feature.hpp:56-427 (BlobDog).
// For scale ir: LoG image into ring slot ir%3 (:170-176); for ir>=2 every voxel
// of scale ir-1 is tested against its 80 neighbours in (x,y,z,scale): strict
// minimum / maximum, all neighbours must be inside the image and un-masked
// (:235-262); minima need score<0, maxima score>0 (:270-271, :289-290).  The
// running best-score filter (:267-303) is order dependent in the reference and
// only ever more permissive than the final filter (:362-417), so only the
// final filter is restated; lists are returned in (scale, z, y, x) order.
// ---------------------------------------------------------------------------
void vo_blob_dog(i64 nx, i64 ny, i64 nz, const float *src, const float *mask,
                 const float *sigmas, int ns, float delta, float truncate_ratio,
                 float minima_threshold, float maxima_threshold,
                 int use_threshold_ratios, i64 capacity, float *min_crds,
                 float *min_sigma, float *min_score, i64 *n_min, float *max_crds,
                 float *max_sigma, float *max_score, i64 *n_max) {
  i64 N = nx * ny * nz;
  std::vector<float> img[3];
  for (int k = 0; k < 3; k++) img[k].resize(N);
  struct Blob { float x, y, z, sigma, score; };
  std::vector<Blob> mins, maxs;
  float gmin = 1.0f, gmax = -1.0f;
  for (int ir = 0; ir < ns; ir++) {
    float s3[3] = {sigmas[ir] * 1.0f, sigmas[ir] * 1.0f, sigmas[ir] * 1.0f};
    vo_apply_log(nx, ny, nz, src, img[ir % 3].data(), mask, s3, delta,
                 truncate_ratio, nullptr, nullptr);
    if (ir < 2) continue;
    const float *I[3] = {img[(ir - 2) % 3].data(), img[(ir - 1) % 3].data(),
                         img[ir % 3].data()};
    for (i64 iz = 0; iz < nz; iz++)
      for (i64 iy = 0; iy < ny; iy++)
        for (i64 ix = 0; ix < nx; ix++) {
          bool is_min = true, is_max = true;
          float e = I[1][IDX(ix, iy, iz)];
          for (int jr = 0; jr < 3 && (is_min || is_max); jr++)
            for (int jz = -1; jz <= 1; jz++)
              for (int jy = -1; jy <= 1; jy++)
                for (int jx = -1; jx <= 1; jx++) {
                  if (!jx && !jy && !jz && jr == 1) continue;
                  i64 X = ix + jx, Y = iy + jy, Z = iz + jz;
                  if (X < 0 || X >= nx || Y < 0 || Y >= ny || Z < 0 || Z >= nz ||
                      (mask && mask[IDX(X, Y, Z)] == 0)) {
                    is_min = is_max = false;
                    continue;
                  }
                  float nb = I[jr][IDX(X, Y, Z)];
                  if (nb <= e) is_min = false;
                  if (nb >= e) is_max = false;
                }
          if (mask && mask[IDX(ix, iy, iz)] == 0) continue;
          if (is_min && e < 0.0f) {
            mins.push_back({(float)ix, (float)iy, (float)iz, sigmas[ir - 1], e});
            if (e < gmin) gmin = e;
          }
          if (is_max && e > 0.0f) {
            maxs.push_back({(float)ix, (float)iy, (float)iz, sigmas[ir - 1], e});
            if (e > gmax) gmax = e;
          }
        }
  }
  bool filt = (minima_threshold != INFINITY) || (maxima_threshold != -INFINITY);
  if (use_threshold_ratios) {
    // Infinite *ratio* thresholds (never produced by filter_mrc together with
    // finite ones for the same list): the reference's running filter (:267-292)
    // multiplies +-inf by the running best score, which admits no maximum at all
    // (-inf * -1.0 = +inf) and a thread-dependent handful of minima; the
    // deterministic reading restated here is "that list is empty".
    if (maxima_threshold == -INFINITY) maxs.clear();
    if (minima_threshold == INFINITY) mins.clear();
  }
  if (filt && use_threshold_ratios) {
    minima_threshold *= gmin;
    maxima_threshold *= gmax;
  }
  i64 a = 0, b = 0;
  for (auto &m : mins)
    if (!filt || m.score <= minima_threshold) {
      if (a < capacity) {
        min_crds[3 * a] = m.x; min_crds[3 * a + 1] = m.y; min_crds[3 * a + 2] = m.z;
        min_sigma[a] = m.sigma; min_score[a] = m.score;
      }
      a++;
    }
  for (auto &m : maxs)
    if (!filt || m.score >= maxima_threshold) {
      if (b < capacity) {
        max_crds[3 * b] = m.x; max_crds[3 * b + 1] = m.y; max_crds[3 * b + 2] = m.z;
        max_sigma[b] = m.sigma; max_score[b] = m.score;
      }
      b++;
    }
  *n_min = a;
  *n_max = b;
}


// ---------------------------------------------------------------------------
// LabelConnected: lib/visfd/connect.hpp:171-1432 with the arguments HandleTV passes
// (bin/filter_mrc/handlers.cpp:1927-2034): unsigned dot products, positive-definite
// tensors, connectivity 1, maxima as seeds, clusters by size, no must-link constraints.
// The voxels' directions are the first eigenvectors of the tensors
// (handlers.cpp:1933-1950: ConvertFlatSym2Evects3, float Shoemake round trip included).
// ---------------------------------------------------------------------------
// TraceProductSym3 as COMPILED (lin3_utils.hpp:502-531): the reference indexes
// MapIndices_linear_to_3x3 (a [6][2] table) with [i][j], i,j in 0..2, which walks the flat
// table {0,0,1,1,2,2,...} and so only ever touches the diagonal entries 0,1,2:
static float trace_product_sym3(const float *A, const float *B) {
  return A[0] * B[0] + A[0] * B[1] + A[1] * B[2] + A[1] * B[0] + A[1] * B[1] + A[2] * B[2] + A[2] * B[1] +
         A[2] * B[2] + A[0] * B[0];
}
static float frobenius_sym3(const float *A) { return std::sqrt(trace_product_sym3(A, A)); }
static float dot3f(const float *a, const float *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

static void first_evec(const float m6[6], int order, float e0[3]) {   // eigen3_simple.hpp:392-405
  float d6[6], ev[3], E[3][3];
  vo_diagonalize_flat_sym3(m6, d6, order);
  vo_diag_flat_to_evects(d6, ev, E);
  e0[0] = E[0][0]; e0[1] = E[0][1]; e0[2] = E[0][2];
}

// labels: N int64 (cluster from 1, -1 undefined, n_maxima + 1 outside the mask: connect.hpp:1398-1401 skips
// those voxels).  direction_out (optional N*3): the standardised directions.  Returns the number of clusters.
i64 vo_label_connected(i64 nx, i64 ny, i64 nz, const float *sal, const float *mask, const float *tensor,
                       int eival_order, float thr_sal, float thr_vs, float thr_vn, float thr_ts, float thr_tn,
                       i64 *labels, float *direction_out) {
  const i64 N = nx * ny * nz;
  static const int nb[6][3] = {{0, 0, -1}, {0, -1, 0}, {-1, 0, 0}, {1, 0, 0}, {0, 1, 0}, {0, 0, 1}};  // :212-240
  if (thr_vs < 0) thr_vs = 0.0f;   // :190-205 (unsigned dot products)
  if (thr_vn < 0) thr_vn = 0.0f;
  std::vector<float> dir((size_t)N * 3, 0.0f);
  for (i64 i = 0; i < N; i++) first_evec(tensor + 6 * i, eival_order, &dir[3 * i]);
  auto masked = [&](i64 i) { return mask && mask[i] == 0.0f; };

  // ---- _FindExtrema (morphology_implementation.hpp:57-515): maxima, plateaus, borders allowed ----
  const float max_thr = (thr_sal == INFINITY) ? -INFINITY : thr_sal;   // :549-550
  std::vector<i64> seed_voxel;
  std::vector<float> seed_score;
  {
    std::vector<char> seen((size_t)N, 0);
    std::vector<i64> q;
    for (i64 i0 = 0; i0 < N; i0++) {
      if (masked(i0) || seen[i0]) continue;
      bool is_max = true;
      q.assign(1, i0);
      seen[i0] = 1;
      for (size_t h = 0; h < q.size(); h++) {
        const i64 v = q[h];
        const i64 x = v % nx, y = (v / nx) % ny, z = v / (nx * ny);
        for (int k = 0; k < 6; k++) {
          const i64 jx = x + nb[k][0], jy = y + nb[k][1], jz = z + nb[k][2];
          if (jx < 0 || jx >= nx || jy < 0 || jy >= ny || jz < 0 || jz >= nz) continue;
          const i64 j = IDX(jx, jy, jz);
          if (masked(j)) continue;
          if (sal[j] == sal[v]) {
            if (!seen[j]) { seen[j] = 1; q.push_back(j); }
          } else if (sal[j] > sal[v]) {
            is_max = false;
          }
        }
      }
      if (is_max && sal[i0] >= max_thr) { seed_voxel.push_back(i0); seed_score.push_back(sal[i0]); }
    }
    // sort(rbegin, rend) of (score, position): :449-470
    std::vector<std::tuple<float, i64> > key(seed_voxel.size());
    for (size_t k = 0; k < key.size(); k++) key[k] = std::make_tuple(seed_score[k], (i64)k);
    std::sort(key.rbegin(), key.rend());
    std::vector<i64> sv(key.size());
    std::vector<float> ss(key.size());
    for (size_t k = 0; k < key.size(); k++) { sv[k] = seed_voxel[std::get<1>(key[k])]; ss[k] = seed_score[std::get<1>(key[k])]; }
    seed_voxel.swap(sv);
    seed_score.swap(ss);
  }
  const i64 nb_ = (i64)seed_voxel.size();
  const i64 UNDEFINED = nb_ + 1, QUEUED = nb_ + 2;
  for (i64 i = 0; i < N; i++) labels[i] = UNDEFINED;
  typedef std::tuple<float, i64, std::tuple<float, float, float> > Entry;   // lexicographic, like the reference's tuple
  std::priority_queue<Entry> q;
  for (i64 b = 0; b < nb_; b++) {
    const i64 v = seed_voxel[b];
    q.push(Entry(seed_score[b], b, std::make_tuple((float)(v % nx), (float)((v / nx) % ny), (float)(v / (nx * ny)))));
    labels[v] = QUEUED;
  }
  std::vector<i64> basin2cluster(nb_);
  std::vector<std::vector<i64> > cluster2basins(nb_);
  for (i64 b = 0; b < nb_; b++) { basin2cluster[b] = b; cluster2basins[b].assign(1, b); }
  std::vector<signed char> polarity(nb_, 1);

  while (!q.empty()) {
    const Entry e = q.top();
    q.pop();
    const float score = std::get<0>(e);
    const float basin_f = (float)std::get<1>(e);   // Scalar i_which_basin, :438
    const i64 basin = (i64)basin_f;
    const i64 x = (i64)std::get<0>(std::get<2>(e)), y = (i64)std::get<1>(std::get<2>(e)), z = (i64)std::get<2>(std::get<2>(e));
    const i64 i = IDX(x, y, z);
    if (-score > thr_sal * -1.0f) { labels[i] = UNDEFINED; continue; }   // :445-449
    if (masked(i)) { labels[i] = UNDEFINED; continue; }
    {
      // CalcHessianFiniteDifferences with the centre moved inside the image (visfd_utils.hpp:579-616), sign flipped (:487-492)
      i64 cx = x, cy = y, cz = z;
      if (cx == 0) cx++; else if (cx == nx - 1) cx--;
      if (cy == 0) cy++; else if (cy == ny - 1) cy--;
      if (cz == 0) cz++; else if (cz == nz - 1) cz--;
      auto F = [&](int dx, int dy, int dz) { return sal[IDX(cx + dx, cy + dy, cz + dz)]; };
      float h[6];
      h[0] = (F(1, 0, 0) + F(-1, 0, 0) - 2 * F(0, 0, 0));
      h[1] = (F(0, 1, 0) + F(0, -1, 0) - 2 * F(0, 0, 0));
      h[2] = (F(0, 0, 1) + F(0, 0, -1) - 2 * F(0, 0, 0));
      h[3] = 0.25 * (F(1, 1, 0) + F(-1, -1, 0) - F(1, -1, 0) - F(-1, 1, 0));
      h[4] = 0.25 * (F(0, 1, 1) + F(0, -1, -1) - F(0, 1, -1) - F(0, -1, 1));
      h[5] = 0.25 * (F(1, 0, 1) + F(-1, 0, -1) - F(-1, 0, 1) - F(1, 0, -1));
      for (int k = 0; k < 6; k++) h[k] *= -1.0;
      bool discard = false;
      const float *T = tensor + 6 * i;
      if (trace_product_sym3(h, T) < thr_ts * frobenius_sym3(h) * frobenius_sym3(T)) discard = true;   // :512-521
      float e0[3];
      first_evec(h, 1, e0);   // decreasing eigenvalues: clusters start at maxima (:173-177)
      const float *V = &dir[3 * i];
      const float d = dot3f(e0, V);
      if (d * d < thr_vs * thr_vs * dot3f(e0, e0) * dot3f(V, V)) discard = true;   // :546-556
      if (discard) {
        labels[i] = UNDEFINED;
        if (i == seed_voxel[basin]) basin2cluster[basin] = -1;   // :580-591
        continue;
      }
    }
    labels[i] = basin;
    for (int k = 0; k < 6; k++) {
      const i64 jx = x + nb[k][0], jy = y + nb[k][1], jz = z + nb[k][2];
      if (jz < 0 || jz >= nz || jy < 0 || jy >= ny || jx < 0 || jx >= nx) continue;
      const i64 j = IDX(jx, jy, jz);
      if (masked(j)) continue;
      const float *Ti = tensor + 6 * i, *Tj = tensor + 6 * j;
      if (trace_product_sym3(Ti, Tj) < thr_tn * frobenius_sym3(Ti) * frobenius_sym3(Tj)) continue;   // :633-643
      float *Vi = &dir[3 * i], *Vj = &dir[3 * j];
      {
        const float d = dot3f(Vi, Vj);
        if (d * d < thr_vn * thr_vn * dot3f(Vi, Vi) * dot3f(Vj, Vj)) continue;   // :662-672
      }
      if (labels[j] == QUEUED) continue;
      if (labels[j] == UNDEFINED) {
        labels[j] = QUEUED;
        q.push(Entry(sal[j], (i64)basin_f, std::make_tuple((float)jx, (float)jy, (float)jz)));
        if (dot3f(Vi, Vj) < 0.0f) { Vj[0] *= -1.0f; Vj[1] *= -1.0f; Vj[2] *= -1.0f; }   // :698-722
        continue;
      }
      const i64 bi = labels[i], bj = labels[j];
      const i64 ci = basin2cluster[bi], cj = basin2cluster[bj];
      const bool polarity_match = !(dot3f(Vi, Vj) * polarity[bi] * polarity[bj] < 0.0f);   // :735-748
      if (ci == cj) continue;
      const i64 keep = std::min(ci, cj), gone = std::max(ci, cj);
      for (i64 b : cluster2basins[gone]) {
        cluster2basins[keep].push_back(b);
        basin2cluster[b] = keep;
        if (!polarity_match) polarity[b] = (signed char)-polarity[b];
      }
      cluster2basins[gone].clear();
    }
  }
  // ---- clusters (:1045-1068), polarity (:1080-1105), sizes, outward normals (:1183-1284), order by size (:1310-1355) ----
  i64 n_clusters = 0;
  std::vector<i64> old2new(nb_);
  for (i64 b = 0; b < nb_; b++) {
    old2new[b] = n_clusters;
    if (basin2cluster[b] == b) n_clusters++;
  }
  for (i64 b = 0; b < nb_; b++)
    if (basin2cluster[b] >= 0) basin2cluster[b] = old2new[basin2cluster[b]];
  auto inside = [&](i64 i) { return !masked(i) && labels[i] != UNDEFINED; };
  for (i64 i = 0; i < N; i++)
    if (inside(i)) for (int d = 0; d < 3; d++) dir[3 * i + d] *= (float)polarity[labels[i]];
  for (i64 i = 0; i < N; i++)
    if (inside(i)) labels[i] = basin2cluster[labels[i]];
  std::vector<long double> size(n_clusters, 0.0L), com(3 * n_clusters, 0.0L), sum(n_clusters, 0.0L);
  for (i64 i = 0; i < N; i++)
    if (inside(i)) {
      size[labels[i]] += 1.0L;
      com[3 * labels[i]] += i % nx; com[3 * labels[i] + 1] += (i / nx) % ny; com[3 * labels[i] + 2] += i / (nx * ny);
    }
  for (i64 c = 0; c < n_clusters; c++) for (int d = 0; d < 3; d++) com[3 * c + d] /= size[c];
  for (i64 i = 0; i < N; i++)
    if (inside(i)) {
      const i64 c = labels[i];
      float r[3];
      r[0] = (i % nx) - com[3 * c]; r[1] = ((i / nx) % ny) - com[3 * c + 1]; r[2] = (i / (nx * ny)) - com[3 * c + 2];
      long double delta = dot3f(r, &dir[3 * i]);
      sum[c] += delta;
    }
  for (i64 i = 0; i < N; i++)
    if (inside(i) && sum[labels[i]] < 0.0L) for (int d = 0; d < 3; d++) dir[3 * i + d] *= -1.0f;
  {
    std::vector<std::tuple<float, i64> > key(n_clusters);
    for (i64 c = 0; c < n_clusters; c++) key[c] = std::make_tuple((float)size[c], c);
    std::sort(key.rbegin(), key.rend());
    std::vector<i64> rank(n_clusters);
    for (i64 r = 0; r < n_clusters; r++) rank[std::get<1>(key[r])] = r;
    for (i64 i = 0; i < N; i++)
      if (inside(i)) labels[i] = rank[labels[i]];
  }
  for (i64 i = 0; i < N; i++) {
    if (masked(i)) continue;
    if (labels[i] == UNDEFINED) labels[i] = -1;
    else labels[i] += 1;
  }
  if (direction_out) memcpy(direction_out, dir.data(), sizeof(float) * 3 * (size_t)N);
  return n_clusters;
}


// ---- oriented point cloud of a detected surface (bin/filter_mrc/handlers.cpp:2039-2309) -----------------------
// For every un-masked voxel of the selected cluster: (1) follow the surface normal in both directions while
// inside the cluster (step ds), take the saliency-weighted mean arc length and the sample next to it (:2097-2215);
// (2) move that point onto the ridge of the saliency along the eigenvector of the saliency's finite-difference
// Hessian with the largest |eigenvalue| (:2224-2295); points further than max_distance from the ridge, with a
// vanishing gradient component, or outside the image are dropped.  labels == NULL: every un-masked voxel, position
// x voxel width, normal = direction (:2053-2066).  rows: {x, y, z, nx, ny, nz} in raster order of the source voxel;
// returns the number of points (only the first `capacity` are stored).
// Deviations, both below the 6 digits the reference prints: the 3x3 eigen-decomposition of the float Hessian is
// done in double (the reference instantiates DiagonalizeSym3 with float here), and a rounded sample position
// that an extrapolation pushed outside the image is clamped (the reference reads out of bounds).
i64 vo_surface_points(i64 nx, i64 ny, i64 nz, const float *sal, const float *dir, const float *labels,
                      const float *mask, int select_cluster, const float voxel_width[3], float ds, int find_ridge,
                      float max_distance, float *rows, i64 capacity) {
  i64 n_out = 0;
  const int size[3] = {(int)nx, (int)ny, (int)nz};
  auto emit = [&](const float xyz[3], const float nrm[3]) {
    if (n_out < capacity) {
      for (int d = 0; d < 3; d++) { rows[6 * n_out + d] = xyz[d]; rows[6 * n_out + 3 + d] = nrm[d]; }
    }
    n_out++;
  };
  auto inside = [&](const int p[3]) { return p[0] >= 0 && p[0] < size[0] && p[1] >= 0 && p[1] < size[1] && p[2] >= 0 && p[2] < size[2]; };
  auto unit = [&](i64 i, float u[3]) {
    const float *v = dir + 3 * i;
    float norm = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);   // length3, visfd_utils.hpp:40-43
    for (int d = 0; d < 3; d++) u[d] = v[d] / norm;
  };
  for (int iz = 0; iz < size[2]; iz++)
    for (int iy = 0; iy < size[1]; iy++)
      for (int ix = 0; ix < size[0]; ix++) {
        const i64 i0 = IDX(ix, iy, iz);
        if (mask && mask[i0] == 0.0f) continue;
        float xyz[3], normal[3];
        if (!labels) {
          xyz[0] = ix * voxel_width[0]; xyz[1] = iy * voxel_width[1]; xyz[2] = iz * voxel_width[2];
          for (int d = 0; d < 3; d++) normal[d] = dir[3 * i0 + d];
          emit(xyz, normal);
          continue;
        }
        if ((float)select_cluster != labels[i0]) continue;
        xyz[0] = ix; xyz[1] = iy; xyz[2] = iz;
        unit(i0, normal);
        for (int d = 0; d < 3; d++) normal[d] *= sal[i0];
        if (ds > 0.0f) {
          std::vector<float> vS, vW, bS, bW;
          std::vector<std::array<float, 3> > vX, bX;
          std::array<float, 3> r = {(float)ix, (float)iy, (float)iz};
          int p[3] = {ix, iy, iz};
          float s = 0.0f, drds[3];
          // (a zero or NaN direction would keep the reference walking on the spot for ever; bounded here)
          const size_t max_steps = (size_t)(4.0 * (nx + ny + nz) / ds) + 16;
          while (vS.size() < max_steps && inside(p) && !(mask && mask[IDX(p[0], p[1], p[2])] == 0.0f) && labels[IDX(p[0], p[1], p[2])] == labels[i0]) {
            const i64 j = IDX(p[0], p[1], p[2]);
            vS.push_back(s); vX.push_back(r); vW.push_back(sal[j]);
            unit(j, drds);
            s += ds;
            for (int d = 0; d < 3; d++) { r[d] += ds * drds[d]; p[d] = (int)std::round(r[d]); }
          }
          r = {(float)ix, (float)iy, (float)iz};
          p[0] = ix; p[1] = iy; p[2] = iz;
          s = 0.0f;
          while (bS.size() < max_steps) {
            unit(IDX(p[0], p[1], p[2]), drds);
            s -= ds;
            for (int d = 0; d < 3; d++) { r[d] -= ds * drds[d]; p[d] = (int)std::round(r[d]); }
            if (!inside(p)) break;
            const i64 j = IDX(p[0], p[1], p[2]);
            if (mask && mask[j] == 0.0f) break;
            if (labels[j] != labels[i0]) break;
            bS.push_back(s); bX.push_back(r); bW.push_back(sal[j]);
          }
          vS.insert(vS.begin(), bS.rbegin(), bS.rend());
          vX.insert(vX.begin(), bX.rbegin(), bX.rend());
          vW.insert(vW.begin(), bW.rbegin(), bW.rend());
          float sum_s = 0.0f, sum_w = 0.0f;
          for (size_t k = 0; k < vS.size(); k++) { sum_s += vW[k] * vS[k]; sum_w += vW[k]; }
          const float ave_s = sum_s / sum_w;
          size_t k = 0;
          while (k + 1 < vS.size()) {
            k++;
            if (vS[k - 1] <= ave_s && ave_s <= vS[k]) break;
          }
          for (int d = 0; d < 3; d++) p[d] = std::min(std::max((int)std::round(vX[k][d]), 0), size[d] - 1);
          unit(IDX(p[0], p[1], p[2]), normal);
          for (int d = 0; d < 3; d++) {
            if (k + 1 < vS.size()) xyz[d] = vX[k][d] + (vX[k + 1][d] - vX[k][d]) * ((ave_s - vS[k]) / (vS[k + 1] - vS[k]));
            else xyz[d] = vX[k][d];
            normal[d] *= sal[i0];
          }
        }
        if (find_ridge) {
          int q[3];
          for (int d = 0; d < 3; d++) q[d] = std::min(std::max((int)std::round(xyz[d]), 0), size[d] - 1);
          i64 x = q[0], y = q[1], z = q[2];
          if (x == 0) x++; else if (x == nx - 1) x--;
          if (y == 0) y++; else if (y == ny - 1) y--;
          if (z == 0) z++; else if (z == nz - 1) z--;
#define F(dx, dy, dz) sal[IDX(x + (dx), y + (dy), z + (dz))]
          const float c = F(0, 0, 0);
          const float g[3] = {0.5f * (F(1, 0, 0) - F(-1, 0, 0)), 0.5f * (F(0, 1, 0) - F(0, -1, 0)), 0.5f * (F(0, 0, 1) - F(0, 0, -1))};
          const float hxx = F(1, 0, 0) + F(-1, 0, 0) - 2 * c, hyy = F(0, 1, 0) + F(0, -1, 0) - 2 * c, hzz = F(0, 0, 1) + F(0, 0, -1) - 2 * c;
          const float hxy = 0.25f * (F(1, 1, 0) + F(-1, -1, 0) - F(1, -1, 0) - F(-1, 1, 0));
          const float hyz = 0.25f * (F(0, 1, 1) + F(0, -1, -1) - F(0, 1, -1) - F(0, -1, 1));
          const float hxz = 0.25f * (F(1, 0, 1) + F(-1, 0, -1) - F(-1, 0, 1) - F(1, 0, -1));
#undef F
          const double M[3][3] = {{hxx, hxy, hxz}, {hxy, hyy, hyz}, {hxz, hyz, hzz}};
          double ev[3], E[3][3];
          vo_diagonalize_sym3(M, ev, E, 0);                  // increasing; then DECREASING_ABS_EIVALS (:252-264)
          if (std::fabs(ev[0]) < std::fabs(ev[2])) {
            std::swap(ev[0], ev[2]);
            for (int d = 0; d < 3; d++) std::swap(E[0][d], E[2][d]);
          }
          float v1[3] = {(float)E[0][0], (float)E[0][1], (float)E[0][2]};
          const float l1 = (float)ev[0];
          float along = g[0] * v1[0] + g[1] * v1[1] + g[2] * v1[2];
          if (along < 0.0f) { along = -along; for (int d = 0; d < 3; d++) v1[d] = -v1[d]; }
          else if (along == 0.0f) continue;
          const float dist = (l1 != 0) ? along / l1 : INFINITY;
          if (max_distance > 0.0f && std::fabs(dist) > max_distance) continue;
          for (int d = 0; d < 3; d++) xyz[d] = q[d] - dist * v1[d];
          if (xyz[0] < 0.0f || size[0] < xyz[0] || xyz[1] < 0.0f || size[1] < xyz[1] || xyz[2] < 0.0f || size[2] < xyz[2]) continue;
          for (int d = 0; d < 3; d++) xyz[d] *= voxel_width[d];
        }
        emit(xyz, normal);
      }
  return n_out;
}

} // extern "C"
