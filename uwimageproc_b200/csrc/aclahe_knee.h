// aclahe_knee.h - the knee search of ParametrosACLAHE (modules/aclahe/python/functions.py:49-93, ACLAHE.py:92-96) in plain
// C++ that compiles for the host and the device: the 49 entropy samples of one block size are fitted with
//   f(u) = p0 exp(-p1 u) + p2 exp(-p3 u),  u = 1 .. 49,
// by scipy.optimize.curve_fit (MINPACK lmdif as scipy.optimize.leastsq calls it: forward-difference Jacobian with step
// sqrt(DBL_EPSILON) |x|, ftol = xtol = 1.49012e-8, gtol = 0, factor = 100, mode = 1, maxfev = 200 (n + 1) = 1000), the fit
// is sampled at u = 1 .. 25 and interpolated by a cubic spline (splrep with s = 0: the not-a-knot interpolant), and the
// curvature |x'y'' - y'x''| / (x'^2 + y'^2)^1.5 of the (clip, entropy) curve is taken at linspace(1, 25, 49); the knee is
// the index of its first maximum.
//
// The arithmetic must round like the reference's double-precision code: build it without floating-point contraction
// (nvcc --fmad=false, g++ -ffp-contract=off).  Only exp and pow come from the platform's libm; they may differ from
// glibc's by an ulp, which can change the number of function evaluations of a fit but has not moved a knee.
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define KNEE_HD __host__ __device__
#else
#define KNEE_HD
#endif

namespace knee {

constexpr int M = 49;   // samples per curve (graficar keeps entries 1..49 of the 51-entry table rows)
constexpr int N = 4;    // parameters of the double exponential
constexpr int NS = 25;  // spline nodes, linspace(1, 25, 25)
constexpr int NE = 49;  // evaluation points, linspace(1, 25, 49)
constexpr int MAXFEV = 200 * (N + 1);
constexpr double FTOL = 1.49012e-8, XTOL = 1.49012e-8, GTOL = 0.0, FACTOR = 100.0;
constexpr double EPSMCH = 2.220446049250313e-16;  // dpmpar(1) = DBL_EPSILON
constexpr double DWARF = 2.2250738585072014e-308; // dpmpar(2) = DBL_MIN

KNEE_HD inline double dmax(double a, double b) { return a > b ? a : b; }
KNEE_HD inline double dmin(double a, double b) { return a < b ? a : b; }

// curve_fit's residual: f(u, *p) - y with the operations in numpy's order
KNEE_HD inline double model(const double* p, double t) { return p[0] * exp(-p[1] * t) + p[2] * exp(-p[3] * t); }
KNEE_HD inline void residual(const double* p, const double* y, double* fv) {
  for (int i = 0; i < M; i++) fv[i] = model(p, (double)(i + 1)) - y[i];
}

// MINPACK enorm: Euclidean norm with the rdwarf / rgiant scaling
KNEE_HD inline double enorm(int n, const double* x) {
  const double rdwarf = 3.834e-20, rgiant = 1.304e19;
  double s1 = 0, s2 = 0, s3 = 0, x1max = 0, x3max = 0;
  const double agiant = rgiant / (double)n;
  for (int i = 0; i < n; i++) {
    const double xabs = fabs(x[i]);
    if (xabs > rdwarf && xabs < agiant) {
      s2 += xabs * xabs;
    } else if (xabs <= rdwarf) {
      if (xabs <= x3max) {
        if (xabs != 0) { const double r = xabs / x3max; s3 += r * r; }
      } else {
        const double r = x3max / xabs;
        s3 = 1.0 + s3 * r * r;
        x3max = xabs;
      }
    } else {
      if (xabs <= x1max) {
        const double r = xabs / x1max;
        s1 += r * r;
      } else {
        const double r = x1max / xabs;
        s1 = 1.0 + s1 * r * r;
        x1max = xabs;
      }
    }
  }
  if (s1 != 0) return x1max * sqrt(s1 + (s2 / x1max) / x1max);
  if (s2 != 0) {
    if (s2 >= x3max) return sqrt(s2 * (1.0 + (x3max / s2) * (x3max * s3)));
    return sqrt(x3max * ((s2 / x3max) + (x3max * s3)));
  }
  return x3max * sqrt(s3);
}

// MINPACK qrfac with column pivoting on the M x N column-major matrix a (leading dimension M)
KNEE_HD inline void qrfac(double* a, int* ipvt, double* rdiag, double* acnorm, double* wa) {
  for (int j = 0; j < N; j++) {
    acnorm[j] = enorm(M, a + j * M);
    rdiag[j] = acnorm[j];
    wa[j] = rdiag[j];
    ipvt[j] = j;
  }
  for (int j = 0; j < N; j++) {
    int kmax = j;
    for (int k = j; k < N; k++)
      if (rdiag[k] > rdiag[kmax]) kmax = k;
    if (kmax != j) {
      for (int i = 0; i < M; i++) { const double t = a[i + j * M]; a[i + j * M] = a[i + kmax * M]; a[i + kmax * M] = t; }
      rdiag[kmax] = rdiag[j];
      wa[kmax] = wa[j];
      const int k = ipvt[j]; ipvt[j] = ipvt[kmax]; ipvt[kmax] = k;
    }
    double ajnorm = enorm(M - j, a + j + j * M);
    if (ajnorm != 0) {
      if (a[j + j * M] < 0) ajnorm = -ajnorm;
      for (int i = j; i < M; i++) a[i + j * M] = a[i + j * M] / ajnorm;
      a[j + j * M] = a[j + j * M] + 1.0;
      for (int k = j + 1; k < N; k++) {
        double sum = 0;
        for (int i = j; i < M; i++) sum += a[i + j * M] * a[i + k * M];
        const double temp = sum / a[j + j * M];
        for (int i = j; i < M; i++) a[i + k * M] -= temp * a[i + j * M];
        if (rdiag[k] != 0) {
          const double t = a[j + k * M] / rdiag[k];
          rdiag[k] = rdiag[k] * sqrt(dmax(0.0, 1.0 - t * t));
          const double q = rdiag[k] / wa[k];
          if (0.05 * (q * q) <= EPSMCH) {
            rdiag[k] = enorm(M - j - 1, a + (j + 1) + k * M);
            wa[k] = rdiag[k];
          }
        }
      }
    }
    rdiag[j] = -ajnorm;
  }
}

// MINPACK qrsolv on the upper triangle of r (leading dimension M)
KNEE_HD inline void qrsolv(double* r, const int* ipvt, const double* diag, const double* qtb, double* x, double* sdiag, double* wa) {
  for (int j = 0; j < N; j++) {
    for (int i = j; i < N; i++) r[i + j * M] = r[j + i * M];
    x[j] = r[j + j * M];
    wa[j] = qtb[j];
  }
  for (int j = 0; j < N; j++) {
    const int l = ipvt[j];
    if (diag[l] != 0) {
      for (int k = j; k < N; k++) sdiag[k] = 0;
      sdiag[j] = diag[l];
      double qtbpj = 0;
      for (int k = j; k < N; k++) {
        if (sdiag[k] == 0) continue;
        double sn, cs;
        if (fabs(r[k + k * M]) < fabs(sdiag[k])) {
          const double cotan = r[k + k * M] / sdiag[k];
          sn = 0.5 / sqrt(0.25 + 0.25 * (cotan * cotan));
          cs = sn * cotan;
        } else {
          const double tn = sdiag[k] / r[k + k * M];
          cs = 0.5 / sqrt(0.25 + 0.25 * (tn * tn));
          sn = cs * tn;
        }
        r[k + k * M] = cs * r[k + k * M] + sn * sdiag[k];
        const double temp = cs * wa[k] + sn * qtbpj;
        qtbpj = -sn * wa[k] + cs * qtbpj;
        wa[k] = temp;
        for (int i = k + 1; i < N; i++) {
          const double t = cs * r[i + k * M] + sn * sdiag[i];
          sdiag[i] = -sn * r[i + k * M] + cs * sdiag[i];
          r[i + k * M] = t;
        }
      }
    }
    sdiag[j] = r[j + j * M];
    r[j + j * M] = x[j];
  }
  int nsing = N;
  for (int j = 0; j < N; j++) {
    if (sdiag[j] == 0 && nsing == N) nsing = j;
    if (nsing < N) wa[j] = 0;
  }
  for (int j = nsing - 1; j >= 0; j--) {
    double sum = 0;
    for (int i = j + 1; i < nsing; i++) sum += r[i + j * M] * wa[i];
    wa[j] = (wa[j] - sum) / sdiag[j];
  }
  for (int j = 0; j < N; j++) x[ipvt[j]] = wa[j];
}

// MINPACK lmpar: Levenberg-Marquardt parameter for the trust region of radius delta
KNEE_HD inline void lmpar(double* r, const int* ipvt, const double* diag, const double* qtb, double delta, double& par, double* x,
                          double* sdiag, double* wa1, double* wa2) {
  int nsing = N;
  for (int j = 0; j < N; j++) {
    wa1[j] = qtb[j];
    if (r[j + j * M] == 0 && nsing == N) nsing = j;
    if (nsing < N) wa1[j] = 0;
  }
  for (int j = nsing - 1; j >= 0; j--) {
    wa1[j] = wa1[j] / r[j + j * M];
    const double temp = wa1[j];
    for (int i = 0; i < j; i++) wa1[i] -= r[i + j * M] * temp;
  }
  for (int j = 0; j < N; j++) x[ipvt[j]] = wa1[j];
  int iter = 0;
  for (int j = 0; j < N; j++) wa2[j] = diag[j] * x[j];
  double dxnorm = enorm(N, wa2);
  double fp = dxnorm - delta;
  if (fp <= 0.1 * delta) {
    par = 0;   // iter == 0
    return;
  }
  double parl = 0;
  if (nsing >= N) {
    for (int j = 0; j < N; j++) { const int l = ipvt[j]; wa1[j] = diag[l] * (wa2[l] / dxnorm); }
    for (int j = 0; j < N; j++) {
      double sum = 0;
      for (int i = 0; i < j; i++) sum += r[i + j * M] * wa1[i];
      wa1[j] = (wa1[j] - sum) / r[j + j * M];
    }
    const double temp = enorm(N, wa1);
    parl = ((fp / delta) / temp) / temp;
  }
  for (int j = 0; j < N; j++) {
    double sum = 0;
    for (int i = 0; i <= j; i++) sum += r[i + j * M] * qtb[i];
    wa1[j] = sum / diag[ipvt[j]];
  }
  const double gnorm = enorm(N, wa1);
  double paru = gnorm / delta;
  if (paru == 0) paru = DWARF / dmin(delta, 0.1);
  par = dmax(par, parl);
  par = dmin(par, paru);
  if (par == 0) par = gnorm / dxnorm;
  for (;;) {
    iter++;
    if (par == 0) par = dmax(DWARF, 0.001 * paru);
    double temp = sqrt(par);
    for (int j = 0; j < N; j++) wa1[j] = temp * diag[j];
    qrsolv(r, ipvt, wa1, qtb, x, sdiag, wa2);
    for (int j = 0; j < N; j++) wa2[j] = diag[j] * x[j];
    dxnorm = enorm(N, wa2);
    temp = fp;
    fp = dxnorm - delta;
    if (fabs(fp) <= 0.1 * delta || (parl == 0 && fp <= temp && temp < 0) || iter == 10) break;
    for (int j = 0; j < N; j++) { const int l = ipvt[j]; wa1[j] = diag[l] * (wa2[l] / dxnorm); }
    for (int j = 0; j < N; j++) {
      wa1[j] = wa1[j] / sdiag[j];
      const double t = wa1[j];
      for (int i = j + 1; i < N; i++) wa1[i] -= r[i + j * M] * t;
    }
    temp = enorm(N, wa1);
    const double parc = ((fp / delta) / temp) / temp;
    if (fp > 0) parl = dmax(parl, par);
    if (fp < 0) paru = dmin(paru, par);
    par = dmax(parl, par + parc);
  }
}

// MINPACK lmdif for the double exponential from p = (7, 0.4, 0.9, 5).  Returns info (1..4: converged; 5: maxfev reached;
// 6..8: tolerances too small), the parameters in p and the number of residual evaluations in *nfev.
KNEE_HD inline int fit(const double* y, double* p, int* nfev_out) {
  double fvec[M], fjac[M * N], wa4[M];
  double diag[N], qtf[N], wa1[N], wa2[N], wa3[N];
  int ipvt[N];
  p[0] = 7; p[1] = 0.4; p[2] = 0.9; p[3] = 5;
  int info = 0, nfev = 0;
  residual(p, y, fvec);
  nfev = 1;
  double fnorm = enorm(M, fvec);
  double par = 0, delta = 0, xnorm = 0;
  int iter = 1;
  const double eps = sqrt(EPSMCH);   // sqrt(max(epsfcn, epsmch)) with scipy's epsfcn = DBL_EPSILON
  for (;;) {
    // fdjac2: forward differences
    for (int j = 0; j < N; j++) {
      const double temp = p[j];
      double h = eps * fabs(temp);
      if (h == 0) h = eps;
      p[j] = temp + h;
      residual(p, y, wa4);
      p[j] = temp;
      for (int i = 0; i < M; i++) fjac[i + j * M] = (wa4[i] - fvec[i]) / h;
    }
    nfev += N;
    qrfac(fjac, ipvt, wa1, wa2, wa3);
    if (iter == 1) {
      for (int j = 0; j < N; j++) {
        diag[j] = wa2[j];
        if (wa2[j] == 0) diag[j] = 1;
      }
      for (int j = 0; j < N; j++) wa3[j] = diag[j] * p[j];
      xnorm = enorm(N, wa3);
      delta = FACTOR * xnorm;
      if (delta == 0) delta = FACTOR;
    }
    for (int i = 0; i < M; i++) wa4[i] = fvec[i];
    for (int j = 0; j < N; j++) {
      if (fjac[j + j * M] != 0) {
        double sum = 0;
        for (int i = j; i < M; i++) sum += fjac[i + j * M] * wa4[i];
        const double temp = -sum / fjac[j + j * M];
        for (int i = j; i < M; i++) wa4[i] += fjac[i + j * M] * temp;
      }
      fjac[j + j * M] = wa1[j];
      qtf[j] = wa4[j];
    }
    double gnorm = 0;
    if (fnorm != 0) {
      for (int j = 0; j < N; j++) {
        const int l = ipvt[j];
        if (wa2[l] != 0) {
          double sum = 0;
          for (int i = 0; i <= j; i++) sum += fjac[i + j * M] * (qtf[i] / fnorm);
          gnorm = dmax(gnorm, fabs(sum / wa2[l]));
        }
      }
    }
    if (gnorm <= GTOL) info = 4;
    if (info != 0) break;
    for (int j = 0; j < N; j++) diag[j] = dmax(diag[j], wa2[j]);
    double ratio;
    do {
      lmpar(fjac, ipvt, diag, qtf, delta, par, wa1, wa2, wa3, wa4);
      for (int j = 0; j < N; j++) {
        wa1[j] = -wa1[j];
        wa2[j] = p[j] + wa1[j];
        wa3[j] = diag[j] * wa1[j];
      }
      const double pnorm = enorm(N, wa3);
      if (iter == 1) delta = dmin(delta, pnorm);
      residual(wa2, y, wa4);
      nfev += 1;
      const double fnorm1 = enorm(M, wa4);
      double actred = -1;
      if (0.1 * fnorm1 < fnorm) { const double q = fnorm1 / fnorm; actred = 1.0 - q * q; }
      for (int j = 0; j < N; j++) {
        wa3[j] = 0;
        const double temp = wa1[ipvt[j]];
        for (int i = 0; i <= j; i++) wa3[i] += fjac[i + j * M] * temp;
      }
      const double temp1 = enorm(N, wa3) / fnorm;
      const double temp2 = (sqrt(par) * pnorm) / fnorm;
      const double prered = temp1 * temp1 + temp2 * temp2 / 0.5;
      const double dirder = -(temp1 * temp1 + temp2 * temp2);
      ratio = 0;
      if (prered != 0) ratio = actred / prered;
      if (ratio <= 0.25) {
        double temp = 0.5;
        if (actred < 0) temp = 0.5 * dirder / (dirder + 0.5 * actred);
        if (0.1 * fnorm1 >= fnorm || temp < 0.1) temp = 0.1;
        delta = temp * dmin(delta, pnorm / 0.1);
        par = par / temp;
      } else if (par == 0 || ratio >= 0.75) {
        delta = pnorm / 0.5;
        par = 0.5 * par;
      }
      if (ratio >= 1e-4) {
        for (int j = 0; j < N; j++) { p[j] = wa2[j]; wa2[j] = diag[j] * p[j]; }
        for (int i = 0; i < M; i++) fvec[i] = wa4[i];
        xnorm = enorm(N, wa2);
        fnorm = fnorm1;
        iter++;
      }
      if (fabs(actred) <= FTOL && prered <= FTOL && 0.5 * ratio <= 1) info = 1;
      if (delta <= XTOL * xnorm) info = 2;
      if (fabs(actred) <= FTOL && prered <= FTOL && 0.5 * ratio <= 1 && info == 2) info = 3;
      if (info != 0) break;
      if (nfev >= MAXFEV) info = 5;
      if (fabs(actred) <= EPSMCH && prered <= EPSMCH && 0.5 * ratio <= 1) info = 6;
      if (delta <= EPSMCH * xnorm) info = 7;
      if (gnorm <= EPSMCH) info = 8;
      if (info != 0) break;
    } while (ratio < 1e-4);
    if (info != 0) break;
  }
  if (nfev_out) *nfev_out = nfev;
  return info;
}

// first and second derivative at linspace(1, 25, 49) of the not-a-knot cubic spline through (k, model(p, k)), k = 1 .. 25
KNEE_HD inline void spline_derivs(const double* p, double* d1, double* d2) {
  double y[NS], mm[NS], c[NS], rhs[NS];
  for (int i = 0; i < NS; i++) y[i] = model(p, (double)(i + 1));
  // unit spacing: M[i-1] + 4 M[i] + M[i+1] = 6 (y[i+1] - 2 y[i] + y[i-1]); not-a-knot (M[0] = 2 M[1] - M[2] and its mirror)
  // turns the first and last rows into 6 M[1] = rhs[1], 6 M[NS-2] = rhs[NS-2]
  for (int i = 1; i < NS - 1; i++) rhs[i] = 6.0 * ((y[i + 1] - y[i]) - (y[i] - y[i - 1]));
  mm[1] = rhs[1] / 6.0;
  mm[NS - 2] = rhs[NS - 2] / 6.0;
  // rows 2 .. NS-3: tridiagonal (1, 4, 1) with the two known ends moved to the right-hand side
  rhs[2] -= mm[1];
  rhs[NS - 3] -= mm[NS - 2];
  c[2] = 1.0 / 4.0;
  rhs[2] = rhs[2] / 4.0;
  for (int i = 3; i <= NS - 3; i++) {
    const double den = 4.0 - c[i - 1];
    c[i] = 1.0 / den;
    rhs[i] = (rhs[i] - rhs[i - 1]) / den;
  }
  mm[NS - 3] = rhs[NS - 3];
  for (int i = NS - 4; i >= 2; i--) mm[i] = rhs[i] - c[i] * mm[i + 1];
  mm[0] = 2.0 * mm[1] - mm[2];
  mm[NS - 1] = 2.0 * mm[NS - 2] - mm[NS - 3];
  for (int j = 0; j < NE; j++) {
    int i = j / 2;
    double t = 0.5 * (j - 2 * i);
    if (i > NS - 2) { i = NS - 2; t = 1.0; }
    const double s = 1.0 - t;
    d1[j] = -mm[i] * (s * s) / 2.0 + mm[i + 1] * (t * t) / 2.0 + (y[i + 1] - y[i]) - (mm[i + 1] - mm[i]) / 6.0;
    d2[j] = mm[i] * s + mm[i + 1] * t;
  }
}

// index of the first maximum of the curvature (numpy's argmax: a NaN wins at its first position)
KNEE_HD inline int curvature_argmax(const double* x1, const double* x2, const double* y1, const double* y2) {
  int best = 0;
  double kb = 0;
  for (int j = 0; j < NE; j++) {
    const double c = x1[j] * y2[j] - y1[j] * x2[j];
    const double s = x1[j] * x1[j] + y1[j] * y1[j];
    const double k = sqrt(c * c) / sqrt(pow(s, 3.0));
    if (k != k) return j;
    if (j == 0 || k > kb) { kb = k; best = j; }
  }
  return best;
}

// derivatives of one fitted curve; false when the fit fails (curve_fit raises: ier not in 1..4)
KNEE_HD inline bool curve_derivs(const double* v, double* d1, double* d2, double* p_out = nullptr, int* nfev = nullptr) {
  double p[N];
  const int info = fit(v, p, nfev);
  if (p_out) for (int j = 0; j < N; j++) p_out[j] = p[j];
  if (info < 1 || info > 4) return false;
  spline_derivs(p, d1, d2);
  return true;
}

// the knee of one entropy curve y[49] (float32 entropies at clip limits 0.5 .. 24.5) given the derivatives of the clip
// curve; -1 when the fit of y fails
KNEE_HD inline int knee_of(const float* yf, const double* x1, const double* x2) {
  double y[M], y1[NE], y2[NE];
  for (int i = 0; i < M; i++) y[i] = (double)yf[i];
  if (!curve_derivs(y, y1, y2)) return -1;
  return curvature_argmax(x1, x2, y1, y2);
}

// the clip curve: float32 clip limits 0.5 .. 24.5 (exact in float32), the same for every frame
KNEE_HD inline bool clip_curve_derivs(double* x1, double* x2) {
  double x[M];
  for (int i = 0; i < M; i++) x[i] = 0.5 * (i + 1);
  return curve_derivs(x, x1, x2);
}

}  // namespace knee
