// k_input.cuh — device kernels for BA::interpInputData (batotp/ba.cpp:95-316) and the
// Spline / util / Robot helpers it calls.  Reference lines are cited per kernel.
//
// Kernel shapes:  T  = one thread per trajectory (strictly sequential walkers)
//                 TR = one thread per (trajectory, coordinate row) (Thomas recurrences)
//                 TP = one thread per (trajectory, point), trajectories fastest (pointwise evaluation)
// All row arrays are point-major [point][trajectory][row] (ba_dev.cuh), accessed through RV views.
#pragma once
#include "ba_dev.cuh"
#include "k_trig.cuh"

// ----------------------------------------------------------------------------- spline primitives
// Thomas elimination factors depend only on the row index, so they are tabulated once on the
// host with the very divisions spline.cpp performs:  natural (spline.cpp:259-268):
// cN[1]=1/4, cN[i]=1/(4-cN[i-1]);  clamped (spline.cpp:229-237): cC[0]=1/2, cC[i]=1/(4-cC[i-1]).
// The elimination denominators 4 - c[i-1] are tabulated with them, together with their correctly rounded
// reciprocals, so that the recurrence divides through sdiv::div (the same quotient as '/', a third of the
// dependent latency).
struct ThomasTabs {
  const double *cN, *dN, *rN;  // natural: factor, denominator of row i, RN(1/denominator)
  const double *cC, *dC, *rC;  // clamped (rows with diagonal 4)
};

// spline.cpp:168-211 + 252-276: y[n] -> second-derivative solution m[n] ("natural", quirk Q4)
template <class VY, class VM>
__host__ __device__ inline void thomas_natural(const VY &y, const VM &m, int npts, const ThomasTabs &tb) {
  const int n = npts - 1;
  m[0] = 0.0;
  m[npts - 1] = 0.0;
  const double a = 1.0, b = 4.0;
  const double *cN = tb.cN;
  // rhs and forward elimination in one pass (each m[i] depends on y[i-1..i+1] and m[i-1] only).  The loads
  // do not depend on the recurrence: they are issued four rows ahead of it.
  double ym = y[0], yc = y[1], prev = 0.0;
  int i = 1;
  for (; i + 3 < npts - 1; i += 4) {
    const double y1 = y[i + 1], y2 = y[i + 2], y3 = y[i + 3], y4 = y[i + 4];
    const double d1 = tb.dN[i], d2 = tb.dN[i + 1], d3 = tb.dN[i + 2], d4 = tb.dN[i + 3];
    const double r1 = tb.rN[i], r2 = tb.rN[i + 1], r3 = tb.rN[i + 2], r4 = tb.rN[i + 3];
    double v = 6 * (ym - 2 * yc + y1);
    if (i == 1)
      v /= b;
    else
      v = sdiv::div(v - a * prev, d1, sdiv::Rcp{r1, true});  // (v - a*prev) / (b - a*cN[i-1])
    m[i] = v;
    prev = v;
    v = sdiv::div(6 * (yc - 2 * y1 + y2) - a * prev, d2, sdiv::Rcp{r2, true});
    m[i + 1] = v;
    prev = v;
    v = sdiv::div(6 * (y1 - 2 * y2 + y3) - a * prev, d3, sdiv::Rcp{r3, true});
    m[i + 2] = v;
    prev = v;
    v = sdiv::div(6 * (y2 - 2 * y3 + y4) - a * prev, d4, sdiv::Rcp{r4, true});
    m[i + 3] = v;
    prev = v;
    ym = y3;
    yc = y4;
  }
  for (; i < npts - 1; ++i) {
    const double yp = y[i + 1];
    double v = 6 * (ym - 2 * yc + yp);
    if (i == 1)
      v /= b;
    else
      v = sdiv::div(v - a * prev, tb.dN[i], sdiv::Rcp{tb.rN[i], true});
    m[i] = v;
    prev = v;
    ym = yc;
    yc = yp;
  }
  double last = (0.0 - a * prev) / (b - a * cN[n - 1]);  // the last unknown is an ordinary row with rhs 0
  m[n] = last;
  int k = n;
  for (; k - 4 >= 1; k -= 4) {  // rows k-1 .. k-4
    const double m1 = m[k - 1], m2 = m[k - 2], m3 = m[k - 3], m4 = m[k - 4];
    const double c1 = cN[k - 1], c2 = cN[k - 2], c3 = cN[k - 3], c4 = cN[k - 4];
    double v = m1 - c1 * last;
    m[k - 1] = v;
    last = v;
    v = m2 - c2 * last;
    m[k - 2] = v;
    last = v;
    v = m3 - c3 * last;
    m[k - 3] = v;
    last = v;
    v = m4 - c4 * last;
    m[k - 4] = v;
    last = v;
  }
  for (; k > 1; --k) {
    const double v = m[k - 1] - cN[k - 1] * last;
    m[k - 1] = v;
    last = v;
  }
}

// spline.cpp:225-243 ("clamped": b0=b_{n-1}=2, back-substitution starts at n-3, quirk Q4)
template <class VY, class VM>
__host__ __device__ inline void thomas_clamped(const VY &y, const VM &m, int n, const ThomasTabs &tb) {
  const double a = 1.0;
  const double *cC = tb.cC;
  double prev = 0.0 / 2.0;
  m[0] = prev;
  double ym = y[0], yc = y[1];
  for (int i = 1; i < n; ++i) {
    double rhs = 0.0;
    if (i < n - 1) {
      const double yp = y[i + 1];
      rhs = 6 * (ym - 2 * yc + yp);
      ym = yc;
      yc = yp;
    }
    double v;
    if (i == n - 1)
      v = (rhs - a * prev) / (2.0 - a * cC[i - 1]);
    else
      v = sdiv::div(rhs - a * prev, tb.dC[i], sdiv::Rcp{tb.rC[i], true});  // / (4.0 - a*cC[i-1])
    m[i] = v;
    prev = v;
  }
  for (int i = n - 2; i-- > 0;) m[i] = m[i] - cC[i] * m[i + 1];
}

// spline.cpp:203-209: coefficients of segment k from knot values and the solution
struct Seg4 {
  double c0, c1, c2, c3;
};
template <class VY, class VM>
__host__ __device__ __forceinline__ Seg4 seg_coef(const VY &y, const VM &m, int k) {
  Seg4 s;
  const double y0 = y[k], y1 = y[k + 1], m0 = m[k], m1 = m[k + 1];
  s.c3 = sdiv::div6(m1 - m0);
  s.c2 = m0 / 2.0;
  s.c1 = y1 - y0 - sdiv::div6(m1 + 2 * m0);
  s.c0 = y0;
  return s;
}
__host__ __device__ __forceinline__ double seg_value(const Seg4 &c, double tau, double tau2, double tau3) {
  return c.c3 * tau3 + c.c2 * tau2 + c.c1 * tau + c.c0;
}

// spline.cpp:64-75 for one output site when the sites are non-decreasing: the monotone cursor
// stops at the first segment with aOut < aIn[seg+1] (capped at nIn-2) == this binary search.
template <class AIn>
__host__ __device__ __forceinline__ int find_seg(const AIn &aIn, int nIn, double aOut) {
  int lo = 0, hi = nIn - 2;  // answer in [lo, hi]
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (aOut < aIn(mid + 1))
      hi = mid;
    else
      lo = mid + 1;
  }
  return lo;
}

// the same answer from a starting guess (sites that are nearly uniform: two or three probes instead of
// log2(n)): the first k with aOut < aIn[k+1] cannot lie below a k with aIn[k] <= aOut
template <class AIn>
__host__ __device__ __forceinline__ int find_seg_from(const AIn &aIn, int nIn, double aOut, int guess) {
  int k = imin_(imax_(guess, 0), nIn - 2);
  while (k > 0 && aOut < aIn(k)) k--;
  while (k < nIn - 2 && !(aOut < aIn(k + 1))) k++;
  return k;
}

struct UniformSites {  // a[k] = res * k   (util.h:101-107 applied to an iota, e.g. ba.cpp:803-805)
  double res;
  __host__ __device__ __forceinline__ double operator()(int k) const { return res * (double)k; }
};
struct ViewSites {
  RV a;
  __host__ __device__ __forceinline__ double operator()(int k) const { return a[k]; }
};

// (trajectory, point) decomposition with trajectories fastest.  The launch (LAUNCH_TP) uses a 3-D grid:
// x covers the nb trajectories of a point (blockDim.x lanes), y/z the points (blockDim.y per block), so no
// thread pays a 64-bit division to find its indices.
#define TP_DECOMP(nb)                                                                      \
  const int bl = (int)(blockIdx.x * blockDim.x + threadIdx.x);                             \
  const int i = (int)((blockIdx.z * gridDim.y + blockIdx.y) * blockDim.y + threadIdx.y);   \
  if (bl >= (nb)) return
// (point, trajectory) decomposition with points fastest (row-contiguous float outputs)
#define PT_DECOMP(npts)                                                                    \
  const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);                              \
  const int bl = (int)((blockIdx.z * gridDim.y + blockIdx.y) * blockDim.y + threadIdx.y);  \
  if (i >= (npts)) return

// ----------------------------------------------------------------------------- load (TP)
// trajReadBIN / trajReadCSV payload -> FP64 rows (ba.cpp:2283-2299, 2417-2437)
template <typename T>
__global__ void k_in_load(WSP, const T *theta, const T *cart, const int *n0, const double *tres,
                          int n0max, int nb) {
  TP_DECOMP(nb);
  const int b = bl;
  if (i >= n0max) return;
  const int n = n0 ? n0[b] : n0max;
  if (i == 0) {
    TrajState &s = w.st[b];
    // a limit row the host rejected (NaN throughout) keeps its trajectory out of every stage
    s.status = (w.lim && w.lim[b].jnt_vel_max[0] != w.lim[b].jnt_vel_max[0]) ? ST_UNSUPPORTED : 0;
    s.nPts = n;
    s.tresInput = tres[b];
    s.sres = tres[b];
    s.scaleType = CFG.c.scale_type;
    s.integRes = CFG.c.integ_res;
    s.isParallelMech = CFG.c.is_parallel;
    for (int q = 0; q < 3; ++q) s.sWeights[q] = CFG.c.s_weights[q];
    for (int q = 0; q < MAXD; ++q) s.cartpt[q] = 0.0;
    s.sLastSec = 0.0;
    s.nRev = s.nFwd = s.nOver = s.nSm = s.nOut = 0;
    s.tRev = s.tFwd = 0.0;
    s.nVerify = 0;
  }
  if (i >= n) return;
  double *dst = w.P + ((size_t)i * w.B + b) * w.R;
  for (int j = 0; j < CFG.J; ++j) dst[j] = theta ? (double)theta[((size_t)b * CFG.J + j) * n0max + i] : 0.0;
  for (int j = 0; j < CFG.R - CFG.J; ++j) {  // the stored Cartesian rows
    double v = 0.0;
    if (cart && j < CFG.Cin) v = (double)cart[((size_t)b * CFG.Cin + j) * n0max + i];
    dst[CFG.J + j] = v;
  }
}

// ----------------------------------------------------------------------------- helpers (T)
// ba.cpp:2768-2794 with nPtsOld <= 3 -> 4 points (interpTrajLinear) ; tiny, done in-thread.
__host__ __device__ inline void traj_linear_to4(const Ws &w, double *base, int b, TrajState &s, int rows) {
  const int nOld = s.nPts, nNew = 4;
  UniformSites so{1.0 / (nOld - 1)}, sn{1.0 / (nNew - 1)};
  int seg[4];
  double tau[4];
  for (int i = 0; i < nNew; ++i) {
    const double a = sn(i);
    seg[i] = find_seg(so, nOld, a);
    tau[i] = (a - so(seg[i])) / (so(seg[i] + 1) - so(seg[i]));
  }
  for (int r = 0; r < rows; ++r) {
    const RV x = rowv(base, w, b, r);
    double o[4];
    for (int i = 0; i < nNew; ++i) o[i] = x[seg[i]] + (x[seg[i] + 1] - x[seg[i]]) * tau[i];
    for (int i = 0; i < nNew; ++i) x[i] = o[i];
  }
  s.sres = s.sres * (nOld - 1) / (nNew - 1);
  s.nPts = nNew;
}

// ----------------------------------------------------------------------------- prepare (T)
// ba.cpp:98-183: timestamp de-duplication, length guards, remClosePts (util.cpp:452-524).
// `ts` (optional) [B][n0max] timestamps of a CSV path; scratch lives in w.sC / w.nrm.
__global__ void k_in_prepare(WSP, const double *ts, int n0max, int hasTheta, int hasCart) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;  // (a rejected limit row, k_in_load)
  const int J = CFG.J, R = CFG.R;
  int nPts = s.nPts;
  const RV scr = RV{w.nrm + (size_t)b * 2, (size_t)w.B * 2};  // per-trajectory scratch vector
  if (ts) {  // ba.cpp:98-127 — the index list is a vector<uint8_t>, so indices wrap at 256
    const double *t = ts + (size_t)b * n0max;
    const RV tt = vecv(w.sC, w, b);  // working copy of the timestamps
    for (int i = 0; i < nPts; ++i) tt[i] = t[i];
    int nRem = 0;
    for (int i = 1; i < nPts; ++i)
      if (tt[i] == tt[i - 1]) scr[nRem++] = (double)(unsigned char)i;
    int n = nPts;
    for (int r = nRem - 1; r >= 0; --r) {
      const int k = (int)scr[r];
      for (int i = k; i < n - 1; ++i) tt[i] = tt[i + 1];
      for (int row = 0; row < R; ++row) {
        const RV x = rowv(w.P, w, b, row);
        for (int i = k; i < n - 1; ++i) x[i] = x[i + 1];
      }
      n--;
    }
    nPts = n;
    s.nPts = nPts;
    s.tresInput = tt[nPts - 1] / (nPts - 1);
    s.sres = s.tresInput;
  }
  if (nPts == 1) {
    s.status |= ST_TOO_SHORT;
    return;
  }
  if (nPts < 4) {
    traj_linear_to4(w, w.P, b, s, R);
    nPts = s.nPts;
  }
  if (CFG.c.is_interp_only) {
    // ba.cpp:139-159: no optimisation, the path is only re-sampled at outRes.  Plan of
    // evalSplineFullTraj(traj, traj.sres, _outRes) (ba.cpp:794-819); the sites are the de-duplicated
    // timestamps when the file had them (already in sC), sres*k otherwise.
    const double oldRes = s.sres;
    int nNew = (int)ceil(oldRes / CFG.c.out_res * (nPts - 1)) + 1;
    nNew = imax_(nNew, 4);
    const RV sC = vecv(w.sC, w, b);
    if (!ts)
      for (int i = 0; i < nPts; ++i) sC[i] = oldRes * (double)i;
    s.sScale = sC[nPts - 1] / (double)(nNew - 1);
    s.nNew = nNew;
    s.nPtsC = nPts;
    s.sresC = s.sres;
    s.vFact = 1 / s.sresC;
    s.aFact = s.vFact * s.vFact;
    s.sres = oldRes * (nPts - 1) / (nNew - 1);
    if (nNew > w.Nc) s.status |= ST_GRID_CAP;
    return;
  }
  s.sLastSec = -1;
  // remClosePts(x = driving rows, y = the others, thresh)
  const bool cartDriven = (CFG.c.path_type == BATOTP_CART);
  const int x0 = cartDriven ? J : 0, nx = cartDriven ? (hasCart ? CFG.Cin : 0) : (hasTheta ? J : 0);
  const double thr = cartDriven ? CFG.c.cart_thresh : CFG.c.jnt_thresh;
  const double thrSQ = thr * thr;
  const RV isRem = scr;
  for (int i = 0; i < nPts; ++i) isRem[i] = 0.0;
  const size_t pst = (size_t)w.B * w.R;
  double *p0 = w.P + (size_t)b * w.R;
  for (;;) {
    bool any = false;
    for (int i = 1; i < nPts; ++i) {
      double sum = 0;
      const double *a = p0 + (size_t)i * pst + x0, *a1 = p0 + (size_t)(i - 1) * pst + x0;
      for (int j = 0; j < nx; ++j) {
        const double d = a[j] - a1[j];
        sum += d * d;
      }
      if (sum < thrSQ && !(isRem[i - 1] != 0.0)) {
        isRem[i] = 1.0;
        any = true;
      }
    }
    if (isRem[nPts - 1] != 0.0 && nPts > 2) {
      isRem[nPts - 1] = 0.0;
      isRem[nPts - 2] = 1.0;
      isRem[nPts - 3] = 0.0;
    }
    if (!any) break;
    int cur = 0;
    for (int i = 0; i < nPts; ++i) {
      if (!(isRem[i] != 0.0)) {
        double *d = p0 + (size_t)cur * pst;
        const double *a = p0 + (size_t)i * pst;
        for (int row = 0; row < R; ++row) d[row] = a[row];
        cur++;
      }
    }
    nPts = cur;
    for (int i = 0; i < nPts; ++i) isRem[i] = 0.0;
  }
  s.nPts = nPts;
  if (nPts == 1) {
    s.status |= ST_TOO_SHORT;
    return;
  }
  if (nPts < 4) traj_linear_to4(w, w.P, b, s, R);
}

// ----------------------------------------------------------------------------- smooth/decimate (TR)
// util.cpp:254-288 (smooth), 343-352 (decimate) as used by ba.cpp:195-242 (quirk Q6: the
// smoothWindow branch smooths with inputDecimFact as the window).  tmp row = Q.
__host__ __device__ inline void smooth_row(const RV &x, const RV &x2, int n, int w) {
  w = imin_(w, n);
  const int wMid = w / 2 + w % 2 - 1;
  w = 2 * wMid + 1;
  x2[0] = x[0];
  x2[n - 1] = x[n - 1];
  for (int i = 1; i < wMid; ++i) {
    double xt = 0, xte = 0;
    const int nT = 2 * i + 1;
    for (int j = 0; j < nT; ++j) {
      xt += x[j];
      xte += x[n - j - 1];
    }
    x2[i] = xt / nT;
    x2[n - i - 1] = xte / nT;
  }
  for (int i = wMid; i < n - wMid; ++i) {
    double xt = 0;
    for (int j = i - wMid; j < i + wMid + 1; ++j) xt += x[j];
    x2[i] = xt / w;
  }
  for (int i = 0; i < n; ++i) x[i] = x2[i];
}

__global__ void k_in_smooth_decimate(WSP) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = t / CFG.R, row = t % CFG.R;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  const int pt = CFG.c.path_type;
  const bool isJ = row < CFG.J;
  const bool active = isJ ? (pt == BATOTP_JOINT || pt == BATOTP_BOTH) : (pt == BATOTP_CART || pt == BATOTP_BOTH);
  if (!active) return;
  const RV x = rowv(w.P, w, b, row), tmp = rowv(w.Q, w, b, row);
  int n = s.nPts;
  const int df = CFG.c.input_decim_fact;
  if (df > 1) {
    smooth_row(x, tmp, n, df);
    const int nOut = (n - 1) / df + 1;
    for (int i = 0; i < nOut; ++i) x[i] = x[df * i];
    if (df * (nOut - 1) + 1 != n) x[nOut - 1] = x[n - 1];
    n = nOut;
  }
  if (CFG.c.smooth_window > 1) smooth_row(x, tmp, n, df);
}
// after k_in_smooth_decimate: nPts, tresInput, sres bookkeeping (ba.cpp:207-223) (T)
__global__ void k_in_decim_fix(WSP) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  const int df = CFG.c.input_decim_fact;
  if (df > 1) {
    s.nPts = (s.nPts - 1) / df + 1;
    s.tresInput *= df;
    s.sres *= df;
  }
}

// ----------------------------------------------------------------------------- Robot point functions (TP)
// mode: 1 = fwdKin (theta rows -> cart rows), 2 = invKin (cart -> theta), 3 = zero cart rows,
//       4 = zero theta rows.  `base` is a point-major array of nb trajectories (b0 = first trajectory
//       of the chunk it holds); evaluated for i < st.nPts (or nOver for the output).
// robot.cpp:105-176 (KUKA; 3x3 products accumulated left to right as in oracle/eigen_standin),
// 185-202 (RR), 243-278 + 291-322 (CSPR inverse kinematics / attachment points).
__host__ __device__ inline void fk_kuka_point(const Trig &tg, const double *th, double *xyz) {
  const double D2R = 3.14159265358979323846 / 180.0;
  double c[7], s[7];
  for (int k = 0; k < 7; ++k) {
    const double tk = D2R * th[k];
    c[k] = tg.c(tk);
    s[k] = tg.s(tk);
  }
  const double c1 = c[0], c2 = c[1], c3 = c[2], c4 = c[3], c5 = c[4], c6 = c[5], c7 = c[6];
  const double s1 = s[0], s2 = s[1], s3 = s[2], s4 = s[3], s5 = s[4], s6 = s[5], s7 = s[6];
  const double Q12[3][3] = {{c1 * c2, -s1, -c1 * s2}, {c2 * s1, c1, -s1 * s2}, {s2, 0, c2}};
  const double Q34[3][3] = {{c3 * c4, -s3, c3 * s4}, {c4 * s3, c3, s3 * s4}, {-s4, 0, c4}};
  const double Q567[3][3] = {{c5 * c6 * c7 - s5 * s7, -c7 * s5 - c5 * c6 * s7, -c5 * s6},
                             {c5 * s7 + c6 * c7 * s5, c5 * c7 - c6 * s5 * s7, -s5 * s6},
                             {c7 * s6, -s6 * s7, c6}};
  double Q1234[3][3], Q[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      Q1234[i][j] = Q12[i][0] * Q34[0][j] + Q12[i][1] * Q34[1][j] + Q12[i][2] * Q34[2][j];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      Q[i][j] = Q1234[i][0] * Q567[0][j] + Q1234[i][1] * Q567[1][j] + Q1234[i][2] * Q567[2][j];
  const double tool[3] = {0, -.08, .545};
  const double a0 = .3105, a1 = .4, a2 = .39;
  const double x1 = a1 * Q12[0][2], y1 = a1 * Q12[1][2], z1 = a1 * Q12[2][2] + a0;
  const double x2 = x1 + a2 * Q1234[0][2], y2 = y1 + a2 * Q1234[1][2], z2 = z1 + a2 * Q1234[2][2];
  xyz[0] = x2 + (Q[0][0] * tool[0] + Q[0][1] * tool[1] + Q[0][2] * tool[2]);
  xyz[1] = y2 + (Q[1][0] * tool[0] + Q[1][1] * tool[1] + Q[1][2] * tool[2]);
  xyz[2] = z2 + (Q[2][0] * tool[0] + Q[2][1] * tool[1] + Q[2][2] * tool[2]);
}
__host__ __device__ inline void fk_rr_point(const Trig &tg, const double *th, double *xy) {
  const double D2R = 3.14159265358979323846 / 180.0;
  const double a1 = .4, a2 = .6;
  const double th1 = D2R * th[0], th2 = D2R * th[1];
  xy[0] = a1 * tg.c(th1) + a2 * tg.c(th1 + th2);
  xy[1] = a1 * tg.s(th1) + a2 * tg.s(th1 + th2);
}
__host__ __device__ inline void ik_cspr_point(const Pmat &pm, const double *xyz, double *rho) {
  for (int k = 0; k < 3; ++k) {
    const double rv[3] = {xyz[0] - pm.p[0][k], xyz[1] - pm.p[1][k], xyz[2] - pm.p[2][k]};
    double sumSQ = 0.0;
    for (int q = 0; q < 3; ++q) sumSQ += rv[q] * rv[q];
    rho[k] = sqrt(sumSQ);
  }
}

__global__ void k_pointfn(WSP, double *base, int b0, int mode, int useOver, Pmat pm, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const TrajState &s = w.st[b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  const int n = useOver ? s.nOver : s.nPts;
  if (i >= n) return;
  const int J = CFG.J, C = CFG.C;
  double *r0 = base + ((size_t)i * nb + bl) * CFG.R;
  if (mode == 1) {
    double th[MAXD], xyz[3];
    for (int j = 0; j < J; ++j) th[j] = r0[j];
    if (CFG.c.robot_type == BATOTP_KUKA) {
      fk_kuka_point(Trig{CFG.trigDev}, th, xyz);
      for (int q = 0; q < 3; ++q) r0[J + q] = xyz[q];
    } else if (CFG.c.robot_type == BATOTP_RR) {
      fk_rr_point(Trig{CFG.trigDev}, th, xyz);
      r0[J + 0] = xyz[0];
      r0[J + 1] = xyz[1];
    }
  } else if (mode == 2) {
    double xyz[3], rho[3];
    for (int q = 0; q < 3; ++q) xyz[q] = r0[J + q];
    ik_cspr_point(pm, xyz, rho);
    for (int q = 0; q < 3; ++q) r0[q] = rho[q];
  } else if (mode == 3) {
    for (int q = 0; q < C; ++q) r0[J + q] = 0.0;
  } else if (mode == 4) {
    for (int q = 0; q < J; ++q) r0[q] = 0.0;
  }
}

// ba.cpp:327-368 aa2qVect (sequential sign continuity) (T);  util.cpp:534-554 aa2q
__host__ __device__ inline void aa2q_dev(const Trig &tg, const double aa[3], double q[4]) {
  const double theta = sqrt(aa[0] * aa[0] + aa[1] * aa[1] + aa[2] * aa[2]);
  if (theta < 1e-6) {
    q[0] = 1.0;
    q[1] = q[2] = q[3] = 0.0;
  } else {
    const double sh = tg.s(0.5 * theta);
    q[0] = tg.c(0.5 * theta);
    for (int i = 0; i < 3; ++i) q[i + 1] = aa[i] * sh / theta;
  }
}
__global__ void k_aa2q(WSP) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  const int J = CFG.J;
  const RV r3 = rowv(w.P, w, b, J + 3), r4 = rowv(w.P, w, b, J + 4), r5 = rowv(w.P, w, b, J + 5),
           r6 = rowv(w.P, w, b, J + 6);
  const Trig tg{CFG.trigDev};
  double aa[3] = {r3[0], r4[0], r5[0]}, q[4], qprev[4];
  aa2q_dev(tg, aa, qprev);
  for (int i = 0; i < s.nPts; ++i) {
    aa[0] = r3[i];
    aa[1] = r4[i];
    aa[2] = r5[i];
    aa2q_dev(tg, aa, q);
    double qdir = 0;
    for (int j = 0; j < 4; ++j) qdir += q[j] * qprev[j];
    if (qdir < 0.0)
      for (int j = 0; j < 4; ++j) q[j] = -q[j];
    for (int j = 0; j < 4; ++j) qprev[j] = q[j];
    r3[i] = q[0];
    r4[i] = q[1];
    r5[i] = q[2];
    r6[i] = q[3];
  }
}

// ----------------------------------------------------------------------------- adjust_s, first half (TP + T)
// ba.cpp:412-590: cumulative norms, optional automatic integration resolution, scale selection,
// the weighted arc-length sites sC, and (regular pass) the resample plan of evalSplineFullTraj
// (ba.cpp:794-819).  ptsOrig is an iota at both call sites (ba.cpp:283, 778) so ptsOrig[i] == i.
// First the increments of the two cumulative norms (ba.cpp:423-446), one thread per (point, trajectory): the square
// roots and the ten coordinate differences of a point are independent of the running sums, so only the additions stay
// sequential (k_adjust_s below reads an increment from the slot its sum goes to).   (TP)
__global__ void k_adjust_inc(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (s.sWeights[1] + s.sWeights[2] < 1e-8) return;
  if (i >= s.nPts - 1) return;
  const int J = CFG.J;
  const bool cartStored = w.R > J;  // otherwise the Cartesian rows are zeros (DevCfg::R)
  const size_t pst = (size_t)w.B * w.R;
  const double *p0 = w.P + (size_t)b * w.R + (size_t)i * pst, *nx = p0 + pst;
  double dthetaSQ = 0;
  for (int j = 0; j < J; ++j) {
    const double d = nx[j] - p0[j];
    dthetaSQ += d * d;
  }
  double dcartSQ = 0;
  for (int j = 0; j < 3; ++j) {
    const double d = cartStored ? nx[J + j] - p0[J + j] : 0.0 - 0.0;
    dcartSQ += d * d;
  }
  double *o = w.nrm + ((size_t)(i + 1) * w.B + b) * 2;
  o[0] = sqrt(dthetaSQ);
  o[1] = sqrt(dcartSQ);
}

// the limit part of the automatic integration step (ba.cpp:493-556); lim: batotp_cfg or batotp_limits
template <class LT>
__host__ __device__ __forceinline__ double auto_integ_res(const LT &lim, int J, double K) {
  double r = K * lim.cart_acc_max / lim.cart_vel_max;
  for (int i = 0; i < J; ++i) r = dmax_(r, K * lim.jnt_acc_max[i] / lim.jnt_vel_max[i]);
  return r;
}

__global__ void k_adjust_s(WSP, int special, int haveInc) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (s.sWeights[1] + s.sWeights[2] < 1e-8) return;  // handled on the host: stage skipped
  const int J = CFG.J;
  double cartNormRes = special ? CFG.c.cart_norm_res : CFG.c.cart_norm_res2;
  const double thetaNormRes = special ? CFG.c.theta_norm_res : CFG.c.theta_norm_res2;
  const int nPts = s.nPts;
  const RV thetaNorm = RV{w.nrm + (size_t)b * 2, (size_t)w.B * 2}, cartPosNorm = RV{w.nrm + (size_t)b * 2 + 1, (size_t)w.B * 2};
  const RV sC = vecv(w.sC, w, b);
  const double sResi = s.sres;
  double MinRatio = 1.0 / CFG.quadThresh;
  double thetaWindow = 5;
  double thetaNormLast = 0, cartPosNormLast = 0;
  const double DEG2RAD = 3.14159265358979323846 / 180.0, RAD2DEG = 180.0 / 3.14159265358979323846;
  if (!CFG.c.are_jnt_deg) thetaWindow *= DEG2RAD;
  double tn = 0.0, cn = 0.0;
  thetaNorm[0] = 0.0;
  cartPosNorm[0] = 0.0;
  // haveInc: the increments sqrt(dthetaSQ), sqrt(dcartSQ) of point i+1 were left in its slots by k_adjust_inc (small
  // chunks: the pass is bound by the latency of one trajectory); otherwise they are formed here (full chunks: one
  // pass over the points instead of two)
  const bool cartStored = w.R > J;  // otherwise the Cartesian rows are zeros (DevCfg::R)
  const size_t pst = (size_t)w.B * w.R;
  const double *p0 = w.P + (size_t)b * w.R;
  double cur[MAXD + 3];
  if (!haveInc) {
    for (int j = 0; j < J; ++j) cur[j] = p0[j];
    for (int j = 0; j < 3; ++j) cur[MAXD + j] = cartStored ? p0[J + j] : 0.0;
  }
  // one point of the two running sums (+ the window bookkeeping of the automatic integration resolution)
  auto add_point = [&](int i, double it, double ic) {
    tn = tn + it;
    thetaNorm[i + 1] = tn;
    cn = cn + ic;
    cartPosNorm[i + 1] = cn;
    if (CFG.c.is_auto_integ_res) {
      const double thetaChange = tn - thetaNormLast;
      const double cartChange = cn - cartPosNormLast;
      if (thetaChange > thetaWindow) {
        MinRatio = dmin_(MinRatio, 3.0 * cartChange / thetaChange);
        thetaNormLast = tn;
        cartPosNormLast = cn;
      }
    }
  };
  if (haveInc) {
    // the additions are the only chain: eight points' increments are fetched ahead of it (independent loads)
    int i = 0;
    for (; i + 8 <= nPts - 1; i += 8) {
      double it[8], ic[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        it[k] = thetaNorm[i + 1 + k];
        ic[k] = cartPosNorm[i + 1 + k];
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) add_point(i + k, it[k], ic[k]);
    }
    for (; i < nPts - 1; ++i) add_point(i, thetaNorm[i + 1], cartPosNorm[i + 1]);
  } else {
    for (int i = 0; i < nPts - 1; ++i) {
      const double *nx = p0 + (size_t)(i + 1) * pst;
      double dthetaSQ = 0;
      for (int j = 0; j < J; ++j) {
        const double v = nx[j];
        const double d = v - cur[j];
        dthetaSQ += d * d;
        cur[j] = v;
      }
      double dcartSQ = 0;
      for (int j = 0; j < 3; ++j) {
        const double v = cartStored ? nx[J + j] : 0.0;
        const double d = v - cur[MAXD + j];
        dcartSQ += d * d;
        cur[MAXD + j] = v;
      }
      add_point(i, sqrt(dthetaSQ), sqrt(dcartSQ));
    }
  }
  const double tnLast = tn, cnLast = cn;
  if (tnLast < thetaNormRes) {
    s.status |= ST_IDENTICAL;
    return;
  }
  double sLast = 0, sResNew = 0;
  if (CFG.c.is_auto_integ_res) {  // ba.cpp:493-556
    if ((cnLast < cartNormRes) && s.scaleType == 2) {
      s.sWeights[1] = s.sWeights[1] + s.sWeights[2];
      s.sWeights[2] = 0;
      s.scaleType = 1;
    }
    const double sW12in = s.sWeights[1] + s.sWeights[2];
    double cartRat = 500.0 * cnLast;
    double thetaRat = tnLast;
    if (!CFG.c.are_jnt_deg) thetaRat *= RAD2DEG;
    const double minIntegRes = 0.004, maxIntegRes = 0.2, K = 0.0003;
    // from the trajectory's own limit row when the batch has them
    double newIntegRes = w.lim ? auto_integ_res(w.lim[b], J, K) : auto_integ_res(CFG.c, J, K);
    newIntegRes = dmin_(newIntegRes, maxIntegRes);
    const double changeRat = cartRat / thetaRat;
    double jointIntegRes = maxIntegRes * changeRat * changeRat;
    double jointWin = maxIntegRes * MinRatio * MinRatio;
    jointWin = dmax_(jointWin, 0.016);
    jointIntegRes = dmin_(jointIntegRes, jointWin);
    if (jointIntegRes < newIntegRes) newIntegRes = jointIntegRes;
    newIntegRes = dmax_(newIntegRes, minIntegRes);
    s.integRes = newIntegRes;
    const double sW12out = cartRat + thetaRat;
    const double outScale = sW12in / sW12out;
    cartRat *= outScale;
    thetaRat *= outScale;
    if (thetaRat > s.sWeights[1]) {
      s.sWeights[1] = thetaRat;
      s.sWeights[2] = cartRat;
    }
    if (s.sWeights[2] > 0) cartNormRes = dmin_(cartNormRes, cartNormRes * s.sWeights[2] / s.sWeights[1]);
  }
  const double ptsLast = (double)(nPts - 1);
  switch (s.scaleType) {
    case 0: sLast = sResi * ptsLast; sResNew = sResi; break;
    case 1: sLast = tnLast; sResNew = thetaNormRes; break;
    case 2: sLast = cnLast; sResNew = cartNormRes; break;
  }
  double cartPosNormFact;
  if (cnLast >= cartNormRes)
    cartPosNormFact = s.sWeights[2] * sLast / cnLast;
  else
    cartPosNormFact = 0;
  const double tTeachFact = s.sWeights[0] * sLast / (sResi * ptsLast);
  const double thetaNormFact = s.sWeights[1] * sLast / tnLast;
  s.sres = sLast / (nPts - 1);
  double prevSC = 0.0;
  bool tooSmall = false;
  for (int i = 0; i < nPts; ++i) {
    const double v = tTeachFact * sResi * (double)i + thetaNormFact * thetaNorm[i] + cartPosNormFact * cartPosNorm[i];
    sC[i] = v;
    if (!special && i > 0 && !tooSmall && (v - prevSC < 1e-12 * s.sres)) tooSmall = true;
    prevSC = v;
  }
  s.sLast = sLast;
  s.sResNew = sResNew;
  s.sResi = sResi;
  s.tTeachFact = tTeachFact;
  s.thetaNormFact = thetaNormFact;
  s.cartPosNormFact = cartPosNormFact;
  if (special) {
    int nPts2 = (int)ceil(sLast / sResNew) + 1;  // ba.cpp:666-667, capacity estimate for the march
    s.nNew = imax_(nPts2, 4);
  } else {
    if (tooSmall) {  // ba.cpp:605-612
      s.status |= ST_SRES_SMALL;
      return;
    }
    // evalSplineFullTraj(traj, traj.sres, sResNew) plan: ba.cpp:794-819
    const double oldRes = s.sres;
    int nNew = (int)ceil(oldRes / sResNew * (nPts - 1)) + 1;
    nNew = imax_(nNew, 4);
    const double newRes = oldRes * (nPts - 1) / (nNew - 1);
    s.sScale = prevSC / (double)(nNew - 1);  // sC[nPts-1] / sMVC[nNew-1]
    s.nNew = nNew;
    s.sresC = s.sres;
    s.vFact = 1 / s.sresC;
    s.aFact = s.vFact * s.vFact;
    s.sres = newRes;
    if (nNew > w.Nc) s.status |= ST_GRID_CAP;
  }
}

// ----------------------------------------------------------------------------- Thomas (TR)
// Spline::getSplineCoeffs on `rows` of the `rowsPerTraj` rows each of nb trajectories holds in the
// point-major array `src` -> solution rows in `dst`.  b0 = chunk index of the first trajectory.
// n source: 0 = st.nPts, 1 = st.nOver, 2 = st.nSm
__global__ void k_thomas_rows(WSP, double *src, double *dst, int nb, int b0, int rows, int rowsPerTraj,
                              int nsel, int clamped, ThomasTabs tabs) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int bl = t / rows, row = t % rows;
  if (bl >= nb) return;
  const TrajState &s = w.st[b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  const int n = nsel == 0 ? s.nPts : (nsel == 1 ? s.nOver : s.nSm);
  const size_t st = (size_t)nb * rowsPerTraj, off = (size_t)bl * rowsPerTraj + row;
  const RV y{src + off, st}, m{dst + off, st};
  if (clamped)
    thomas_clamped(y, m, n, tabs);
  else
    thomas_natural(y, m, n, tabs);
}

// ----------------------------------------------------------------------------- interpSpecial (T)
// ba.cpp:651-781: constant-ds march along the weighted arc length.  Source rows P (+M), emits Q.
// evalSplinePartials (ba.cpp:1341-1380) supplies the values; the Cartesian rows are refreshed
// only when a Cartesian constraint is on, otherwise Traj::cartpt keeps its previous content.
// JT / CT: joints and stored Cartesian rows as compile-time constants (JT = 0: both from the configuration), so
// that the joint loops unroll and `last` / `cartpt` stay in registers instead of local memory.  CT = 0: the
// Cartesian rows of a joint-only generic robot are not stored, their knots are read as a literal 0.0.
template <int JT, int CT>
__global__ void k_march(WSP) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  const int J = JT ? JT : CFG.J, C = JT ? CT : w.R - J, R = J + C;
  const int nPts = s.nPts;
  const RV sC = vecv(w.sC, w, b);
  const size_t pst = (size_t)w.B * w.R;
  const double *P = w.P + (size_t)b * w.R, *M = w.M + (size_t)b * w.R;
  double *Q = w.Q + (size_t)b * w.R;
  const int Nc = w.Nc;
  double last[MAXD + 3];  // the previously emitted point (theta rows, cart xyz)
  #pragma unroll
  for (int r = 0; r < R; ++r) Q[r] = P[r];
  #pragma unroll
  for (int j = 0; j < J; ++j) last[j] = P[j];
  #pragma unroll
  for (int j = 0; j < 3; ++j) last[MAXD + j] = C ? P[J + j] : 0.0;
  double sPrv = 0, prv_ds = 0;
  int CurNewPt = 1, CurOldPt = 1;
  int seg = 0;
  bool isDone = false;
  const int lastSeg = nPts - 2;
  const bool cartEval = CFG.cartOn != 0;
  double cartpt[MAXD];
  #pragma unroll
  for (int q = 0; q < MAXD; ++q) cartpt[q] = s.cartpt[q];
  const double sCend = sC[nPts - 1];
  while (!isDone) {
    const double *po = P + (size_t)CurOldPt * pst;
    double dthetaSQ = 0;
    #pragma unroll
    for (int j = 0; j < J; ++j) {
      const double d = po[j] - last[j];
      dthetaSQ += d * d;
    }
    double dcartSQ = 0;
    #pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double d = (C ? po[J + j] : 0.0) - last[MAXD + j];
      dcartSQ += d * d;
    }
    const double cur_ds = s.tTeachFact * s.sResi * (double)CurOldPt + s.thetaNormFact * sqrt(dthetaSQ) +
                          s.cartPosNormFact * sqrt(dcartSQ);
    if (cur_ds > s.sResNew) {
      const double sNew = sPrv + s.sResNew - prv_ds;
      prv_ds = 0;
      sPrv = sNew;
      const double sCur = sPrv;
      if (sCur > sCend) isDone = true;
      if (!isDone) {
        // updateCurSeg (ba.cpp:1617-1652) on the non-uniform sites
        double sSeg, sNext;
        int guard = 0;
        for (;;) {
          sSeg = sC[seg];
          sNext = sC[seg + 1];
          if (sCur >= sSeg && sCur <= sNext) break;
          if (sCur > sSeg) {
            if (seg >= lastSeg) {
              seg = lastSeg;
              break;
            }
            seg++;
          }
          if (sCur < sSeg) {
            if (seg <= 0) {
              seg = 0;
              break;
            }
            seg--;
          }
          if (++guard > 4 * nPts + 16) {
            s.status |= ST_NUMERIC;
            return;
          }
        }
        const double tau = (sCur - sSeg) / (sC[seg + 1] - sSeg);
        const double tau2 = tau * tau, tau3 = tau2 * tau;
        if (CurNewPt >= Nc - 1) {
          s.status |= ST_GRID_CAP;
          return;
        }
        const double *y0 = P + (size_t)seg * pst, *y1 = y0 + pst, *m0 = M + (size_t)seg * pst, *m1 = m0 + pst;
        double *qo = Q + (size_t)CurNewPt * pst;
        #pragma unroll
        for (int j = 0; j < J; ++j) {
          Seg4 c;
          c.c3 = sdiv::div6(m1[j] - m0[j]);
          c.c2 = m0[j] / 2.0;
          c.c1 = y1[j] - y0[j] - sdiv::div6(m1[j] + 2 * m0[j]);
          c.c0 = y0[j];
          const double v = seg_value(c, tau, tau2, tau3);
          qo[j] = v;
          last[j] = v;
        }
        if (cartEval)
          #pragma unroll
          for (int j = 0; j < C; ++j) {
            const int r = J + j;
            Seg4 c;
            c.c3 = sdiv::div6(m1[r] - m0[r]);
            c.c2 = m0[r] / 2.0;
            c.c1 = y1[r] - y0[r] - sdiv::div6(m1[r] + 2 * m0[r]);
            c.c0 = y0[r];
            cartpt[j] = seg_value(c, tau, tau2, tau3);
          }
        #pragma unroll
        for (int j = 0; j < C; ++j) qo[J + j] = cartpt[j];
        #pragma unroll
        for (int j = 0; j < 3; ++j) last[MAXD + j] = cartpt[j];
        CurOldPt = seg + 1;
        CurNewPt++;
      }
    } else {
      if (CurOldPt == nPts - 1) {
        isDone = true;
      } else {
        prv_ds = cur_ds;
        sPrv = sC[CurOldPt];
        CurOldPt++;
      }
    }
  }
  {
    const double *pe = P + (size_t)(nPts - 1) * pst;
    double *qo = Q + (size_t)CurNewPt * pst;
    #pragma unroll
    for (int r = 0; r < R; ++r) qo[r] = pe[r];
  }
  #pragma unroll
  for (int q = 0; q < MAXD; ++q) s.cartpt[q] = cartpt[q];
  s.nPts = CurNewPt + 1;
  s.sres = s.sResNew;
  if (s.nPts < 4) traj_linear_to4(w, w.Q, b, s, R);
}

// The same march with MG lanes per trajectory: lane r owns coordinate row r (its previously emitted value, its
// knot gathers, its segment coefficients and its store), the scalar control (arc-length bookkeeping, cursor, tau) is
// computed redundantly by every lane of the group.  k_march is bound by the latency of one iteration (two square
// roots, a division, 7..10 rows of coefficient arithmetic, three dependent gathers) at one warp per 32 trajectories;
// here an iteration costs a lane one row, and the machine holds MG times as many warps.  Bit-exactness: the squared
// row differences are summed in the reference's order (ba.cpp:681-690: joint 0 first) from values every lane
// fetches by shuffle; all other expressions are k_march's, row by row.  Shuffles name the group's own lanes, so the
// two groups of a warp may diverge.  Rows: r < J joints; J <= r < J + MAXD the Cartesian rows / Traj::cartpt.
#define MG 16
__global__ void k_march_group(WSP) {
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = gt / MG, r = gt % MG;
  const int lane = (int)(threadIdx.x & 31u), gbase = lane & ~(MG - 1);
  const unsigned gmask = ((MG == 32) ? 0xffffffffu : ((1u << MG) - 1u)) << gbase;
  if (b >= w.B) return;  // (a whole group leaves together)
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  // C: the stored Cartesian rows; a joint-only generic robot stores none and reads rows J..J+2 as a literal 0.0
  const int J = CFG.J, C = w.R - J, R = J + C;
  const bool isJ = r < J, isC = r >= J && r < R, isC3 = r >= J && r < J + 3, isCp = r >= J && r - J < MAXD;
  const int nPts = s.nPts;
  const RV sC = vecv(w.sC, w, b);
  const size_t pst = (size_t)w.B * w.R;
  const double *P = w.P + (size_t)b * w.R, *M = w.M + (size_t)b * w.R;
  double *Q = w.Q + (size_t)b * w.R;
  const int Nc = w.Nc;
  if (r < R) Q[r] = P[r];
  double last = (isJ || (isC3 && C)) ? P[r] : 0.0;  // the previously emitted point: theta rows, cart xyz
  double cartpt = isCp ? s.cartpt[r - J] : 0.0;
  double sPrv = 0, prv_ds = 0;
  int CurNewPt = 1, CurOldPt = 1;
  int seg = 0;
  bool isDone = false;
  const int lastSeg = nPts - 2;
  const bool cartEval = CFG.cartOn != 0;
  const double sCend = sC[nPts - 1];
  const double teach = s.tTeachFact * s.sResi, thetaNormFact = s.thetaNormFact, cartPosNormFact = s.cartPosNormFact;
  const double sResNew = s.sResNew;
  while (!isDone) {
    const double *po = P + (size_t)CurOldPt * pst;
    double dsq = 0.0;
    if (isJ || isC3) {
      const double d = (isJ || C ? po[r] : 0.0) - last;
      dsq = d * d;
    }
    double dthetaSQ = 0;
    for (int j = 0; j < J; ++j) dthetaSQ += __shfl_sync(gmask, dsq, gbase + j);
    double dcartSQ = 0;
    for (int j = 0; j < 3; ++j) dcartSQ += __shfl_sync(gmask, dsq, gbase + J + j);
    const double cur_ds = teach * (double)CurOldPt + thetaNormFact * sqrt(dthetaSQ) + cartPosNormFact * sqrt(dcartSQ);
    if (cur_ds > sResNew) {
      const double sNew = sPrv + sResNew - prv_ds;
      prv_ds = 0;
      sPrv = sNew;
      const double sCur = sPrv;
      if (sCur > sCend) isDone = true;
      if (!isDone) {
        // updateCurSeg (ba.cpp:1617-1652) on the non-uniform sites
        double sSeg, sNext;
        int guard = 0;
        for (;;) {
          sSeg = sC[seg];
          sNext = sC[seg + 1];
          if (sCur >= sSeg && sCur <= sNext) break;
          if (sCur > sSeg) {
            if (seg >= lastSeg) {
              seg = lastSeg;
              break;
            }
            seg++;
          }
          if (sCur < sSeg) {
            if (seg <= 0) {
              seg = 0;
              break;
            }
            seg--;
          }
          if (++guard > 4 * nPts + 16) {
            if (r == 0) s.status |= ST_NUMERIC;
            return;
          }
        }
        const double tau = (sCur - sSeg) / (sC[seg + 1] - sSeg);
        const double tau2 = tau * tau, tau3 = tau2 * tau;
        if (CurNewPt >= Nc - 1) {
          if (r == 0) s.status |= ST_GRID_CAP;
          return;
        }
        double *qo = Q + (size_t)CurNewPt * pst;
        if (isJ || (isC && cartEval)) {
          const double *y0 = P + (size_t)seg * pst, *y1 = y0 + pst, *m0 = M + (size_t)seg * pst, *m1 = m0 + pst;
          Seg4 c;
          c.c3 = sdiv::div6(m1[r] - m0[r]);
          c.c2 = m0[r] / 2.0;
          c.c1 = y1[r] - y0[r] - sdiv::div6(m1[r] + 2 * m0[r]);
          c.c0 = y0[r];
          const double v = seg_value(c, tau, tau2, tau3);
          if (isJ) {
            qo[r] = v;
            last = v;
          } else
            cartpt = v;
        }
        if (isC) qo[r] = cartpt;
        if (isC3) last = cartpt;
        CurOldPt = seg + 1;
        CurNewPt++;
      }
    } else {
      if (CurOldPt == nPts - 1) {
        isDone = true;
      } else {
        prv_ds = cur_ds;
        sPrv = sC[CurOldPt];
        CurOldPt++;
      }
    }
  }
  if (r < R) Q[(size_t)CurNewPt * pst + r] = P[(size_t)(nPts - 1) * pst + r];
  if (isCp) s.cartpt[r - J] = cartpt;
  __syncwarp(gmask);  // the rows of every lane are in place before lane 0 re-reads them (fewer than 4 points)
  if (r == 0) {
    s.nPts = CurNewPt + 1;
    s.sres = sResNew;
    if (s.nPts < 4) traj_linear_to4(w, w.Q, b, s, R);
  }
}

// ----------------------------------------------------------------------------- resample (TP)
// evalSplineFullTraj, regular pass (ba.cpp:835-859): sites sMVC[i] = sScale*i located in the
// non-uniform sC by findInterpSegs, values by interp1spline.  Source P/M/sC -> Q.
__global__ void k_resample(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nNew) return;
  const RV sC = vecv(w.sC, w, b);
  const int nOld = s.nPts;
  const double aOut = s.sScale * (double)i;
  ViewSites in{sC};
  // the sites are the arc lengths of the constant-ds march: nearly uniform, so the search starts at the
  // proportional position (a NaN or out-of-range estimate only costs probes)
  const double est = aOut / sC[nOld - 1] * (double)(nOld - 1);
  const int seg = find_seg_from(in, nOld, aOut, (est > 0.0 && est < 2.0e9) ? (int)est : 0);
  const double lo = sC[seg];
  const double den = sC[seg + 1] - lo;
  const double tau = (aOut - lo) / den;
  const double tau2 = tau * tau, tau3 = tau2 * tau;
  const size_t pst = (size_t)w.B * w.R;
  const double *y0 = w.P + (size_t)seg * pst + (size_t)b * w.R, *y1 = y0 + pst;
  const double *m0 = w.M + (size_t)seg * pst + (size_t)b * w.R, *m1 = m0 + pst;
  double *qo = w.Q + (size_t)i * pst + (size_t)b * w.R;
  for (int r = 0; r < CFG.R; ++r) {
    Seg4 c;
    c.c3 = sdiv::div6(m1[r] - m0[r]);
    c.c2 = m0[r] / 2.0;
    c.c1 = y1[r] - y0[r] - sdiv::div6(m1[r] + 2 * m0[r]);
    c.c0 = y0[r];
    qo[r] = seg_value(c, tau, tau2, tau3);
  }
}
// spline.cpp:78-87: a zero-length input segment aborts findInterpSegs (status only) (T)
// one thread per (input segment, trajectory) flags the trajectory (TP), then the commit (T)
__global__ void k_resample_check(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  TrajState &s = w.st[bl];
  if (s.status & ST_FATAL_MASK & ~ST_DIV0) return;
  if (i >= s.nPts - 1) return;
  const RV sC = vecv(w.sC, w, bl);
  if (sC[i + 1] - sC[i] < 1e-20) atomicOr(&s.status, (int)ST_DIV0);
}
__global__ void k_resample_commit(WSP) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;  // includes ST_DIV0 from k_resample_check
  s.nPts = s.nNew;
}

// ba.cpp:155-157 after the interpolation-only resample: the result IS the output (sres = outRes)  (T)
__global__ void k_interp_only_finish(WSP) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  s.nOut = s.nSm = s.nPts;
  s.nCartOut = s.nPts;
  s.isReinterp = 0;
  s.sres = CFG.c.out_res;
  s.sresOut = CFG.c.out_res;
  s.nRev = s.nFwd = 0;
  s.tRev = s.tFwd = 0.0;
  if (s.nOut > w.OutC) s.status |= ST_STEP_CAP;
}

// ----------------------------------------------------------------------------- final grid (T + TP)
// ba.cpp:297-300: sC.clear(); evalSplineFullTraj(traj, sres, sres) -> uniform sites sres*k.
__global__ void k_final_plan(WSP) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  const int nOld = s.nPts;
  const double oldRes = s.sres, newResIn = s.sres;
  int nNew = (int)ceil(oldRes / newResIn * (nOld - 1)) + 1;
  nNew = imax_(nNew, 4);
  const double newRes = oldRes * (nOld - 1) / (nNew - 1);
  const double sBack = s.sres * (double)(nOld - 1);  // sC[nOld-1]
  s.sScale = sBack / (double)(nNew - 1);
  s.nPtsC = nOld;
  s.nNew = nNew;
  s.sresC = s.sres;
  s.vFact = 1 / s.sresC;
  s.aFact = s.vFact * s.vFact;
  s.sres = newRes;
  s.nPts = nNew;
  if (nNew > w.Nc) s.status |= ST_GRID_CAP;
}

// Segment table (TP over segments): per (segment k, row r) the four spline coefficients {c3, c2, c1, c0}
// (spline.cpp:205-208) of the kinematic rows (joints, then Cartesian xyz when a Cartesian constraint is on)
// and, with torque limits, of the dynamics rows a1..a4 (ba.cpp:1387-1405).  The sweep forms the products
// evalSplinePartials starts from (3*c3, 2*c2, 6*c3; ba.cpp:1359-1360) when it loads a segment; the output
// phase evaluates theta(t) from the same rows, so no consumer repeats the /6 divisions.
__global__ void k_build_table(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nPtsC - 1) return;
  const int J = CFG.J;
  double *t = w.tab + ((size_t)b * w.Nc + i) * (size_t)w.RT * 4;
  int rt = 0;
  const int nKin = J + (CFG.cartOn ? 3 : 0);
  for (int r = 0; r < nKin; ++r, ++rt) {
    const Seg4 c = seg_coef(rowv(w.P, w, b, r), rowv(w.M, w, b, r), i);
    t[rt * 4 + 0] = c.c3;
    t[rt * 4 + 1] = c.c2;
    t[rt * 4 + 2] = c.c1;
    t[rt * 4 + 3] = c.c0;
  }
  if (CFG.trqOn) {
    for (int a = 0; a < 4; ++a)
      for (int j = 0; j < J; ++j, ++rt) {
        const Seg4 c = seg_coef(arowv(w.A, w, b, a, j), arowv(w.AM, w, b, a, j), i);
        t[rt * 4 + 0] = c.c3;
        t[rt * 4 + 1] = c.c2;
        t[rt * 4 + 2] = c.c1;
        t[rt * 4 + 3] = c.c0;
      }
  }
}

// The same table built through shared-memory tiles of BT_SEGS segments x TRAJ trajectories: the knots are read with
// trajectories fastest (the point-major order of P/M and A/AM), the table is written one trajectory at a time as
// contiguous BT_SEGS*RT*32-byte runs.  Block (TRAJ, BT_SEGS).  Two shapes: 8 trajectories x 10 rows (kinematic rows
// only: GEN7DOF, KUKA, UR5) and 4 trajectories x 18 rows (with the 4*J dynamics rows of the 2- and 3-joint robots: RR, CSPR3DOF; 7-joint robots
// with a caller-supplied model take the untiled k_build_table).
#define BT_TRAJ 8
#define BT_SEGS 16
#define BT_ROWS 10
#define BT_TRAJ_DYN 4
#define BT_ROWS_DYN 18
template <int TRAJ, int ROWS>
__global__ void k_build_table_tile(WSP, int npts, int nb) {
  EMU_SHARED double tile[TRAJ][BT_SEGS][ROWS * 4];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int b0 = (int)blockIdx.x * TRAJ, i0 = (int)(blockIdx.z * gridDim.y + blockIdx.y) * BT_SEGS;
  const int RT = w.RT;
  const int nKin = CFG.J + (CFG.cartOn ? 3 : 0);
  {
    const int b = b0 + tx, i = i0 + ty;
    if (b < nb && i < npts) {
      const TrajState &s = w.st[b];
      if (!(s.status & ST_FATAL_MASK) && i < s.nPtsC - 1) {
        for (int r = 0; r < RT; ++r) {
          Seg4 c;
          if (r < nKin)
            c = seg_coef(rowv(w.P, w, b, r), rowv(w.M, w, b, r), i);
          else {
            const int q = r - nKin, a = q / CFG.J, j = q - a * CFG.J;
            c = seg_coef(arowv(w.A, w, b, a, j), arowv(w.AM, w, b, a, j), i);
          }
          tile[tx][ty][r * 4 + 0] = c.c3;
          tile[tx][ty][r * 4 + 1] = c.c2;
          tile[tx][ty][r * 4 + 2] = c.c1;
          tile[tx][ty][r * 4 + 3] = c.c0;
        }
      }
    }
  }
  __syncthreads();
  const int tid = ty * TRAJ + tx, per = RT * 4;
  for (int bl = 0; bl < TRAJ; ++bl) {
    const int b = b0 + bl;
    if (b >= nb) break;
    const TrajState &s = w.st[b];
    if (s.status & ST_FATAL_MASK) continue;
    const int nSeg = imin_(imin_(s.nPtsC - 1, npts) - i0, BT_SEGS);  // valid segments of this tile
    if (nSeg <= 0) continue;
    double *t = w.tab + ((size_t)b * w.Nc + i0) * (size_t)per;
    for (int e = tid; e < nSeg * per; e += TRAJ * BT_SEGS) t[e] = tile[bl][e / per][e % per];
  }
}

// Values and s-derivatives on the final grid (ba.cpp:840-855), needed by the dynamic model
// (findDynModel, ba.cpp:905-938).  Source P/M -> Q (values), GD, GD2.   (TP)
__global__ void k_eval_grid(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nNew) return;
  UniformSites in{s.sresC};
  const double aOut = s.sScale * (double)i;
  const int seg = find_seg(in, s.nPtsC, aOut);
  const double den = in(seg + 1) - in(seg);
  const double tau = (aOut - in(seg)) / den;
  const double tau2 = tau * tau, tau3 = tau2 * tau;
  const double vfact = 1.0 / s.sresC;  // interp1spline's own 1/tfact with tfact = oldRes (spline.cpp:142-143)
  const double afact = vfact * vfact;
  for (int r = 0; r < CFG.R; ++r) {
    const Seg4 c = seg_coef(rowv(w.P, w, b, r), rowv(w.M, w, b, r), seg);
    rowv(w.Q, w, b, r)[i] = seg_value(c, tau, tau2, tau3);
    rowv(w.GD, w, b, r)[i] = (3 * c.c3 * tau2 + 2 * c.c2 * tau + c.c1) * vfact;
    rowv(w.GD2, w, b, r)[i] = (6 * c.c3 * tau + 2 * c.c2) * afact;
  }
}
