// k_output.cuh — device kernels for BA::interpOutputData (batotp/ba.cpp:1661-1931), the
// dynamic model (findDynModel ba.cpp:873-949, Robot::dynRR robot.cpp:377-431, dynCSPR3DOF
// 487-517, setA 534-558, solveLinSys util.cpp:413-442) and result packing
// (trajWriteBIN ba.cpp:2617-2647, sdotWrite 2735-2749).
#pragma once
#include "k_input.cuh"

// ----------------------------------------------------------------------------- small dense solve
// util.cpp:413-442 with isSVD=0: x = A.lu().solve(b).  Eigen (un-vendored dependency, "3.3.4",
// README.md:32-50) PartialPivLU restated: first-max partial pivoting, sub-column divided by the
// pivot, rank-1 trailing update, column-oriented unit-lower then upper substitution.  Pinned by
// the prebuilt bin/batest CSPR3DOF fingerprints through the oracle (DESIGN.md §oracle).
__host__ __device__ inline void lu3_solve(const double A[3][3], const double b[3], double x[3]) {
  double lu[3][3];
  int perm[3] = {0, 1, 2};
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) lu[i][j] = A[i][j];
  for (int k = 0; k < 3; ++k) {
    int p = k;
    double best = fabs(lu[k][k]);
    for (int i = k + 1; i < 3; ++i) {
      const double v = fabs(lu[i][k]);
      if (v > best) {
        best = v;
        p = i;
      }
    }
    if (p != k) {
      for (int j = 0; j < 3; ++j) {
        const double t = lu[k][j];
        lu[k][j] = lu[p][j];
        lu[p][j] = t;
      }
      const int t = perm[k];
      perm[k] = perm[p];
      perm[p] = t;
    }
    if (best != 0.0) {
      const double piv = lu[k][k];
      for (int i = k + 1; i < 3; ++i) lu[i][k] /= piv;
    }
    for (int i = k + 1; i < 3; ++i)
      for (int j = k + 1; j < 3; ++j) lu[i][j] -= lu[i][k] * lu[k][j];
  }
  for (int i = 0; i < 3; ++i) x[i] = b[perm[i]];
  for (int i = 0; i < 3; ++i)
    for (int r = i + 1; r < 3; ++r) x[r] -= x[i] * lu[r][i];
  for (int i = 2; i >= 0; --i) {
    x[i] /= lu[i][i];
    for (int r = 0; r < i; ++r) x[r] -= x[i] * lu[r][i];
  }
}

// robot.cpp:377-431 at one point (theta in degrees; thetaD/thetaD2 are s- or t-derivatives)
__host__ __device__ inline void dyn_rr_point(const Trig &tg, const double th[2], const double thD[2],
                                             const double thD2[2], double a1[2], double a2[2], double a3[2],
                                             double a4[2]) {
  const double D2R = 3.14159265358979323846 / 180.0, g = 9.81;
  const double A1 = .4, A2 = .6, m1 = 4, m2 = 8;
  const double th1 = D2R * th[0], th2 = D2R * th[1];
  const double dth1 = D2R * thD[0], dth2 = D2R * thD[1];
  const double ddth1 = D2R * thD2[0], ddth2 = D2R * thD2[1];
  const double c1 = tg.c(th1), c2 = tg.c(th2), c12 = tg.c(th1 + th2);
  const double A11 = .25 * m1 * A1 * A1 + m2 * (A1 * A1 + .25 * A2 * A2 + A1 * A2 * c2);
  const double A12 = .5 * m2 * (.5 * A2 * A2 + A1 * A2 * c2);
  const double A22 = .25 * m2 * A2 * A2;
  a1[0] = A11 * dth1 + A12 * dth2;
  a1[1] = A12 * dth1 + A22 * dth2;
  const double ccFact = m2 * A1 * A2 * tg.s(th2);
  a2[0] = A11 * ddth1 + A12 * ddth2 - ccFact * dth2 * (dth1 + .5 * dth2);
  a2[1] = A12 * ddth1 + A22 * ddth2 - .5 * ccFact * dth1 * dth1;
  a3[0] = 10 * dth1;
  a3[1] = 10 * dth2;
  a4[0] = .5 * g * (m1 * A1 * c1 + m2 * (2.0 * A1 * c1 + A2 * c12));
  a4[1] = .5 * g * m2 * A2 * c12;
}

// findDynModel on the grid (TP): values in Q, s-derivatives in GD/GD2 -> A rows (+Par2Ser)
__global__ void k_dyn_grid(WSP, Pmat pm, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = bl;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nPts) return;
  const int J = CFG.J;
  double a[4][MAXD];
  for (int k = 0; k < 4; ++k)
    for (int q = 0; q < MAXD; ++q) a[k][q] = 0.0;
  const size_t off = ((size_t)i * w.B + b) * w.R;
  const double *q0 = w.Q + off, *g1 = w.GD + off, *g2 = w.GD2 + off;
  if (CFG.c.is_parallel) {  // dynCSPR3DOF (robot.cpp:487-517)
    for (int q = 0; q < 3; ++q) {
      a[0][q] = -g1[J + q];
      a[1][q] = -g2[J + q];
    }
    a[3][2] = 9.81;
    if (CFG.c.is_par2ser) {  // ba.cpp:916-938: a_k <- A^-1 a_k with A from setA
      double Am[3][3], cart[3], th[3];
      for (int q = 0; q < 3; ++q) {
        cart[q] = q0[J + q];
        th[q] = q0[q];
      }
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) Am[r][c] = (cart[r] - pm.p[r][c]) / th[c];
      for (int k = 0; k < 4; ++k) {
        double x[3], bb[3] = {a[k][0], a[k][1], a[k][2]};
        lu3_solve(Am, bb, x);
        for (int q = 0; q < 3; ++q) a[k][q] = x[q];
      }
    }
  } else {  // dynRR
    double th[2], d1[2], d2[2];
    for (int q = 0; q < 2; ++q) {
      th[q] = q0[q];
      d1[q] = g1[q];
      d2[q] = g2[q];
    }
    dyn_rr_point(Trig{CFG.trigDev}, th, d1, d2, a[0], a[1], a[2], a[3]);
  }
  double *Ab = w.A + ((size_t)i * w.B + b) * 4 * w.AD;
  for (int k = 0; k < 4; ++k)
    for (int q = 0; q < w.AD; ++q) Ab[k * w.AD + q] = a[k][q];
}

// ----------------------------------------------------------------------------- output plan (T)
// ba.cpp:1664-1706: output resolution bookkeeping, oversampled size, natural spline of sMVC(t), for every
// trajectory of the resident chunk.  The output kernels after it work on the sub-chunk [w.b0, w.b0 + w.Bo).
__global__ void k_out_plan(WSP, ThomasTabs tabs) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= w.B) return;
  TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  const double outResT = CFG.c.out_res;
  double outRes = outResT, outSmooth = CFG.c.out_smooth_fact;
  int isReinterp = 0;
  if (outRes < s.integRes) {
    isReinterp = 1;
    outRes = s.integRes;
    outSmooth *= dmax_(outResT / outRes, 1.);
  }
  const double tLast = s.tStep * (double)(s.nFwd - 1);
  int nOver = (int)(outSmooth * ceil(tLast / outRes + 1.));
  nOver = imax_(nOver, 4);
  s.isReinterp = isReinterp;
  s.outResEff = outRes;
  s.outSmooth = outSmooth;
  s.outResT = outResT;
  s.nOver = nOver;
  s.segWalk = 0;
  if (nOver > w.Oc) {
    s.status |= ST_STEP_CAP;
    return;
  }
  double *sF = w.hist + (size_t)b * 4 * w.Sc + 2 * (size_t)w.Sc;
  const RV y{sF, 1}, m{w.mS + (size_t)b * w.Sc, 1};
  thomas_natural(y, m, s.nFwd, tabs);
}

// tMVCout[i] (ba.cpp:1693-1699) -> s at that time (TP)
__host__ __device__ __forceinline__ double tmvc_out(int i, int n, double tLast) {
  const double last = (double)(n - 3);
  double v;
  if (i == 0)
    v = 0;
  else if (i == 1)
    v = 1.0 / 3.0;
  else if (i == n - 1)
    v = last;
  else if (i == n - 2)
    v = last - 1.0 / 3.0;
  else
    v = (double)(i - 1);
  return (tLast / last) * v;
}

__global__ void k_out_s(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = w.b0 + bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nOver) return;
  const double tLast = s.tStep * (double)(s.nFwd - 1);
  const double t = tmvc_out(i, s.nOver, tLast);
  UniformSites in{s.tStep};
  const int seg = find_seg(in, s.nFwd, t);
  const double tau = (t - in(seg)) / (in(seg + 1) - in(seg));
  double *sF = w.hist + (size_t)b * 4 * w.Sc + 2 * (size_t)w.Sc;
  const Seg4 c = seg_coef(RV{sF, 1}, RV{w.mS + (size_t)b * w.Sc, 1}, seg);
  const double tau2 = tau * tau, tau3 = tau2 * tau;
  w.sOut[(size_t)i * w.Bo + bl] = seg_value(c, tau, tau2, tau3);
}

// findInterpSegs(traj.sC, sMVCout) (ba.cpp:1708, spline.cpp:56-99).  The reference walks a forward-only
// cursor: seg[i] = min(nIn-2, max_{i' <= i} f(a[i'])) with f(a) = the first k with a < sC[k+1].  s(t) is
// monotone in practice, so k_out_segs_par (TP) evaluates f(a[i]) directly from the uniform sites and flags
// a trajectory when f decreases anywhere; only flagged trajectories take the sequential walk (T) after it.
__host__ __device__ __forceinline__ int first_seg_uniform(double res, int nIn, double a) {
  const int last = nIn - 2;
  int k = 0;
  const float g = (float)a / (float)res;  // estimate only: corrected against the products the reference compares with
  if (g > 0.0f) k = (g < (float)last) ? (int)g : last;
  while (k > 0 && a < res * (double)k) k--;
  while (k < last && !(a < res * (double)(k + 1))) k++;
  return k;
}
__global__ void k_out_segs_par(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nOver) return;
  const size_t at = (size_t)i * w.Bo + bl;
  const double a = w.sOut[at];
  const int nIn = s.nPtsC;
  const double res = s.sresC;
  const int k = first_seg_uniform(res, nIn, a);
  if (i > 0) {
    const int kp = first_seg_uniform(res, nIn, w.sOut[at - w.Bo]);
    if (kp > k) s.segWalk = 1;  // the running maximum differs from f here: sequential walk needed
  }
  w.segO[at] = k;
  const double lo = res * (double)k, hiEdge = res * (double)(k + 1);
  w.tauO[at] = (a - lo) / (hiEdge - lo);
}
__global__ void k_out_segs(WSP) {
  const int bl = blockIdx.x * blockDim.x + threadIdx.x;
  if (bl >= w.Bo) return;
  TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  if (!s.segWalk) return;  // k_out_segs_par's result stands
  s.segWalk = 0;
  const int nIn = s.nPtsC;
  const double res = s.sresC;
  int cur = 0;
  double hiEdge = res * (double)(cur + 1);
  for (int i = 0; i < s.nOver; ++i) {
    const size_t at = (size_t)i * w.Bo + bl;
    const double a = w.sOut[at];
    while (!(a < hiEdge || cur == nIn - 2)) {
      cur++;
      hiEdge = res * (double)(cur + 1);
    }
    w.segO[at] = cur;
    const double lo = res * (double)cur;
    w.tauO[at] = (a - lo) / (hiEdge - lo);
  }
}

// k_out_s + k_out_segs_par in one pass over 32x32 tiles (sites x trajectories).  s(t) is read from the
// trajectory-major history rows, so a warp takes 32 consecutive sites of ONE trajectory (its four gathers hit
// one or two segments of that row); the tile is turned in shared memory and written with trajectories
// fastest, the order the point-major consumers read.  The monotonicity test compares with the lane to the
// left (the site before the tile is recomputed).  Block (32, 8).
__global__ void k_out_s_segs(WSP, int npts, int nb) {
  EMU_SHARED double tS[32][33], tTau[32][33];
  EMU_SHARED int tSeg[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int bl0 = (int)blockIdx.x * 32, i0 = (int)(blockIdx.z * gridDim.y + blockIdx.y) * 32;
  for (int k = 0; k < 4; ++k) {
    const int bll = ty + 8 * k, bl = bl0 + bll, i = i0 + tx;
    bool valid = bl < nb && i < npts;
    double a = 0, tau = 0;
    int kseg = 0;
    if (valid) {
      TrajState &s = w.st[w.b0 + bl];
      valid = !(s.status & ST_FATAL_MASK) && i < s.nOver;
      if (valid) {
        const int b = w.b0 + bl;
        const double tLast = s.tStep * (double)(s.nFwd - 1);
        UniformSites in{s.tStep};
        const double *sF = w.hist + (size_t)b * 4 * w.Sc + 2 * (size_t)w.Sc;
        const RV ys{const_cast<double *>(sF), 1}, ms{w.mS + (size_t)b * w.Sc, 1};
        const float rStep = 1.0f / (float)s.tStep;  // only steers the search
        auto s_at = [&](int ii) {
          const double t = tmvc_out(ii, s.nOver, tLast);
          const int seg = find_seg_from(in, s.nFwd, t, (int)((float)t * rStep));
          const double ta = (t - in(seg)) / (in(seg + 1) - in(seg));
          const Seg4 c = seg_coef(ys, ms, seg);
          const double ta2 = ta * ta, ta3 = ta2 * ta;
          return seg_value(c, ta, ta2, ta3);
        };
        a = s_at(i);
        const int nIn = s.nPtsC;
        const double res = s.sresC;
        kseg = first_seg_uniform(res, nIn, a);
        const double lo = res * (double)kseg, hiEdge = res * (double)(kseg + 1);
        tau = (a - lo) / (hiEdge - lo);
        if (tx == 0 && i > 0) {
          if (first_seg_uniform(res, nIn, s_at(i - 1)) > kseg) s.segWalk = 1;
        }
      }
    }
    // the running maximum of findInterpSegs differs from f(a) where f decreases: sequential walk needed
    const int kleft = __shfl_up_sync(0xffffffffu, valid ? kseg : -1, 1);
    if (valid && tx > 0 && kleft > kseg) w.st[w.b0 + bl].segWalk = 1;
    tS[bll][tx] = a;
    tTau[bll][tx] = tau;
    tSeg[bll][tx] = valid ? kseg : -1;
  }
  __syncthreads();
  for (int k = 0; k < 4; ++k) {
    const int il = ty + 8 * k, i = i0 + il, bl = bl0 + tx;
    if (bl < nb && i < npts && tSeg[tx][il] >= 0) {
      const size_t at = (size_t)i * w.Bo + bl;
      w.sOut[at] = tS[tx][il];
      w.segO[at] = tSeg[tx][il];
      w.tauO[at] = tTau[tx][il];
    }
  }
}

// theta(t) / cart(t) at the oversampled sites (ba.cpp:1713-1742).  One thread per (point, trajectory, row),
// rows fastest: the four knot gathers and the store of a point are contiguous R*8-byte runs.  Rows that are
// not path-driven are filled by the kinematics kernel afterwards (or are the generic robot's zeros).
__global__ void k_out_eval(WSP, int npts, int nb) {
  // x covers (trajectory, row) pairs, rows fastest; nb = Bo * R
  const int R = w.R;
  const int xr = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  const int i = (int)((blockIdx.z * gridDim.y + blockIdx.y) * blockDim.y + threadIdx.y);
  if (xr >= nb) return;
  const int bl = xr / R, r = xr - bl * R;
  if (i >= npts) return;
  const int b = w.b0 + bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nOver) return;
  const size_t at = (size_t)i * w.Bo + bl;
  const int pt = CFG.c.path_type;
  const bool isJ = r < CFG.J;
  const bool driven = isJ ? (pt == BATOTP_JOINT || pt == BATOTP_BOTH) : (pt == BATOTP_CART || pt == BATOTP_BOTH);
  double v = 0.0;
  if (driven) {
    const int seg = w.segO[at];
    const double tau = w.tauO[at];
    const double tau2 = tau * tau, tau3 = tau2 * tau;
    const size_t pst = (size_t)w.B * R;
    const size_t k0 = (size_t)seg * pst + (size_t)b * R + r;
    const double y0 = w.P[k0], y1 = w.P[k0 + pst], m0 = w.M[k0], m1 = w.M[k0 + pst];
    Seg4 c;
    c.c3 = sdiv::div6(m1 - m0);
    c.c2 = m0 / 2.0;
    c.c1 = y1 - y0 - sdiv::div6(m1 + 2 * m0);
    c.c0 = y0;
    v = seg_value(c, tau, tau2, tau3);
  }
  w.O5[at * R + r] = v;
}

// Torque branch, part 1 (ba.cpp:1746-1765 / 1807-1812): values and time derivatives of the
// re-splined rows at their own knots (seg=i-1, tau=1; i=0: seg=0, tau=0).  O5/OM -> OA, OD, OD2.  (TP)
// (torque runs use Os == Oc, so OA/OM share O5's pitch)
__global__ void k_out_knot_eval(WSP, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nOver) return;
  const int J = CFG.J;
  const int seg = (i == 0) ? 0 : i - 1;
  const double tau = (i == 0) ? 0.0 : 1.0;
  const double tau2 = tau * tau, tau3 = tau2 * tau;
  const double tfact = s.outResEff / s.outSmooth;
  const double vfact = 1.0 / tfact, afact = vfact * vfact;
  for (int r = 0; r < CFG.R; ++r) {
    const bool resplined = (r < J) || CFG.c.is_parallel;
    if (resplined) {
      const Seg4 c = seg_coef(orowv(w.O5, w, bl, r), orowv(w.OM, w, bl, r), seg);
      orowv(w.OA, w, bl, r)[i] = seg_value(c, tau, tau2, tau3);
      orowv(w.OD, w, bl, r)[i] = (3 * c.c3 * tau2 + 2 * c.c2 * tau + c.c1) * vfact;
      orowv(w.OD2, w, bl, r)[i] = (6 * c.c3 * tau + 2 * c.c2) * afact;
    } else {
      orowv(w.OA, w, bl, r)[i] = orowv(w.O5, w, bl, r)[i];
    }
  }
}

// Torque branch, part 2 (ba.cpp:1770-1803 / 1815-1825): generalized forces at the output sites (TP)
__global__ void k_out_trq(WSP, Pmat pm, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nOver) return;
  const int J = CFG.J;
  const size_t off = ((size_t)i * w.Bo + bl) * w.R;
  const double *oa = w.OA + off, *od = w.OD + off, *od2 = w.OD2 + off;
  double *trq = w.Trq + ((size_t)i * w.Bo + bl) * MAXD;
  if (CFG.c.is_parallel) {
    double a2[3], a3[3] = {0, 0, 0}, a4[3] = {0, 0, 9.81}, cart[3], th[3], bStar[3], x[3], Am[3][3];
    for (int q = 0; q < 3; ++q) {
      a2[q] = -od2[J + q];
      cart[q] = oa[J + q];
      th[q] = oa[q];
    }
    for (int q = 0; q < 3; ++q) bStar[q] = a2[q] + a3[q] + a4[q];
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) Am[r][c] = (cart[r] - pm.p[r][c]) / th[c];
    lu3_solve(Am, bStar, x);
    for (int q = 0; q < J; ++q) trq[q] = x[q];
  } else {
    double th[2], d1[2], d2[2], a1[2], a2[2], a3[2], a4[2];
    for (int q = 0; q < 2; ++q) {
      th[q] = oa[q];
      d1[q] = od[q];
      d2[q] = od2[q];
    }
    dyn_rr_point(Trig{CFG.trigDev}, th, d1, d2, a1, a2, a3, a4);
    for (int q = 0; q < 2; ++q) trq[q] = a2[q] + a3[q] + a4[q];
  }
}

// ----------------------------------------------------------------------------- smoothing (TP)
// util.cpp:254-288 evaluated pointwise: x2[p] for a row of length n, window w (valid for n >= 2*wMid).
template <class V>
__host__ __device__ __forceinline__ double smooth_at(V &&x, int n, int wIn, int p) {
  int w = imin_(wIn, n);
  const int wMid = w / 2 + w % 2 - 1;
  w = 2 * wMid + 1;
  if (p >= wMid && p < n - wMid) {
    double xt = 0;
    for (int j = p - wMid; j < p + wMid + 1; ++j) xt += x[j];
    return xt / w;
  }
  if (p == 0) return x[0];
  if (p == n - 1) return x[n - 1];
  if (p < wMid) {
    double xt = 0;
    const int nT = 2 * p + 1;
    for (int j = 0; j < nT; ++j) xt += x[j];
    return xt / nT;
  }
  const int q = n - 1 - p;
  double xte = 0;
  const int nT = 2 * q + 1;
  for (int j = 0; j < nT; ++j) xte += x[n - j - 1];
  return xte / nT;
}

// ba.cpp:1838-1871 plan (T): nSm
__global__ void k_out_smooth_plan(WSP) {
  const int bl = blockIdx.x * blockDim.x + threadIdx.x;
  if (bl >= w.Bo) return;
  TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  if (s.outSmooth > 1.5) {
    const int nIn = s.nOver;
    s.nSm = imax_((int)((nIn - 1) / s.outSmooth) + 1, 4);
    int wv = imin_((int)s.outSmooth, nIn);
    const int wMid = wv / 2 + wv % 2 - 1;
    if (nIn < 2 * wMid + 1) s.status |= ST_UNSUPPORTED;  // degenerate window/length combination
  } else
    s.nSm = s.nOver;
}

// smooth + linear decimation of every row (src -> dst) and of the torque rows (TP over nSm).
// Trajectories whose smoothing factor is <= 1.5 (ba.cpp:1838) are copied through unchanged.
// src/dst are point-major sub-chunk arrays [.][Bo][R].
__global__ void k_out_smooth(WSP, double *src, double *dst, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nSm) return;
  const bool sm = s.outSmooth > 1.5;
  const int nIn = s.nOver, nOut = s.nSm;
  int seg = i;
  double tau = 0;
  if (sm) {
    const double aOut = ((double)(nIn - 1) / (double)(nOut - 1)) * (double)i;
    UniformSites in{1.0};
    seg = find_seg(in, nIn, aOut);
    tau = (aOut - (double)seg) / ((double)(seg + 1) - (double)seg);
  }
  const int wv = (int)s.outSmooth;
  for (int r = 0; r < CFG.R; ++r) {
    const RV x = orowv(src, w, bl, r);
    double v;
    if (sm) {
      const double v0 = smooth_at(x, nIn, wv, seg), v1 = smooth_at(x, nIn, wv, seg + 1);
      v = v0 + (v1 - v0) * tau;
    } else
      v = x[i];
    orowv(dst, w, bl, r)[i] = v;
  }
  if (CFG.trqOn)
    for (int r = 0; r < CFG.J; ++r) {
      const RV x = trqv(w.Trq, w, bl, r);
      double v;
      if (sm) {
        const double v0 = smooth_at(x, nIn, wv, seg), v1 = smooth_at(x, nIn, wv, seg + 1);
        v = v0 + (v1 - v0) * tau;
      } else
        v = x[i];
      trqv(w.Trq2, w, bl, r)[i] = v;
    }
}

// Fused evaluation + smoothing + decimation (ba.cpp:1713-1742 then 1838-1871) for runs whose oversampled rows
// have no other consumer (no torque branch, no kinematics at the output sites, smoothing on for the whole
// batch): one thread per (decimated point, trajectory, row) evaluates the 2*wMid+2 oversampled values its
// two smoothing windows need — the same seg_value expressions k_out_eval forms, summed in smooth()'s
// order — so the oversampled rows (the largest array of the output phase) never travel through HBM.
struct OverEval {  // x[j]: row r of trajectory b at oversampled site j; caches the segment coefficients
  const double *P, *M, *tauO;
  const int *segO;
  size_t pst, rowOff;  // B * R;  b * R + r
  int Bo, bl, cseg;
  Seg4 c;
  __host__ __device__ __forceinline__ double operator[](int j) {
    const size_t at = (size_t)j * Bo + bl;
    const int sg = segO[at];
    const double ta = tauO[at];
    if (sg != cseg) {
      const size_t k0 = (size_t)sg * pst + rowOff;
      const double y0 = P[k0], y1 = P[k0 + pst], m0 = M[k0], m1 = M[k0 + pst];
      c.c3 = sdiv::div6(m1 - m0);
      c.c2 = m0 / 2.0;
      c.c1 = y1 - y0 - sdiv::div6(m1 + 2 * m0);
      c.c0 = y0;
      cseg = sg;
    }
    const double ta2 = ta * ta, ta3 = ta2 * ta;
    return seg_value(c, ta, ta2, ta3);
  }
};
// WM = wMid of smooth() (util.cpp:262): the window is 2*WM+1 points
template <int WM>
__global__ void k_out_eval_smooth(WSP, double *dst, int npts, int nb) {
  // x covers (trajectory, row) pairs, rows fastest (nb = Bo * R); y/z the decimated points
  const int R = w.R;
  const int xr = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  const int i = (int)((blockIdx.z * gridDim.y + blockIdx.y) * blockDim.y + threadIdx.y);
  if (xr >= nb) return;
  const int bl = xr / R, r = xr - bl * R;
  if (i >= npts) return;
  const int b = w.b0 + bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nSm) return;
  const int pt = CFG.c.path_type;
  const bool isJ = r < CFG.J;
  const bool driven = isJ ? (pt == BATOTP_JOINT || pt == BATOTP_BOTH) : (pt == BATOTP_CART || pt == BATOTP_BOTH);
  double v = 0.0;  // non-driven rows are zeros here (generic robot), and smoothing zeros gives zeros
  if (driven) {
    const int nIn = s.nOver, nOut = s.nSm;
    const int wv = (int)s.outSmooth;
    const double aOut = ((double)(nIn - 1) / (double)(nOut - 1)) * (double)i;
    UniformSites in{1.0};
    const int seg = find_seg(in, nIn, aOut);
    const double tau = (aOut - (double)seg) / ((double)(seg + 1) - (double)seg);
    OverEval X{w.P, w.M, w.tauO, w.segO, (size_t)w.B * R, (size_t)b * R + r, w.Bo, bl, -1, Seg4{0, 0, 0, 0}};
    int ww = imin_(wv, nIn);
    const int wMid = ww / 2 + ww % 2 - 1;
    double v0, v1;
    if (wMid == WM && seg >= WM && seg + 1 < nIn - WM) {
      // both windows are interior (util.cpp:268-273): their 2*WM+2 sites are evaluated once, in registers
      double x[2 * WM + 2];
#pragma unroll
      for (int q = 0; q < 2 * WM + 2; ++q) x[q] = X[seg - WM + q];
      double t0 = 0, t1 = 0;
#pragma unroll
      for (int q = 0; q < 2 * WM + 1; ++q) {
        t0 += x[q];
        t1 += x[q + 1];
      }
      v0 = t0 / (2 * WM + 1);
      v1 = t1 / (2 * WM + 1);
    } else {
      v0 = smooth_at(X, nIn, wv, seg);
      v1 = smooth_at(X, nIn, wv, seg + 1);
    }
    v = v0 + (v1 - v0) * tau;
  }
  dst[((size_t)i * w.Bo + bl) * R + r] = v;
}

// The same for joint-driven paths with one thread per (decimated point, trajectory): the NR = nJoints driven
// rows share the site lookups (segO/tauO are read once instead of once per row) and give the thread NR
// independent chains.  Rows NR..R-1 are the generic robot's zeros.  (TP)
template <int WM, int NR>
__global__ void k_out_eval_smooth_rows(WSP, double *dst, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = w.b0 + bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nSm) return;
  const int R = w.R;
  const int nIn = s.nOver, nOut = s.nSm;
  const int wv = (int)s.outSmooth;
  const double aOut = ((double)(nIn - 1) / (double)(nOut - 1)) * (double)i;
  UniformSites in{1.0};
  const int seg = find_seg(in, nIn, aOut);
  const double tau = (aOut - (double)seg) / ((double)(seg + 1) - (double)seg);
  double *o = dst + ((size_t)i * w.Bo + bl) * R;
  const size_t pst = (size_t)w.B * R;
  int ww = imin_(wv, nIn);
  const int wMid = ww / 2 + ww % 2 - 1;
  if (wMid == WM && seg >= WM && seg + 1 < nIn - WM) {
    // sites of the two windows first (independent loads), then one pass per distinct segment among them — the
    // sites are in ascending segment order, so the sums still run over ascending q as smooth() does — with the
    // coefficients {c3,c2,c1,c0} read from the segment table (no division left in this kernel's main path)
    int sgq[2 * WM + 2];
    double taq[2 * WM + 2];
#pragma unroll
    for (int q = 0; q < 2 * WM + 2; ++q) {
      const size_t at = (size_t)(seg - WM + q) * w.Bo + bl;
      sgq[q] = w.segO[at];
      taq[q] = w.tauO[at];
    }
    double t0[NR], t1[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) t0[r] = t1[r] = 0.0;
    int sgc = sgq[0];
    for (;;) {
      const double *t = w.tab + ((size_t)b * w.Nc + sgc) * (size_t)w.RT * 4;
      double c3[NR], c2[NR], c1[NR], c0[NR];
#pragma unroll
      for (int r = 0; r < NR; ++r) {
#ifdef BATOTP_HOST_EMU
        c3[r] = t[r * 4 + 0];
        c2[r] = t[r * 4 + 1];
        c1[r] = t[r * 4 + 2];
        c0[r] = t[r * 4 + 3];
#else
        const double2 lo = *reinterpret_cast<const double2 *>(t + r * 4);
        const double2 hi = *reinterpret_cast<const double2 *>(t + r * 4 + 2);
        c3[r] = lo.x;
        c2[r] = lo.y;
        c1[r] = hi.x;
        c0[r] = hi.y;
#endif
      }
      int nx = 0x7fffffff;
#pragma unroll
      for (int q = 0; q < 2 * WM + 2; ++q) {
        if (sgq[q] == sgc) {
          const double ta = taq[q], ta2 = ta * ta, ta3 = ta2 * ta;
#pragma unroll
          for (int r = 0; r < NR; ++r) {
            const double x = c3[r] * ta3 + c2[r] * ta2 + c1[r] * ta + c0[r];  // seg_value
            if (q <= 2 * WM) t0[r] += x;
            if (q >= 1) t1[r] += x;
          }
        } else if (sgq[q] > sgc) {
          nx = imin_(nx, sgq[q]);
        }
      }
      if (nx == 0x7fffffff) break;
      sgc = nx;
    }
    const sdiv::Rcp rw = {1.0 / (double)(2 * WM + 1), true};  // RN(1/w): folded at compile time
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const double v0 = sdiv::div(t0[r], (double)(2 * WM + 1), rw), v1 = sdiv::div(t1[r], (double)(2 * WM + 1), rw);
      o[r] = v0 + (v1 - v0) * tau;
    }
  } else {
    for (int r = 0; r < NR; ++r) {
      OverEval X{w.P, w.M, w.tauO, w.segO, pst, (size_t)b * R + r, w.Bo, bl, -1, Seg4{0, 0, 0, 0}};
      const double v0 = smooth_at(X, nIn, wv, seg), v1 = smooth_at(X, nIn, wv, seg + 1);
      o[r] = v0 + (v1 - v0) * tau;
    }
  }
  for (int r = NR; r < R; ++r) o[r] = 0.0;
}

// ----------------------------------------------------------------------------- final (T + TP)
// ba.cpp:1873-1921: final sizes
__global__ void k_out_final_plan(WSP) {
  const int bl = blockIdx.x * blockDim.x + threadIdx.x;
  if (bl >= w.Bo) return;
  TrajState &s = w.st[w.b0 + bl];
  if (s.status & ST_FATAL_MASK) return;
  const double tLast = s.tStep * (double)(s.nFwd - 1);
  if (s.isReinterp) {
    s.nOut = imax_((int)(ceil(tLast / s.outResT)), 4);
    s.sresOut = s.outResT;
    s.nCartOut = CFG.c.robot_type == BATOTP_GENJNT ? s.nSm : s.nOut;
  } else {
    s.nOut = s.nSm;
    s.sresOut = s.outResEff;
    s.nCartOut = s.nSm;
  }
  if (s.nOut > w.OutC) s.status |= ST_STEP_CAP;
}

// util.cpp:563-580
__host__ __device__ inline void q2aa_dev(const double q[4], double aa[3]) {
  const double nrm = sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (nrm < 1e-6) {
    aa[0] = aa[1] = aa[2] = 0.0;
  } else {
    const double theta = 2.0 * atan2(nrm, q[0]) / nrm;
    for (int i = 0; i < 3; ++i) aa[i] = theta * q[i + 1];
  }
}

// Final resample (when outRes < integRes, ba.cpp:1880-1915) and float32 packing in trajWriteBIN
// row order.  src rows hold nSm points, srcM their natural-spline solutions (point-major sub-chunk
// arrays); outputs are trajectory-major [Bo][row][OutC] as the caller's buffers.  (TP over OutC,
// points fastest so that the float rows are written coalesced)
// `pitch` = row stride (points) of the float32 outputs: the caller's out_cap when the rows travel on, so that a
// sub-chunk leaves in one contiguous copy; the FP64 side outputs (cartOutD, outD) keep the capacity w.OutC.
// `rag` (optional): ragged layout - trajectory bl's joint / torque block starts at (rag[bl] - rag0)*J floats and is
// [J][nOut] with no padding (cartOut must be NULL then); see batotp_batch_out.row_offset.
// outD: [Bo][J + C + J][OutC] (theta, Cartesian, torque rows), also when the Cartesian rows are not stored (zeros).
__global__ void k_out_pack(WSP, double *src, double *srcM, double *trqSrc, double *trqM, float *thetaOut,
                           float *cartOut, float *trqOut, double *cartOutD, double *outD, int pitch,
                           const long long *rag, long long rag0, int npts, int nb) {
  PT_DECOMP(npts);
  if (bl >= nb) return;
  const TrajState &s = w.st[w.b0 + bl];
  const int J = CFG.J, C = CFG.C, Cin = CFG.Cin, RD = J + C + J;
  const bool cartStored = w.R > J;  // otherwise the Cartesian rows are zeros (DevCfg::R)
  const bool fatal = (s.status & ST_FATAL_MASK) != 0;
  // float rows: pitched [bl][row][pitch], or ragged [rag[bl]*J + row*nOut]
  const size_t fBase = rag ? (size_t)(rag[bl] - rag0) * J : (size_t)bl * J * pitch;
  const size_t fRow = rag ? (size_t)(fatal ? 0 : s.nOut) : (size_t)pitch;
  const bool inF = rag ? (!fatal && i < s.nOut) : (i < pitch), inD = i < w.OutC;
  if (!inF && !inD) return;
  // rows are zero beyond their length (and for trajectories that were not optimised)
  if ((fatal || i >= s.nOut) && inF) {
    for (int r = 0; r < J; ++r) thetaOut[fBase + (size_t)r * fRow + i] = 0.f;
    if (trqOut && CFG.trqOn)
      for (int r = 0; r < J; ++r) trqOut[fBase + (size_t)r * fRow + i] = 0.f;
  }
  if (fatal || i >= s.nCartOut) {
    if (cartOut && inF)
      for (int r = 0; r < Cin; ++r) cartOut[((size_t)bl * Cin + r) * pitch + i] = 0.f;
    if (cartOutD && C == 7 && inD)
      for (int r = 0; r < 7; ++r) cartOutD[((size_t)bl * 7 + r) * w.OutC + i] = 0.0;
  }
  if (fatal) return;
  const bool generic = CFG.c.robot_type == BATOTP_GENJNT;
  int seg = 0;
  double tau = 0, tau2 = 0, tau3 = 0;
  const bool re = s.isReinterp != 0;
  if (re && i < s.nOut) {
    UniformSites s1{1. / (double)(s.nSm - 1)}, s2{1. / (double)(s.nOut - 1)};
    const double a = s2(i);
    seg = find_seg(s1, s.nSm, a);
    tau = (a - s1(seg)) / (s1(seg + 1) - s1(seg));
    tau2 = tau * tau;
    tau3 = tau2 * tau;
  }
  if (i < s.nOut) {
    for (int r = 0; r < J; ++r) {
      double v;
      if (re)
        v = seg_value(seg_coef(orowv(src, w, bl, r), orowv(srcM, w, bl, r), seg), tau, tau2, tau3);
      else
        v = orowv(src, w, bl, r)[i];
      if (inF) thetaOut[fBase + (size_t)r * fRow + i] = (float)v;
      if (outD) outD[((size_t)bl * RD + r) * w.OutC + i] = v;
    }
    if (trqOut && CFG.trqOn)
      for (int r = 0; r < J; ++r) {
        double v;
        if (re)
          v = seg_value(seg_coef(trqv(trqSrc, w, bl, r), trqv(trqM, w, bl, r), seg), tau, tau2, tau3);
        else
          v = trqv(trqSrc, w, bl, r)[i];
        if (inF) trqOut[fBase + (size_t)r * fRow + i] = (float)v;
        if (outD) outD[((size_t)bl * RD + J + C + r) * w.OutC + i] = v;
      }
  }
  if (i < s.nCartOut && (cartOut || cartOutD || outD)) {
    double cv[MAXD];
    for (int r = 0; r < C; ++r) {
      if (!cartStored)
        cv[r] = 0.0;
      else if (re && !generic)
        cv[r] = seg_value(seg_coef(orowv(src, w, bl, J + r), orowv(srcM, w, bl, J + r), seg), tau, tau2, tau3);
      else
        cv[r] = orowv(src, w, bl, J + r)[i];
    }
    if (outD)
      for (int r = 0; r < C; ++r) outD[((size_t)bl * RD + J + r) * w.OutC + i] = cv[r];
    if (C == 7) {
      if (cartOutD) {  // strict-parity path: the host applies q2aa with its own libm
        for (int r = 0; r < 7; ++r) cartOutD[((size_t)bl * 7 + r) * w.OutC + i] = cv[r];
      } else {
        double aa[3];
        q2aa_dev(cv + 3, aa);
        for (int r = 0; r < 3; ++r) cv[3 + r] = aa[r];
      }
    }
    if (cartOut && inF && !(C == 7 && cartOutD))
      for (int r = 0; r < Cin; ++r) cartOut[((size_t)bl * Cin + r) * pitch + i] = (float)cv[r];
  }
}

// k_out_pack for a generic robot without torque rows and without the FP64 copy (GEN7DOF / GENJNT batches): one warp
// per (trajectory, 32 consecutive output points).  The source rows are point-major, so the knots a tile needs -
// the points seg(i0) .. seg(i0+31)+1 of ONE trajectory, J contiguous doubles each - are staged cooperatively in
// shared memory (lanes run over (point, row), rows fastest: each request touches a few 8*J-byte runs instead of
// 32 scattered sectors), then every lane evaluates its output point for all rows with the expressions of
// k_out_pack and the float rows are written coalesced.  The Cartesian rows of a generic robot are plain copies
// of the source rows at the same index (k_out_pack: `re && !generic`), staged the same way.  A tile whose
// source range does not fit the staging buffer (output much coarser than the source) reads the knots directly.
// Block (32, OP_WARPS).
#define OP_WARPS 8
#define OP_CAP 40
struct SView {
  const double *p;
  int st;
  __host__ __device__ __forceinline__ double operator[](int i) const { return p[i * st]; }
};
__global__ void k_out_pack_rows(WSP, double *src, double *srcM, float *thetaOut, float *cartOut, int pitch,
                                const long long *rag, long long rag0, int npts, int nb) {
  EMU_SHARED double sY[OP_WARPS][OP_CAP * MAXD];
  EMU_SHARED double sM[OP_WARPS][OP_CAP * MAXD];
  const int lane = threadIdx.x, wy = threadIdx.y;
  const int i0 = (int)blockIdx.x * 32, i = i0 + lane;
  const int bl = (int)(blockIdx.z * gridDim.y + blockIdx.y) * OP_WARPS + wy;
  if (bl >= nb) return;  // the whole warp
  const TrajState &s = w.st[w.b0 + bl];
  const int J = CFG.J, Cin = CFG.Cin;
  const bool fatal = (s.status & ST_FATAL_MASK) != 0;
  const bool inRange = i < npts;
  const size_t pst = (size_t)w.Bo * w.R;
  // ---------------- joint rows
  const int nOut = fatal ? 0 : imin_(s.nOut, npts);
  const bool live = i < nOut;
  // float rows: pitched [bl][row][pitch], or ragged (rag[bl]*J + row*nOut: no padding, nothing beyond the length)
  const size_t fBase = rag ? (size_t)(rag[bl] - rag0) * J : (size_t)bl * J * pitch;
  const size_t fRow = rag ? (size_t)(fatal ? 0 : s.nOut) : (size_t)pitch;
  if (i0 < nOut) {  // warp-uniform
    const bool re = s.isReinterp != 0;
    int seg = live ? i : nOut - 1;
    double tau = 0, tau2 = 0, tau3 = 0;
    if (re) {
      UniformSites s1{1. / (double)(s.nSm - 1)}, s2{1. / (double)(s.nOut - 1)};
      const double a = s2(live ? i : nOut - 1);
      seg = find_seg(s1, s.nSm, a);
      tau = (a - s1(seg)) / (s1(seg + 1) - s1(seg));
      tau2 = tau * tau;
      tau3 = tau2 * tau;
    }
    const int lastLive = imin_(nOut - 1 - i0, 31);
    const int segLo = __shfl_sync(0xffffffffu, seg, 0);
    const int segHi = __shfl_sync(0xffffffffu, seg, lastLive) + (re ? 1 : 0);
    const int np = segHi - segLo + 1;
    // every live lane's knots inside the staged range (they are, for the non-decreasing seg of regular sites)
    const bool inside = !live || (seg >= segLo && seg + (re ? 1 : 0) <= segHi);
    if (__all_sync(0xffffffffu, inside) && np <= OP_CAP && np > 0) {  // warp-uniform
      const double *py = src + (size_t)bl * w.R + (size_t)segLo * pst;
      const double *pm = srcM + (size_t)bl * w.R + (size_t)segLo * pst;
      for (int e = lane; e < np * J; e += 32) {
        const int p = e / J, r = e - p * J;
        sY[wy][e] = py[(size_t)p * pst + r];
        if (re) sM[wy][e] = pm[(size_t)p * pst + r];
      }
      __syncwarp();
      if (live) {
        const int o = (seg - segLo) * J;
        for (int r = 0; r < J; ++r) {
          double v;
          if (re)
            v = seg_value(seg_coef(SView{&sY[wy][o + r], J}, SView{&sM[wy][o + r], J}, 0), tau, tau2, tau3);
          else
            v = sY[wy][o + r];
          thetaOut[fBase + (size_t)r * fRow + i] = (float)v;
        }
      }
      __syncwarp();  // the staging buffer is reused below
    } else if (live) {
      for (int r = 0; r < J; ++r) {
        double v;
        if (re)
          v = seg_value(seg_coef(orowv(src, w, bl, r), orowv(srcM, w, bl, r), seg), tau, tau2, tau3);
        else
          v = orowv(src, w, bl, r)[i];
        thetaOut[fBase + (size_t)r * fRow + i] = (float)v;
      }
    }
  }
  if (!live && inRange && !rag)  // rows are zero beyond their length (and for trajectories that were not optimised)
    for (int r = 0; r < J; ++r) thetaOut[fBase + (size_t)r * fRow + i] = 0.f;
  // ---------------- Cartesian rows (generic robot: the source rows J.. at the same index, no re-interpolation;
  //                  zeros when they are not stored)
  if (Cin > 0 && cartOut && w.R == J) {
    if (inRange)
      for (int r = 0; r < Cin; ++r) cartOut[((size_t)bl * Cin + r) * pitch + i] = 0.f;
  } else if (Cin > 0 && cartOut) {
    const int nC = fatal ? 0 : imin_(s.nCartOut, npts);
    const bool liveC = i < nC;
    if (i0 < nC) {  // warp-uniform
      const int npc = imin_(nC - i0, 32);
      const double *pc = src + (size_t)bl * w.R + J + (size_t)i0 * pst;
      for (int e = lane; e < npc * Cin; e += 32) {
        const int p = e / Cin, r = e - p * Cin;
        sY[wy][e] = pc[(size_t)p * pst + r];
      }
      __syncwarp();
      if (liveC)
        for (int r = 0; r < Cin; ++r) cartOut[((size_t)bl * Cin + r) * pitch + i] = (float)sY[wy][lane * Cin + r];
    }
    if (!liveC && inRange)
      for (int r = 0; r < Cin; ++r) cartOut[((size_t)bl * Cin + r) * pitch + i] = 0.f;
  }
}

// s-sdot histories in sdotWrite order (ascending s for the reverse sweep) as float32 (TP over Sc,
// points fastest); also clears the switching flags beyond the recorded steps.
// `pitch` = row stride (points) of histOut (the caller's hist_cap, or w.Sc); npts covers max(pitch, w.Sc).
__global__ void k_pack_hist(WSP, float *histOut, int pitch, int npts, int nb) {
  PT_DECOMP(npts);
  if (bl >= nb) return;
  const int b = w.b0 + bl;
  const TrajState &s = w.st[b];
  const bool fatal = (s.status & ST_FATAL_MASK) != 0;
  const int nRev = fatal ? 0 : s.nRev, nFwd = fatal ? 0 : s.nFwd;
  const double *hb = w.hist + (size_t)b * 4 * w.Sc;
  float *o = histOut + (size_t)bl * 4 * pitch;
  unsigned char *fl = w.flags + (size_t)b * 2 * w.Sc;
  const bool inF = i < pitch, inS = i < w.Sc;
  if (i < nRev) {
    if (inF) {
      o[i] = (float)hb[(w.Sc - nRev) + i];
      o[(size_t)pitch + i] = (float)hb[(size_t)w.Sc + (w.Sc - nRev) + i];
    }
  } else {
    if (inF) {
      o[i] = 0.f;
      o[(size_t)pitch + i] = 0.f;
    }
    if (inS) fl[i] = 0;
  }
  if (i < nFwd) {
    if (inF) {
      o[2 * (size_t)pitch + i] = (float)hb[2 * (size_t)w.Sc + i];
      o[3 * (size_t)pitch + i] = (float)hb[3 * (size_t)w.Sc + i];
    }
  } else {
    if (inF) {
      o[2 * (size_t)pitch + i] = 0.f;
      o[3 * (size_t)pitch + i] = 0.f;
    }
    if (inS) fl[(size_t)w.Sc + i] = 0;
  }
}

// per-trajectory scalars of the output sub-chunk -> the caller's arrays when those live on the device
// (batotp_batch_out.on_device); `first` = index of the resident chunk's first trajectory in the caller's batch (T)
struct ScalarOut {
  int *status, *n_rev, *n_fwd, *n_out, *n_cart_out, *n_grid;
  double *t_total, *t_rev, *s_last_sec, *out_sres;
};
__global__ void k_fetch_scalars(WSP, ScalarOut o, int first, int b0, int nb) {
  const int bl = blockIdx.x * blockDim.x + threadIdx.x;
  if (bl >= nb) return;
  const TrajState &s = w.st[b0 + bl];
  const int g = first + b0 + bl;
  const bool fatal = (s.status & ST_FATAL_MASK) != 0;
  if (o.status) o.status[g] = s.status;
  if (o.n_rev) o.n_rev[g] = s.nRev;
  if (o.n_fwd) o.n_fwd[g] = s.nFwd;
  if (o.n_out) o.n_out[g] = fatal ? 0 : s.nOut;
  if (o.n_cart_out) o.n_cart_out[g] = fatal ? 0 : s.nCartOut;
  if (o.n_grid) o.n_grid[g] = s.nPtsC;
  if (o.t_total) o.t_total[g] = s.tFwd;
  if (o.t_rev) o.t_rev[g] = s.tRev;
  if (o.s_last_sec) o.s_last_sec[g] = s.sLastSec;
  if (o.out_sres) o.out_sres[g] = s.sresOut;
}
