// k_mvc.cuh — derived product (SURVEY §8a A10): the per-sample maximum-velocity curve.
// One thread per (trajectory, grid knot): the sweep's own per-point functions
// (evalSplinePartials ba.cpp:1341, the velocity caps of sdotLim ba.cpp:1216-1229 without the
// MVC term, applyAccelConstraintsBisectionPt ba.cpp:1248) evaluated independently at every
// knot s_k, starting from `sdotStart`.  The reference has no such stage (its MVC is the
// reverse sweep); the oracle's orc_mvc_per_sample defines the expected values.
#pragma once
#include "k_sweep.cuh"

// LIM: trajectory b's limit row (w.lim) instead of the cfg's limits
template <int J, bool CART, bool TRQ, bool LIM = false>
__global__ void k_mvc(WSP, double sdotStart, double *out, int cap, int npts, int nb) {
  TP_DECOMP(nb);
  if (i >= npts) return;
  const int b = bl;
  const TrajState &s = w.st[b];
  if (s.status & ST_FATAL_MASK) return;
  if (i >= s.nPtsC || i >= cap) return;
  constexpr int NK = J + (CART ? 3 : 0);
  constexpr int RT = NK + (TRQ ? 4 * J : 0);
  const double absh = s.integRes;
  const double sBack = s.sresC * (double)(s.nPtsC - 1);
  const auto &lim = LimSrc<LIM>::get(w, LIM ? w.lim + b : nullptr);
  TrajConsts C;
  traj_consts(C, CFG, lim, s, sBack, absh);
  int seg = imin_(i, s.nPtsC - 2);
  const double sCur = s.sresC * (double)i;
  double sSeg;
  cursor_uniform(C.sresC, s.nPtsC - 2, sCur, seg, sSeg);
  const double tau = (sCur - sSeg) / (C.sresC * (double)(seg + 1) - sSeg);
  struct KGlobal {  // the segment table holds {c3,c2,c1,c0}; kinematic rows are read as {3c3, 2c2, c1, 6c3}
    const double *t;
    __host__ __device__ __forceinline__ double raw(int r, int q) const { return t[r * 4 + q]; }
    __host__ __device__ __forceinline__ double operator()(int r, int q) const {
      if (r >= NK) return t[r * 4 + q];
      return q == 0 ? 3 * t[r * 4] : (q == 1 ? 2 * t[r * 4 + 1] : (q == 2 ? t[r * 4 + 2] : 6 * t[r * 4]));
    }
  };
  const KGlobal K{w.tab + ((size_t)b * w.Nc + seg) * (size_t)RT * 4};
  PointVals<J, CART, TRQ> P;
  eval_point<J, CART, TRQ>(P, K, tau, C, CFG, lim);
  // sdotLim without the MVC term and with _sdotMin = 0
  double sd = sdotStart;
  sd = dmin_(sd, sBack / absh);
  sd = dmax_(sd, 0.0);
  sd = dmin_(sd, P.velLim);
  Bisect bis;
  bis.begin(sd);
  double Lo, Hi;
  for (;;) {
    const bool viol = verify_point<J, CART, TRQ>(P, C, CFG, lim, bis.sdotCur, Lo, Hi);
    if (bis.step(viol) != 0) break;
  }
  out[(size_t)b * cap + i] = bis.sdotIn;
}
