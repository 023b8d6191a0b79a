// k_sweep_group.cuh — the sweeps of the Bisection Algorithm with a GROUP of lanes per trajectory.
//
// Reference: the same functions as k_sweep.cuh (BA::sweep ba.cpp:979-1195, sdotLim 1204-1236,
// applyAccelConstraintsBisectionPt 1248-1332, evalSplinePartials 1341-1413, evalCartQuadCoeffs 1423-1439,
// verifySecondOrderConstraints 1449-1581, evalsdot 1590-1607, updateCurSeg 1617-1652).
//
// Why a second kernel.  k_sweep.cuh gives every lane its own trajectory: the cheapest mapping per trajectory
// (all 32 lanes do useful arithmetic), but one trajectory then costs ~2000 dependent instructions per point and the
// launch lasts (steps of the longest path) x 6 stages x that latency however few paths there are.  A batch that
// cannot fill the machine (the KUKA x4096 configuration: 128 warps for 592 warp schedulers; a single path: one
// lane) is bound by exactly that latency.  Here G = 8 (or 4) lanes share one trajectory: lane j owns joint j - its
// kinematic row and, with torque limits, its four dynamics rows - lanes 0..2 evaluate the Cartesian rows as a second
// job, and the per-joint loops of evalSplinePartials / sdotLim / verifySecondOrderConstraints become one pass plus a
// three-step shuffle reduction.  The scalar control (Runge-Kutta combine, MVC cursor, bisection bracket) is computed
// redundantly by every lane of the group, so nothing needs to be broadcast.  Per point a warp issues roughly a
// quarter of the instructions, four times as many warps are in flight for the same batch, and the coefficients
// live in registers.  Per trajectory it costs more issue slots (8 lanes carry one trajectory), so large batches stay
// with k_sweep.cuh; batotp_cuda.cu picks by chunk size.
//
// Bit-exactness.  Every value is formed by the expressions of k_sweep.cuh's exact path (eval_point / verify_point:
// reference operand order, shared-reciprocal divisions that equal '/').  The only new step is the reduction:
//   H = min over joints, L = max over joints, velocity cap = min over joints
// std::min / std::max are exact selections, so the fold order can only matter for ties between +0 and -0 and for
// NaN operands.  A lane folds its own quotients into the clamp +-sddotmax first (a NaN quotient is dropped there,
// as in the reference's H = min(H, x)), so no NaN enters the tree, and each tree step keeps the lower lane's value
// on a tie - the element the reference's left-to-right loop over the joints would have kept.
#pragma once
#include "k_sweep.cuh"

#ifndef SWG_NT
#ifdef BATOTP_HOST_EMU
#define SWG_NT 32  // the emulation pays for every fibre of a CTA at every collective: one warp per CTA
#else
#define SWG_NT 128
#endif
#endif

template <int J, bool CART>
struct GroupShape {
  static constexpr int NEED = (J > (CART ? 3 : 1)) ? J : (CART ? 3 : 1);
  static constexpr int G = NEED > 4 ? 8 : 4;  // lanes per trajectory
};

// min / max over the lanes of a group, ties resolved towards the lower lane (= the reference's loop order)
template <int G>
__device__ __forceinline__ double group_min(double v, int lane) {
#pragma unroll
  for (int m = 1; m < G; m <<= 1) {
    const double x = __shfl_xor_sync(0xffffffffu, v, m);
    v = (lane & m) ? dmin_(x, v) : dmin_(v, x);
  }
  return v;
}
template <int G>
__device__ __forceinline__ double group_max(double v, int lane) {
#pragma unroll
  for (int m = 1; m < G; m <<= 1) {
    const double x = __shfl_xor_sync(0xffffffffu, v, m);
    v = (lane & m) ? dmax_(x, v) : dmax_(v, x);
  }
  return v;
}

// LIM: every trajectory has its own limit row (w.lim): a lane loads its joint's four values and the Cartesian ones when
// its group picks a trajectory up
template <int J, bool CART, bool TRQ, bool LIM = false>
__global__ void __launch_bounds__(SWG_NT) k_sweep_group(WSP) {
  constexpr int G = GroupShape<J, CART>::G;
  constexpr int NK = J + (CART ? 3 : 0);
  constexpr int RT = NK + (TRQ ? 4 * J : 0);
#ifdef BATOTP_HOST_EMU
  static double smem_[14 * SWG_NT];
#else
  __shared__ double smem_[14 * SWG_NT];
#endif
  double (*sS)[SWG_NT] = reinterpret_cast<double (*)[SWG_NT]>(smem_);  // sdotArr[0..6], sddotArr[0..6], per lane
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int gl = lane & (G - 1);      // role inside the group
  const int gbase = lane & ~(G - 1);  // first lane of the group
  const bool jointLane = gl < J;
  const bool cartLane = CART && gl < 3;
  const unsigned gmask = ((G == 32) ? 0xffffffffu : ((1u << G) - 1u)) << gbase;  // (for ballots)
#define SD(k) sS[(k)][tid]
#define SDD(k) sS[7 + (k)][tid]
  // this lane's limits
  const int jj = jointLane ? gl : 0;
  const batotp_limits *lrow = nullptr;  // LIM: the row of trajectory b
#define LIMS LimSrc<LIM>::get(w, lrow)
  double velMax = CFG.c.jnt_vel_max[jj], accMax = CFG.c.jnt_acc_max[jj];
  double trqMax = CFG.c.jnt_trq_max[jj], trqMin = CFG.c.jnt_trq_min[jj];
  double cartVelMax = CFG.c.cart_vel_max;
  const bool accOn = CFG.c.is_jnt_acc_on != 0, cartAccOn = CART && CFG.c.is_cart_acc_on != 0;
  const bool cartVelOn = CART && CFG.c.is_cart_vel_on != 0;

  // ---- group state (identical in every lane of a group unless noted)
  int b = -1, dir = -1, istep = 0;
  int seg = 0, segLoaded = -1, lastSeg = 0, nM = 0, segM = 0, segMLoaded = -1;
  int nLim = 0, nBis = 0, limT = 0, isOn = 0, status = 0;
  unsigned nVerify = 0;
  double absh = 0, h = 0, sBack = 0, sLast = 0, sdotCap = 0, sdotMin = 0;
  double sArr0 = 0, sCur = 0, prevS = 0, prevSd = 0, sLastSec = 0;
  double m0 = 0, m1 = 0, d0 = 0, d1 = 0;
  sdiv::Rcp rTau = {0, false};
  double denTau = 1;
  double Lb = 0, Hb = 0;
  double velLim = 1.0 / 0.0;
  const double *tab = nullptr, *sM = nullptr, *sdM = nullptr;
  double *hs = nullptr, *hsd = nullptr;
  unsigned char *hflags = nullptr;
  TrajConsts C;
  C.sresC = C.vFact = C.aFact = C.sddotmax = C.thrV = C.thrA = C.thrQ = C.thrQ2 = C.amaxSQ = 0;
  Bisect bis;
  bis.begin(0.0);
  bool have = false, needPro = false, drained = false;
  // ---- per-lane rows: cached segment coefficients and the values at the current point
  // own joint row {3c3, 2c2, c1}; a lane without a joint keeps theta' = (tau + 1) vFact, theta'' = aFact: its
  // results are masked out everywhere, but the compiler evaluates some quotients of theta', theta'' ahead of
  // their conditions, and zeros there would send every such division down the slow path
  double kr0 = 0, kr1 = 1, kr2 = 1;
  double cr0 = 0, cr1 = 0, cr2 = 0;  // own Cartesian row (lanes 0..2)
  double dr[TRQ ? 4 : 1][4];          // own dynamics rows a1..a4 {c3,c2,c1,c0}
  double thD = 0, thDD = 0;
  sdiv::Rcp rD = {0, false};
  double a1 = 0, a2 = 0, a3 = 0, a4 = 0;
  sdiv::Rcp rA1 = {0, false};
  double Q0 = 0, Q1 = 0, Q2 = 0;
  sdiv::Rcp r2A = {0, false};
#pragma unroll
  for (int a = 0; a < (TRQ ? 4 : 1); ++a)
#pragma unroll
    for (int q = 0; q < 4; ++q) dr[a][q] = 0;

  // nRevKnown: the reverse sweep's point count as every lane knows it (the leader's store to TrajState may not be
  // visible to the other lanes yet)
  auto sweep_begin = [&](int d, int nRevKnown) {
    const TrajState &s = w.st[b];
    dir = d;
    absh = s.integRes;
    h = d * absh;
    lastSeg = s.nPtsC - 2;
    sBack = s.sresC * (double)(s.nPtsC - 1);
    sdotCap = sBack / absh;
    traj_consts(C, CFG, LIMS, s, sBack, absh);
    tab = w.tab + (size_t)b * w.Nc * (size_t)w.RT * 4;
    double *hb = w.hist + (size_t)b * 4 * w.Sc;
    if (d == 1) {
      hs = hb + 2 * (size_t)w.Sc;
      hsd = hb + 3 * (size_t)w.Sc;
      hflags = w.flags + ((size_t)b * 2 + 1) * w.Sc;
      nM = nRevKnown;
      sM = hb + (w.Sc - nRevKnown);
      sdM = hb + (size_t)w.Sc + (w.Sc - nRevKnown);
      seg = 0;
      sArr0 = 0;
      sLast = sBack;
    } else {
      hs = hb;
      hsd = hb + (size_t)w.Sc;
      hflags = w.flags + (size_t)b * 2 * w.Sc;
      nM = 0;
      sM = sdM = nullptr;
      seg = s.nPtsC - 2;
      sArr0 = sBack;
      sLast = 0;
    }
    segM = 0;
    segMLoaded = -1;
    segLoaded = -1;
    for (int q = 0; q < 14; ++q) sS[q][tid] = 0.0;
    sCur = sArr0;
    istep = 0;
    limT = 0;
    isOn = 0;
    nLim = nBis = 0;
    needPro = true;
  };
  // Every collective of this kernel is warp-wide and sits in convergent code, the queue fetch included: the groups
  // that need a trajectory draw one (their leader lane), all lanes take part in the broadcast, and the draw is
  // repeated while some group drew a trajectory that interpInputData has already rejected.
  auto fetch_all = [&]() {
    bool need = !have && !drained;
    while (__any_sync(0xffffffffu, need)) {
      int bb = 0;
      if (need && gl == 0) bb = atomicAdd(w.queue, 1);
      bb = __shfl_sync(0xffffffffu, bb, gbase);
      if (need) {
        b = bb;
        if (b >= w.B) {
          drained = true;
          need = false;
        } else if (!(w.st[b].status & ST_FATAL_MASK)) {
          need = false;
          have = true;
          status = 0;
          nVerify = 0;
          sLastSec = w.st[b].sLastSec;
          if (LIM) {
            lrow = w.lim + b;
            velMax = lrow->jnt_vel_max[jj];
            accMax = lrow->jnt_acc_max[jj];
            if (TRQ) {
              trqMax = lrow->jnt_trq_max[jj];
              trqMin = lrow->jnt_trq_min[jj];
            }
            if (CART) cartVelMax = lrow->cart_vel_max;
          }
          sweep_begin(-1, 0);
        }
      }
    }
  };
  auto mvc_window = [&]() {
    if (segM != segMLoaded) {
      m0 = sM[segM];
      m1 = sM[segM + 1];
      d0 = sdM[segM];
      d1 = sdM[segM + 1];
      segMLoaded = segM;
    }
  };
  auto mvc_cursor = [&](double s) {
    const int last = nM - 2;
    int guard = 0;
    for (;;) {
      mvc_window();
      if (s >= m0 && s <= m1) break;
      if (s > m0) {
        if (segM >= last) {
          segM = last;
          break;
        }
        segM++;
      }
      if (s < m0) {
        if (segM <= 0) {
          segM = 0;
          break;
        }
        segM--;
      }
      if (++guard > 4 * nM + 16) {
        status |= ST_NUMERIC;
        break;
      }
    }
    mvc_window();
  };
  auto sdot_lim = [&](double sd) {
    const double sdoti = sd;
    if (dir == 1) {
      mvc_cursor(sCur);
      const double tauM = (sCur - m0) / (m1 - m0);
      const double mv = dmax_(d0 + tauM * (d1 - d0), sdotMin);
      if (sd > mv) {
        isOn = 1;
        sd = mv;
      } else
        isOn = 0;
    }
    sd = dmin_(sd, sdotCap);
    sd = dmax_(sd, sdotMin);
    sd = dmin_(sd, velLim);
    if (sd < sdoti) limT = 1;
    return sd;
  };

  // verifySecondOrderConstraints (ba.cpp:1449-1581) for the group: this lane's joint, then the reduction, then the
  // Cartesian part (every lane forms it from the shared quadratic coefficients)
  auto verify = [&](double sdot, double &Lo, double &Hi) -> bool {
    double L = -C.sddotmax, H = C.sddotmax;
    const double sq = sdot * sdot;
    bool viol = false;
    if (TRQ && jointLane) {  // ba.cpp:1495-1509
      const double tmp1 = a3 * sdot + a4;
      if (!(fabs(a1) < C.thrV)) {
        const double tmp2 = a2 * sq + tmp1;
        const double s0 = sdiv::div(trqMax - tmp2, a1, rA1);
        const double s1 = sdiv::div(trqMin - tmp2, a1, rA1);
        H = dmin_(H, dmax_(s0, s1));
        L = dmax_(L, dmin_(s0, s1));
      }
    }
    if (accOn && jointLane) {  // ba.cpp:1514-1533
      const double v = thD;
      if (fabs(v) < C.thrV) {  // rare: the joint (nearly) stands still, only the curvature bounds sdot
        if (!(fabs(thDD) < C.thrA)) {
          double den = fabs(thDD);
#ifdef __CUDA_ARCH__
          asm volatile("" : "+d"(den));  // keeps the division inside its condition (it is loop-invariant and pure,
                                         // so it would be hoisted to every point otherwise)
#endif
          if (sq > accMax / den) viol = true;
        }
      } else {
        const int sg = (0.0 < v) - (v < 0.0);
        const double vT = thDD * sq;
        H = dmin_(H, sdiv::div((double)sg * accMax - vT, v, rD));
        L = dmax_(L, sdiv::div((double)(-sg) * accMax - vT, v, rD));
      }
    }
    H = group_min<G>(H, lane);
    L = group_max<G>(L, lane);
    viol = (__ballot_sync(0xffffffffu, viol) & gmask) != 0;
    viol |= (L > H);
    if (cartAccOn) {  // ba.cpp:1535-1578 + solveQuadratic util.cpp:361-383
      const double A = Q0;
      if (A > C.thrQ) {
        const double Bq = Q1 * sq;
        const double Cq = Q2 * sq * sq - C.amaxSQ;
        double s1 = 0, s2 = 0;
        bool haveRoots = true;
        if (fabs(A) < 1e-308) {
          if (fabs(Bq) < 1e-308)
            haveRoots = false;
          else {
            s1 = -Cq / Bq;
            s2 = s1;
          }
        } else {
          const double rad = Bq * Bq - 4 * A * Cq;
          if (rad < 0) {
            viol = true;
            haveRoots = false;
          } else {
            const double den = 2 * A;
            const double F1 = sdiv::div(-Bq, den, r2A), F2 = sdiv::div(sqrt(rad), den, r2A);
            s1 = F1 + F2;
            s2 = F1 - F2;
          }
        }
        if (haveRoots) {
          H = dmin_(H, dmax_(s1, s2));
          L = dmax_(L, dmin_(s1, s2));
          viol |= (L > H);
        }
      } else {
        double Cq = Q2;
        if (!(Cq < C.thrQ2)) {
#ifdef __CUDA_ARCH__
          asm volatile("" : "+d"(Cq));  // as above: not ahead of its condition
#endif
          if (sq * sq > C.amaxSQ / Cq) viol = true;
        }
      }
    }
    Lo = L;
    Hi = H;
    return viol;
  };

  // ================= one point for the groups with `act` (kind / j are warp-uniform) =================
  auto run_point = [&](const int kind, const int j, const bool act) {
    int r = BR_SETTLED;
    double sd = 0.0;
    if (act) {
      if (kind == TK_PRO1) {  // ba.cpp:1026-1035
        sd = .1 * h * SDD(0);
        sdotMin = sd;
      } else if (kind == TK_PRO2) {  // ba.cpp:1039-1041
        sd = bis.sdotIn;
      } else if (kind == TK_STAGE) {  // ba.cpp:1055-1089
        if (j == 0) {
          if (dir == 1) mvc_cursor(sArr0 + h * SD(0));
          nLim = 0;
          nBis = 0;
        }
        limT = 0;
        double sdotT = 0, sddotT = 0;
        for (int k = 0; k <= j; ++k) {
          const double bk = CFG.B[k][j];
          sdotT += bk * SD(k);
          sddotT += bk * SDD(k);
        }
        sCur = sArr0 + h * sdotT;
        sd = SD(0) + h * sddotT;
        sd = dmax_(sd, 0.0);
      }
      if (kind != TK_BEGIN) sd = sdot_lim(sd);
      if (kind == TK_PRO1) {
        sdotMin = sd;
        SD(0) = sd;
        if (gl == 0) hs[dir == 1 ? 0 : w.Sc - 1] = sArr0;
      }
      if (kind == TK_PRO2) {
        SD(0) = sd;
        if (gl == 0) {
          hsd[dir == 1 ? 0 : w.Sc - 1] = sd;
          hflags[0] = 0;
        }
        prevS = sArr0;
        prevSd = sd;
        istep = 1;
        needPro = false;
      }
    }
    if (kind == TK_PRO2) return;  // warp-uniform
    // ---------------- evalSplinePartials at sCur (ba.cpp:1341-1413).  The lanes of an idle group run the arithmetic
    // on whatever they hold (no memory access, results unused) so that the shuffles below stay warp-wide.
    double tau = 0;
    if (act) {
      double sSeg;
      if (!cursor_uniform(C.sresC, lastSeg, sCur, seg, sSeg)) status |= ST_NUMERIC;
      if (seg != segLoaded) {
        const double *t = tab + (size_t)seg * RT * 4;
        if (jointLane) {
          const double *p = t + gl * 4;
          kr0 = 3 * p[0];
          kr1 = 2 * p[1];
          kr2 = p[2];
        }
        if (cartLane) {
          const double *p = t + (J + gl) * 4;
          cr0 = 3 * p[0];
          cr1 = 2 * p[1];
          cr2 = p[2];
        }
        if (TRQ && jointLane) {
#pragma unroll
          for (int a = 0; a < (TRQ ? 4 : 1); ++a) {
            const double *p = t + (NK + a * J + gl) * 4;
#pragma unroll
            for (int q = 0; q < 4; ++q) dr[a][q] = p[q];
          }
        }
        denTau = C.sresC * (double)(seg + 1) - sSeg;
        rTau = sdiv::prep(denTau);
        segLoaded = seg;
#ifndef BATOTP_HOST_EMU
        {
          const int nx = seg + dir;
          if (nx >= 0 && nx <= lastSeg && gl * 128 < RT * 32)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char *>(tab + (size_t)nx * RT * 4) + gl * 128));
        }
#endif
      }
      tau = sdiv::div(sCur - sSeg, denTau, rTau);
      bis.begin(sd);
      r = BR_ITER;
    }
    {
      const double tau2 = tau * tau;
      double vl = 1.0 / 0.0;
      // joint row of this lane (ba.cpp:1359-1360)
      thD = (kr0 * tau2 + kr1 * tau + kr2) * C.vFact;
      thDD = ((2 * kr0) * tau + kr1) * C.aFact;
      rD = sdiv::prep(thD);
      if (jointLane && fabs(thD) > C.thrV) vl = fabs(sdiv::div(velMax, thD, rD));
      vl = group_min<G>(vl, lane);
      if (CART) {
        // Cartesian rows x, y, z on lanes 0..2 of the group, quadratic coefficients in every lane (ba.cpp:1434-1436)
        const double vo = (cr0 * tau2 + cr1 * tau + cr2) * C.vFact;
        const double ao = ((2 * cr0) * tau + cr1) * C.aFact;
        const double vx = __shfl_sync(0xffffffffu, vo, gbase), vy = __shfl_sync(0xffffffffu, vo, gbase + 1),
                     vz = __shfl_sync(0xffffffffu, vo, gbase + 2);
        const double ax = __shfl_sync(0xffffffffu, ao, gbase), ay = __shfl_sync(0xffffffffu, ao, gbase + 1),
                     az = __shfl_sync(0xffffffffu, ao, gbase + 2);
        Q0 = vx * vx + vy * vy + vz * vz;
        Q1 = 2 * (vx * ax + vy * ay + vz * az);
        Q2 = ax * ax + ay * ay + az * az;
        r2A = sdiv::prep(2 * Q0);
        if (cartVelOn && Q0 > C.thrQ) vl = dmin_(vl, cartVelMax / sqrt(Q0));
      }
      if (TRQ) {  // ba.cpp:1387-1405
        const double tau3 = tau2 * tau;
        a1 = dr[0][0] * tau3 + dr[0][1] * tau2 + dr[0][2] * tau + dr[0][3];
        a2 = dr[TRQ ? 1 : 0][0] * tau3 + dr[TRQ ? 1 : 0][1] * tau2 + dr[TRQ ? 1 : 0][2] * tau + dr[TRQ ? 1 : 0][3];
        a3 = dr[TRQ ? 2 : 0][0] * tau3 + dr[TRQ ? 2 : 0][1] * tau2 + dr[TRQ ? 2 : 0][2] * tau + dr[TRQ ? 2 : 0][3];
        a4 = dr[TRQ ? 3 : 0][0] * tau3 + dr[TRQ ? 3 : 0][1] * tau2 + dr[TRQ ? 3 : 0][2] * tau + dr[TRQ ? 3 : 0][3];
        rA1 = sdiv::prep(a1);
      }
      if (act) velLim = vl;
    }
    // ---------------- applyAccelConstraintsBisectionPt (ba.cpp:1270-1321)
    while (__any_sync(0xffffffffu, r == BR_ITER)) {
      double lo_, hi_;
      const bool viol = verify(bis.sdotCur, lo_, hi_);  // warp-wide (shuffles); idle groups discard the result
      if (r == BR_ITER) {
        Lb = lo_;
        Hb = hi_;
        nVerify++;
        r = bis.step_any(viol);
      }
    }
    // ---------------- the point is settled (ba.cpp:1090-1093)
    if (act) {
      const bool failed = (r == BR_FAILED);
      bis.sdotIn = failed ? sd : bis.sdotCur;
      if (bis.nIter > 0 && dir == -1 && sLastSec < 0) sLastSec = sCur;
      const double sddotRes = (dir == 1) ? Hb : Lb;
      if (failed) status |= ST_BISECT_FAIL;
      if (kind == TK_STAGE) {
        SD(j + 1) = bis.sdotIn;
        if (!failed) SDD(j + 1) = sddotRes;
        if (limT) nLim++;
        if (bis.nIter > 0) nBis++;
      } else {
        if (!failed) SDD(0) = sddotRes;
      }
    }
  };

  // ================= persistent warp loop =================
  for (;;) {
    __syncwarp();  // the leader's history stores of the last step are visible to the group (MVC reads)
    fetch_all();
    if (!__any_sync(0xffffffffu, have)) break;
    const bool pro = have && needPro;
    for (int p = __any_sync(0xffffffffu, pro) ? -3 : 0; p < 6; ++p)
      run_point(p < 0 ? p + 3 : TK_STAGE, p < 0 ? 0 : p, p < 0 ? pro : have);
    // ---- step end (ba.cpp:1096-1122)
    if (have) {
      bool sweepDone = false, trajAbort = false;
      int nPtsDone = 0;
      sArr0 = sCur;
      SD(0) = SD(6);
      SDD(0) = SDD(6);
      const int i = istep;
      if (i >= w.Sc) {
        status |= ST_STEP_CAP;
        trajAbort = true;
      } else {
        const int at = (dir == 1) ? i : (w.Sc - 1 - i);
        const double sd6 = SD(0);
        if (gl == 0) hflags[i] = (unsigned char)(nLim | (nBis << 3) | (isOn << 6));
        if (sCur * dir > sLast) {  // integration has completed: ba.cpp:1109-1141
          const int nPts = i + 1;
          const double sRat = (sLast - prevS) / (sArr0 - prevS);
          double sdLast = prevSd + sRat * (sd6 - prevSd);
          if (dir == 1) sdLast = sdM[nM - 1];
          if (gl == 0) {
            hs[at] = sLast;
            hsd[at] = sdLast;
            TrajState &s = w.st[b];
            if (dir == 1) {
              s.nFwd = nPts;
              s.tFwd = absh * i;
            } else {
              s.nRev = nPts;
              s.tRev = absh * i;
            }
          }
          nPtsDone = nPts;
          sweepDone = true;
        } else {
          if (gl == 0) {
            hs[at] = sArr0;
            hsd[at] = sd6;
          }
          prevS = sArr0;
          prevSd = sd6;
          const int maxIntegSteps = (int)floor(CFG.c.max_integ_time / absh) + 1;
          if (i > maxIntegSteps || (status & ST_NUMERIC)) {
            if (!(status & ST_NUMERIC)) status |= ST_MAX_INTEG_TIME;
            trajAbort = true;
          } else {
            istep = i + 1;
          }
        }
      }
      if (sweepDone || trajAbort) {  // rare path
        bool next = false;
        if (sweepDone && !trajAbort) {
          if (nPtsDone < 4) {  // ba.cpp:1171-1184: stretch a 2..3 point result to 4 points, linear in t
            if (gl == 0) stretch_to4(hs, hsd, w.Sc, nPtsDone, dir, absh, w.st[b]);
            nPtsDone = 4;
          } else if (dir == 1) {
            if (gl == 0) w.st[b].tStep = absh;
          }
          if (dir == -1) {
            sweep_begin(1, nPtsDone);
            next = true;
          }
        }
        if (!next) {
          if (gl == 0) {
            TrajState &s = w.st[b];
            s.status |= status;
            s.sLastSec = sLastSec;
            s.nVerify = (long long)nVerify;
          }
          have = false;
        }
      }
    }
  }
#undef SD
#undef SDD
#undef LIMS
}
