// tg_poly.cuh -- polynomial evaluation, Jenkins-Traub root finder and the per-segment magnitude extremum.
// One thread per (segment, quantity).
// Replaces Polynomial::evaluate / getCoefficients / convolve / computeMinMaxCandidates
// (reference: eth/polynomial.h:108-163, eth/polynomial.cpp:36-85,176-192), findRootsJenkinsTraub + rpoly_ak1
// (eth/rpoly/rpoly_ak1.cpp:59-120,148-932) and Segment::computeMinMaxMagnitudeCandidates /
// Trajectory::computeMinMaxMagnitude (eth/segment.cpp:113-212, eth/trajectory.cpp:211-243).
//
// B200 mapping: the reference's root finder walks five work arrays of up to 16 doubles with data-dependent bounds.
// Indexed dynamically they live in per-thread local memory and the kernel becomes L1/L2-traffic bound (round-1 ncu:
// profiles/).  Here the maximum degree M is a template parameter (it is fixed per quantity: 15/13/11 for |v|,|a|,|j| of
// the horizontal pair, 7/6/5 for a single dimension), every loop is fully unrolled to M with a predicate on the live
// degree, and all array indices are compile-time constants, so the arrays stay in REGISTERS.  The arithmetic
// performed for the live entries -- and therefore every root -- is identical to the dynamic formulation (and to the
// oracle, which is checked bit for bit against the reference's own file).
#ifndef TG_POLY_CUH_
#define TG_POLY_CUH_

#include "tg_common.cuh"

namespace tg {

// Horner from the top coefficient, one multiply and one add per step (eth/polynomial.h:150-163)
TG_HD double poly_eval(const double* __restrict__ c, double t, int deriv) {
  double acc = bcoef(deriv, TG_N - 1) * c[TG_N - 1];
  for (int j = TG_N - 2; j >= deriv; --j) {
    acc = acc * t;
    acc = acc + bcoef(deriv, j) * c[j];
  }
  return acc;
}
template <int DERIV, int N = TG_N>
TG_HD double poly_eval_s(const double* __restrict__ c, double t) {
  double acc = bcoef(DERIV, N - 1) * c[N - 1];
#pragma unroll
  for (int j = N - 2; j >= DERIV; --j) {
    acc = acc * t;
    acc = acc + bcoef(DERIV, j) * c[j];
  }
  return acc;
}

// Strided view of a per-thread work array.  On the device the five Jenkins-Traub work arrays live in SHARED memory,
// element i of thread t at base[i * blockDim + t] (conflict-free, no local-memory traffic); tests/host_emu uses stride 1.
#if defined(TG_JT_STATS)
static thread_local long long tg_jt_stats[16];
#endif
// The device kernels that use it run ONE WARP per block (cuda_backend.cu asserts it), so the stride is a compile-time
// constant there and an element address is one shift-add.  One warp per block because a block keeps its shared memory
// until its slowest thread is done, and Jenkins-Traub run times vary 3x between polynomials: with 128-thread blocks the
// SMs averaged 3.4 resident warps out of 12 (profiles/r01_extrema_s10.md).
#define TG_WARR_DEVICE_STRIDE 32
struct WArr {
  double* b;
  int st;
#if defined(__CUDA_ARCH__)
  TG_HD double& operator[](int i) const { return b[i * TG_WARR_DEVICE_STRIDE]; }
#else
  TG_HD double& operator[](int i) const { return b[(size_t)i * st]; }
#endif
};

// Jenkins-Traub three-stage iteration (TOMS 493) as an explicit per-thread STATE MACHINE.
//
// The reference code (rpoly_ak1.cpp:148-932) is a nest of data-dependent loops with early returns.  Run one thread per
// polynomial, the 32 lanes of a warp drift into different loops and the SIMT hardware serialises them (round-1 ncu of
// the direct transcription: 3.5 active lanes per instruction, I-cache misses the top stall -- profiles/).  Here every
// lane carries a `state`, and one pass of the driver loop executes each state's block once for the lanes that are in
// it, so lanes that are in the same stage -- whatever iteration they are at -- execute together.  The arithmetic inside
// a block, its order, the convergence tests and iteration caps are those of the reference, so the zeros are
// bit-identical to the oracle's (which is itself checked bit for bit against the reference file).
#ifndef TG_JT_REP
#define TG_JT_REP 1
#endif
#ifndef TG_JT_SCHED
#define TG_JT_SCHED 1  // 0: majority state first, 1: oldest first
#endif
// FP64 division, square root and the sign-preserving helpers are the bulk of the machine's code when inlined at ~40
// sites (an IEEE division is ~25 SASS instructions); one out-of-line copy measured fastest.  Measured and rejected in round 2
// (profiles/r02_extrema_jt.md): the compiler's fast division path written out inline with the reciprocal of a shared denominator
// computed once (calcSC divides three numerators by the same d) -- 42.8 vs 39.7 ms for the horizontal-acceleration launches.
#if defined(__CUDA_ARCH__) && !defined(TG_JT_INLINE_DIV)
__device__ __noinline__ double tg_jt_div(double a, double b) { return a / b; }
__device__ __noinline__ double tg_jt_sqrt(double a) { return tgdm::dsqrt(a); }
#define TG_DIV(a, b) tg_jt_div((a), (b))
#define TG_SQRT(a) tg_jt_sqrt(a)
#else
#define TG_DIV(a, b) ((a) / (b))
#define TG_SQRT(a) tgdm::dsqrt(a)
#endif
struct JtMachine {
  enum State { kRootBegin, kChop, kNewton, kKInit, kShiftBegin, kFsPrep, kFixedStep, kQuadStep, kRealStep, kDone };
  WArr p, qp, K, qk;  // shared-memory work arrays (degree + 1 entries each)
  double* svk;        // per-thread save areas (rarely touched): svk[0..M], tmp[0..M]
  double* tmp;
  int N, NN, state, nfound;
  int fl;  // floating-point operations executed for the current polynomial (counted per block, see step(); feeds the roofline)
  // calcSC scalars
  double a, b, c, d, e, f, g, h, a1, a3, a7;
  double szr, szi, lzr, lzi;
  // rpoly main
  double xx, yy, bnd, x, xm, dx, ff;
  int jj;
  // fixed shift
  double u, v, ui, vi, betas, betav, oss, ots, otv, ovv, s, ss, ts, tss, tv, tvv, vv;
  int j, L2, tFlag, spass, vpass, stry, vtry, first, prep_tail;
  // quadratic iteration
  double qu, qv, qomp, qrelstp;
  int qj, qtried;
  // real iteration
  double rs, rt, romp;
  int rj;
#if defined(TG_JT_STATS)
  int npass[16] = {0};
#endif

  TG_HD static void quad_sd(int nn, double uu, double vv_, const WArr& pp, const WArr& q, double* ra, double* rb) {
    double bb, aa;
    q[0] = bb = pp[0];
    q[1] = aa = -(bb * uu) + pp[1];
#pragma unroll 1
    for (int i = 2; i < nn; i++) {
      const double t = -(aa * uu + bb * vv_) + pp[i];
      q[i] = t;
      bb = aa;
      aa = t;
    }
    *ra = aa;
    *rb = bb;
  }
  TG_HD int calc_sc(double uu, double vv_) {  // rpoly_ak1.cpp:561-602
    quad_sd(N, uu, vv_, K, qk, &c, &d);
    if (dabs(c) <= (10.0 * TG_DBL_EPSILON * dabs(K[N - 1]))) {
      if (dabs(d) <= (10.0 * TG_DBL_EPSILON * dabs(K[N - 2]))) return 3;
    }
    h = vv_ * b;
    if (dabs(d) >= dabs(c)) {
      e = TG_DIV(a, d);
      f = TG_DIV(c, d);
      g = uu * b;
      a3 = e * (g + a) + h * TG_DIV(b, d);
      a1 = -a + f * b;
      a7 = h + (f + uu) * a;
      return 2;
    }
    e = TG_DIV(a, c);
    f = TG_DIV(d, c);
    g = e * uu;
    a3 = e * a + (g + TG_DIV(h, c)) * b;
    a1 = -(a * f) + b;  // f is TG_DIV(d, c), the quotient the reference computes a second time here
    a7 = g * d + h * f + a;
    return 1;
  }
  TG_HD void next_k(int tf) {  // rpoly_ak1.cpp:604-645
    if (tf == 3) {
      K[1] = K[0] = 0.0;
#pragma unroll 1
      for (int i = 2; i < N; i++) K[i] = qk[i - 2];
      return;
    }
    const double temp = ((tf == 1) ? b : a);
    if (dabs(a1) > (10.0 * TG_DBL_EPSILON * dabs(temp))) {
      a7 = TG_DIV(a7, a1);
      a3 = TG_DIV(a3, a1);
      K[0] = qp[0];
      K[1] = -(a7 * qp[0]) + qp[1];
#pragma unroll 1
      for (int i = 2; i < N; i++) K[i] = -(a7 * qp[i - 1]) + a3 * qk[i - 2] + qp[i];
    } else {
      K[0] = 0.0;
      K[1] = -a7 * qp[0];
#pragma unroll 1
      for (int i = 2; i < N; i++) K[i] = -(a7 * qp[i - 1]) + a3 * qk[i - 2];
    }
  }
  TG_HD void newest(int tf, double uu, double vv_, double* ou, double* ov) const {  // rpoly_ak1.cpp:647-683
    *ov = *ou = 0.0;
    if (tf == 3) return;
    double a4, a5;
    if (tf != 2) {
      a4 = a + uu * b + h * f;
      a5 = c + (uu + vv_ * f) * d;
    } else {
      a4 = (a + g) * f + h;
      a5 = (f + uu) * c + vv_ * d;
    }
    const double pN = p[N], pN1 = p[N - 1], kN1 = K[N - 1], kN2 = K[N - 2];
    const double b1 = TG_DIV(-kN1, pN);
    const double b2 = TG_DIV(-(kN2 + b1 * pN1), pN);
    const double c1 = vv_ * b2 * a1;
    const double c2 = b1 * a7;
    const double c3 = b1 * b1 * a3;
    const double c4 = -(c2 + c3) + c1;
    const double temp = -c4 + a5 + b1 * a4;
    if (temp != 0.0) {
      *ou = -TG_DIV(uu * (c3 + c2) + vv_ * (b1 * a1 + b2 * a7), temp) + uu;
      *ov = vv_ * (1.0 + TG_DIV(c4, temp));
    }
  }
  TG_HD static void quad(double qa, double b1, double qc, double* sr, double* si, double* lr, double* li) {  // rpoly_ak1.cpp:881-932
    *sr = *si = *lr = *li = 0.0;
    if (qa == 0) {
      *sr = ((b1 != 0) ? -TG_DIV(qc, b1) : *sr);
      return;
    }
    if (qc == 0) {
      *lr = -TG_DIV(b1, qa);
      return;
    }
    const double bb = b1 / 2.0;
    double dd, ee;
    if (dabs(bb) < dabs(qc)) {
      ee = ((qc >= 0) ? qa : -qa);
      ee = -ee + bb * TG_DIV(bb, dabs(qc));
      dd = TG_SQRT(dabs(ee)) * TG_SQRT(dabs(qc));
    } else {
      ee = -(TG_DIV(qa, bb) * TG_DIV(qc, bb)) + 1.0;
      dd = TG_SQRT(dabs(ee)) * (dabs(bb));
    }
    if (ee >= 0) {
      dd = ((bb >= 0) ? -dd : dd);
      *lr = TG_DIV(-bb + dd, qa);
      *sr = ((*lr != 0) ? TG_DIV(TG_DIV(qc, *lr), qa) : *sr);
    } else {
      *lr = *sr = -TG_DIV(bb, qa);
      *si = dabs(TG_DIV(dd, qa));
      *li = -(*si);
    }
  }

  // ---- control-flow glue of Fxshfr_ak1's third-stage do-while (rpoly_ak1.cpp:459-523) --------------------------
  TG_HD void restore_k() {
#pragma unroll 1
    for (int i = 0; i < N; i++) K[i] = svk[i];
  }
  TG_HD void begin_quad() {
    qj = 0;
    qtried = 0;
    qu = ui;
    qv = vi;
    qomp = 0.0;
    qrelstp = 0.0;
    state = kQuadStep;
  }
  TG_HD void begin_real() {
    rj = 0;
    rs = s;
    rt = 0.0;
    romp = 0.0;
    state = kRealStep;
  }
  TG_HD void stage3_top() {  // start of one pass of the do { } while (vpass && !vtry)
    const bool shortcut = first && ((spass) && (!vpass || (tss < tvv)));
    first = 0;
    if (!shortcut) begin_quad();
    else begin_real();
  }
  TG_HD void stage3_cond() {
    if (vpass && !vtry) {
      stage3_top();
    } else {
      prep_tail = 1;  // re-compute qp and the scalars, then finish this fixed-shift step
      state = kFsPrep;
    }
  }
  TG_HD void quad_failed() {
    vtry = 1;
    betav = betav * 0.25;
    if (stry || (!spass)) {
      restore_k();
      stage3_cond();
    } else {
      restore_k();
      begin_real();
    }
  }
  TG_HD void real_failed(int iFlag) {
    stry = 1;
    betas = betas * 0.25;
    if (iFlag != 0) {
      ui = -(s + s);
      vi = s * s;
      stage3_cond();  // `continue`: straight to the loop condition, K is NOT restored
    } else {
      restore_k();
      stage3_cond();
    }
  }
  template <class Sink>
  TG_HD void root_found(int nz, Sink& sink) {  // rpoly_ak1.cpp:338-356
    sink(szr, szi);
    if (nz != 1) sink(lzr, lzi);
    nfound += nz;
    NN = NN - nz;
    N = NN - 1;
#pragma unroll 1
    for (int i = 0; i < NN; i++) p[i] = qp[i];
    state = kRootBegin;
  }

  // One pass of the block of state `cur` (the caller guarantees state == cur).
  template <class Sink>
  TG_HD void step(int cur, Sink& sink, int* shifts) {
    const double lb2 = 0x1.62e42fefa39efp-1;   // log(2.0)
    const double lo = TG_FLT_MIN / TG_DBL_EPSILON;
    const double cosr = -0x1.1db8f6d6a512ap-4;  // cos(94 deg) as glibc returns it for 94.0 * (3.14159265358979323846 / 180)
    const double sinr = 0x1.fec0b7170fff6p-1;   // sin(94 deg)
    if (cur == kRootBegin) {
      fl += 2 * N + 90;   // moduli scan, scaling, log / exp of the starting radius
      if (N < 1) {
        state = kDone;
      } else if (N <= 2) {
        if (N < 2) {
          sink(-TG_DIV(p[1], p[0]), 0.0);
        } else {
          double sr_, si_, lr_, li_;
          quad(p[0], p[1], p[2], &sr_, &si_, &lr_, &li_);
          sink(sr_, si_);
          sink(lr_, li_);
        }
        state = kDone;
      } else {
        double moduli_max = 0.0, moduli_min = TG_FLT_MAX;
#pragma unroll 1
        for (int i = 0; i < NN; i++) {
          const double xa = dabs(p[i]);
          if (xa > moduli_max) moduli_max = xa;
          if ((xa != 0) && (xa < moduli_min)) moduli_min = xa;
        }
        double sc = TG_DIV(lo, moduli_min);
        if (((sc <= 1.0) && (moduli_max >= 10)) || ((sc > 1.0) && (TG_DIV(TG_FLT_MAX, sc) >= moduli_max))) {
          sc = ((sc == 0) ? TG_FLT_MIN : sc);
          const int l = (int)(TG_DIV(tgdm::dlog_k(sc), lb2) + 0.5);
          const double factor = tgdm::scalb(1.0, l);
          if (factor != 1.0)
#pragma unroll 1
            for (int i = 0; i < NN; i++) p[i] = p[i] * factor;
        }
        // upper estimate of the lower bound on the zero moduli; pt[i] = |p[i]|, pt[N] = -|p[N]|
        const double ptN = -dabs(p[N]), pt0 = dabs(p[0]), ptNM1 = dabs(p[N - 1]);
        x = tgdm::dexp_k(TG_DIV(tgdm::dlog_k(-ptN) - tgdm::dlog_k(pt0), (double)N));
        if (ptNM1 != 0) {
          const double xm_ = TG_DIV(-ptN, ptNM1);
          x = ((xm_ < x) ? xm_ : x);
        }
        xm = x;
        state = kChop;
      }
    }
    else if (cur == kChop) {
      fl += 2 * N + 1;
       // one pass of: do { x = xm; xm = 0.1 x; ff = pt(xm) } while (ff > 0)
      x = xm;
      xm = 0.1 * x;
      ff = dabs(p[0]);
#pragma unroll 1
      for (int i = 1; i < N; i++) ff = ff * xm + dabs(p[i]);
      ff = ff * xm + (-dabs(p[N]));
      if (!(ff > 0)) {
        dx = x;
        state = kNewton;
      }
    }
    else if (cur == kNewton) {
      fl += 4 * N + 3;
       // one pass of: while (|dx/x| > 0.005) { Newton step }
      if (dabs(TG_DIV(dx, x)) > 0.005) {
        double df;
        df = ff = dabs(p[0]);
#pragma unroll 1
        for (int i = 1; i < N; i++) {
          ff = x * ff + dabs(p[i]);
          df = x * df + ff;
        }
        ff = x * ff + (-dabs(p[N]));
        dx = TG_DIV(ff, df);
        x = x - dx;
      } else {
        bnd = x;
        state = kKInit;
      }
    }
    else if (cur == kKInit) {
      fl += 12 * N;
       // K = p'/N and five no-shift steps (rpoly_ak1.cpp:285-320)
      const int NM1 = N - 1;
#pragma unroll 1
      for (int i = 1; i < N; i++) K[i] = TG_DIV((double)(N - i) * p[i], (double)N);
      K[0] = p[0];
      const double aa = p[N], bb = p[NM1];
      int zerok = ((K[NM1] == 0) ? 1 : 0);
#pragma unroll 1
      for (int q = 0; q < 5; q++) {
        const double cc = K[NM1];
        if (zerok) {
#pragma unroll 1
          for (int i = 0; i < NM1; i++) {
            const int jx = NM1 - i;
            K[jx] = K[jx - 1];
          }
          K[0] = 0;
          zerok = ((K[NM1] == 0) ? 1 : 0);
        } else {
          const double t = TG_DIV(-aa, cc);
#pragma unroll 1
          for (int i = 0; i < NM1; i++) {
            const int jx = NM1 - i;
            K[jx] = t * K[jx - 1] + p[jx];
          }
          K[0] = p[0];
          zerok = ((dabs(K[NM1]) <= dabs(bb) * TG_DBL_EPSILON * 10.0) ? 1 : 0);
        }
      }
#pragma unroll 1
      for (int i = 0; i < N; i++) tmp[i] = K[i];
      jj = 1;
      state = kShiftBegin;
    }
    else if (cur == kShiftBegin) {
      fl += 10;
       // next shift of the jj loop (rpoly_ak1.cpp:324-336) + Fxshfr prologue (404-411)
      if (jj > 20) {
        state = kDone;  // no convergence after 20 shifts: the zeros found so far stand
      } else {
        const double xxx = -(sinr * yy) + cosr * xx;
        yy = sinr * xx + cosr * yy;
        xx = xxx;
        const double sr = bnd * xx;
        if (shifts) ++*shifts;
        betav = betas = 0.25;
        u = -(2.0 * sr);
        oss = sr;
        ovv = v = bnd;
        ots = otv = 0.0;
        j = 0;
        L2 = 20 * jj;
        prep_tail = 0;
        state = kFsPrep;
      }
    }
    else if (cur == kFsPrep) {
      fl += 8 * N + 7;    // quad_sd on p (4 per coefficient) + calc_sc
       // quad_sd on p + calc_sc: Fxshfr prologue (411-413) and stage-3 epilogue (527-528)
      quad_sd(NN, u, v, p, qp, &a, &b);
      tFlag = calc_sc(u, v);
      if (prep_tail) {
        ovv = vv;
        oss = ss;
        otv = tv;
        ots = ts;
        j++;
      }
      state = kFixedStep;
    }
    else if (cur == kFixedStep) {
      fl += 8 * N + 49;   // next_k + calc_sc + newest + convergence tests
       // one pass of the fixed-shift loop (rpoly_ak1.cpp:415-538)
      if (j >= L2) {
#pragma unroll 1
        for (int i = 0; i < N; i++) K[i] = tmp[i];  // unsuccessful shift: restore K, next jj
        jj++;
        state = kShiftBegin;
      } else {
        next_k(tFlag);
        tFlag = calc_sc(u, v);
        newest(tFlag, u, v, &ui, &vi);
        vv = vi;
        const double kN1 = K[N - 1];
        ss = ((kN1 != 0.0) ? -TG_DIV(p[N], kN1) : 0.0);
        ts = tv = 1.0;
        bool stage3 = false;
        if ((j != 0) && (tFlag != 3)) {
          tv = ((vv != 0.0) ? dabs(TG_DIV(vv - ovv, vv)) : tv);
          ts = ((ss != 0.0) ? dabs(TG_DIV(ss - oss, ss)) : ts);
          tvv = ((tv < otv) ? tv * otv : 1.0);
          tss = ((ts < ots) ? ts * ots : 1.0);
          vpass = ((tvv < betav) ? 1 : 0);
          spass = ((tss < betas) ? 1 : 0);
          if ((spass) || (vpass)) {
#pragma unroll 1
            for (int i = 0; i < N; i++) svk[i] = K[i];
            s = ss;
            stry = vtry = 0;
            first = 1;
            stage3 = true;
            stage3_top();
          }
        }
        if (!stage3) {
          ovv = vv;
          oss = ss;
          otv = tv;
          ots = ts;
          j++;
        }
      }
    }
    else if (cur == kQuadStep) {
      fl += 18 * N + 100; // quad, quad_sd, error bound, 2 x calc_sc, next_k, newest
       // one pass of QuadIT_ak1's do-while (rpoly_ak1.cpp:698-779)
      int nz = -1;  // -1: keep iterating
      quad(1.0, qu, qv, &szr, &szi, &lzr, &lzi);
      if (dabs(dabs(szr) - dabs(lzr)) > 0.01 * dabs(lzr)) {
        nz = 0;
      } else {
        quad_sd(NN, qu, qv, p, qp, &a, &b);
        const double mp = dabs(-(szr * b) + a) + dabs(szi * b);
        const double zm = TG_SQRT(dabs(qv));
        double ee = 2.0 * dabs(qp[0]);
        const double t = -(szr * b);
#pragma unroll 1
        for (int i = 1; i < N; i++) ee = ee * zm + dabs(qp[i]);
        ee = ee * zm + dabs(a + t);
        ee = (9.0 * ee + 2.0 * dabs(t) - 7.0 * (dabs(a + t) + zm * dabs(b))) * TG_DBL_EPSILON;
        if (mp <= 20.0 * ee) {
          nz = 2;
        } else {
          qj++;
          if (qj > 20) {
            nz = 0;
          } else {
            if (qj >= 2) {
              if ((qrelstp <= 0.01) && (mp >= qomp) && (!qtried)) {
                // a cluster stalls the convergence: five fixed-shift steps close to it
                qrelstp = ((qrelstp < TG_DBL_EPSILON) ? TG_SQRT(TG_DBL_EPSILON) : TG_SQRT(qrelstp));
                qu = qu - qu * qrelstp;
                qv = qv + qv * qrelstp;
                quad_sd(NN, qu, qv, p, qp, &a, &b);
#pragma unroll 1
                for (int i = 0; i < 5; i++) {
                  const int tf = calc_sc(qu, qv);
                  next_k(tf);
                }
                qtried = 1;
                qj = 0;
              }
            }
            qomp = mp;
            int tf = calc_sc(qu, qv);
            next_k(tf);
            tf = calc_sc(qu, qv);
            double qui, qvi;
            newest(tf, qu, qv, &qui, &qvi);
            if (qvi != 0) {
              qrelstp = dabs(TG_DIV(-qv + qvi, qvi));
              qu = qui;
              qv = qvi;
            } else {
              nz = 0;
            }
          }
        }
      }
      if (nz > 0) root_found(nz, sink);
      else if (nz == 0) quad_failed();
    }
    else if (cur == kRealStep) {
      fl += 10 * N + 10;  // two synthetic divisions, error bound, K update, K evaluation
       // one pass of RealIT_ak1's loop (rpoly_ak1.cpp:798-875)
      const int nm1 = N - 1;
      double pv;
      qp[0] = pv = p[0];
#pragma unroll 1
      for (int i = 1; i < NN; i++) qp[i] = pv = pv * rs + p[i];
      const double mp = dabs(pv);
      const double ms = dabs(rs);
      double ee = 0.5 * dabs(qp[0]);
#pragma unroll 1
      for (int i = 1; i < NN; i++) ee = ee * ms + dabs(qp[i]);
      if (mp <= 20.0 * TG_DBL_EPSILON * (2.0 * ee - mp)) {
        szr = rs;
        szi = 0.0;
        root_found(1, sink);
      } else {
        rj++;
        if (rj > 10) {
          real_failed(0);
        } else if ((rj >= 2) && ((dabs(rt) <= 0.001 * dabs(-rt + rs)) && (mp > romp))) {
          s = rs;  // a cluster near the real axis: hand the iterate to the quadratic iteration
          real_failed(1);
        } else {
          romp = mp;
          double kv;
          qk[0] = kv = K[0];
#pragma unroll 1
          for (int i = 1; i < N; i++) qk[i] = kv = kv * rs + K[i];
          if (dabs(kv) > dabs(K[nm1]) * 10.0 * TG_DBL_EPSILON) {
            rt = -TG_DIV(pv, kv);
            K[0] = qp[0];
#pragma unroll 1
            for (int i = 1; i < N; i++) K[i] = rt * qk[i - 1] + qp[i];
          } else {
            K[0] = 0.0;
#pragma unroll 1
            for (int i = 1; i < N; i++) K[i] = qk[i - 1];
          }
          kv = K[0];
#pragma unroll 1
          for (int i = 1; i < N; i++) kv = kv * rs + K[i];
          rt = ((dabs(kv) > (dabs(K[nm1]) * 10.0 * TG_DBL_EPSILON)) ? -TG_DIV(pv, kv) : 0.0);
          rs = rs + rt;
        }
      }
    }
  }
  // start of a polynomial of the given degree whose coefficients are already in p[0..degree]
  TG_HD void begin(int degree) {
    N = degree;
    NN = N + 1;
    xx = 0x1.6a09e667f3bcdp-1;  // sqrt(0.5)
    yy = -xx;
    state = kRootBegin;
    nfound = 0;
    fl = 0;
  }

  // Runs the machine to completion.  p[0..degree] holds the coefficients (decreasing powers, p[0] != 0 and zeros at the
  // origin already stripped by the caller).
  template <class Sink>
  TG_HD void run(int degree, Sink& sink, int* shifts) {
    begin(degree);
#if defined(__CUDA_ARCH__)
    const unsigned lanes = __activemask();  // the lanes that run this machine together
#endif
    for (;;) {
      // Warp-level scheduling: every pass executes ONE block, chosen uniformly for the warp (the state that most
      // unfinished lanes are in); lanes in other states sit the pass out.  All lanes in a block therefore execute it
      // together -- no reliance on the compiler's reconvergence of a divergent goto graph (which measured 2.6 active
      // lanes per instruction).  Lanes are independent, so the schedule cannot change any result.
      int cur = state;
#if defined(__CUDA_ARCH__)
#if TG_JT_SCHED == 0
      const unsigned same = __match_any_sync(lanes, state);
      const unsigned key = (state == kDone) ? 0u : (((unsigned)__popc(same) << 8) | (unsigned)(state + 1));
      const unsigned win = __reduce_max_sync(lanes, key);
      if (win == 0u) break;
      cur = (int)(win & 0xffu) - 1;
#else
      // oldest first: the lanes that are furthest behind (fewest zeros found, then earliest stage of the round) run;
      // lanes that are ahead wait for them, which keeps the warp in step round after round instead of letting it
      // split into groups that time-share the SM
      const unsigned key = (state == kDone) ? 0xffffffffu : (((unsigned)nfound << 8) | (unsigned)state);
      const unsigned win = __reduce_min_sync(lanes, key);
      if (win == 0xffffffffu) break;
      cur = (int)(win & 0xffu);
      if (key != win) continue;
#endif
#else
      if (cur == kDone) break;
#endif
      if (state != cur) continue;
      // a few consecutive steps of the same block per scheduling decision: amortises the warp vote and keeps the
      // instruction stream in one code region (round-1 ncu: instruction-fetch stalls dominated with one step per pass)
#pragma unroll 1
      for (int rep = 0; rep < TG_JT_REP && state == cur; ++rep) {
#if defined(TG_JT_STATS)
      npass[cur]++;
#endif
#if defined(TG_JT_TRACE)
      tg_jt_trace(cur, N);
#endif
      step(cur, sink, shifts);
      }  // rep
    }
  }
};

// doubles of strided scratch a thread needs for polynomials of degree <= M
template <int M>
struct JtScratch {
  static constexpr int kShared = 4 * (M + 1);  // p, qp, K, qk
};

// findRootsJenkinsTraub (rpoly_ak1.cpp:76-120) on INCREASING coefficients ci[0..M]: trims trailing |c| < DBL_MIN,
// reverses, strips the zeros at the origin (rpoly_ak1.cpp:174-180) and runs the machine.
template <int M, class Sink>
TG_HD void find_roots_jt(const double (&ci)[M + 1], double* scratch, int stride, Sink& sink, int* shifts, int* flops = nullptr) {
  int last = -1;
#pragma unroll
  for (int i = 0; i <= M; i++)
    if (dabs(ci[i]) >= TG_DBL_MIN) last = i;
  if (last < 1) return;  // all zero, or a constant: no roots
  // zeros at the origin = exactly-zero low-order coefficients (rpoly_ak1.cpp:174-180 tests op[N] == 0)
  int low = last;
#pragma unroll
  for (int i = M; i >= 0; i--)
    if (i <= last && ci[i] != 0.0) low = i;  // descending scan: ends at the lowest non-zero coefficient
  for (int z = 0; z < low; ++z) sink(0.0, 0.0);
  const int degree = last - low;
  double svk[M + 1], tmp[M + 1];
  JtMachine m;
  m.p = WArr{scratch, stride};
  m.qp = WArr{scratch + (size_t)(M + 1) * stride, stride};
  m.K = WArr{scratch + (size_t)2 * (M + 1) * stride, stride};
  m.qk = WArr{scratch + (size_t)3 * (M + 1) * stride, stride};
  m.svk = svk;
  m.tmp = tmp;
  // decreasing order: p[i] = ci[last - i], i = 0..degree
#pragma unroll
  for (int i = 0; i <= M; i++) {
    const int dst = last - i;
    if (dst >= 0 && dst <= degree) m.p[dst] = ci[i];
  }
  m.run(degree, sink, shifts);
  if (flops) *flops += m.fl;  // operations of the executed stage-machine blocks (profiling launches only)
#if defined(TG_JT_STATS)
  for (int i = 0; i < 10; ++i) tg_jt_stats[i] += m.npass[i];
#endif
}

// The same preparation without running the machine: m's work arrays are bound already; on return m.state is kRootBegin
// (polynomial loaded) or kDone (no zeros to iterate for).  Used by the persistent kernel that refills idle lanes.
template <int M, class Sink>
TG_HD void jt_load(const double (&ci)[M + 1], JtMachine& m, Sink& sink) {
  m.state = JtMachine::kDone;
  int last = -1;
#pragma unroll
  for (int i = 0; i <= M; i++)
    if (dabs(ci[i]) >= TG_DBL_MIN) last = i;
  if (last < 1) return;
  int low = last;
#pragma unroll
  for (int i = M; i >= 0; i--)
    if (i <= last && ci[i] != 0.0) low = i;
  for (int z = 0; z < low; ++z) sink(0.0, 0.0);
  const int degree = last - low;
#pragma unroll
  for (int i = 0; i <= M; i++) {
    const int dst = last - i;
    if (dst >= 0 && dst <= degree) m.p[dst] = ci[i];
  }
  m.begin(degree);
}

// candidate sink: magnitude of the DERIV-th derivative over dims [D0, D0+ND) at every real zero inside [0, T]
// (eth/polynomial.cpp:36-63 filter, eth/segment.cpp:172-178 magnitude, 203-209 maximum).  N: coefficients per polynomial (the
// general-shape path of tg_generic.cuh instantiates 6, 8, 10 and 12; every other caller the default).
template <int DERIV, int D0, int ND, int N = TG_N>
struct MaxSink {
  const double* coef;
  double T;
  double best;
  TG_HD void consider(double t) {
    double mag = 0.0;
#pragma unroll
    for (int dim = D0; dim < D0 + ND; ++dim) {
      const double v = poly_eval_s<DERIV, N>(coef + dim * N, t);
      mag = mag + v * v;
    }
    mag = dsqrt(mag);
    if (best < mag) best = mag;
  }
  TG_HD void operator()(double re, double im) {
    if (dabs(im) > TG_DBL_EPSILON) return;
    if (re < 0.0 || re > T) return;
    consider(re);
  }
};

// horizontal pair (dims 0,1): zeros of sum_d conv(p_d^(k), p_d^(k+1))  (eth/segment.cpp:122-145)
template <int DERIV, int N = TG_N>
TG_HD double segment_max_horizontal(const double* __restrict__ coef, double T, double* scratch, int stride, int* shifts, int* flops = nullptr) {
  constexpr int n_d = N - DERIV, n_dd = n_d - 1, len = n_d + n_dd - 1, M = len - 1;
  double acc[M + 1];
#pragma unroll
  for (int i = 0; i < len; ++i) acc[i] = 0.0;
#pragma unroll
  for (int dim = 0; dim < 2; ++dim) {
    const double* c = coef + dim * N;
    double dc[n_d], ddc[n_dd];
#pragma unroll
    for (int jx = 0; jx < n_d; ++jx) dc[jx] = c[jx + DERIV] * bcoef(DERIV, jx + DERIV);
#pragma unroll
    for (int jx = 0; jx < n_dd; ++jx) ddc[jx] = c[jx + DERIV + 1] * bcoef(DERIV + 1, jx + DERIV + 1);
#pragma unroll
    for (int i = 0; i < len; ++i) {
      double cv = 0.0;
      const int data_idx = i - n_dd + 1;
      const int lower = (0 > -data_idx) ? 0 : -data_idx, upper = (n_dd < n_d - data_idx) ? n_dd : n_d - data_idx;
#pragma unroll
      for (int kidx = lower; kidx < upper; ++kidx) cv = cv + ddc[n_dd - 1 - kidx] * dc[data_idx + kidx];
      acc[i] = acc[i] + cv;
    }
  }
  MaxSink<DERIV, 0, 2, N> sink{coef, T, TG_DBL_LOWEST};
  if (0.0 > T) return sink.best;
  sink.consider(0.0);
  sink.consider(T);
  find_roots_jt<M>(acc, scratch, stride, sink, shifts, flops);
  return sink.best;
}

// single dimension DIM: zeros of p^(k+1) (eth/polynomial.cpp:69-85)
template <int DERIV, int DIM, int N = TG_N>
TG_HD double segment_max_single(const double* __restrict__ coef, double T, double* scratch, int stride, int* shifts, int* flops = nullptr) {
  constexpr int M = N - DERIV - 2;  // degree of the (k+1)-th derivative
  const double* c = coef + DIM * N;
  double ddc[M + 1];
#pragma unroll
  for (int jx = 0; jx <= M; ++jx) ddc[jx] = c[jx + DERIV + 1] * bcoef(DERIV + 1, jx + DERIV + 1);
  MaxSink<DERIV, DIM, 1, N> sink{coef, T, TG_DBL_LOWEST};
  if (0.0 > T) return sink.best;
  sink.consider(0.0);
  sink.consider(T);
  find_roots_jt<M>(ddc, scratch, stride, sink, shifts, flops);
  return sink.best;
}

// computeMaximumOfMagnitude (lin_impl.h:477-508) on one segment: magnitude of the DERIV-th derivative over ALL dimensions
// (lin_impl.h:407-409) at t = 0, t = T and the real zeros of sum_d conv(p_d^(k), p_d^(k+1)) inside [0, T], in that order;
// a candidate replaces the running one only when strictly larger, so the first of equal maxima wins (operator< of
// Extremum compares values).  Leaves value = lowest() when the segment has no candidate (T < 0).
template <int DERIV, int N = TG_N>
struct MaxAllSink {
  const double* coef;
  double T;
  double best, best_t;
  TG_HD void consider(double t) {
    double mag = 0.0;
#pragma unroll
    for (int dim = 0; dim < TG_D; ++dim) {
      const double v = poly_eval_s<DERIV, N>(coef + dim * N, t);
      mag = mag + v * v;
    }
    mag = dsqrt(mag);
    if (best < mag) {
      best = mag;
      best_t = t;
    }
  }
  TG_HD void operator()(double re, double im) {
    if (dabs(im) > TG_DBL_EPSILON) return;
    if (re < 0.0 || re > T) return;
    consider(re);
  }
};
template <int DERIV, int N = TG_N>
struct MaxAllDegree {
  static constexpr int value = 2 * (N - DERIV) - 3;
};
template <int DERIV, int N = TG_N>
TG_HD void segment_max_all_dims(const double* __restrict__ coef, double T, double* scratch, int stride, double* value, double* time) {
  constexpr int n_d = N - DERIV, n_dd = n_d - 1, len = n_d + n_dd - 1, M = len - 1;
  double acc[M + 1];
#pragma unroll
  for (int i = 0; i < len; ++i) acc[i] = 0.0;
#pragma unroll 1
  for (int dim = 0; dim < TG_D; ++dim) {
    const double* c = coef + dim * N;
    double dc[n_d], ddc[n_dd];
#pragma unroll
    for (int jx = 0; jx < n_d; ++jx) dc[jx] = c[jx + DERIV] * bcoef(DERIV, jx + DERIV);
#pragma unroll
    for (int jx = 0; jx < n_dd; ++jx) ddc[jx] = c[jx + DERIV + 1] * bcoef(DERIV + 1, jx + DERIV + 1);
#pragma unroll
    for (int i = 0; i < len; ++i) {
      double cv = 0.0;
      const int data_idx = i - n_dd + 1;
      const int lower = (0 > -data_idx) ? 0 : -data_idx, upper = (n_dd < n_d - data_idx) ? n_dd : n_d - data_idx;
#pragma unroll
      for (int kidx = lower; kidx < upper; ++kidx) cv = cv + ddc[n_dd - 1 - kidx] * dc[data_idx + kidx];
      acc[i] = acc[i] + cv;
    }
  }
  MaxAllSink<DERIV, N> sink{coef, T, TG_DBL_LOWEST, 0.0};
  if (!(0.0 > T)) {
    sink.consider(0.0);
    sink.consider(T);
    find_roots_jt<M>(acc, scratch, stride, sink, nullptr);
  }
  *value = sink.best;
  *time = sink.best_t;
}

// Quantity Q in 0..8 : (group, derivative) = (horizontal|vertical|heading, velocity|acceleration|jerk) in the order
// the reference asks for them (eth/trajectory.cpp:616-622).  coef: [4][N] of one segment.
template <int Q, int N = TG_N>
TG_HD double segment_max_q(const double* __restrict__ coef, double T, double* scratch, int stride, int* shifts, int* flops = nullptr) {
  if constexpr (Q == 0) return segment_max_horizontal<1, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 1) return segment_max_horizontal<2, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 2) return segment_max_horizontal<3, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 3) return segment_max_single<1, 2, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 4) return segment_max_single<2, 2, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 5) return segment_max_single<3, 2, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 6) return segment_max_single<1, 3, N>(coef, T, scratch, stride, shifts, flops);
  else if constexpr (Q == 7) return segment_max_single<2, 3, N>(coef, T, scratch, stride, shifts, flops);
  else return segment_max_single<3, 3, N>(coef, T, scratch, stride, shifts, flops);
}

template <int Q, int N = TG_N>
TG_HD double segment_max_impl(const double* __restrict__ coef, double T, double* scratch, int stride, int* shifts, int* flops = nullptr) {
  return segment_max_q<Q, N>(coef, T, scratch, stride, shifts, flops);
}

// maximum polynomial degree met by quantity Q (scratch sizing): 2(N-k)-3 for the horizontal pair, N-k-2 for one dimension
// (N = 12: 19 for the horizontal velocity, the largest of any shape)
template <int Q, int N = TG_N>
struct QuantityDegree {
  static constexpr int kDeriv = Q % 3 + 1;
  static constexpr int value = (Q < 3) ? 2 * (N - kDeriv) - 3 : N - kDeriv - 2;
};

// What the persistent extrema kernel needs to know about quantity Q: the polynomial whose real zeros are the candidate
// times (eth/segment.cpp:122-145 for the horizontal pair, eth/polynomial.cpp:69-85 for one dimension) and the sink that
// evaluates the magnitude at them.
template <int Q, int N = TG_N>
struct QuantityJob {
  static constexpr int kDeriv = Q % 3 + 1;
  static constexpr bool kPair = Q < 3;
  static constexpr int kD0 = kPair ? 0 : (Q < 6 ? 2 : 3);
  static constexpr int kND = kPair ? 2 : 1;
  static constexpr int M = QuantityDegree<Q, N>::value;
  typedef MaxSink<kDeriv, kD0, kND, N> Sink;
  TG_HD static void poly(const double* __restrict__ coef, double (&ci)[M + 1]) {
    if constexpr (kPair) {
      constexpr int n_d = N - kDeriv, n_dd = n_d - 1, len = n_d + n_dd - 1;
      static_assert(len == M + 1, "degree");
#pragma unroll
      for (int i = 0; i < len; ++i) ci[i] = 0.0;
#pragma unroll
      for (int dim = 0; dim < 2; ++dim) {
        const double* c = coef + dim * N;
        double dc[n_d], ddc[n_dd];
#pragma unroll
        for (int jx = 0; jx < n_d; ++jx) dc[jx] = c[jx + kDeriv] * bcoef(kDeriv, jx + kDeriv);
#pragma unroll
        for (int jx = 0; jx < n_dd; ++jx) ddc[jx] = c[jx + kDeriv + 1] * bcoef(kDeriv + 1, jx + kDeriv + 1);
#pragma unroll
        for (int i = 0; i < len; ++i) {
          double cv = 0.0;
          const int data_idx = i - n_dd + 1;
          const int lower = (0 > -data_idx) ? 0 : -data_idx, upper = (n_dd < n_d - data_idx) ? n_dd : n_d - data_idx;
#pragma unroll
          for (int kidx = lower; kidx < upper; ++kidx) cv = cv + ddc[n_dd - 1 - kidx] * dc[data_idx + kidx];
          ci[i] = ci[i] + cv;
        }
      }
    } else {
      const double* c = coef + kD0 * N;
#pragma unroll
      for (int jx = 0; jx <= M; ++jx) ci[jx] = c[jx + kDeriv + 1] * bcoef(kDeriv + 1, jx + kDeriv + 1);
    }
  }
};

}  // namespace tg

#endif  // TG_POLY_CUH_

