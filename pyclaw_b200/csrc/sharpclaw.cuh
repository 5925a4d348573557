// sharpclaw.cuh -- SharpClaw: WENO5 reconstruction + interface / in-cell Riemann
// solves + fluctuation sum, fused with the SSP Runge-Kutta stage update (sm_100a).
//
// Replaces  src/fortran/2d/sharpclaw/flux2.f90:2-96 -> src/fortran/1d/sharpclaw/flux1.f90:2-195
//           -> reconstruct.f90:85-116 (weno_comp) -> weno.f90:5-102 (PyWENO weno5)
//           or reconstruct.f90:120-185 (hand-written weno5, lim_type 3)
// and the numpy stage arithmetic of src/pyclaw/sharpclaw.py:172-206.
//
// One thread per column i.  The x-direction of a row is done through shared memory
// (neighbouring threads hold neighbouring cells), the y-direction is a rolling 5-row
// window private to the thread, so q is read once and the stage result written once.
// dq = (0 + dq_x) + dq_y exactly as flux2.f90 accumulates it.
#pragma once
#include "launch.cuh"

struct WenoTab;
struct ScArgs {
    const double *q;  // stage state, ghost cells filled
    const double *qa; // second register of the RK combination (or null)
    double *out;
    double *dq_out;
    long long mstride;
    int pitch;
    int mx, my, mbc;
    double dtdx, dtdy;
    RpParams rp;
    // PyWENO coefficients (weno.f90:35-90), already rounded the way the chosen
    // variant reads the literals
    double c333, c1033, c366, c833, c633, c133, c433, c166;
    double d01, d06, d03, eps;
    double r183, r116, r0333, r0833, r0166;
    double epweno; // reconstruct.f90:7
    int mode;
    double ca, cb, div;
    unsigned long long *cfl_bits;
    int rows_per_cta;
    // capacity function (flux1.f90:59-63): dtdx(i) = dt / (dx * aux(mcapa, i))
    const double *capa; // the capa component of aux, padded like q (or null)
    double dt, dx, dy;
    // aux array for solvers that read it (flux1.f90:128,177-186): the interface solve sees
    // aux(i-1), aux(i); the in-cell solve sees aux(i) on both sides
    const double *aux;
    long long amstride;
    const struct WenoTab *tab; // weno_variant = tables: device memory owned by the caller
    // lim_type = 1 (flux1.f90:79-83): second-order TVD reconstruction, limiter id per COMPONENT
    int tvd;
    int mthlim[8];
    // 3-D (sharpclaw3.cuh): doubles per z-plane, mz, dt/dz
    long long plane;
    int mz;
    double dtdz;
};

// aux of the cell at array offset `off` (row offset + clamped column)
__device__ __forceinline__ AuxCell sc_aux(const ScArgs &A, long long off)
{
    return AuxCell{A.aux + off, A.amstride};
}

// dt / (d * capa) with one correctly rounded division, fast path first
__device__ __forceinline__ double sc_dtd(double dt, double d, double capa)
{
    FastArith fa;
    double den = d * capa;
    double v = fa.div(dt, den);
    if (fa.bad()) v = dt / den;
    return v;
}

// a product / a sum that nvcc never contracts into an FMA, whatever -fmad says
__device__ __forceinline__ double xm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xa(double a, double b) { return __dadd_rn(a, b); }

// weno.f90:35-98 for one component of one cell: ql = value at the left edge, qr at the right.
// The six weights are quotients over three denominators and two normalisations, i.e. five
// reciprocals for twelve divisions.
template <class AR>
__device__ __forceinline__ void weno5_pyweno(AR &ar, const ScArgs &A, double qm2, double qm1, double q0,
                                             double qp1, double qp2, double &ql, double &qr)
{
    // Smoothness indicators: sums of products that cancel to (nearly) zero wherever q is smooth,
    // over an eps of 1e-36 -- the non-linear weights are ill-conditioned in their rounding.  They
    // are therefore evaluated product by product and sum by sum in every build (xm / xa are never
    // contracted into an FMA): with contraction allowed here the fma build drifts from the strict
    // one by 1.5e-11 over the shallow-water test run, without it by round-off (profiles/README.md).
    double sigma0 = xa(xa(xa(xa(xa(xm(xm(A.c333, q0), q0), xm(xm(-A.c1033, q0), qp1)), xm(xm(A.c366, q0), qp2)),
                             xm(xm(A.c833, qp1), qp1)), xm(xm(-A.c633, qp1), qp2)), xm(xm(A.c133, qp2), qp2));
    double sigma1 = xa(xa(xa(xa(xa(xm(xm(A.c133, qm1), qm1), xm(xm(-A.c433, qm1), q0)), xm(xm(A.c166, qm1), qp1)),
                             xm(xm(A.c433, q0), q0)), xm(xm(-A.c433, q0), qp1)), xm(xm(A.c133, qp1), qp1));
    double sigma2 = xa(xa(xa(xa(xa(xm(xm(A.c133, qm2), qm2), xm(xm(-A.c633, qm2), qm1)), xm(xm(A.c366, qm2), q0)),
                             xm(xm(A.c833, qm1), qm1)), xm(xm(-A.c1033, qm1), q0)), xm(xm(A.c333, q0), q0));
    const Recip e0 = ar.rcp((sigma0 + A.eps) * (sigma0 + A.eps));
    const Recip e1 = ar.rcp((sigma1 + A.eps) * (sigma1 + A.eps));
    const Recip e2 = ar.rcp((sigma2 + A.eps) * (sigma2 + A.eps));
    // The twelve quotients need no validity tests of their own (div_nz): the numerators d0k are
    // positive constants, each reciprocal has passed its window test (2^-500 <= r < 2^500, or the
    // whole block is redone with the IEEE operators), so every omega lies in [2^-504, 2^500], acc in
    // [2^-504, 2^502], and a normalised weight omega / acc in [2^-1006, 1] because acc is a sum of
    // positive terms that contains omega: all normal, none zero.
    double acc = 0.0;
    double omega0 = ar.div_nz(A.d01, e0);
    acc = acc + omega0;
    double omega1 = ar.div_nz(A.d06, e1);
    acc = acc + omega1;
    double omega2 = ar.div_nz(A.d03, e2);
    acc = acc + omega2;
    const Recip ra = ar.rcp_nc(acc); // acc in [2^-504, 2^502]: its window test is implied
    omega0 = ar.div_nz(omega0, ra);
    omega1 = ar.div_nz(omega1, ra);
    omega2 = ar.div_nz(omega2, ra);
    acc = 0.0;
    double omega3 = ar.div_nz(A.d03, e0);
    acc = acc + omega3;
    double omega4 = ar.div_nz(A.d06, e1);
    acc = acc + omega4;
    double omega5 = ar.div_nz(A.d01, e2);
    acc = acc + omega5;
    const Recip rb = ar.rcp_nc(acc);
    omega3 = ar.div_nz(omega3, rb);
    omega4 = ar.div_nz(omega4, rb);
    omega5 = ar.div_nz(omega5, rb);
    double fr0 = (A.r183) * q0 + (-A.r116) * qp1 + (A.r0333) * qp2;
    double fr1 = (A.r0333) * qm1 + (A.r0833) * q0 + (-A.r0166) * qp1;
    double fr2 = (-A.r0166) * qm2 + (A.r0833) * qm1 + (A.r0333) * q0;
    double fr3 = (A.r0333) * q0 + (A.r0833) * qp1 + (-A.r0166) * qp2;
    double fr4 = (-A.r0166) * qm1 + (A.r0833) * q0 + (A.r0333) * qp1;
    double fr5 = (A.r0333) * qm2 + (-A.r116) * qm1 + (A.r183) * q0;
    ql = omega0 * fr0 + omega1 * fr1 + omega2 * fr2;
    qr = omega3 * fr3 + omega4 * fr4 + omega5 * fr5;
}

// reconstruct.f90:136-181 for one side.  (t1,t2,t3,e1,e2,e3) are the side's differences.
template <class AR>
__device__ __forceinline__ double weno5_old_side(AR &ar, double epweno, double t1, double t2, double t3,
                                                 double e1, double e2, double e3, double qa, double qb,
                                                 double qc, double qd)
{
    double tt1 = 13. * (t1 * t1) + 3. * (e1 * e1);
    double tt2 = 13. * (t2 * t2) + 3. * (e2 * e2);
    double tt3 = 13. * (t3 * t3) + 3. * (e3 * e3);
    tt1 = (epweno + tt1) * (epweno + tt1);
    tt2 = (epweno + tt2) * (epweno + tt2);
    tt3 = (epweno + tt3) * (epweno + tt3);
    double s1 = tt2 * tt3;
    double s2 = 6. * tt1 * tt3;
    double s3 = 3. * tt1 * tt2;
    double t0 = ar.div(1., s1 + s2 + s3);
    s1 = s1 * t0;
    s3 = s3 * t0;
    // (-q(i-2) + 7 (q(i-1) + q(i)) - q(i+1)) / 12
    return ar.div(s1 * (t2 - t1) + (0.5 * s3 - 0.25) * (t3 - t2), 3.) +
           ar.div(-qa + 7. * (qb + qc) - qd, 12.);
}

template <class AR>
__device__ __forceinline__ void weno5_old(AR &ar, const ScArgs &A, double a, double b, double c, double d,
                                          double e, double &ql, double &qr)
{
    double d1 = b - a, d2 = c - b, d3 = d - c, d4 = e - d; // dq1m(c-1), dq1m(c), dq1m(c+1), dq1m(c+2)
    // ql(c): m1 = 2 (im = -1) evaluated at position c
    ql = weno5_old_side(ar, A.epweno, -(d4 - d3), -(d3 - d2), -(d2 - d1), d4 - 3. * d3, d3 + d2,
                        3. * d2 - d1, a, b, c, d);
    // qr(c): m1 = 1 (im = +1) evaluated at position c+1
    qr = weno5_old_side(ar, A.epweno, (d1 - d2), (d2 - d3), (d3 - d4), d1 - 3. * d2, d2 + d3,
                        3. * d3 - d4, b, c, d, e);
}

// gfortran's MIN / MAX: "mvar = a1; if (a2 < mvar .or. isnan(mvar)) mvar = a2" -- a NaN argument
// is dropped in favour of the other one.  tvd2 divides by a jump that is zero in flat regions
// (r = 0/0), so the NaN rule decides the result there.
__device__ __forceinline__ double fmin_g(double a1, double a2) { return (a2 < a1 || a1 != a1) ? a2 : a1; }
__device__ __forceinline__ double fmax_g(double a1, double a2) { return (a2 > a1 || a1 != a1) ? a2 : a1; }

// reconstruct.f90:568-625 (tvd2) for one component of one cell: dqm = q(i) - q(i-1),
// dqp = q(i+1) - q(i), r = dqp / dqm, ql / qr = q(i) -/+ 0.5 phi(r) dqm.  The Fortran carries
// dqm over from the previous iteration (dqm = dqp), which for the FIRST cell of a slice is a
// variable that was never assigned; here every cell, the first included, uses its own backward
// difference (the only defined reading; DESIGN.md).
template <class AR>
__device__ __forceinline__ void tvd2(AR &ar, int meth, double b, double c, double d, double &ql, double &qr)
{
    const double dqm = c - b;
    const double dqp = d - c;
    const double r = ar.div(dqp, dqm);
    double qlimitr;
    switch (meth) {
    case 1: qlimitr = fmax_g(0.0, fmin_g(1.0, r)); break;
    case 2: qlimitr = fmax_g(fmax_g(0.0, fmin_g(1.0, 2.0 * r)), fmin_g(2.0, r)); break;
    case 3: qlimitr = ar.div(r + fabs(r), 1.0 + fabs(r)); break;
    case 4: {
        double cc = (1.0 + r) / 2.0;
        qlimitr = fmax_g(0.0, fmin_g(fmin_g(cc, 2.0), 2.0 * r));
    } break;
    case 5: { // Cada & Torrilhon, simple version
        const double beta = 2.0, xgamma = 2.0, alpha = 1.0 / 3.0;
        double pp = (2.0 + r) / 3.0;
        double amax = fmax_g(fmax_g(-alpha * r, 0.0), fmin_g(fmin_g(beta * r, pp), xgamma));
        qlimitr = fmax_g(0.0, fmin_g(pp, amax));
    } break;
    default: qlimitr = 0.0; // "select case" without a matching case leaves qlimitr as it was; 0 = first order
    }
    qr = c + 0.5 * qlimitr * dqm;
    ql = c - 0.5 * qlimitr * dqm;
}

template <bool OLD, class AR>
__device__ __forceinline__ void weno5(AR &ar, const ScArgs &A, double a, double b, double c, double d,
                                      double e, double &ql, double &qr, int m = 0)
{
    if (OLD) weno5_old(ar, A, a, b, c, d, e, ql, qr);
    else if (A.tvd) tvd2(ar, A.mthlim[m], b, c, d, ql, qr);
    else weno5_pyweno(ar, A, a, b, c, d, e, ql, qr);
}

__device__ __forceinline__ void sc_cfl_commit(double cfl, unsigned long long *cfl_bits)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double other = __shfl_xor_sync(0xffffffffu, cfl, o);
        cfl = dmax2(cfl, other);
    }
    if ((threadIdx.x & 31) == 0 && cfl > 0.0)
        atomicMax(cfl_bits, (unsigned long long)__double_as_longlong(cfl));
}

template <int MEQN>
__device__ __forceinline__ void stage_store(const ScArgs &A, long long idx, const double (&q)[MEQN],
                                            const double (&dq)[MEQN])
{
#pragma unroll
    for (int m = 0; m < MEQN; m++) {
        const long long o = m * A.mstride + idx;
        if (A.dq_out) A.dq_out[o] = dq[m];
        if (A.mode == 0) {
            double v = dq[m];
            if (A.div != 1.0) { // dq/6 of SSP104: zero increments are common, keep them off the slow path
                FastArith fa;
                v = fa.div(dq[m], A.div);
                if (fa.bad()) v = dq[m] / A.div;
            }
            A.out[o] = q[m] + v;
        } else if (A.mode == 1) {
            A.out[o] = A.ca * A.qa[o] + A.cb * (q[m] + dq[m]);
        } else if (A.mode == 2) {
            A.out[o] = (A.qa[o] + A.ca * q[m]) + A.cb * dq[m];
        }
    }
}

// x-direction of one row, shared by the 1-D and 2-D kernels.  On entry qs holds the
// staged row (index k <-> cell i0-3+k).  Returns dq_x for the thread's cell; full=false
// computes only the interface solve (rows 0 and my+1 contribute to the CFL number only).
// Everything of flux1.f90 after the reconstruction (:129-192), for the cell / interface of
// thread t: interface solve with the left neighbour's right-edge value, CFL, in-cell solve,
// fluctuation sum.
template <class RP, int NT>
__device__ __forceinline__ void sc_xrow_solve(const ScArgs &A, const double (&ql)[RP::MEQN],
                                              const double (&qr)[RP::MEQN], double *x1, double *x2,
                                              int t, bool iface_cfl, bool full, double &cfl,
                                              double (&dqx)[RP::MEQN], double dtdx_c, double dtdx_l,
                                              const AuxCell &axl, const AuxCell &axc);

template <class RP, bool OLD, int NT>
__device__ __forceinline__ void sc_xrow(const ScArgs &A, const double *qs, double *x1, double *x2,
                                        int t, bool iface_cfl, bool full, double &cfl,
                                        double (&dqx)[RP::MEQN], double dtdx_c, double dtdx_l,
                                        const AuxCell &axl, const AuxCell &axc)
{
    constexpr int MEQN = RP::MEQN;
    constexpr int QS = NT + 4;
    double ql[MEQN], qr[MEQN];
    with_arith_fz([&](auto &ar) {
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            const double *row = qs + m * QS + t;
            weno5<OLD>(ar, A, row[0], row[1], row[2], row[3], row[4], ql[m], qr[m], m);
        }
    });
    sc_xrow_solve<RP, NT>(A, ql, qr, x1, x2, t, iface_cfl, full, cfl, dqx, dtdx_c, dtdx_l, axl, axc);
}

template <class RP, int NT>
__device__ __forceinline__ void sc_xrow_solve(const ScArgs &A, const double (&ql)[RP::MEQN],
                                              const double (&qr)[RP::MEQN], double *x1, double *x2,
                                              int t, bool iface_cfl, bool full, double &cfl,
                                              double (&dqx)[RP::MEQN], double dtdx_c, double dtdx_l,
                                              const AuxCell &axl, const AuxCell &axc)
{
    constexpr int MEQN = RP::MEQN, MW = RP::MWAVES, NROE = RP::NROE;
#pragma unroll
    for (int m = 0; m < MEQN; m++) x1[m * NT + t] = qr[m];
    __syncthreads();
    double wave[MEQN][MW], s[MW], amdq[MEQN], apdq[MEQN], roe[NROE];
    double left[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) left[m] = x1[m * NT + (t > 0 ? t - 1 : 0)];
    with_arith_fz([&](auto &ar) { RP::solve(ar, A.rp, left, ql, axl, axc, wave, s, amdq, apdq, roe); });
    if (iface_cfl) {
#pragma unroll
        for (int mw = 0; mw < MW; mw++) cfl = dmax2(dmax2(cfl, dtdx_c * s[mw]), -dtdx_l * s[mw]);
    }
#pragma unroll
    for (int m = 0; m < MEQN; m++) x2[m * NT + t] = amdq[m];
    __syncthreads();
    if (full) {
        double amdq2[MEQN], apdq2[MEQN];
        with_arith_fz([&](auto &ar) { RP::solve(ar, A.rp, ql, qr, axc, axc, wave, s, amdq2, apdq2, roe); });
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            double an = x2[m * NT + (t < NT - 1 ? t + 1 : t)];
            dqx[m] = 0.0 - dtdx_c * (an + apdq[m] + amdq2[m] + apdq2[m]);
        }
    }
}

// ---------------------------------------------------------------------------
// 2-D: thread t <-> column ic = i0-1+t, output columns t = 1 .. NT-2.
// D3: the x and y directions of one z-plane k = blockIdx.z of [0, mz+1] of a 3-D field
// (sharpclaw3.cuh).  The ghost planes 0 and mz+1 add to the Courant number only.
// ---------------------------------------------------------------------------
#ifndef CLAW_SC_MINB
#define CLAW_SC_MINB 3 // 168 registers, 44 B of spills: 35.96 -> 32.49 ms per step (strict), 25.8 -> 21.6 ms (fma) at 8192^2; 4 CTAs spill 270 B
#endif
template <class RPX, class RPY, bool OLD, int NT, bool CAPA = false, bool D3 = false>
__global__ void __launch_bounds__(NT, (RPX::MEQN <= 3) ? CLAW_SC_MINB : 2) sc2d_kernel(const ScArgs A)
{
    constexpr int MEQN = RPX::MEQN, MW = RPX::MWAVES, NROE = RPX::NROE;
    constexpr int NC = NT - 2;
    constexpr int QS = NT + 4;
    extern __shared__ double sm[];
    double *qs0 = sm;                 // [2][MEQN][NT+4] staged rows (double buffered)
    double *x1 = qs0 + 2 * MEQN * QS; // [MEQN][NT]
    double *x2 = x1 + MEQN * NT;      // [MEQN][NT]

    const int t = threadIdx.x;
    const int mbc = A.mbc;
    const int i0 = 1 + blockIdx.x * NC;
    const int ic = i0 - 1 + t;
    const int imax = A.mx + mbc;
    const int icl = min(ic, imax) + mbc - 1;
    const int cstage = min(i0 - 3 + t, imax) + mbc - 1;
    const int cstage2 = min(i0 - 3 + NT + t, imax) + mbc - 1; // threads 0..3
    const bool col_out = (t >= 1) && (t <= NC) && (ic <= A.mx);
    const bool xiface = (t >= 1) && (ic >= 1) && (ic <= A.mx + 1);
    const bool ycol = (ic >= 0) && (ic <= A.mx + 1);
    const int j0 = 1 + blockIdx.y * A.rows_per_cta;
    const int j1 = min(j0 + A.rows_per_cta, A.my + 1);
    const long long po = D3 ? A.plane * (long long)(blockIdx.z + mbc - 1) : 0; // plane offset
    const bool gp = D3 && (blockIdx.z == 0 || blockIdx.z == A.mz + 1);         // ghost plane

    double cfl = 0.0;
    double dtdy_c = A.dtdy, dtdy_p = A.dtdy; // dt/(dy capa) of rows c and c-1
    double w0[MEQN], w1[MEQN], w2[MEQN], w3[MEQN], w4[MEQN];
    double dx1[MEQN], dx2[MEQN], dx3[MEQN], dx4[MEQN];
    double qr_prev[MEQN], apdq_prev[MEQN], amdq2_prev[MEQN], apdq2_prev[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) {
        w0[m] = w1[m] = w2[m] = w3[m] = w4[m] = 1.0;
        dx1[m] = dx2[m] = dx3[m] = dx4[m] = 0.0;
        qr_prev[m] = 1.0; apdq_prev[m] = amdq2_prev[m] = apdq2_prev[m] = 0.0;
    }

    // cp.async staging: row k+1 is requested into the other half of a double-buffered
    // shared-memory row before row k is processed (index kk <-> cell i0-3+kk)
    {
        const long long ro = (long long)A.pitch * (j0 - 3 + mbc - 1) + po;
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            cp_async8(&qs0[m * QS + t], &A.q[m * A.mstride + ro + cstage]);
            if (t < 4) cp_async8(&qs0[m * QS + NT + t], &A.q[m * A.mstride + ro + cstage2]);
        }
        cp_async_commit();
    }
    int qb = 0;
    for (int k = j0 - 3; k <= j1 + 2; k++) {
        const long long rowoff = (long long)A.pitch * (k + mbc - 1) + po;
        cp_async_wait_all();
        __syncthreads();
        const double *qs = qs0 + qb * (MEQN * QS);
        if (k < j1 + 2) {
            double *qsn = qs0 + (qb ^ 1) * (MEQN * QS);
            const long long ro = rowoff + A.pitch;
#pragma unroll
            for (int m = 0; m < MEQN; m++) {
                cp_async8(&qsn[m * QS + t], &A.q[m * A.mstride + ro + cstage]);
                if (t < 4) cp_async8(&qsn[m * QS + NT + t], &A.q[m * A.mstride + ro + cstage2]);
            }
            cp_async_commit();
        }
        qb ^= 1;
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            w0[m] = w1[m]; w1[m] = w2[m]; w2[m] = w3[m]; w3[m] = w4[m];
            w4[m] = qs[m * QS + t + 2]; // this thread's own column
            dx4[m] = dx3[m]; dx3[m] = dx2[m]; dx2[m] = dx1[m];
        }
        const bool xfull = (k >= j0) && (k < j1) && !gp;
        const bool xcfl_only = (k == 0 && j0 == 1) || (k == A.my + 1 && j1 == A.my + 1) || (gp && k >= j0 && k < j1);
        if (xfull || xcfl_only) {
            double dtdx_c = A.dtdx, dtdx_l = A.dtdx;
            if (CAPA) {
                const int il = min(max(ic - 1, 1 - mbc), imax) + mbc - 1;
                dtdx_c = sc_dtd(A.dt, A.dx, __ldg(&A.capa[rowoff + icl]));
                dtdx_l = sc_dtd(A.dt, A.dx, __ldg(&A.capa[rowoff + il]));
            }
            const AuxCell nocell{nullptr, 0};
            const bool AUXRP = (RPX::MAUX > 0);
            const int ilc = min(max(ic - 1, 1 - mbc), imax) + mbc - 1;
            sc_xrow<RPX, OLD, NT>(A, qs, x1, x2, t, xiface, xfull, cfl, dx1, dtdx_c, dtdx_l,
                                  AUXRP ? sc_aux(A, rowoff + ilc) : nocell, AUXRP ? sc_aux(A, rowoff + icl) : nocell);
        }

        // y-direction: reconstruct cell c = k-2 from rows k-4 .. k
        const int c = k - 2;
        if (c >= j0 - 1) {
            if (CAPA) {
                dtdy_p = dtdy_c;
                dtdy_c = sc_dtd(A.dt, A.dy, __ldg(&A.capa[(long long)A.pitch * (c + mbc - 1) + icl]));
            }
            double ql[MEQN], qr[MEQN];
            with_arith_fz([&](auto &ar) {
#pragma unroll
                for (int m = 0; m < MEQN; m++)
                    weno5<OLD>(ar, A, w0[m], w1[m], w2[m], w3[m], w4[m], ql[m], qr[m], m);
            });
            double wave[MEQN][MW], s[MW], amdq[MEQN], apdq[MEQN], roe[NROE];
            double amdq2[MEQN], apdq2[MEQN];
#pragma unroll
            for (int m = 0; m < MEQN; m++) { amdq[m] = apdq[m] = amdq2[m] = apdq2[m] = 0.0; }
            if (c >= j0) {
                const AuxCell nocell{nullptr, 0};
                const bool AUXRP = (RPY::MAUX > 0);
                const long long offc = (long long)A.pitch * (c + mbc - 1) + icl + po;
                const AuxCell ayc = AUXRP ? sc_aux(A, offc) : nocell;
                const AuxCell aym = AUXRP ? sc_aux(A, offc - A.pitch) : nocell;
                with_arith_fz([&](auto &ar) { RPY::solve(ar, A.rp, qr_prev, ql, aym, ayc, wave, s, amdq, apdq, roe); });
                if (ycol && c >= 1 && c <= A.my + 1) {
#pragma unroll
                    for (int mw = 0; mw < MW; mw++)
                        cfl = dmax2(dmax2(cfl, dtdy_c * s[mw]), -dtdy_p * s[mw]);
                }
                if (c < j1 && !gp)
                    with_arith_fz([&](auto &ar) { RPY::solve(ar, A.rp, ql, qr, ayc, ayc, wave, s, amdq2, apdq2, roe); });
                // cell c-1 = k-3 is complete
                const int jc = c - 1;
                if (jc >= j0 && jc < j1 && col_out && !gp) {
                    double dq[MEQN];
#pragma unroll
                    for (int m = 0; m < MEQN; m++) {
                        double dqy = 0.0 - dtdy_p * (amdq[m] + apdq_prev[m] + amdq2_prev[m] + apdq2_prev[m]);
                        dq[m] = (0.0 + dx4[m]) + dqy;
                    }
                    stage_store<MEQN>(A, (long long)A.pitch * (jc + mbc - 1) + icl + po, w1, dq);
                }
            }
#pragma unroll
            for (int m = 0; m < MEQN; m++) {
                qr_prev[m] = qr[m]; apdq_prev[m] = apdq[m];
                amdq2_prev[m] = amdq2[m]; apdq2_prev[m] = apdq2[m];
            }
        }
    }
    sc_cfl_commit(cfl, A.cfl_bits);
}

// ---------------------------------------------------------------------------
// 1-D: one row, x-direction only.
// ---------------------------------------------------------------------------
template <class RP, bool OLD, int NT, bool CAPA = false>
__global__ void __launch_bounds__(NT) sc1d_kernel(const ScArgs A)
{
    constexpr int MEQN = RP::MEQN;
    constexpr int NC = NT - 2;
    constexpr int QS = NT + 4;
    extern __shared__ double sm[];
    double *qs = sm;
    double *x1 = qs + MEQN * QS;
    double *x2 = x1 + MEQN * NT;
    const int t = threadIdx.x;
    const int mbc = A.mbc;
    const int i0 = 1 + blockIdx.x * NC;
    const int ic = i0 - 1 + t;
    const int imax = A.mx + mbc;
    const int icl = min(ic, imax) + mbc - 1;
    const int cstage = min(i0 - 3 + t, imax) + mbc - 1;
    const int cstage2 = min(i0 - 3 + NT + t, imax) + mbc - 1;
    const bool col_out = (t >= 1) && (t <= NC) && (ic <= A.mx);
    const bool xiface = (t >= 1) && (ic >= 1) && (ic <= A.mx + 1);
    double cfl = 0.0;
    double q0[MEQN], dqx[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) {
        qs[m * QS + t] = A.q[m * A.mstride + cstage];
        if (t < 4) qs[m * QS + NT + t] = A.q[m * A.mstride + cstage2];
        q0[m] = A.q[m * A.mstride + icl];
        dqx[m] = 0.0;
    }
    __syncthreads();
    double dtdx_c = A.dtdx, dtdx_l = A.dtdx;
    if (CAPA) {
        const int il = min(max(ic - 1, 1 - mbc), imax) + mbc - 1;
        dtdx_c = sc_dtd(A.dt, A.dx, __ldg(&A.capa[icl]));
        dtdx_l = sc_dtd(A.dt, A.dx, __ldg(&A.capa[il]));
    }
    const AuxCell nocell{nullptr, 0};
    const bool AUXRP = (RP::MAUX > 0);
    const int ilc = min(max(ic - 1, 1 - mbc), imax) + mbc - 1;
    sc_xrow<RP, OLD, NT>(A, qs, x1, x2, t, xiface, true, cfl, dqx, dtdx_c, dtdx_l,
                         AUXRP ? sc_aux(A, ilc) : nocell, AUXRP ? sc_aux(A, icl) : nocell);
    if (col_out) stage_store<MEQN>(A, icl, q0, dqx);
    sc_cfl_commit(cfl, A.cfl_bits);
}

// ---- launchers of the WENO5 stage kernels, for the built-in solvers (sharpclaw.cu), the user
// solver (sweep_user.cu) and the plane kernel of the 3-D stage (sharpclaw3.cuh).  old selects the
// literal reading of weno5 (weno_variant), CAPA the capacity-function form.
constexpr int SNT = 128; // threads per CTA

template <class RP, bool CAPA = false>
static int sc_launch1(bool old, const ScArgs &A, cudaStream_t st)
{
    constexpr int NC = SNT - 2;
    size_t smem = sizeof(double) * (RP::MEQN * (SNT + 4) + 2 * RP::MEQN * SNT);
    auto k = old ? sc1d_kernel<RP, true, SNT, CAPA> : sc1d_kernel<RP, false, SNT, CAPA>;
    k<<<(A.mx + NC - 1) / NC, SNT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

template <class RPX>
constexpr size_t sc2d_smem() { return sizeof(double) * (2 * RPX::MEQN * (SNT + 4) + 2 * RPX::MEQN * SNT); }

template <class RPX, class RPY, bool CAPA = false>
static int sc_launch2(bool old, ScArgs A, cudaStream_t st)
{
    constexpr int NC = SNT - 2;
    constexpr size_t smem = sc2d_smem<RPX>();
    auto k = old ? sc2d_kernel<RPX, RPY, true, SNT, CAPA> : sc2d_kernel<RPX, RPY, false, SNT, CAPA>;
    CUDA_OK(set_smem(k, smem));
    const int nxcta = (A.mx + NC - 1) / NC;
    A.rows_per_cta = pick_rows(A.my, nxcta, false);
    dim3 grid(nxcta, (A.my + A.rows_per_cta - 1) / A.rows_per_cta);
    k<<<grid, SNT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------
// 1-D, char_decomp = 1 (flux1.f90:95-105): wave-based WENO5, reconstruct.f90:393-471 (weno5_wave)
// and :474-565 (weno5_fwave, solver.fwave = True).  A Riemann solve between CELL AVERAGES gives
// the waves of every interface; the smoothness indicators are built from the projections of the
// neighbouring interfaces' waves (i-2 .. i+2) onto this interface's wave, family by family, and
// the reconstructed jump is added along the wave.  Thread t <-> cell / interface ic = i0-3+t;
// the waves travel through shared memory, both edge values of an interface (the right edge of
// cell t-1, the left edge of cell t) are produced by thread t itself.  Cells t = 3 .. NT-4 are
// output.  (The reference's 2-D flux1.f90 cannot run this branch: it calls rpn2 without ixy and
// then both reconstructions, src/fortran/2d/sharpclaw/flux1.f90:102-106.)
// ---------------------------------------------------------------------------
template <class RP, bool FW, int NT>
__global__ void __launch_bounds__(NT) sc1d_wave_kernel(const ScArgs A)
{
    constexpr int MEQN = RP::MEQN, MW = RP::MWAVES, NROE = RP::NROE;
    constexpr int NC = NT - 6;
    constexpr int QS = NT + 1;
    constexpr bool AUXRP = (RP::MAUX > 0);
    extern __shared__ double sm[];
    double *qs = sm;                   // [MEQN][NT+1], index k <-> cell i0-4+k
    double *wsm = qs + MEQN * QS;      // [MEQN*MW][NT] waves (f-waves / s) of interface t
    double *x1 = wsm + MEQN * MW * NT; // [MEQN][NT] right-edge value of cell t-1
    double *x2 = x1 + MEQN * NT;       // [MEQN][NT] amdq of interface t
    const int t = threadIdx.x;
    const int mbc = A.mbc;
    const int i0 = 1 + blockIdx.x * NC;
    const int ic = i0 - 3 + t;
    const int imax = A.mx + mbc;
    auto col = [&](int i) { return min(max(i, 1 - mbc), imax) + mbc - 1; };
    const int icl = col(ic), ill = col(ic - 1);
    const bool col_out = (t >= 3) && (t <= NT - 4) && (ic >= 1) && (ic <= A.mx);
    const bool xiface = (t >= 2) && (t <= NT - 3) && (ic >= 1) && (ic <= A.mx + 1);
    const double epweno = A.epweno, tiny = (double)1.e-14f;
#pragma unroll
    for (int m = 0; m < MEQN; m++) {
        qs[m * QS + t] = A.q[m * A.mstride + col(i0 - 4 + t)];
        if (t == 0) qs[m * QS + NT] = A.q[m * A.mstride + col(i0 - 4 + NT)];
    }
    __syncthreads();
    const AuxCell nocell{nullptr, 0};
    const AuxCell axl = AUXRP ? sc_aux(A, ill) : nocell, axc = AUXRP ? sc_aux(A, icl) : nocell;
    double qm[MEQN], q0[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) { qm[m] = qs[m * QS + t]; q0[m] = qs[m * QS + t + 1]; }
    // ---- waves between the cell averages (rp1(q1d, q1d, aux, aux)) ----
    double wv[MEQN][MW];
    {
        double s[MW], am[MEQN], ap[MEQN], roe[NROE];
        with_arith_fz([&](auto &ar) { RP::solve(ar, A.rp, qm, q0, axl, axc, wv, s, am, ap, roe); });
        if (FW) { // weno5_fwave: fwave / s, plain IEEE division (s = 0 gives Inf / NaN as in the Fortran)
#pragma unroll
            for (int m = 0; m < MEQN; m++)
#pragma unroll
                for (int mw = 0; mw < MW; mw++) wv[m][mw] = wv[m][mw] / s[mw];
        }
    }
#pragma unroll
    for (int m = 0; m < MEQN; m++)
#pragma unroll
        for (int mw = 0; mw < MW; mw++) wsm[(m * MW + mw) * NT + t] = wv[m][mw];
    __syncthreads();
    // ---- reconstruction at interface t: qrl = right edge of cell t-1, qll = left edge of cell t ----
    double qrl[MEQN], qll[MEQN];
    const int tm2 = max(t - 2, 0), tm1 = max(t - 1, 0), tp1 = min(t + 1, NT - 1), tp2 = min(t + 2, NT - 1);
    with_arith_fz([&](auto &ar) {
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            if (FW) {
                qrl[m] = qm[m];
                qll[m] = q0[m];
            } else {
                const double a = qs[m * QS + tm1], d = qs[m * QS + min(t + 2, NT)];
                qrl[m] = ar.div(-a + 7. * (qm[m] + q0[m]) - d, 12.);
                qll[m] = qrl[m];
            }
        }
#pragma unroll
        for (int mw = 0; mw < MW; mw++) {
            // projections of the neighbouring interfaces' waves on this one
            double wnorm2 = 0.0, dm2 = 0.0, dm1 = 0.0, dp1 = 0.0, dp2 = 0.0;
#pragma unroll
            for (int m = 0; m < MEQN; m++) {
                const double w = wv[m][mw];
                const double *row = wsm + (m * MW + mw) * NT;
                if (m == 0) {
                    wnorm2 = w * w; dm2 = row[tm2] * w; dm1 = row[tm1] * w; dp1 = row[tp1] * w; dp2 = row[tp2] * w;
                } else {
                    wnorm2 = wnorm2 + w * w; dm2 = dm2 + row[tm2] * w; dm1 = dm1 + row[tm1] * w;
                    dp1 = dp1 + row[tp1] * w; dp2 = dp2 + row[tp2] * w;
                }
            }
            double u[2], wn = 0.0;
#pragma unroll
            for (int m1 = 0; m1 < 2; m1++) {
                const double im = (m1 == 0) ? 1.0 : -1.0;
                const double theta1 = (m1 == 0) ? dm2 : dp2; // i + intwo
                const double theta2 = (m1 == 0) ? dm1 : dp1; // i + inone
                const double theta3 = (m1 == 0) ? dp1 : dm1; // i + ione
                const double t1 = im * (theta1 - theta2);
                const double t2 = im * (theta2 - wnorm2);
                const double t3 = im * (wnorm2 - theta3);
                double tt1 = 13. * (t1 * t1) + 3. * ((theta1 - 3. * theta2) * (theta1 - 3. * theta2));
                double tt2 = 13. * (t2 * t2) + 3. * ((theta2 + wnorm2) * (theta2 + wnorm2));
                double tt3 = 13. * (t3 * t3) + 3. * ((3. * wnorm2 - theta3) * (3. * wnorm2 - theta3));
                tt1 = (epweno + tt1) * (epweno + tt1);
                tt2 = (epweno + tt2) * (epweno + tt2);
                tt3 = (epweno + tt3) * (epweno + tt3);
                double s1 = tt2 * tt3;
                const double s2 = 6. * tt1 * tt3;
                double s3 = 3. * tt1 * tt2;
                const double t0 = ar.div(1., s1 + s2 + s3);
                s1 = s1 * t0;
                s3 = s3 * t0;
                if (wnorm2 > tiny) {
                    double uu = ar.div(s1 * (t2 - t1) + (0.5 * s3 - 0.25) * (t3 - t2), 3.);
                    if (FW) uu = uu + ar.div(im * (theta2 + 6.0 * wnorm2 - theta3), 12.0);
                    u[m1] = uu;
                    wn = ar.div(1.0, wnorm2);
                } else {
                    u[m1] = 0.0;
                    wn = 0.0;
                }
            }
#pragma unroll
            for (int m = 0; m < MEQN; m++) {
                qrl[m] = qrl[m] + u[0] * wv[m][mw] * wn;
                qll[m] = qll[m] + u[1] * wv[m][mw] * wn;
            }
        }
    });
    // ---- flux1.f90:129-192: interface solve, CFL, in-cell solve, fluctuation sum ----
    double cfl = 0.0;
    double wave[MEQN][MW], s[MW], amdq[MEQN], apdq[MEQN], roe[NROE];
    with_arith_fz([&](auto &ar) { RP::solve(ar, A.rp, qrl, qll, axl, axc, wave, s, amdq, apdq, roe); });
    if (xiface) {
#pragma unroll
        for (int mw = 0; mw < MW; mw++) cfl = dmax2(dmax2(cfl, A.dtdx * s[mw]), -A.dtdx * s[mw]);
    }
#pragma unroll
    for (int m = 0; m < MEQN; m++) { x1[m * NT + t] = qrl[m]; x2[m * NT + t] = amdq[m]; }
    __syncthreads();
    double qrc[MEQN], dqx[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) qrc[m] = x1[m * NT + tp1]; // right edge of this cell
    {
        double amdq2[MEQN], apdq2[MEQN];
        with_arith_fz([&](auto &ar) { RP::solve(ar, A.rp, qll, qrc, axc, axc, wave, s, amdq2, apdq2, roe); });
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            const double an = x2[m * NT + tp1];
            dqx[m] = 0.0 - A.dtdx * (an + apdq[m] + amdq2[m] + apdq2[m]);
        }
    }
    if (col_out) stage_store<MEQN>(A, icl, q0, dqx);
    sc_cfl_commit(cfl, A.cfl_bits);
}

// ---------------------------------------------------------------------------
// WENO of order 7 .. 17 (weno.f90:104-2425), 1-D.  The generated subroutines all have the
// shape of weno5 with k = (order+1)/2 stencils; the kernel walks coefficient tables held in
// caller-owned device memory (ScArgs::tab; regenerated on the host from the formulas' definition,
// pyclaw_b200/weno_tables.py) in the order the generated code evaluates its terms.
// ---------------------------------------------------------------------------
struct WenoTab { // all doubles: the packed buffer of clawb200_pack_weno_tables
    double k, eps;
    double S[9][45], CL[9][9], CR[9][9], WL[9], WR[9];
};

template <class AR>
__device__ __forceinline__ void weno_tab(AR &ar, const WenoTab &c_weno, const double *row /* cell i at row[0] */,
                                         double &ql, double &qr)
{
    const int k = (int)c_weno.k;
    const double eps = c_weno.eps;
    double sigma[9], omega[18];
    for (int r = 0; r < k; r++) {
        double sg = 0.0;
        int n = 0;
        for (int a = 0; a < k; a++)
            for (int b = a; b < k; b++) {
                double tt = xm(xm(c_weno.S[r][n], row[a - r]), row[b - r]); // never contracted (see weno5_pyweno)
                sg = (n == 0) ? tt : xa(sg, tt);
                n++;
            }
        sigma[r] = sg;
    }
    // as in weno5_pyweno: the linear weights are positive, each reciprocal passes its window test,
    // so the quotients (and the reciprocal of their sum) need none of their own
    Recip re[9];
    for (int r = 0; r < k; r++) re[r] = ar.rcp((sigma[r] + eps) * (sigma[r] + eps));
    double acc = 0.0;
    for (int r = 0; r < k; r++) {
        omega[r] = ar.div_nz(c_weno.WL[r], re[r]);
        acc = acc + omega[r];
    }
    {
        const Recip ra = ar.rcp_nc(acc);
        for (int r = 0; r < k; r++) omega[r] = ar.div_nz(omega[r], ra);
    }
    acc = 0.0;
    for (int r = 0; r < k; r++) {
        omega[k + r] = ar.div_nz(c_weno.WR[r], re[r]);
        acc = acc + omega[k + r];
    }
    {
        const Recip ra = ar.rcp_nc(acc);
        for (int r = 0; r < k; r++) omega[k + r] = ar.div_nz(omega[k + r], ra);
    }
    double fs0 = 0.0, fs1 = 0.0;
    for (int r = 0; r < k; r++) {
        double fl = 0.0, fq = 0.0;
        for (int j = 0; j < k; j++) {
            double tl = (c_weno.CL[r][j]) * row[j - r];
            double tr = (c_weno.CR[r][j]) * row[j - r];
            fl = (j == 0) ? tl : fl + tl;
            fq = (j == 0) ? tr : fq + tr;
        }
        double t0 = (omega[r]) * (fl), t1 = (omega[k + r]) * (fq);
        fs0 = (r == 0) ? t0 : fs0 + t0;
        fs1 = (r == 0) ? t1 : fs1 + t1;
    }
    ql = fs0;
    qr = fs1;
}

template <class RP, int NT>
__global__ void __launch_bounds__(NT) sc1d_tab_kernel(const ScArgs A)
{
    constexpr int MEQN = RP::MEQN;
    constexpr int NC = NT - 2;
    const WenoTab &c_weno = *A.tab;
    const int k = (int)c_weno.k;
    const int H = k - 1;            // halo cells of the stencil on each side
    const int QS = NT + 2 * H;
    extern __shared__ double sm[];
    double *qs = sm;                // [MEQN][NT + 2H], index e <-> cell i0-1-H+e
    double *x1 = qs + MEQN * QS;
    double *x2 = x1 + MEQN * NT;
    const int t = threadIdx.x;
    const int mbc = A.mbc;
    const int i0 = 1 + blockIdx.x * NC;
    const int ic = i0 - 1 + t;
    const int imax = A.mx + mbc;
    const int icl = min(ic, imax) + mbc - 1;
    const bool col_out = (t >= 1) && (t <= NC) && (ic <= A.mx);
    const bool xiface = (t >= 1) && (ic >= 1) && (ic <= A.mx + 1);
    for (int e = t; e < QS; e += NT) {
        const int c = min(max(i0 - 1 - H + e, 1 - mbc), imax) + mbc - 1;
#pragma unroll
        for (int m = 0; m < MEQN; m++) qs[m * QS + e] = A.q[m * A.mstride + c];
    }
    __syncthreads();
    double cfl = 0.0;
    double q0[MEQN], ql[MEQN], qr[MEQN], dqx[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) { q0[m] = qs[m * QS + t + H]; dqx[m] = 0.0; }
    with_arith_fz([&](auto &ar) {
#pragma unroll
        for (int m = 0; m < MEQN; m++) weno_tab(ar, c_weno, qs + m * QS + t + H, ql[m], qr[m]);
    });
    const AuxCell nocell{nullptr, 0};
    const bool AUXRP = (RP::MAUX > 0);
    const int ilc = min(max(ic - 1, 1 - mbc), imax) + mbc - 1;
    sc_xrow_solve<RP, NT>(A, ql, qr, x1, x2, t, xiface, true, cfl, dqx, A.dtdx, A.dtdx,
                          AUXRP ? sc_aux(A, ilc) : nocell, AUXRP ? sc_aux(A, icl) : nocell);
    if (col_out) stage_store<MEQN>(A, icl, q0, dqx);
    sc_cfl_commit(cfl, A.cfl_bits);
}

// ---------------------------------------------------------------------------
// WENO of order 7 .. 17 in 2-D (flux2.f90:2-96 over the table-driven reconstruction).
// Same decomposition as sc2d_kernel -- thread t <-> column ic, rows walked in order, the
// x-direction of a row through shared memory -- but the y-stencil (2k-1 rows) is gathered
// from global memory at every row instead of living in a rolling register window: these
// orders are a capability (no application of the reference selects them), not a tuned path.
// ---------------------------------------------------------------------------
template <class RPX, class RPY, int NT>
__global__ void __launch_bounds__(NT) sc2d_tab_kernel(const ScArgs A)
{
    constexpr int MEQN = RPX::MEQN, MW = RPX::MWAVES, NROE = RPX::NROE;
    constexpr int NC = NT - 2;
    const WenoTab &c_weno = *A.tab;
    const int kk = (int)c_weno.k;
    const int H = kk - 1;
    const int QS = NT + 2 * H;
    extern __shared__ double sm[];
    double *qs = sm;                // [MEQN][NT + 2H], index e <-> column i0-1-H+e
    double *x1 = qs + MEQN * QS;
    double *x2 = x1 + MEQN * NT;
    const int t = threadIdx.x;
    const int mbc = A.mbc;
    const int i0 = 1 + blockIdx.x * NC;
    const int ic = i0 - 1 + t;
    const int imax = A.mx + mbc;
    const int icl = min(ic, imax) + mbc - 1;
    const int ilc = min(max(ic - 1, 1 - mbc), imax) + mbc - 1;
    const bool col_out = (t >= 1) && (t <= NC) && (ic <= A.mx);
    const bool xiface = (t >= 1) && (ic >= 1) && (ic <= A.mx + 1);
    const bool ycol = (ic >= 0) && (ic <= A.mx + 1);
    const int j0 = 1 + blockIdx.y * A.rows_per_cta;
    const int j1 = min(j0 + A.rows_per_cta, A.my + 1);
    const AuxCell nocell{nullptr, 0};
    constexpr bool AUXX = (RPX::MAUX > 0), AUXY = (RPY::MAUX > 0);

    double cfl = 0.0;
    double dqx_prev[MEQN], q_prev[MEQN];
    double qr_prev[MEQN], apdq_prev[MEQN], amdq2_prev[MEQN], apdq2_prev[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) {
        dqx_prev[m] = 0.0; q_prev[m] = 1.0;
        qr_prev[m] = 1.0; apdq_prev[m] = amdq2_prev[m] = apdq2_prev[m] = 0.0;
    }
    for (int c = j0 - 1; c <= j1; c++) {
        const long long rowoff = (long long)A.pitch * (c + mbc - 1);
        // ---- x-direction of row c (rows 0 and my+1 only contribute to the CFL number)
        const bool xfull = (c >= j0) && (c < j1);
        const bool xcfl_only = (c == 0 && j0 == 1) || (c == A.my + 1 && j1 == A.my + 1);
        double dqx[MEQN], qc[MEQN];
#pragma unroll
        for (int m = 0; m < MEQN; m++) { dqx[m] = 0.0; qc[m] = A.q[m * A.mstride + rowoff + icl]; }
        if (xfull || xcfl_only) { // uniform over the CTA
            __syncthreads();
            for (int e = t; e < QS; e += NT) {
                const int col = min(max(i0 - 1 - H + e, 1 - mbc), imax) + mbc - 1;
#pragma unroll
                for (int m = 0; m < MEQN; m++) qs[m * QS + e] = A.q[m * A.mstride + rowoff + col];
            }
            __syncthreads();
            double ql[MEQN], qr[MEQN];
            with_arith_fz([&](auto &ar) {
#pragma unroll
                for (int m = 0; m < MEQN; m++) weno_tab(ar, c_weno, qs + m * QS + t + H, ql[m], qr[m]);
            });
            sc_xrow_solve<RPX, NT>(A, ql, qr, x1, x2, t, xiface, xfull, cfl, dqx, A.dtdx, A.dtdx,
                                   AUXX ? sc_aux(A, rowoff + ilc) : nocell, AUXX ? sc_aux(A, rowoff + icl) : nocell);
        }
        // ---- y-direction: reconstruct cell (ic, c) from rows c-H .. c+H
        double ql[MEQN], qr[MEQN];
        with_arith_fz([&](auto &ar) {
#pragma unroll
            for (int m = 0; m < MEQN; m++) {
                double col[17];
                for (int e = 0; e <= 2 * H; e++) {
                    const int row = min(max(c - H + e, 1 - mbc), A.my + mbc) + mbc - 1;
                    col[e] = A.q[m * A.mstride + (long long)A.pitch * row + icl];
                }
                weno_tab(ar, c_weno, col + H, ql[m], qr[m]);
            }
        });
        double wave[MEQN][MW], s[MW], amdq[MEQN], apdq[MEQN], roe[NROE];
        double amdq2[MEQN], apdq2[MEQN];
#pragma unroll
        for (int m = 0; m < MEQN; m++) { amdq[m] = apdq[m] = amdq2[m] = apdq2[m] = 0.0; }
        if (c >= j0) {
            const long long offc = rowoff + icl;
            const AuxCell ayc = AUXY ? sc_aux(A, offc) : nocell;
            const AuxCell aym = AUXY ? sc_aux(A, offc - A.pitch) : nocell;
            with_arith_fz([&](auto &ar) { RPY::solve(ar, A.rp, qr_prev, ql, aym, ayc, wave, s, amdq, apdq, roe); });
            if (ycol && c >= 1 && c <= A.my + 1) {
#pragma unroll
                for (int mw = 0; mw < MW; mw++) cfl = dmax2(dmax2(cfl, A.dtdy * s[mw]), -A.dtdy * s[mw]);
            }
            if (c < j1)
                with_arith_fz([&](auto &ar) { RPY::solve(ar, A.rp, ql, qr, ayc, ayc, wave, s, amdq2, apdq2, roe); });
            const int jc = c - 1; // this row's lower interface completes cell row c-1
            if (jc >= j0 && jc < j1 && col_out) {
                double dq[MEQN];
#pragma unroll
                for (int m = 0; m < MEQN; m++) {
                    double dqy = 0.0 - A.dtdy * (amdq[m] + apdq_prev[m] + amdq2_prev[m] + apdq2_prev[m]);
                    dq[m] = (0.0 + dqx_prev[m]) + dqy;
                }
                stage_store<MEQN>(A, (long long)A.pitch * (jc + mbc - 1) + icl, q_prev, dq);
            }
        } // c == j0-1: only the reconstruction (its right-edge value feeds interface j0)
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            qr_prev[m] = qr[m]; apdq_prev[m] = apdq[m];
            amdq2_prev[m] = amdq2[m]; apdq2_prev[m] = apdq2[m];
            dqx_prev[m] = dqx[m]; q_prev[m] = qc[m];
        }
    }
    sc_cfl_commit(cfl, A.cfl_bits);
}
