// rp.cuh -- pointwise Riemann solvers as inlined device functions (sm_100a).
//
// One struct per (equation set, sweep direction).  The sweeps in classic.cuh /
// sharpclaw.cuh instantiate them as template parameters, so the normal solve
// (rpn2 / rp1) and the transverse solve (rpt2) are inlined into the fused sweep
// kernels; what the reference passes through the `comroe` common block
// (development/rp_approaches/rpn2_euler_5wave.f:49-52) travels in registers as
// the `roe[]` array instead.
//
// Arithmetic follows the reference statement by statement, left to right, and the
// translation unit is compiled with -fmad=false, so results are bit-identical to
// the strict-IEEE CPU oracle (oracle/claw_oracle.c), which is itself pinned to the
// reference's golden files.
//
// Interface convention (rpn2_euler_5wave.f:24-25): the Riemann problem at interface i
// has left state qr(:,i-1) and right state ql(:,i); here simply `l[]` and `r[]`.
//
// Every division and square root goes through an arithmetic policy `AR` (arith.cuh):
// same correctly-rounded results, but divisions by a common denominator share one
// refined reciprocal and no operation carries its own slow-path branch.
#pragma once
#include "arith.cuh"

#define CLAW_RP_ACOUSTICS 1
#define CLAW_RP_ADVECTION 2
#define CLAW_RP_EULER5 3
#define CLAW_RP_SHALLOW 4

#define CLAW_RP_SPHERE 5
#define CLAW_RP_NEL_FWAVE 6
#define CLAW_RP_PSYSTEM 7
#define CLAW_RP_ACOUSTICS3D_VC 8
#define CLAW_RP_VC_ACOUSTICS 9
#define CLAW_RP_BURGERS 10
#define CLAW_RP_ADVECTION_COLOR 11
#define CLAW_RP_VC_ADVECTION 12
#define CLAW_RP_EULER1D 13
#define CLAW_RP_ADVECTION3D 14
#define CLAW_RP_EULER3D 15
#define CLAW_RP_ADVECTION3D_VC_FWAVE 16
#define CLAW_RP_SHALLOW_BATHY_FWAVE 17
#define CLAW_RP_USER 100 // a solver compiled in from a user header (sweep_user.cu)

// Solvers that return f-waves (jumps in the flux) instead of waves: the sweeps then use the
// second-order correction of step1fw.f:135-136 / flux2fw.f:151-152.  A member FWAVE = true
// in the solver struct selects it; solvers without the member are wave solvers.
template <class RP, class = void>
struct rp_is_fwave { static constexpr bool value = false; };
template <class RP>
struct rp_is_fwave<RP, decltype((void)RP::FWAVE)> { static constexpr bool value = RP::FWAVE; };

// Solvers whose y-sweep window fits in registers declare Y_REGS = true (classic.cuh, y-engine).
template <class RP, class = void>
struct rp_y_regs { static constexpr bool value = false; };
template <class RP>
struct rp_y_regs<RP, decltype((void)RP::Y_REGS)> { static constexpr bool value = RP::Y_REGS; };

// CTAs per SM the single-pass kernel (fused.cuh) is compiled for; solvers may override F_MINB.
template <class RP, class = void>
struct rp_f_minb { static constexpr int value = 3; };
template <class RP>
struct rp_f_minb<RP, decltype((void)RP::F_MINB)> { static constexpr int value = RP::F_MINB; };

struct RpParams {
    double p[8];
};

// One cell of the aux array (structure of arrays, component stride `ms`); read through
// the read-only path.  A null cell is passed to solvers that use no aux data.
struct AuxCell {
    const double *p;
    long long ms;
    __device__ __forceinline__ double operator()(int ma) const { return __ldg(p + ma * ms); }
};

// The same cell staged in shared memory (x-engine, solvers with RP::X_AUX_SMEM): component stride
// = padded row length of the staging ring.
struct AuxCellS {
    const double *p;
    int ms;
    __device__ __forceinline__ double operator()(int ma) const { return p[ma * ms]; }
};
// solvers that read so many aux components per interface (the sphere: ~70) that the x-engine stages
// the aux rows in shared memory with cp.async, like q
template <class RP, class = void>
struct rp_x_aux_smem { static constexpr bool value = false; };
template <class RP>
struct rp_x_aux_smem<RP, decltype((void)RP::X_AUX_SMEM)> { static constexpr bool value = RP::X_AUX_SMEM; };

__device__ __forceinline__ double dmax2(double a, double b) { return (a > b) ? a : b; }
__device__ __forceinline__ double dmin2(double a, double b) { return (a < b) ? a : b; }

// ---------------------------------------------------------------------------
// Acoustics.  clawpack/riemann rp1_acoustics.f, rpn2_acoustics.f, rpt2_acoustics.f
// (external repository; SURVEY.md appendix B.1).  cparam{rho,bulk,cc,zz}.
// NDIM = 1: meqn 2 (p,u); NDIM = 2: meqn 3 (p,u,v).
// ---------------------------------------------------------------------------
template <int NDIM, int IXY>
struct RpAcoustics {
    static constexpr int ID = CLAW_RP_ACOUSTICS;
    static constexpr int MEQN = NDIM + 1, MWAVES = 2, NROE = 1;
#ifndef CLAW_AC_X_MINB
#define CLAW_AC_X_MINB 5
#define CLAW_AC_Y_MINB 3
#endif
#ifdef CLAW_AC_F_MINB
    static constexpr int F_MINB = CLAW_AC_F_MINB;
#endif
    static constexpr int X_MINB = CLAW_AC_X_MINB, Y_MINB = CLAW_AC_Y_MINB;
#ifndef CLAW_AC_Y_REGS
#define CLAW_AC_Y_REGS 1
#endif
    static constexpr bool Y_REGS = CLAW_AC_Y_REGS;
    static constexpr int MAUX = 0; // aux components read by the solver
    static constexpr bool QCOR = false; // CTAs/SM the sweeps are compiled for
    static constexpr int MU = (IXY == 2) ? 2 : 1, MV = (IXY == 2) ? 1 : 2;
    __host__ __device__ static constexpr bool nz(int m, int mw) { return m == 0 || m == MU; }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[MEQN],
                                                 const double (&r)[MEQN], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[MEQN][MWAVES],
                                                 double (&s)[MWAVES], double (&amdq)[MEQN],
                                                 double (&apdq)[MEQN], double (&roe)[NROE])
    {
        const double cc = P.p[2], zz = P.p[3];
        const Recip r2z = ar.rcp(2.0 * zz);
        double delta1 = r[0] - l[0];
        double delta2 = r[MU] - l[MU];
        double a1 = ar.div(-delta1 + zz * delta2, r2z);
        double a2 = ar.div(delta1 + zz * delta2, r2z);
        wave[0][0] = -a1 * zz;
        wave[MU][0] = a1;
        s[0] = -cc;
        wave[0][1] = a2 * zz;
        wave[MU][1] = a2;
        s[1] = cc;
        if (NDIM == 2) {
            wave[NDIM == 2 ? MV : 0][0] = 0.0;
            wave[NDIM == 2 ? MV : 0][1] = 0.0;
        }
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            amdq[m] = s[0] * wave[m][0];
            apdq[m] = s[1] * wave[m][1];
        }
        roe[0] = 0.0;
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[MEQN], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[MEQN],
                                                      double (&bm)[MEQN], double (&bp)[MEQN])
    {
        const double cc = P.p[2], zz = P.p[3];
        constexpr int mv = (NDIM == 2) ? MV : 0, mu = (NDIM == 2) ? MU : 0;
        const Recip r2z = ar.rcp(2.0 * zz);
        double a1 = ar.div(-asdq[0] + zz * asdq[mv], r2z);
        double a2 = ar.div(asdq[0] + zz * asdq[mv], r2z);
        bm[0] = cc * a1 * zz;
        bm[mu] = 0.0;
        bm[mv] = -cc * a1;
        bp[0] = cc * a2 * zz;
        bp[mu] = 0.0;
        bp[mv] = cc * a2;
    }
};

// ---------------------------------------------------------------------------
// Scalar advection.  clawpack/riemann rp1_advection.f, rpn2_advection.f,
// rpt2_advection.f (external; SURVEY.md B.2).  cparam{u} / {u,v}.
// ---------------------------------------------------------------------------
template <int NDIM, int IXY>
struct RpAdvection {
    static constexpr int ID = CLAW_RP_ADVECTION;
    static constexpr int MEQN = 1, MWAVES = 1, NROE = 1;
    static constexpr int X_MINB = 6, Y_MINB = 6;
    static constexpr int MAUX = 0;
    static constexpr bool QCOR = false;
    __host__ __device__ static constexpr bool nz(int, int) { return true; }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[1],
                                                 const double (&r)[1], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[1][1],
                                                 double (&s)[1], double (&amdq)[1],
                                                 double (&apdq)[1], double (&roe)[NROE])
    {
        wave[0][0] = r[0] - l[0];
        s[0] = (IXY == 2) ? P.p[1] : P.p[0];
        amdq[0] = dmin2(s[0], 0.0) * wave[0][0];
        apdq[0] = dmax2(s[0], 0.0) * wave[0][0];
        roe[0] = 0.0;
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[1], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[1], double (&bm)[1],
                                                      double (&bp)[1])
    {
        double stran = (IXY == 2) ? P.p[0] : P.p[1];
        double stranm = dmin2(stran, 0.0), stranp = dmax2(stran, 0.0);
        bm[0] = stranm * asdq[0];
        bp[0] = stranp * asdq[0];
    }
};

// ---------------------------------------------------------------------------
// Euler, Roe solver, 4 acoustic/shear/entropy waves + tracer wave, entropy fix.
// development/rp_approaches/rpn2_euler_5wave.f:5-302, rpt2_euler_5wave.f:4-98.
// cparam{gamma,gamma1}.  roe[] = {u2v2,u,v,enth,a,g1a2,euv} (common /comroe/).
// ---------------------------------------------------------------------------
template <int IXY>
struct RpEuler5 {
    static constexpr int ID = CLAW_RP_EULER5;
    static constexpr int MEQN = 5, MWAVES = 5, NROE = 8; // 7 Roe quantities + 1/(2a)
#ifndef CLAW_EU_X_MINB
#define CLAW_EU_X_MINB 3
#define CLAW_EU_Y_MINB 2
#endif
    static constexpr int X_MINB = CLAW_EU_X_MINB, Y_MINB = CLAW_EU_Y_MINB;
    static constexpr int MAUX = 0;
    static constexpr bool QCOR = false;
    static constexpr int MU = (IXY == 2) ? 2 : 1, MV = (IXY == 2) ? 1 : 2;
    // sparsity of wave(m,mw) as written at rpn2_euler_5wave.f:124-163
    __host__ __device__ static constexpr bool nz(int m, int mw)
    {
        return (mw == 4) ? (m == 4) : (mw == 1) ? (m == MV || m == 3) : (m != 4);
    }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[5],
                                                 const double (&r)[5], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[5][5],
                                                 double (&s)[5], double (&amdq)[5],
                                                 double (&apdq)[5], double (&roe)[NROE])
    {
        const double gamma = P.p[0], gamma1 = P.p[1];
        // :87-104
        double rhsqrtl, rhsqrtr;
        Recip rsl, rsr, rl0, rr0; // 1 / sqrt(rho), 1 / rho of the two states
        ar.sqrt_rcps(l[0], rhsqrtl, rsl, rl0);
        ar.sqrt_rcps(r[0], rhsqrtr, rsr, rr0);
        double pl = gamma1 * (l[3] - ar.div(0.5 * (l[1] * l[1] + l[2] * l[2]), rl0));
        double pr = gamma1 * (r[3] - ar.div(0.5 * (r[1] * r[1] + r[2] * r[2]), rr0));
        double rhsq2 = rhsqrtl + rhsqrtr;
        const Recip rs2 = ar.rcp(rhsq2);
        double u = ar.div(ar.div(l[MU], rsl) + ar.div(r[MU], rsr), rs2);
        double v = ar.div(ar.div(l[MV], rsl) + ar.div(r[MV], rsr), rs2);
        double enth = ar.div((ar.div(l[3] + pl, rsl) + ar.div(r[3] + pr, rsr)), rs2);
        double u2v2 = u * u + v * v;
        double a2r = gamma1 * (enth - .5 * u2v2);
        double a;
        Recip r2a, ra2; // 1 / (2 a), 1 / a^2
        ar.sqrt_rcp2s(a2r, a, r2a, ra2);
        double g1a2 = ar.div(gamma1, ra2);
        double euv = enth - u2v2;
        roe[0] = u2v2; roe[1] = u; roe[2] = v; roe[3] = enth; roe[4] = a; roe[5] = g1a2; roe[6] = euv;
        roe[7] = r2a.r;
        // :110-119
        double d1 = r[0] - l[0];
        double d2 = r[MU] - l[MU];
        double d3 = r[MV] - l[MV];
        double d4 = r[3] - l[3];
        double a3 = g1a2 * (euv * d1 + u * d2 + v * d3 - d4);
        double a2 = d3 - v * d1;
        double a4 = ar.div(d2 + (a - u) * d1 - a * a3, r2a);
        double a1 = d1 - a3 - a4;
        // :124-163
        wave[0][0] = a1;
        wave[MU][0] = a1 * (u - a);
        wave[MV][0] = a1 * v;
        wave[3][0] = a1 * (enth - u * a);
        wave[4][0] = 0.0;
        s[0] = u - a;
        wave[0][1] = 0.0;
        wave[MU][1] = 0.0;
        wave[MV][1] = a2;
        wave[3][1] = a2 * v;
        wave[4][1] = 0.0;
        s[1] = u;
        wave[0][2] = a3;
        wave[MU][2] = a3 * u;
        wave[MV][2] = a3 * v;
        wave[3][2] = a3 * 0.5 * u2v2;
        wave[4][2] = 0.0;
        s[2] = u;
        wave[0][3] = a4;
        wave[MU][3] = a4 * (u + a);
        wave[MV][3] = a4 * v;
        wave[3][3] = a4 * (enth + u * a);
        wave[4][3] = 0.0;
        s[3] = u + a;
        wave[0][4] = 0.0;
        wave[MU][4] = 0.0;
        wave[MV][4] = 0.0;
        wave[3][4] = 0.0;
        wave[4][4] = r[4] - l[4];
        s[4] = u;
        // :205-286 entropy fix.  pim1 / pi below are bitwise equal to pl / pr above (the
        // sums of squares differ only in the order of a commutative addition), so they and
        // the divisions by rho(i-1), rho(i) are not repeated.
        bool done = false;
        {
            double pim1 = pl;
            double cim1 = ar.sqrt(ar.div(gamma * pim1, rl0));
            double s0 = ar.div(l[MU], rl0) - cim1;
            if (s0 >= 0.0 && s[0] > 0.0) {
#pragma unroll
                for (int m = 0; m < 5; m++) amdq[m] = 0.0;
                done = true;
            }
            if (!done) {
                double rho1 = l[0] + wave[0][0];
                double rhou1 = l[MU] + wave[MU][0];
                double rhov1 = l[MV] + wave[MV][0];
                double en1 = l[3] + wave[3][0];
                const Recip rr1 = ar.rcp(rho1);
                double p1 = gamma1 * (en1 - ar.div(0.5 * (rhou1 * rhou1 + rhov1 * rhov1), rr1));
                double c1 = ar.sqrt(ar.div(gamma * p1, rr1));
                double s1 = ar.div(rhou1, rr1) - c1;
                double sfract;
                if (s0 < 0.0 && s1 > 0.0)
                    sfract = ar.div(s0 * (s1 - s[0]), s1 - s0);
                else if (s[0] < 0.0)
                    sfract = s[0];
                else
                    sfract = 0.0;
#pragma unroll
                for (int m = 0; m < 5; m++) amdq[m] = sfract * wave[m][0];
                if (s[1] >= 0.0) done = true;
            }
        }
        if (!done) {
#pragma unroll
            for (int m = 0; m < 5; m++) {
                amdq[m] = amdq[m] + s[1] * wave[m][1];
                amdq[m] = amdq[m] + s[2] * wave[m][2];
                amdq[m] = amdq[m] + s[4] * wave[m][4];
            }
            double pi = pr;
            double ci = ar.sqrt(ar.div(gamma * pi, rr0));
            double s3 = ar.div(r[MU], rr0) + ci;
            double rho2 = r[0] - wave[0][3];
            double rhou2 = r[MU] - wave[MU][3];
            double rhov2 = r[MV] - wave[MV][3];
            double en2 = r[3] - wave[3][3];
            const Recip rr2 = ar.rcp(rho2);
            double p2 = gamma1 * (en2 - ar.div(0.5 * (rhou2 * rhou2 + rhov2 * rhov2), rr2));
            double c2 = ar.sqrt(ar.div(gamma * p2, rr2));
            double s2 = ar.div(rhou2, rr2) + c2;
            double sfract = 0.0;
            bool add4 = true;
            if (s2 < 0.0 && s3 > 0.0)
                sfract = ar.div(s2 * (s3 - s[3]), s3 - s2);
            else if (s[3] < 0.0)
                sfract = s[3];
            else
                add4 = false;
            if (add4) {
#pragma unroll
                for (int m = 0; m < 5; m++) amdq[m] = amdq[m] + sfract * wave[m][3];
            }
        }
        // :291-298
#pragma unroll
        for (int m = 0; m < 5; m++) {
            double df = 0.0;
#pragma unroll
            for (int mw = 0; mw < 5; mw++)
                if (nz(m, mw)) df = df + s[mw] * wave[m][mw]; // zero entries add +-0 to a sum that starts at +0
            apdq[m] = df - amdq[m];
        }
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[5], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[5], double (&bm)[5],
                                                      double (&bp)[5])
    {
        const double u2v2 = roe[0], u = roe[1], v = roe[2], enth = roe[3], a = roe[4],
                     g1a2 = roe[5], euv = roe[6];
        const Recip r2a{2.0 * a, roe[7]}; // refined in solve() (already validated there)
        double a3 = g1a2 * (euv * asdq[0] + u * asdq[MU] + v * asdq[MV] - asdq[3]);
        double a2 = asdq[MU] - u * asdq[0];
        double a4 = ar.div(asdq[MV] + (a - v) * asdq[0] - a * a3, r2a);
        double a1 = asdq[0] - a3 - a4;
        double waveb[5][4], sb[4];
        waveb[0][0] = a1;
        waveb[MU][0] = a1 * u;
        waveb[MV][0] = a1 * (v - a);
        waveb[3][0] = a1 * (enth - v * a);
        waveb[4][0] = 0.0;
        sb[0] = v - a;
        waveb[0][1] = a3;
        waveb[MU][1] = a3 * u + a2;
        waveb[MV][1] = a3 * v;
        waveb[3][1] = a3 * 0.5 * u2v2 + a2 * u;
        waveb[4][1] = 0.0;
        sb[1] = v;
        waveb[0][2] = a4;
        waveb[MU][2] = a4 * u;
        waveb[MV][2] = a4 * (v + a);
        waveb[3][2] = a4 * (enth + v * a);
        waveb[4][2] = 0.0;
        sb[2] = v + a;
        waveb[0][3] = 0.0;
        waveb[MU][3] = 0.0;
        waveb[MV][3] = 0.0;
        waveb[3][3] = 0.0;
        waveb[4][3] = asdq[4];
        sb[3] = v;
        // waveb(5,1:3) and waveb(1:4,4) are literal zeros (rpt2_euler_5wave.f:57-80): adding
        // their +-0 products to sums that start at +0 changes nothing, so they are skipped
#pragma unroll
        for (int m = 0; m < 5; m++) {
            bm[m] = 0.0;
            bp[m] = 0.0;
#pragma unroll
            for (int mw = 0; mw < 4; mw++) {
                if ((mw == 3) == (m == 4)) {
                    bm[m] = bm[m] + dmin2(sb[mw], 0.0) * waveb[m][mw];
                    bp[m] = bp[m] + dmax2(sb[mw], 0.0) * waveb[m][mw];
                }
            }
        }
    }
};

// ---------------------------------------------------------------------------
// Shallow water, Roe solver with entropy fix.
// clawpack/riemann rpn2_shallow_roe_with_efix.f, rpt2_shallow_roe_with_efix.f
// (external; SURVEY.md B.3).  cparam{grav}.  roe[] = {u,v,a}.
// ---------------------------------------------------------------------------
template <int IXY>
struct RpShallow {
    static constexpr int ID = CLAW_RP_SHALLOW;
    static constexpr int MEQN = 3, MWAVES = 3, NROE = 4; // u, v, a, 0.5/a
#ifndef CLAW_SW_X_MINB
#define CLAW_SW_X_MINB 4
#define CLAW_SW_Y_MINB 3
#endif
    static constexpr int X_MINB = CLAW_SW_X_MINB, Y_MINB = CLAW_SW_Y_MINB;
    static constexpr int F_MINB = 2; // single-pass kernel: 3 CTAs/SM (168 registers) spills
    static constexpr int MAUX = 0;
    static constexpr bool QCOR = false;
    static constexpr int MU = (IXY == 2) ? 2 : 1, MV = (IXY == 2) ? 1 : 2;
    __host__ __device__ static constexpr bool nz(int m, int mw)
    {
        return (mw == 1) ? (m == MV) : true;
    }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[3],
                                                 const double (&r)[3], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[3][3],
                                                 double (&s)[3], double (&amdq)[3],
                                                 double (&apdq)[3], double (&roe)[NROE])
    {
        const double grav = P.p[0];
        double h = (l[0] + r[0]) * 0.50;
        double hsqrtl, hsqrtr;
        Recip rsl, rsr;
        ar.sqrt_rcp(l[0], hsqrtl, rsl);
        ar.sqrt_rcp(r[0], hsqrtr, rsr);
        double hsq2 = hsqrtl + hsqrtr;
        const Recip rs2 = ar.rcp(hsq2);
        double u = ar.div(ar.div(l[MU], rsl) + ar.div(r[MU], rsr), rs2);
        double v = ar.div(ar.div(l[MV], rsl) + ar.div(r[MV], rsr), rs2);
        double a;
        Recip ra;
        ar.sqrt_rcp(grav * h, a, ra);
        double hoa = ar.div(0.50, ra);
        roe[0] = u; roe[1] = v; roe[2] = a; roe[3] = hoa;
        double d1 = r[0] - l[0];
        double d2 = r[MU] - l[MU];
        double d3 = r[MV] - l[MV];
        double a1 = ((u + a) * d1 - d2) * hoa;
        double a2 = -v * d1 + d3;
        double a3 = (-(u - a) * d1 + d2) * hoa;
        wave[0][0] = a1;
        wave[MU][0] = a1 * (u - a);
        wave[MV][0] = a1 * v;
        s[0] = u - a;
        wave[0][1] = 0.0;
        wave[MU][1] = 0.0;
        wave[MV][1] = a2;
        s[1] = u;
        wave[0][2] = a3;
        wave[MU][2] = a3 * (u + a);
        wave[MV][2] = a3 * v;
        s[2] = u + a;
        bool done = false;
        double him1 = l[0];
        double s0 = ar.div(l[MU], him1) - ar.sqrt(grav * him1);
        if (s0 > 0.0 && s[0] > 0.0) {
#pragma unroll
            for (int m = 0; m < 3; m++) amdq[m] = 0.0;
            done = true;
        }
        if (!done) {
            double h1 = l[0] + wave[0][0];
            double hu1 = l[MU] + wave[MU][0];
            double s1 = ar.div(hu1, h1) - ar.sqrt(grav * h1);
            double sfract;
            if (s0 < 0.0 && s1 > 0.0)
                sfract = s0 * ar.div(s1 - s[0], s1 - s0);
            else if (s[0] < 0.0)
                sfract = s[0];
            else
                sfract = 0.0;
#pragma unroll
            for (int m = 0; m < 3; m++) amdq[m] = sfract * wave[m][0];
            if (s[1] > 0.0) done = true;
        }
        if (!done) {
#pragma unroll
            for (int m = 0; m < 3; m++) amdq[m] = amdq[m] + s[1] * wave[m][1];
            double hi = r[0];
            double s03 = ar.div(r[MU], hi) + ar.sqrt(grav * hi);
            double h3 = r[0] - wave[0][2];
            double hu3 = r[MU] - wave[MU][2];
            double s3 = ar.div(hu3, h3) + ar.sqrt(grav * h3);
            double sfract = 0.0;
            bool add3 = true;
            if (s3 < 0.0 && s03 > 0.0)
                sfract = s3 * ar.div(s03 - s[2], s03 - s3);
            else if (s[2] < 0.0)
                sfract = s[2];
            else
                add3 = false;
            if (add3) {
#pragma unroll
                for (int m = 0; m < 3; m++) amdq[m] = amdq[m] + sfract * wave[m][2];
            }
        }
#pragma unroll
        for (int m = 0; m < 3; m++) {
            double df = 0.0;
#pragma unroll
            for (int mw = 0; mw < 3; mw++)
                if (nz(m, mw)) df = df + s[mw] * wave[m][mw];
            apdq[m] = df - amdq[m];
        }
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[3], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[3], double (&bm)[3],
                                                      double (&bp)[3])
    {
        const double u = roe[0], v = roe[1], a = roe[2], hoa = roe[3]; // hoa = 0.5/a from solve()
        double a1 = hoa * ((v + a) * asdq[0] - asdq[MV]);
        double a2 = asdq[MU] - u * asdq[0];
        double a3 = hoa * (-(v - a) * asdq[0] + asdq[MV]);
        double waveb[3][3], sb[3];
        waveb[0][0] = a1;
        waveb[MU][0] = a1 * u;
        waveb[MV][0] = a1 * (v - a);
        sb[0] = v - a;
        waveb[0][1] = 0.0;
        waveb[MU][1] = a2;
        waveb[MV][1] = 0.0;
        sb[1] = v;
        waveb[0][2] = a3;
        waveb[MU][2] = a3 * u;
        waveb[MV][2] = a3 * (v + a);
        sb[2] = v + a;
        // waveb(1,2) and waveb(mv,2) are literal zeros: skipped (sums start at +0)
#pragma unroll
        for (int m = 0; m < 3; m++) {
            bm[m] = 0.0;
            bp[m] = 0.0;
#pragma unroll
            for (int mw = 0; mw < 3; mw++) {
                if (mw != 1 || m == MU) {
                    bm[m] = bm[m] + dmin2(sb[mw], 0.0) * waveb[m][mw];
                    bp[m] = bp[m] + dmax2(sb[mw], 0.0) * waveb[m][mw];
                }
            }
        }
    }
};


// ---------------------------------------------------------------------------
// Shallow water on the sphere (3-D Cartesian momentum, 16 aux components).
// clawpack/riemann rpn2_shallow_sphere.f, rpt2_shallow_sphere.f (external; SURVEY.md B.4)
// with apps/shallow-sphere/qcor.f:2-72 for the step2qcor correction.
// params: p[0] = g (common /sw/), p[1] = dxcom, p[2] = dycom (common /comxyt/).
// aux (0-based): 0 kappa | 1-3 normal, 4-6 tangent of the LEFT edge | 7-9 normal,
// 10-12 tangent of the BOTTOM edge | 13-15 radial unit vector at the cell centre
// (apps/shallow-sphere/setaux.f:9-25).  The oracle restatement of this solver reproduces
// test/swsphere_height to 2e-17.
// ---------------------------------------------------------------------------
template <int IXY>
struct RpSphere {
    static constexpr int ID = CLAW_RP_SPHERE;
    static constexpr int MEQN = 4, MWAVES = 3, NROE = 1;
    static constexpr int X_MINB = 2, Y_MINB = 2;
    static constexpr int MAUX = 16;
    static constexpr bool QCOR = true;
    static constexpr bool X_AUX_SMEM = true;
    static constexpr int IOFF = (IXY == 2) ? 7 : 1;   // edge data of the sweep direction
    static constexpr int IOFFT = (IXY == 2) ? 1 : 7;  // edge data of the transverse direction
    __host__ __device__ static constexpr bool nz(int m, int mw) { return !(m == 0 && mw == 1); }

    // axl = cell i-1 (its radial vector projects amdq), axr = cell i (owns the edge)
    template <class AR, class AX>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[4],
                                                 const double (&r)[4], const AX &axl, const AX &axr,
                                                 double (&wave)[4][3], double (&s)[3], double (&amdq)[4],
                                                 double (&apdq)[4], double (&roe)[NROE])
    {
        const double g = P.p[0];
        const double dy = (IXY == 2) ? P.p[1] : P.p[2];
        const double enx = axr(IOFF + 0), eny = axr(IOFF + 1), enz = axr(IOFF + 2);
        double etx = axr(IOFF + 3), ety = axr(IOFF + 4), etz = axr(IOFF + 5);
        double gamma;
        Recip rg;
        ar.sqrt_rcp(etx * etx + ety * ety + etz * etz, gamma, rg);
        etx = ar.div(etx, rg); ety = ar.div(ety, rg); etz = ar.div(etz, rg);
        // "ql" of the Fortran is the right cell, "qr" the left cell
        double hunl = enx * r[1] + eny * r[2] + enz * r[3];
        double hunr = enx * l[1] + eny * l[2] + enz * l[3];
        double hutl = etx * r[1] + ety * r[2] + etz * r[3];
        double hutr = etx * l[1] + ety * l[2] + etz * l[3];
        double hl = r[0], hr = l[0];
        double h = (hl + hr) * 0.50;
        double hsqr, hsql;
        Recip rsr, rsl;
        ar.sqrt_rcp(hr, hsqr, rsr);
        ar.sqrt_rcp(hl, hsql, rsl);
        double hsq = hsqr + hsql;
        const Recip rsq = ar.rcp(hsq);
        double u = ar.div(ar.div(hunr, rsr) + ar.div(hunl, rsl), rsq);
        double v = ar.div(ar.div(hutr, rsr) + ar.div(hutl, rsl), rsq);
        double a;
        Recip ra;
        ar.sqrt_rcp(g * h, a, ra);
        double hoa = ar.div(0.50, ra);
        double d1 = hl - hr, d2 = hunl - hunr, d3 = hutl - hutr;
        double a1 = ((u + a) * d1 - d2) * hoa;
        double a2 = -v * d1 + d3;
        double a3 = (-(u - a) * d1 + d2) * hoa;
        const Recip rdy = ar.rcp(dy);
        wave[0][0] = a1;
        wave[1][0] = a1 * (u - a) * enx + a1 * v * etx;
        wave[2][0] = a1 * (u - a) * eny + a1 * v * ety;
        wave[3][0] = a1 * (u - a) * enz + a1 * v * etz;
        s[0] = ar.div((u - a) * gamma, rdy);
        wave[0][1] = 0.0;
        wave[1][1] = a2 * etx;
        wave[2][1] = a2 * ety;
        wave[3][1] = a2 * etz;
        s[1] = ar.div(u * gamma, rdy);
        wave[0][2] = a3;
        wave[1][2] = a3 * (u + a) * enx + a3 * v * etx;
        wave[2][2] = a3 * (u + a) * eny + a3 * v * ety;
        wave[3][2] = a3 * (u + a) * enz + a3 * v * etz;
        s[2] = ar.div((u + a) * gamma, rdy);
        // entropy fix
        bool done = false;
        double him1 = l[0];
        double s0 = ar.div((ar.div(hunr, him1) - ar.sqrt(g * him1)) * gamma, rdy);
        if (s0 > 0.0 && s[0] > 0.0) {
#pragma unroll
            for (int m = 0; m < 4; m++) amdq[m] = 0.0;
            done = true;
        }
        if (!done) {
            double h1 = l[0] + wave[0][0];
            double hu1 = hunr + (enx * wave[1][0] + eny * wave[2][0] + enz * wave[3][0]);
            double s1 = ar.div((ar.div(hu1, h1) - ar.sqrt(g * h1)) * gamma, rdy);
            double sfract;
            if (s0 < 0.0 && s1 > 0.0)
                sfract = s0 * ar.div(s1 - s[0], s1 - s0);
            else if (s[0] < 0.0)
                sfract = s[0];
            else
                sfract = 0.0;
#pragma unroll
            for (int m = 0; m < 4; m++) amdq[m] = sfract * wave[m][0];
            if (s[1] > 0.0) done = true;
        }
        if (!done) {
#pragma unroll
            for (int m = 0; m < 4; m++) amdq[m] = amdq[m] + s[1] * wave[m][1];
            double hi = r[0];
            double s03 = ar.div((ar.div(hunl, hi) + ar.sqrt(g * hi)) * gamma, rdy);
            double h3 = r[0] - wave[0][2];
            double hu3 = hunl - (enx * wave[1][2] + eny * wave[2][2] + enz * wave[3][2]);
            double s3 = ar.div((ar.div(hu3, h3) + ar.sqrt(g * h3)) * gamma, rdy);
            double sfract = 0.0;
            bool add3 = true;
            if (s3 < 0.0 && s03 > 0.0)
                sfract = s3 * ar.div(s03 - s[2], s03 - s3);
            else if (s[2] < 0.0)
                sfract = s[2];
            else
                add3 = false;
            if (add3) {
#pragma unroll
                for (int m = 0; m < 4; m++) amdq[m] = amdq[m] + sfract * wave[m][2];
            }
        }
#pragma unroll
        for (int m = 0; m < 4; m++) {
            double df = 0.0;
#pragma unroll
            for (int mw = 0; mw < 3; mw++) df = df + s[mw] * wave[m][mw];
            apdq[m] = df - amdq[m];
        }
        // project the momentum components onto the tangent plane
        {
            double erx = axl(13), ery = axl(14), erz = axl(15);
            double amn = erx * amdq[1] + ery * amdq[2] + erz * amdq[3];
            amdq[1] = amdq[1] - amn * erx;
            amdq[2] = amdq[2] - amn * ery;
            amdq[3] = amdq[3] - amn * erz;
            erx = axr(13); ery = axr(14); erz = axr(15);
            double apn = erx * apdq[1] + ery * apdq[2] + erz * apdq[3];
            apdq[1] = apdq[1] - apn * erx;
            apdq[2] = apdq[2] - apn * ery;
            apdq[3] = apdq[3] - apn * erz;
        }
        roe[0] = 0.0;
    }

    // one side of rpt2: edge data from `axe`, radial vector from `axp`, state of the cell
    template <class AR, bool UP, class AX>
    __device__ __forceinline__ static void side(AR &ar, double g, double dx, const double (&qc)[4],
                                                const AX &axe, const AX &axp,
                                                const double (&asdq)[4], double (&b)[4])
    {
        const double enx = axe(IOFFT + 0), eny = axe(IOFFT + 1), enz = axe(IOFFT + 2);
        double etx = axe(IOFFT + 3), ety = axe(IOFFT + 4), etz = axe(IOFFT + 5);
        double gamma;
        Recip rg;
        ar.sqrt_rcp(etx * etx + ety * ety + etz * etz, gamma, rg);
        etx = ar.div(etx, rg); ety = ar.div(ety, rg); etz = ar.div(etz, rg);
        const double h = qc[0];
        const Recip rh = ar.rcp(h);
        double u = ar.div(enx * qc[1] + eny * qc[2] + enz * qc[3], rh);
        double v = ar.div(etx * qc[1] + ety * qc[2] + etz * qc[3], rh);
        double a;
        Recip ra;
        ar.sqrt_rcp(g * h, a, ra);
        double hoa = ar.div(0.50, ra);
        double d2 = enx * asdq[1] + eny * asdq[2] + enz * asdq[3];
        double d3 = etx * asdq[1] + ety * asdq[2] + etz * asdq[3];
        double d1 = asdq[0];
        double a1 = ((u + a) * d1 - d2) * hoa;
        double a2 = -v * d1 + d3;
        double a3 = (-(u - a) * d1 + d2) * hoa;
        double waveb[4][3], sb[3];
        const Recip rdx = ar.rcp(dx);
        waveb[0][0] = a1;
        waveb[1][0] = a1 * (u - a) * enx + a1 * v * etx;
        waveb[2][0] = a1 * (u - a) * eny + a1 * v * ety;
        waveb[3][0] = a1 * (u - a) * enz + a1 * v * etz;
        sb[0] = ar.div((u - a) * gamma, rdx);
        waveb[0][1] = 0.0;
        waveb[1][1] = a2 * etx;
        waveb[2][1] = a2 * ety;
        waveb[3][1] = a2 * etz;
        sb[1] = ar.div(u * gamma, rdx);
        waveb[0][2] = a3;
        waveb[1][2] = a3 * (u + a) * enx + a3 * v * etx;
        waveb[2][2] = a3 * (u + a) * eny + a3 * v * ety;
        waveb[3][2] = a3 * (u + a) * enz + a3 * v * etz;
        sb[2] = ar.div((u + a) * gamma, rdx);
#pragma unroll
        for (int m = 0; m < 4; m++) {
            b[m] = 0.0;
#pragma unroll
            for (int mw = 0; mw < 3; mw++)
                b[m] = b[m] + (UP ? dmax2(sb[mw], 0.0) : dmin2(sb[mw], 0.0)) * waveb[m][mw];
        }
        double erx = axp(13), ery = axp(14), erz = axp(15);
        double bn = erx * b[1] + ery * b[2] + erz * b[3];
        b[1] = b[1] - bn * erx;
        b[2] = b[2] - bn * ery;
        b[3] = b[3] - bn * erz;
    }

    // qc = state of the cell the fluctuation moves into; ax1/ax2/ax3 = that cell in the
    // previous / current / next slice
    template <class AR, class AX>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[4], const AX &ax1,
                                                      const AX &ax2, const AX &ax3,
                                                      const double (&asdq)[4], double (&bm)[4], double (&bp)[4])
    {
        const double g = P.p[0];
        const double dx = (IXY == 2) ? P.p[2] : P.p[1];
        side<AR, true, AX>(ar, g, dx, qc, ax3, ax3, asdq, bp);
        side<AR, false, AX>(ar, g, dx, qc, ax2, ax1, asdq, bm);
    }

    // apps/shallow-sphere/qcor.f:2-72: axi = this cell, axn = the next cell along the sweep
    template <class AR, class AX>
    __device__ __forceinline__ static void qcor(AR &ar, const RpParams &P, const double (&q)[4],
                                                const AX &axi, const AX &axn, double (&qcv)[4])
    {
        const double g = P.p[0];
        const double dy = (IXY == 2) ? P.p[1] : P.p[2];
        const Recip rdy = ar.rcp(dy);
        double etxl = axi(IOFF + 3), etyl = axi(IOFF + 4), etzl = axi(IOFF + 5);
        double gammal = ar.div(ar.sqrt(etxl * etxl + etyl * etyl + etzl * etzl), rdy);
        double enxl = axi(IOFF + 0) * gammal, enyl = axi(IOFF + 1) * gammal, enzl = axi(IOFF + 2) * gammal;
        double etxr = axn(IOFF + 3), etyr = axn(IOFF + 4), etzr = axn(IOFF + 5);
        double gammar = ar.div(ar.sqrt(etxr * etxr + etyr * etyr + etzr * etzr), rdy);
        double enxr = axn(IOFF + 0) * gammar, enyr = axn(IOFF + 1) * gammar, enzr = axn(IOFF + 2) * gammar;
        const double q1 = q[0], q2 = q[1], q3 = q[2], q4 = q[3];
        const Recip r1 = ar.rcp(q1);
        const double hg = 0.5 * g * (q1 * q1);
        qcv[0] = (enxr - enxl) * q2 + (enyr - enyl) * q3 + (enzr - enzl) * q4;
        qcv[1] = (enxr - enxl) * (ar.div(q2 * q2, r1) + hg) + (enyr - enyl) * ar.div(q2 * q3, r1) +
                 (enzr - enzl) * ar.div(q2 * q4, r1);
        qcv[2] = (enxr - enxl) * ar.div(q2 * q3, r1) + (enyr - enyl) * (ar.div(q3 * q3, r1) + hg) +
                 (enzr - enzl) * ar.div(q3 * q4, r1);
        qcv[3] = (enxr - enxl) * ar.div(q2 * q4, r1) + (enyr - enyl) * ar.div(q3 * q4, r1) +
                 (enzr - enzl) * (ar.div(q4 * q4, r1) + hg);
        double erx = axi(13), ery = axi(14), erz = axi(15);
        double qcn = erx * qcv[1] + ery * qcv[2] + erz * qcv[3];
        qcv[1] = qcv[1] - qcn * erx;
        qcv[2] = qcv[2] - qcn * ery;
        qcv[3] = qcv[3] - qcn * erz;
    }
};


// ---------------------------------------------------------------------------
// 1-D shallow water, Roe solver with entropy fix.  clawpack/riemann
// rp1_shallow_roe_with_efix.f (external; app apps/shallow/1d).  cparam{grav}.
// ---------------------------------------------------------------------------
struct RpShallow1D {
    static constexpr int ID = CLAW_RP_SHALLOW;
    static constexpr int MEQN = 2, MWAVES = 2, NROE = 1;
    static constexpr int X_MINB = 4, Y_MINB = 4;
    static constexpr int MAUX = 0;
    static constexpr bool QCOR = false;
    __host__ __device__ static constexpr bool nz(int, int) { return true; }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[2],
                                                 const double (&r)[2], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[2][2], double (&s)[2], double (&amdq)[2],
                                                 double (&apdq)[2], double (&roe)[NROE])
    {
        const double grav = P.p[0];
        const double hl = l[0], hr = r[0], hul = l[1], hur = r[1];
        double hsqrtl = ar.sqrt(hl);
        double hsqrtr = ar.sqrt(hr);
        double hsq2 = hsqrtl + hsqrtr;
        double ubar = ar.div(ar.div(hul, hsqrtl) + ar.div(hur, hsqrtr), hsq2);
        double cbar = ar.sqrt(0.5 * grav * (hl + hr));
        const Recip rc = ar.rcp(cbar);
        double d1 = hr - hl;
        double d2 = hur - hul;
        double a1 = ar.div(0.5 * (-d2 + (ubar + cbar) * d1), rc);
        double a2 = ar.div(0.5 * (d2 - (ubar - cbar) * d1), rc);
        wave[0][0] = a1;
        wave[1][0] = a1 * (ubar - cbar);
        s[0] = ubar - cbar;
        wave[0][1] = a2;
        wave[1][1] = a2 * (ubar + cbar);
        s[1] = ubar + cbar;
        bool done = false;
        double s0 = ar.div(hul, hl) - ar.sqrt(grav * hl);
        if (s0 > 0.0 && s[0] > 0.0) {
            amdq[0] = 0.0; amdq[1] = 0.0;
            done = true;
        }
        if (!done) {
            double h1 = hl + wave[0][0];
            double hu1 = hul + wave[1][0];
            double s1 = ar.div(hu1, h1) - ar.sqrt(grav * h1);
            double sfract;
            if (s0 < 0.0 && s1 > 0.0)
                sfract = s0 * ar.div(s1 - s[0], s1 - s0);
            else if (s[0] < 0.0)
                sfract = s[0];
            else
                sfract = 0.0;
            amdq[0] = sfract * wave[0][0];
            amdq[1] = sfract * wave[1][0];
            double s03 = ar.div(hur, hr) + ar.sqrt(grav * hr);
            double h3 = hr - wave[0][1];
            double hu3 = hur - wave[1][1];
            double s3 = ar.div(hu3, h3) + ar.sqrt(grav * h3);
            bool add = true;
            if (s3 < 0.0 && s03 > 0.0)
                sfract = s3 * ar.div(s03 - s[1], s03 - s3);
            else if (s[1] < 0.0)
                sfract = s[1];
            else
                add = false;
            if (add) {
                amdq[0] = amdq[0] + sfract * wave[0][1];
                amdq[1] = amdq[1] + sfract * wave[1][1];
            }
        }
#pragma unroll
        for (int m = 0; m < 2; m++) {
            double df = 0.0;
#pragma unroll
            for (int mw = 0; mw < 2; mw++) df = df + s[mw] * wave[m][mw];
            apdq[m] = df - amdq[m];
        }
        roe[0] = 0.0;
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &, const double (&)[NROE],
                                                      const double (&)[2], const AuxCell &, const AuxCell &,
                                                      const AuxCell &, const double (&)[2], double (&bm)[2],
                                                      double (&bp)[2])
    {
        bm[0] = bm[1] = bp[0] = bp[1] = 0.0;
    }
};

// ---------------------------------------------------------------------------
// Elasticity in a heterogeneous medium, f-wave solvers.
//   1-D (NDIM = 1): eps_t - u_x = 0, (rho u)_t - sigma(eps, x)_x = 0
//        clawpack/riemann rp1_nonlinear_elasticity_fwave.f (external); app
//        apps/elasticity/1d/stegoton/stegoton.py: aux = {rho, K}, stress law from rp_params[0]
//   2-D (NDIM = 2): the p-system, clawpack/riemann rpn2_psystem.f / rpt2_psystem.f (external);
//        app test/psystem/psystem.py: aux = {rho, E, stress law, copy of eps}
// Stress law 1: sigma = E eps ; law 2: sigma = exp(E eps) - 1.
// The flux jump (-du, -dsigma) is split into b1 (1, z_{i-1}) at speed -c_{i-1} and
// b2 (1, -z_i) at speed +c_i with c = sqrt(sigma'/rho), z = rho c.
// exp() is the CUDA library's (<= 1 ulp): for law 2 parity with the CPU oracle is to
// rounding error, for law 1 it is bit for bit.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double el_sigma(double eps, double E, double law)
{
    return (law == 1.0) ? E * eps : exp(E * eps) - 1.0;
}
__device__ __forceinline__ double el_sigmap(double eps, double E, double law)
{
    return (law == 1.0) ? E : E * exp(E * eps);
}

template <int NDIM, int IXY>
struct RpElasticFwave {
    static constexpr int ID = (NDIM == 1) ? CLAW_RP_NEL_FWAVE : CLAW_RP_PSYSTEM;
    static constexpr int MEQN = NDIM + 1, MWAVES = 2, NROE = 1;
    static constexpr int X_MINB = 4, Y_MINB = 3;
    static constexpr int MAUX = (NDIM == 1) ? 2 : 4;
    static constexpr bool QCOR = false;
    static constexpr bool FWAVE = true;
    static constexpr int MU = (IXY == 2) ? 2 : 1, MV = (IXY == 2) ? 1 : 2;
    __host__ __device__ static constexpr bool nz(int m, int mw) { return m == 0 || m == MU; }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[MEQN],
                                                 const double (&r)[MEQN], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[MEQN][MWAVES],
                                                 double (&s)[MWAVES], double (&amdq)[MEQN],
                                                 double (&apdq)[MEQN], double (&roe)[NROE])
    {
        const double rhoi = axr(0), rhoim = axl(0);
        const double Ei = axr(1), Eim = axl(1);
        const double lawi = (NDIM == 2) ? axr(2) : P.p[0];
        const double lawim = (NDIM == 2) ? axl(2) : P.p[0];
        const double epsi = r[0], epsim = l[0];
        const double urhoi = r[MU], urhoim = l[MU];
        const Recip rri = ar.rcp(rhoi), rrim = ar.rcp(rhoim);
        double bulki = el_sigmap(epsi, Ei, lawi);
        double bulkim = el_sigmap(epsim, Eim, lawim);
        double ci = ar.sqrt(ar.div(bulki, rri));
        double cim = ar.sqrt(ar.div(bulkim, rrim));
        double zi = ci * rhoi;
        double zim = cim * rhoim;
        double du = ar.div(urhoi, rri) - ar.div(urhoim, rrim);
        double dsig = el_sigma(epsi, Ei, lawi) - el_sigma(epsim, Eim, lawim);
        const Recip rz = ar.rcp(zim + zi);
        double b1 = ar.div(-(zi * du + dsig), rz);
        double b2 = ar.div(-(zim * du - dsig), rz);
        wave[0][0] = b1;
        wave[MU][0] = b1 * zim;
        s[0] = -cim;
        wave[0][1] = b2;
        wave[MU][1] = b2 * (-zi);
        s[1] = ci;
        if (NDIM == 2) {
            wave[NDIM == 2 ? MV : 0][0] = 0.0;
            wave[NDIM == 2 ? MV : 0][1] = 0.0;
        }
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            amdq[m] = wave[m][0];
            apdq[m] = wave[m][1];
        }
        roe[0] = 0.0;
    }

    // rpt2: asdq split with the transverse eigenvectors (1, z) at -c and (1, -z) at +c, using
    // the impedance of the cell it leaves (ax2) and of the one it enters (ax1 below, ax3 above)
    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[MEQN], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[MEQN],
                                                      double (&bm)[MEQN], double (&bp)[MEQN])
    {
        constexpr int mv = (NDIM == 2) ? MV : 0, mu = (NDIM == 2) ? MU : 0;
        const double rm = ax1(0), rc = ax2(0), rp = ax3(0);
        double cm = ar.sqrt(ar.div(el_sigmap(ax1(3), ax1(1), ax1(2)), rm));
        double cc = ar.sqrt(ar.div(el_sigmap(ax2(3), ax2(1), ax2(2)), rc));
        double cp = ar.sqrt(ar.div(el_sigmap(ax3(3), ax3(1), ax3(2)), rp));
        double zm = cm * rm, zz = cc * rc, zp = cp * rp;
        double a1 = ar.div(zz * asdq[0] + asdq[mv], zm + zz);
        double a2 = ar.div(zz * asdq[0] - asdq[mv], zz + zp);
        bm[0] = -cm * a1;
        bm[mu] = 0.0;
        bm[mv] = -cm * a1 * zm;
        bp[0] = cp * a2;
        bp[mu] = 0.0;
        bp[mv] = cp * a2 * (-zp);
    }
};

// ---------------------------------------------------------------------------
// Shallow water over bathymetry, f-wave solver (Bale, LeVeque, Mitran & Rossmanith 2002, SIAM J.
// Sci. Comput. 24; LeVeque 2002 sec. 15.5): the source -g h b_x is folded into the flux jump of each
// interface, so at a lake at rest (u = v = 0, h + b constant) every f-wave is round-off and the step
// keeps the lake at rest (well balanced).  Restated, parity unpinned.
// q = (h, hu) (NDIM = 1) or (h, hu, hv); aux = {b}, the bottom elevation; params {grav, dry_tolerance}.
//   velocity u = hu / h where h > dry_tolerance, else 0; phi = hu u + g h^2 / 2
//   u^ = (sqrt(h_l) u_l + sqrt(h_r) u_r) / (sqrt(h_l) + sqrt(h_r)) (v^ alike), c^ = sqrt(g (h_l + h_r) / 2),
//   with h clamped at 0 under every square root
//   s1 = min(u_l - sqrt(g h_l), u^ - c^), s3 = max(u_r + sqrt(g h_r), u^ + c^) (Einfeldt); 2-D: s2 = u^
//   d1 = hu_r - hu_l, d2 = phi_r - phi_l + g (h_l + h_r) (b_r - b_l) / 2, 2-D: d3 = hu_r v_r - hu_l v_l
//   b1 = (s3 d1 - d2) / (s3 - s1), b3 = (d2 - s1 d1) / (s3 - s1)
//   Z1 = b1 (1, s1, v_l), Z2 = (0, 0, d3 - b1 v_l - b3 v_r) (2-D only), Z3 = b3 (1, s3, v_r)
//   amdq / apdq = sum of the f-waves with s < 0 / s > 0, half of each wave with s = 0 to either side.
// An interface dry on both sides has no waves.  roe[] = {u^, v^, c^, 0.5 / c^}: the transverse solve is
// RpShallow's at these averages (it reads no aux; the bathymetry enters through the normal f-waves).
// ---------------------------------------------------------------------------
template <int NDIM, int IXY>
struct RpShallowBathyFwave {
    static constexpr int ID = CLAW_RP_SHALLOW_BATHY_FWAVE;
    static constexpr int MEQN = NDIM + 1, MWAVES = NDIM + 1, NROE = 4;
    static constexpr int X_MINB = 3, Y_MINB = 3; // -Xptxas -v: the unsplit x-sweep spills at 4 CTAs/SM (128 registers)
    static constexpr int MAUX = 1;
    static constexpr bool QCOR = false;
    static constexpr bool FWAVE = true;
    static constexpr int MU = (IXY == 2) ? 2 : 1, MV = (IXY == 2) ? 1 : 2;
    // the 2-D shear wave has its MV component only
    __host__ __device__ static constexpr bool nz(int m, int mw) { return !(NDIM == 2 && mw == 1 && m != MV); }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[MEQN],
                                                 const double (&r)[MEQN], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[MEQN][MWAVES],
                                                 double (&s)[MWAVES], double (&amdq)[MEQN],
                                                 double (&apdq)[MEQN], double (&roe)[NROE])
    {
        constexpr int mv = (NDIM == 2) ? MV : 0, NW = MWAVES;
        const double grav = P.p[0], dry = P.p[1];
        const double hl = l[0], hr = r[0];
        const bool wetl = hl > dry, wetr = hr > dry;
        if (!wetl && !wetr) {
#pragma unroll
            for (int m = 0; m < MEQN; m++) {
#pragma unroll
                for (int mw = 0; mw < NW; mw++) wave[m][mw] = 0.0;
                amdq[m] = 0.0;
                apdq[m] = 0.0;
            }
#pragma unroll
            for (int mw = 0; mw < NW; mw++) s[mw] = 0.0;
            roe[0] = roe[1] = roe[2] = roe[3] = 0.0;
            return;
        }
        // a dry cell's quotient is discarded: divide by 1 there so that it stays finite
        const Recip rhl = ar.rcp(wetl ? hl : 1.0), rhr = ar.rcp(wetr ? hr : 1.0);
        const double ul = wetl ? ar.div(l[MU], rhl) : 0.0, ur = wetr ? ar.div(r[MU], rhr) : 0.0;
        double vl = 0.0, vr = 0.0;
        if (NDIM == 2) {
            vl = wetl ? ar.div(l[mv], rhl) : 0.0;
            vr = wetr ? ar.div(r[mv], rhr) : 0.0;
        }
        const double phil = l[MU] * ul + 0.5 * grav * (hl * hl);
        const double phir = r[MU] * ur + 0.5 * grav * (hr * hr);
        const double hl0 = dmax2(hl, 0.0), hr0 = dmax2(hr, 0.0);
        const double sql = ar.sqrt(hl0), sqr = ar.sqrt(hr0);
        const Recip rsq = ar.rcp(sql + sqr);
        const double ubar = ar.div(sql * ul + sqr * ur, rsq);
        const double vbar = (NDIM == 2) ? ar.div(sql * vl + sqr * vr, rsq) : 0.0;
        double cbar;
        Recip rc;
        ar.sqrt_rcp(0.5 * grav * (hl0 + hr0), cbar, rc);
        const double s1 = dmin2(ul - ar.sqrt(grav * hl0), ubar - cbar);
        const double s3 = dmax2(ur + ar.sqrt(grav * hr0), ubar + cbar);
        const double d1 = r[MU] - l[MU];
        const double d2 = phir - phil + 0.5 * grav * (hl + hr) * (axr(0) - axl(0));
        const Recip rds = ar.rcp(s3 - s1);
        const double b1 = ar.div(s3 * d1 - d2, rds);
        const double b3 = ar.div(d2 - s1 * d1, rds);
        wave[0][0] = b1;
        wave[MU][0] = b1 * s1;
        s[0] = s1;
        wave[0][NW - 1] = b3;
        wave[MU][NW - 1] = b3 * s3;
        s[NW - 1] = s3;
        if (NDIM == 2) {
            const double d3 = r[MU] * vr - l[MU] * vl;
            wave[mv][0] = b1 * vl;
            wave[0][1] = 0.0;
            wave[MU][1] = 0.0;
            wave[mv][1] = d3 - b1 * vl - b3 * vr;
            s[1] = ubar;
            wave[mv][NW - 1] = b3 * vr;
        }
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            double am = 0.0, ap = 0.0;
#pragma unroll
            for (int mw = 0; mw < NW; mw++) {
                if (!nz(m, mw)) continue; // literal zeros: adding them to sums that start at +0 changes nothing
                const double z = wave[m][mw];
                if (s[mw] < 0.0) am = am + z;
                else if (s[mw] > 0.0) ap = ap + z;
                else { am = am + 0.5 * z; ap = ap + 0.5 * z; }
            }
            amdq[m] = am;
            apdq[m] = ap;
        }
        roe[0] = ubar; roe[1] = vbar; roe[2] = cbar; roe[3] = ar.div(0.50, rc);
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[MEQN], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[MEQN],
                                                      double (&bm)[MEQN], double (&bp)[MEQN])
    {
        if constexpr (NDIM == 2) {
            if (roe[2] != 0.0) {
                RpShallow<IXY>::transverse(ar, P, roe, qc, ax1, ax2, ax3, asdq, bm, bp);
                return;
            }
        }
#pragma unroll
        for (int m = 0; m < MEQN; m++) { bm[m] = 0.0; bp[m] = 0.0; }
    }
};


// ---------------------------------------------------------------------------
// 3-D acoustics in a heterogeneous medium.  clawpack/riemann rpn3_vc_acoustics.f (external;
// test/acoustics/3d).  q = (p, u, v, w); aux = {impedance Z, sound speed c} of each cell.
// IXYZ = 1, 2, 3 is the sweep direction.  The 3-D interface (transverse<ICOOR> = rpt3,
// double_transverse<ICOOR> = rptt3) is defined below with the other 3-D solvers.
// ---------------------------------------------------------------------------
template <int IXYZ>
struct RpAcoustics3D {
    static constexpr int ID = CLAW_RP_ACOUSTICS3D_VC;
    static constexpr int MEQN = 4, MWAVES = 2, NROE = 1;
    static constexpr int MAUX = 2;
    static constexpr int MU = IXYZ;

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[4],
                                                 const double (&r)[4], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[4][2], double (&s)[2], double (&amdq)[4],
                                                 double (&apdq)[4], double (&roe)[NROE])
    {
        const double zi = axr(0), zim = axl(0);
        double delta1 = r[0] - l[0];
        double delta2 = r[MU] - l[MU];
        const Recip rz = ar.rcp(zim + zi);
        double a1 = ar.div(-delta1 + zi * delta2, rz);
        double a2 = ar.div(delta1 + zim * delta2, rz);
#pragma unroll
        for (int m = 0; m < 4; m++) { wave[m][0] = 0.0; wave[m][1] = 0.0; }
        wave[0][0] = -a1 * zim;
        wave[MU][0] = a1;
        s[0] = -axl(1);
        wave[0][1] = a2 * zi;
        wave[MU][1] = a2;
        s[1] = axr(1);
#pragma unroll
        for (int m = 0; m < 4; m++) {
            amdq[m] = s[0] * wave[m][0];
            apdq[m] = s[1] * wave[m][1];
        }
        roe[0] = 0.0;
    }

    // rpt3 / rptt3_vc_acoustics: asdq split along the line of three cells through (e0, f0) of the
    // transverse aux neighbourhood in direction ICOOR (velocity component rp3_dir(IXYZ, ICOOR))
    template <int ICOOR, class AR, class AX>
    __device__ __forceinline__ static void split(AR &ar, const AX &aux, int e0, int f0, const double (&asdq)[4],
                                                 double (&bm)[4], double (&bp)[4]);
    template <int ICOOR, class AR, class AX>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &, const double (&)[NROE],
                                                      const double (&)[4], const double (&)[4], const AX &aux, int,
                                                      const double (&asdq)[4], double (&bm)[4], double (&bp)[4])
    {
        split<ICOOR>(ar, aux, 0, 0, asdq, bm, bp);
    }
    // the material of the plane (ICOOR = 2) or row (ICOOR = 3) the first split moved into
    template <int ICOOR, class AR, class AX>
    __device__ __forceinline__ static void double_transverse(AR &ar, const RpParams &, const double (&)[NROE],
                                                             const double (&)[4], const double (&)[4], const AX &aux,
                                                             int, int impt, const double (&bsasdq)[4], double (&cm)[4],
                                                             double (&cp)[4])
    {
        const int off = (impt == 1) ? -1 : 1;
        if (ICOOR == 2) split<ICOOR>(ar, aux, 0, off, bsasdq, cm, cp);
        else split<ICOOR>(ar, aux, off, 0, bsasdq, cm, cp);
    }
};


// ---------------------------------------------------------------------------
// Further solvers of the reference's applications (all external: clawpack/riemann,
// un-vendored; restated from the published algorithms, parity unpinned).
// ---------------------------------------------------------------------------

// 2-D acoustics in a heterogeneous medium: rpn2_vc_acoustics.f / rpt2_vc_acoustics.f
// (apps/acoustics/2d/variable).  aux = {density, sound speed}.
template <int IXY>
struct RpVcAcoustics {
    static constexpr int ID = CLAW_RP_VC_ACOUSTICS;
    static constexpr int MEQN = 3, MWAVES = 2, NROE = 1;
    static constexpr int X_MINB = 4, Y_MINB = 3;
    static constexpr int MAUX = 2;
    static constexpr bool QCOR = false;
    static constexpr int MU = (IXY == 2) ? 2 : 1, MV = (IXY == 2) ? 1 : 2;
    __host__ __device__ static constexpr bool nz(int m, int mw) { return m == 0 || m == MU; }

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[3],
                                                 const double (&r)[3], const AuxCell &axl, const AuxCell &axr,
                                                 double (&wave)[3][2], double (&s)[2], double (&amdq)[3],
                                                 double (&apdq)[3], double (&roe)[NROE])
    {
        const double ci = axr(1), cim = axl(1);
        const double zi = axr(0) * ci, zim = axl(0) * cim;
        double delta1 = r[0] - l[0];
        double delta2 = r[MU] - l[MU];
        const Recip rz = ar.rcp(zim + zi);
        double a1 = ar.div(-delta1 + zi * delta2, rz);
        double a2 = ar.div(delta1 + zim * delta2, rz);
        wave[0][0] = -a1 * zim; wave[MU][0] = a1; wave[MV][0] = 0.0; s[0] = -cim;
        wave[0][1] = a2 * zi;   wave[MU][1] = a2; wave[MV][1] = 0.0; s[1] = ci;
#pragma unroll
        for (int m = 0; m < 3; m++) { amdq[m] = s[0] * wave[m][0]; apdq[m] = s[1] * wave[m][1]; }
        roe[0] = 0.0;
    }

    template <class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&qc)[3], const AuxCell &ax1,
                                                      const AuxCell &ax2, const AuxCell &ax3,
                                                      const double (&asdq)[3], double (&bm)[3], double (&bp)[3])
    {
        const double cm = ax1(1), cp = ax3(1);
        const double zm = ax1(0) * cm, zz = ax2(0) * ax2(1), zp = ax3(0) * cp;
        double a1 = ar.div(-asdq[0] + asdq[MV] * zz, zm + zz);
        double a2 = ar.div(asdq[0] + asdq[MV] * zz, zz + zp);
        bm[0] = cm * a1 * zm; bm[MU] = 0.0; bm[MV] = -cm * a1;
        bp[0] = cp * a2 * zp; bp[MU] = 0.0; bp[MV] = cp * a2;
    }
};

// 1-D Burgers with the transonic entropy fix: rp1_burgers.f90 (apps/burgers/1d)
struct RpBurgers {
    static constexpr int ID = CLAW_RP_BURGERS;
    static constexpr int MEQN = 1, MWAVES = 1, NROE = 1;
    static constexpr int X_MINB = 6, Y_MINB = 6;
    static constexpr int MAUX = 0;
    static constexpr bool QCOR = false;
    __host__ __device__ static constexpr bool nz(int, int) { return true; }
    template <class AR>
    __device__ __forceinline__ static void solve(AR &, const RpParams &, const double (&l)[1], const double (&r)[1],
                                                 const AuxCell &, const AuxCell &, double (&wave)[1][1],
                                                 double (&s)[1], double (&amdq)[1], double (&apdq)[1],
                                                 double (&roe)[NROE])
    {
        wave[0][0] = r[0] - l[0];
        s[0] = 0.5 * (l[0] + r[0]);
        amdq[0] = dmin2(s[0], 0.0) * wave[0][0];
        apdq[0] = dmax2(s[0], 0.0) * wave[0][0];
        if (l[0] < 0.0 && r[0] > 0.0) {
            amdq[0] = -0.5 * (l[0] * l[0]);
            apdq[0] = 0.5 * (r[0] * r[0]);
        }
        roe[0] = 0.0;
    }
    template <class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &, const double (&)[NROE],
                                                      const double (&)[1], const AuxCell &, const AuxCell &,
                                                      const AuxCell &, const double (&)[1], double (&bm)[1],
                                                      double (&bp)[1])
    {
        bm[0] = 0.0; bp[0] = 0.0;
    }
};

// Colour equation q_t + u q_x (+ v q_y) = 0 with edge velocities in aux:
// rp1_advection_color.f (NDIM = 1, apps/advection/1d/variable) and rpn2_vc_advection.f /
// rpt2_vc_advection.f (NDIM = 2, apps/advection/2d/annulus).
template <int NDIM, int IXY>
struct RpColor {
    static constexpr int ID = (NDIM == 1) ? CLAW_RP_ADVECTION_COLOR : CLAW_RP_VC_ADVECTION;
    static constexpr int MEQN = 1, MWAVES = 1, NROE = 1;
    static constexpr int X_MINB = 6, Y_MINB = 6;
    static constexpr int MAUX = NDIM;
    static constexpr bool QCOR = false;
    static constexpr int MA = (IXY == 2) ? 1 : 0; // edge velocity of the sweep direction
    static constexpr int KV = (IXY == 2) ? 0 : 1; // ... of the transverse direction
    __host__ __device__ static constexpr bool nz(int, int) { return true; }
    template <class AR>
    __device__ __forceinline__ static void solve(AR &, const RpParams &, const double (&l)[1], const double (&r)[1],
                                                 const AuxCell &axl, const AuxCell &axr, double (&wave)[1][1],
                                                 double (&s)[1], double (&amdq)[1], double (&apdq)[1],
                                                 double (&roe)[NROE])
    {
        const double u = axr(MA);
        wave[0][0] = r[0] - l[0];
        s[0] = u;
        amdq[0] = dmin2(u, 0.0) * wave[0][0];
        apdq[0] = dmax2(u, 0.0) * wave[0][0];
        roe[0] = 0.0;
    }
    template <class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &, const double (&)[NROE],
                                                      const double (&)[1], const AuxCell &ax1, const AuxCell &ax2,
                                                      const AuxCell &ax3, const double (&asdq)[1], double (&bm)[1],
                                                      double (&bp)[1])
    {
        bm[0] = dmin2(ax2(NDIM == 2 ? KV : 0), 0.0) * asdq[0];
        bp[0] = dmax2(ax3(NDIM == 2 ? KV : 0), 0.0) * asdq[0];
    }
};

// 1-D Euler, Roe solver with entropy fix: rp1_euler_with_efix.f (apps/euler/1d/wcblast);
// the 1-D twin of RpEuler5.  cparam{gamma, gamma1}.
struct RpEuler1D {
    static constexpr int ID = CLAW_RP_EULER1D;
    static constexpr int MEQN = 3, MWAVES = 3, NROE = 1;
    static constexpr int X_MINB = 3, Y_MINB = 3;
    static constexpr int MAUX = 0;
    static constexpr bool QCOR = false;
    __host__ __device__ static constexpr bool nz(int, int) { return true; }
    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[3], const double (&r)[3],
                                                 const AuxCell &, const AuxCell &, double (&wave)[3][3],
                                                 double (&s)[3], double (&amdq)[3], double (&apdq)[3],
                                                 double (&roe)[NROE])
    {
        const double gamma1 = P.p[1];
        const double rl = l[0], rr = r[0], ml = l[1], mr = r[1], el = l[2], er = r[2];
        double rhsqrtl = ar.sqrt(rl), rhsqrtr = ar.sqrt(rr);
        const Recip rrl = ar.rcp(rl), rrr = ar.rcp(rr);
        double pl = gamma1 * (el - ar.div(0.5 * (ml * ml), rrl));
        double pr = gamma1 * (er - ar.div(0.5 * (mr * mr), rrr));
        double rhsq2 = rhsqrtl + rhsqrtr;
        const Recip rsl = ar.rcp(rhsqrtl), rsr = ar.rcp(rhsqrtr), rs2 = ar.rcp(rhsq2);
        double u = ar.div(ar.div(ml, rsl) + ar.div(mr, rsr), rs2);
        double enth = ar.div((ar.div(el + pl, rsl) + ar.div(er + pr, rsr)), rs2);
        double a2s = gamma1 * (enth - 0.5 * (u * u));
        double a = ar.sqrt(a2s);
        double d1 = rr - rl, d2 = mr - ml, d3 = er - el;
        double a2 = ar.div(gamma1, a * a) * ((enth - u * u) * d1 + u * d2 - d3);
        double a3 = ar.div(d2 + (a - u) * d1 - a * a2, 2.0 * a);
        double a1 = d1 - a2 - a3;
        wave[0][0] = a1; wave[1][0] = a1 * (u - a); wave[2][0] = a1 * (enth - u * a); s[0] = u - a;
        wave[0][1] = a2; wave[1][1] = a2 * u;       wave[2][1] = a2 * 0.5 * (u * u);  s[1] = u;
        wave[0][2] = a3; wave[1][2] = a3 * (u + a); wave[2][2] = a3 * (enth + u * a); s[2] = u + a;
        bool done = false;
        double ul = ar.div(ml, rrl);
        double cl = ar.sqrt(gamma1 * (gamma1 + 1.0) * (ar.div(el, rrl) - 0.5 * (ul * ul)));
        double s0 = ul - cl;
        if (s0 >= 0.0 && s[0] > 0.0) {
#pragma unroll
            for (int m = 0; m < 3; m++) amdq[m] = 0.0;
            done = true;
        }
        if (!done) {
            double rho1 = rl + wave[0][0], rhou1 = ml + wave[1][0], en1 = el + wave[2][0];
            const Recip r1 = ar.rcp(rho1);
            double p1 = gamma1 * (en1 - ar.div(0.5 * (rhou1 * rhou1), r1));
            double c1 = ar.sqrt(ar.div((gamma1 + 1.0) * p1, r1));
            double s1 = ar.div(rhou1, r1) - c1;
            double sfract;
            if (s0 < 0.0 && s1 > 0.0) sfract = ar.div(s0 * (s1 - s[0]), s1 - s0);
            else if (s[0] < 0.0) sfract = s[0];
            else sfract = 0.0;
#pragma unroll
            for (int m = 0; m < 3; m++) amdq[m] = sfract * wave[m][0];
            if (s[1] >= 0.0) done = true;
        }
        if (!done) {
#pragma unroll
            for (int m = 0; m < 3; m++) amdq[m] = amdq[m] + s[1] * wave[m][1];
            double ur = ar.div(mr, rrr);
            double cr = ar.sqrt(gamma1 * (gamma1 + 1.0) * (ar.div(er, rrr) - 0.5 * (ur * ur)));
            double s3 = ur + cr;
            double rho2 = rr - wave[0][2], rhou2 = mr - wave[1][2], en2 = er - wave[2][2];
            const Recip r2 = ar.rcp(rho2);
            double p2 = gamma1 * (en2 - ar.div(0.5 * (rhou2 * rhou2), r2));
            double c2 = ar.sqrt(ar.div((gamma1 + 1.0) * p2, r2));
            double s2 = ar.div(rhou2, r2) + c2;
            double sfract = 0.0;
            bool add = true;
            if (s2 < 0.0 && s3 > 0.0) sfract = ar.div(s2 * (s3 - s[2]), s3 - s2);
            else if (s[2] < 0.0) sfract = s[2];
            else add = false;
            if (add) {
#pragma unroll
                for (int m = 0; m < 3; m++) amdq[m] = amdq[m] + sfract * wave[m][2];
            }
        }
#pragma unroll
        for (int m = 0; m < 3; m++) {
            double df = 0.0;
#pragma unroll
            for (int mw = 0; mw < 3; mw++) df = df + s[mw] * wave[m][mw];
            apdq[m] = df - amdq[m];
        }
        roe[0] = 0.0;
    }
    template <class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &, const double (&)[NROE],
                                                      const double (&)[3], const AuxCell &, const AuxCell &,
                                                      const AuxCell &, const double (&)[3], double (&bm)[3],
                                                      double (&bp)[3])
    {
#pragma unroll
        for (int m = 0; m < 3; m++) { bm[m] = 0.0; bp[m] = 0.0; }
    }
};


// ===========================================================================
// 3-D solvers of the unsplit and dimensionally split 3-D steps (step3.cuh).  One struct per sweep
// direction IXYZ = 1, 2, 3 with the three routines of clawpack/riemann's 3-D interface:
//
//   solve(ar, P, l, r, axl, axr, wave, s, amdq, apdq, roe)            rpn3 at one interface (the
//       signature of the 2-D solve above; roe[] carries what rpt3 / rptt3 need of the interface)
//   transverse<ICOOR>(ar, P, roe, ql, qr, aux, imp, asdq, bm, bp)     rpt3: asdq split in the
//       y-like (ICOOR = 2) or z-like (ICOOR = 3) direction of the sweep into its down- / up-going
//       parts; imp = 1 for amdq (it enters the cell left of the interface), 2 for apdq
//   double_transverse<ICOOR>(ar, P, roe, ql, qr, aux, imp, impt, bsasdq, cm, cp)   rptt3: a
//       fluctuation already split in the OTHER transverse direction (impt = 1 / 2: its down- /
//       up-going part) split again in direction ICOOR
//
// ql / qr are the states left and right of the interface.  `aux` holds the aux data of the 3x3
// cells around the cell the fluctuation enters, in the plane normal to the sweep: aux(ma, e, f),
// e / f = -1..1 the offset in the y-like / z-like direction (flux3.f's aux1 / aux2 / aux3 slices:
// auxN <-> e = N - 2, their third index k <-> f = k - 2).  "y-like" is direction IXYZ % 3 + 1,
// "z-like" the remaining one.
// ===========================================================================
template <int MAUX>
struct AuxNbhd {
    double v[MAUX > 0 ? MAUX : 1][3][3];
    __device__ __forceinline__ double operator()(int ma, int e, int f) const { return v[ma][e + 1][f + 1]; }
};

// velocity component (1, 2, 3) of the direction ICOOR (1 = the sweep, 2 = y-like, 3 = z-like)
__host__ __device__ constexpr int rp3_dir(int ixyz, int icoor) { return (ixyz - 1 + icoor - 1) % 3 + 1; }

template <int IXYZ>
template <int ICOOR, class AR, class AX>
__device__ __forceinline__ void RpAcoustics3D<IXYZ>::split(AR &ar, const AX &aux, int e0, int f0, const double (&asdq)[4],
                                                          double (&bm)[4], double (&bp)[4])
{
    constexpr int IU = rp3_dir(IXYZ, ICOOR);
    constexpr int de = (ICOOR == 2) ? 1 : 0, df = (ICOOR == 3) ? 1 : 0;
    const double zm = aux(0, e0 - de, f0 - df), zz = aux(0, e0, f0), zp = aux(0, e0 + de, f0 + df);
    const double cm = aux(1, e0 - de, f0 - df), cp = aux(1, e0 + de, f0 + df);
    const double a1 = ar.div(-asdq[0] + asdq[IU] * zz, zm + zz);
    const double a2 = ar.div(asdq[0] + asdq[IU] * zz, zz + zp);
#pragma unroll
    for (int m = 0; m < 4; m++) { bm[m] = 0.0; bp[m] = 0.0; }
    bm[0] = cm * a1 * zm;
    bp[0] = cp * a2 * zp;
    bm[IU] = -cm * a1;
    bp[IU] = cp * a2;
}

// 3-D constant-coefficient advection q_t + u q_x + v q_y + w q_z = 0 (rpn3 / rpt3 /
// rptt3_advection, clawpack/riemann; external, restated): params {u, v, w}.
template <int IXYZ>
struct RpAdvection3 {
    static constexpr int ID = CLAW_RP_ADVECTION3D;
    static constexpr int MEQN = 1, MWAVES = 1, NROE = 1, MAUX = 0;

    template <class AR>
    __device__ __forceinline__ static void solve(AR &, const RpParams &P, const double (&l)[1], const double (&r)[1],
                                                 const AuxCell &, const AuxCell &, double (&wave)[1][1],
                                                 double (&s)[1], double (&amdq)[1], double (&apdq)[1],
                                                 double (&roe)[NROE])
    {
        wave[0][0] = r[0] - l[0];
        s[0] = P.p[IXYZ - 1];
        amdq[0] = dmin2(s[0], 0.0) * wave[0][0];
        apdq[0] = dmax2(s[0], 0.0) * wave[0][0];
        roe[0] = 0.0;
    }
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &P, const double (&)[NROE],
                                                      const double (&)[1], const double (&)[1], const AuxNbhd<MAUX> &,
                                                      int, const double (&asdq)[1], double (&bm)[1], double (&bp)[1])
    {
        const double st = P.p[rp3_dir(IXYZ, ICOOR) - 1];
        bm[0] = dmin2(st, 0.0) * asdq[0];
        bp[0] = dmax2(st, 0.0) * asdq[0];
    }
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void double_transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                             const double (&ql)[1], const double (&qr)[1],
                                                             const AuxNbhd<MAUX> &aux, int imp, int,
                                                             const double (&bsasdq)[1], double (&cm)[1], double (&cp)[1])
    {
        transverse<ICOOR>(ar, P, roe, ql, qr, aux, imp, bsasdq, cm, cp);
    }
};

// 3-D conservative transport q_t + (u q)_x + (v q)_y + (w q)_z = 0 in a cell-centred velocity field,
// f-wave form (the 3-D f-wave step, DESIGN.md §1): aux = {u, v, w} of each cell; restated, parity
// unpinned.
//   rpn3, direction IXYZ, velocity component d = rp3_dir(IXYZ, 1):
//     ul = aux_l(d), ur = aux_r(d);  fwave = (ur*qr) - (ul*ql);  s = 0.5*(ul + ur)
//     s > 0: apdq = fwave, amdq = 0;  s < 0: amdq = fwave, apdq = 0;  s == 0: amdq = apdq = 0.5*fwave
//     so amdq + apdq == fwave == f(q_r) - f(q_l) exactly, and the step conserves q for any velocity
//     field.  The products and the difference of fwave never contract into an FMA, in either build.
//   rpt3, direction ICOOR: vt = velocity component rp3_dir(IXYZ, ICOOR) of the line of three cells
//     through the cell asdq enters (aux(ma, e, f) around that cell):
//       bm = min(0.5*(vt(-1) + vt(0)), 0) * asdq    (the lower edge of that cell)
//       bp = max(0.5*(vt(0) + vt(+1)), 0) * asdq    (the upper edge)
//   rptt3: the same split along the line through the cell the first split sent bsasdq to (impt = 1 /
//     2: one cell down / up in the other transverse direction), the convention of RpAcoustics3D.
template <int IXYZ>
struct RpVcAdvectionFwave3 {
    static constexpr int ID = CLAW_RP_ADVECTION3D_VC_FWAVE;
    static constexpr int MEQN = 1, MWAVES = 1, NROE = 1, MAUX = 3;
    static constexpr bool FWAVE = true;

    template <class AR>
    __device__ __forceinline__ static void solve(AR &, const RpParams &, const double (&l)[1], const double (&r)[1],
                                                 const AuxCell &axl, const AuxCell &axr, double (&wave)[1][1],
                                                 double (&s)[1], double (&amdq)[1], double (&apdq)[1],
                                                 double (&roe)[NROE])
    {
        constexpr int D = rp3_dir(IXYZ, 1);
        const double ul = axl(D - 1), ur = axr(D - 1);
        const double fwave = __dsub_rn(__dmul_rn(ur, r[0]), __dmul_rn(ul, l[0]));
        const double sp = 0.5 * (ul + ur);
        wave[0][0] = fwave;
        s[0] = sp;
        if (sp > 0.0) { amdq[0] = 0.0; apdq[0] = fwave; }
        else if (sp < 0.0) { amdq[0] = fwave; apdq[0] = 0.0; }
        else { amdq[0] = 0.5 * fwave; apdq[0] = 0.5 * fwave; }
        roe[0] = 0.0;
    }
    // asdq split along the line of three cells through (e0, f0) in direction ICOOR
    template <int ICOOR>
    __device__ __forceinline__ static void split(const AuxNbhd<MAUX> &aux, int e0, int f0, const double (&asdq)[1],
                                                 double (&bm)[1], double (&bp)[1])
    {
        constexpr int MA = rp3_dir(IXYZ, ICOOR) - 1;
        constexpr int de = (ICOOR == 2) ? 1 : 0, df = (ICOOR == 3) ? 1 : 0;
        const double vm = aux(MA, e0 - de, f0 - df), v0 = aux(MA, e0, f0), vp = aux(MA, e0 + de, f0 + df);
        bm[0] = dmin2(0.5 * (vm + v0), 0.0) * asdq[0];
        bp[0] = dmax2(0.5 * (v0 + vp), 0.0) * asdq[0];
    }
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &, const double (&)[NROE],
                                                      const double (&)[1], const double (&)[1], const AuxNbhd<MAUX> &aux,
                                                      int, const double (&asdq)[1], double (&bm)[1], double (&bp)[1])
    {
        split<ICOOR>(aux, 0, 0, asdq, bm, bp);
    }
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void double_transverse(AR &, const RpParams &, const double (&)[NROE],
                                                             const double (&)[1], const double (&)[1],
                                                             const AuxNbhd<MAUX> &aux, int, int impt,
                                                             const double (&bsasdq)[1], double (&cm)[1], double (&cp)[1])
    {
        const int off = (impt == 1) ? -1 : 1;
        if (ICOOR == 2) split<ICOOR>(aux, 0, off, bsasdq, cm, cp);
        else split<ICOOR>(aux, off, 0, bsasdq, cm, cp);
    }
};

// 3-D Euler equations, Roe solver with the Harten-Hyman entropy fix (rpn3 / rpt3 / rptt3_euler,
// clawpack/riemann; external, restated from the published algorithm, LeVeque 2002 sec. 15.3 and
// 18.8).  q = (rho, rho u, rho v, rho w, E); params {gamma, gamma1}.  Three waves: u - c, u (the
// entropy jump and both shear jumps), u + c.  With v = w = 0 the normal solve performs the
// operations of RpEuler1D (rp1_euler_with_efix) on the same values.
// roe[] = {u, v, w, enth, a, u^2 + v^2 + w^2} of the interface.
template <class AR>
__device__ __forceinline__ void euler3_roe(AR &ar, double gamma1, const double (&l)[5], const double (&r)[5],
                                           double (&roe)[6])
{
    const double rhsqrtl = ar.sqrt(l[0]), rhsqrtr = ar.sqrt(r[0]);
    const Recip rrl = ar.rcp(l[0]), rrr = ar.rcp(r[0]);
    const double pl = gamma1 * (l[4] - ar.div(0.5 * (l[1] * l[1] + l[2] * l[2] + l[3] * l[3]), rrl));
    const double pr = gamma1 * (r[4] - ar.div(0.5 * (r[1] * r[1] + r[2] * r[2] + r[3] * r[3]), rrr));
    const double rhsq2 = rhsqrtl + rhsqrtr;
    const Recip rsl = ar.rcp(rhsqrtl), rsr = ar.rcp(rhsqrtr), rs2 = ar.rcp(rhsq2);
#pragma unroll
    for (int k = 0; k < 3; k++) roe[k] = ar.div(ar.div(l[1 + k], rsl) + ar.div(r[1 + k], rsr), rs2);
    const double enth = ar.div((ar.div(l[4] + pl, rsl) + ar.div(r[4] + pr, rsr)), rs2);
    const double uvw2 = roe[0] * roe[0] + roe[1] * roe[1] + roe[2] * roe[2];
    roe[3] = enth;
    roe[4] = ar.sqrt(gamma1 * (enth - 0.5 * uvw2));
    roe[5] = uvw2;
}

// d (a jump or a fluctuation) split into the eigenvectors of the Roe matrix of direction MT
// (velocity component 1, 2, 3): wave 0 at un - a, wave 1 at un, wave 2 at un + a
template <int MT, class AR>
__device__ __forceinline__ void euler3_waves(AR &ar, double gamma1, const double (&roe)[6], const double (&d)[5],
                                             double (&wave)[5][3], double (&s)[3])
{
    constexpr int M1 = MT % 3 + 1, M2 = (MT + 1) % 3 + 1; // the two momenta across direction MT
    const double un = roe[MT - 1], u1 = roe[M1 - 1], u2 = roe[M2 - 1];
    const double enth = roe[3], a = roe[4], uvw2 = roe[5];
    const double a3 = ar.div(gamma1, a * a) *
                      ((enth - uvw2) * d[0] + roe[0] * d[1] + roe[1] * d[2] + roe[2] * d[3] - d[4]);
    const double b1 = d[M1] - u1 * d[0], b2 = d[M2] - u2 * d[0];
    const double a5 = ar.div(d[MT] + (a - un) * d[0] - a * a3, 2.0 * a);
    const double a1 = d[0] - a3 - a5;
    wave[0][0] = a1; wave[MT][0] = a1 * (un - a); wave[M1][0] = a1 * u1; wave[M2][0] = a1 * u2;
    wave[4][0] = a1 * (enth - un * a); s[0] = un - a;
    wave[0][1] = a3; wave[MT][1] = a3 * un; wave[M1][1] = a3 * u1 + b1; wave[M2][1] = a3 * u2 + b2;
    wave[4][1] = a3 * 0.5 * uvw2 + b1 * u1 + b2 * u2; s[1] = un;
    wave[0][2] = a5; wave[MT][2] = a5 * (un + a); wave[M1][2] = a5 * u1; wave[M2][2] = a5 * u2;
    wave[4][2] = a5 * (enth + un * a); s[2] = un + a;
}

template <int IXYZ>
struct RpEuler3 {
    static constexpr int ID = CLAW_RP_EULER3D;
    static constexpr int MEQN = 5, MWAVES = 3, NROE = 6, MAUX = 0;
    static constexpr int MU = IXYZ;

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &P, const double (&l)[5], const double (&r)[5],
                                                 const AuxCell &, const AuxCell &, double (&wave)[5][3],
                                                 double (&s)[3], double (&amdq)[5], double (&apdq)[5],
                                                 double (&roe)[NROE])
    {
        const double gamma1 = P.p[1];
        euler3_roe(ar, gamma1, l, r, roe);
        double d[5];
#pragma unroll
        for (int m = 0; m < 5; m++) d[m] = r[m] - l[m];
        euler3_waves<MU>(ar, gamma1, roe, d, wave, s);
        // Harten-Hyman entropy fix on the acoustic waves, left-going fluctuation first
        const Recip rrl = ar.rcp(l[0]), rrr = ar.rcp(r[0]);
        bool done = false;
        const double ulx = ar.div(l[1], rrl), uly = ar.div(l[2], rrl), ulz = ar.div(l[3], rrl);
        const double cl = ar.sqrt(gamma1 * (gamma1 + 1.0) * (ar.div(l[4], rrl) - 0.5 * (ulx * ulx + uly * uly + ulz * ulz)));
        const double s0 = ar.div(l[MU], rrl) - cl;
        if (s0 >= 0.0 && s[0] > 0.0) {
#pragma unroll
            for (int m = 0; m < 5; m++) amdq[m] = 0.0;
            done = true;
        }
        if (!done) {
            double q1[5];
#pragma unroll
            for (int m = 0; m < 5; m++) q1[m] = l[m] + wave[m][0];
            const Recip r1 = ar.rcp(q1[0]);
            const double p1 = gamma1 * (q1[4] - ar.div(0.5 * (q1[1] * q1[1] + q1[2] * q1[2] + q1[3] * q1[3]), r1));
            const double c1 = ar.sqrt(ar.div((gamma1 + 1.0) * p1, r1));
            const double s1 = ar.div(q1[MU], r1) - c1;
            double sfract;
            if (s0 < 0.0 && s1 > 0.0) sfract = ar.div(s0 * (s1 - s[0]), s1 - s0);
            else if (s[0] < 0.0) sfract = s[0];
            else sfract = 0.0;
#pragma unroll
            for (int m = 0; m < 5; m++) amdq[m] = sfract * wave[m][0];
            if (s[1] >= 0.0) done = true;
        }
        if (!done) {
#pragma unroll
            for (int m = 0; m < 5; m++) amdq[m] = amdq[m] + s[1] * wave[m][1];
            const double urx = ar.div(r[1], rrr), ury = ar.div(r[2], rrr), urz = ar.div(r[3], rrr);
            const double cr = ar.sqrt(gamma1 * (gamma1 + 1.0) * (ar.div(r[4], rrr) - 0.5 * (urx * urx + ury * ury + urz * urz)));
            const double s3 = ar.div(r[MU], rrr) + cr;
            double q2[5];
#pragma unroll
            for (int m = 0; m < 5; m++) q2[m] = r[m] - wave[m][2];
            const Recip r2 = ar.rcp(q2[0]);
            const double p2 = gamma1 * (q2[4] - ar.div(0.5 * (q2[1] * q2[1] + q2[2] * q2[2] + q2[3] * q2[3]), r2));
            const double c2 = ar.sqrt(ar.div((gamma1 + 1.0) * p2, r2));
            const double s2 = ar.div(q2[MU], r2) + c2;
            double sfract = 0.0;
            bool add = true;
            if (s2 < 0.0 && s3 > 0.0) sfract = ar.div(s2 * (s3 - s[2]), s3 - s2);
            else if (s[2] < 0.0) sfract = s[2];
            else add = false;
            if (add) {
#pragma unroll
                for (int m = 0; m < 5; m++) amdq[m] = amdq[m] + sfract * wave[m][2];
            }
        }
#pragma unroll
        for (int m = 0; m < 5; m++) {
            double df = 0.0;
#pragma unroll
            for (int mw = 0; mw < 3; mw++) df = df + s[mw] * wave[m][mw];
            apdq[m] = df - amdq[m];
        }
    }
    // rpt3 / rptt3: asdq split with the eigenvectors of the Roe matrix of direction ICOOR at the
    // interface's Roe averages (no aux data: both routines are the same split)
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                      const double (&)[5], const double (&)[5], const AuxNbhd<MAUX> &,
                                                      int, const double (&asdq)[5], double (&bm)[5], double (&bp)[5])
    {
        double wave[5][3], s[3];
        euler3_waves<rp3_dir(IXYZ, ICOOR)>(ar, P.p[1], roe, asdq, wave, s);
#pragma unroll
        for (int m = 0; m < 5; m++) {
            bm[m] = dmin2(s[0], 0.0) * wave[m][0] + dmin2(s[1], 0.0) * wave[m][1] + dmin2(s[2], 0.0) * wave[m][2];
            bp[m] = dmax2(s[0], 0.0) * wave[m][0] + dmax2(s[1], 0.0) * wave[m][1] + dmax2(s[2], 0.0) * wave[m][2];
        }
    }
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void double_transverse(AR &ar, const RpParams &P, const double (&roe)[NROE],
                                                             const double (&ql)[5], const double (&qr)[5],
                                                             const AuxNbhd<MAUX> &aux, int imp, int,
                                                             const double (&bsasdq)[5], double (&cm)[5], double (&cp)[5])
    {
        transverse<ICOOR>(ar, P, roe, ql, qr, aux, imp, bsasdq, cm, cp);
    }
};
