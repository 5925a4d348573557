// rp_point.cu -- the Riemann solvers as stand-alone pointwise operators.
//
// The reference's plugin seam for a Riemann solver is
//     rp(q_l, q_r, aux_l, aux_r, aux_global) -> (wave, s, amdq, apdq)          (doc/rp.rst:7-62,
//     src/pyclaw/clawpack.py:349) and, in Fortran, rpn2 / rpt2 (flux2.f:99-100, 167-168, 180-181).
// These entry points evaluate exactly the device functions that are inlined into the sweeps
// (rp.cuh) on arrays of left / right states, one thread per interface, so that the solvers can
// be checked on their own -- against the oracle, and against properties that do not depend on
// any restatement (sum of waves = jump, conservation, B(q^) asdq = bm + bp).
//
// Layout: structure of arrays, ql[m][n], wave[(m * mwaves + mw)][n], s[mw][n].
#include "launch.cuh"

// TRANS = false: solvers without the 2-D transverse solve (the 3-D ones)
template <class RP, bool TRANS>
__global__ void rp_point_kernel(long long n, RpParams P, const double *__restrict__ ql,
                                const double *__restrict__ qr, const double *__restrict__ auxl,
                                const double *__restrict__ auxr, double *__restrict__ wave,
                                double *__restrict__ s, double *__restrict__ amdq,
                                double *__restrict__ apdq, int imp, const double *__restrict__ asdq,
                                double *__restrict__ bm, double *__restrict__ bp)
{
    constexpr int MEQN = RP::MEQN, MW = RP::MWAVES, NROE = RP::NROE;
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double l[MEQN], r[MEQN], w[MEQN][MW], sp[MW], am[MEQN], ap[MEQN], roe[NROE];
#pragma unroll
    for (int m = 0; m < MEQN; m++) { l[m] = ql[m * n + i]; r[m] = qr[m * n + i]; }
    const AuxCell nocell{nullptr, 0};
    // aux_l / aux_r of the reference's contract: [maux][n], the cell on either side of interface i
    const AuxCell axl = auxl ? AuxCell{auxl + i, n} : nocell, axr = auxr ? AuxCell{auxr + i, n} : nocell;
    with_arith([&](auto &ar) { RP::solve(ar, P, l, r, axl, axr, w, sp, am, ap, roe); });
    if (wave) {
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
#pragma unroll
            for (int mw = 0; mw < MW; mw++) wave[(m * MW + mw) * n + i] = w[m][mw];
            amdq[m * n + i] = am[m];
            apdq[m * n + i] = ap[m];
        }
#pragma unroll
        for (int mw = 0; mw < MW; mw++) s[mw * n + i] = sp[mw];
    }
    if constexpr (TRANS) {
    if (asdq) { // rpt2: split asdq with the Roe data of this interface (imp = 1: the cell on the left)
        double a[MEQN], b1[MEQN], b2[MEQN];
#pragma unroll
        for (int m = 0; m < MEQN; m++) a[m] = asdq[m * n + i];
        with_arith([&](auto &ar) { RP::transverse(ar, P, roe, (imp == 1) ? l : r, nocell, nocell, nocell, a, b1, b2); });
#pragma unroll
        for (int m = 0; m < MEQN; m++) { bm[m * n + i] = b1[m]; bp[m * n + i] = b2[m]; }
    }
    }
}

template <class RP, bool TRANS = true>
static int rp_point_launch(long long n, const RpParams &P, const double *ql, const double *qr, const double *auxl,
                           const double *auxr, double *wave,
                           double *s, double *amdq, double *apdq, int imp, const double *asdq, double *bm,
                           double *bp, cudaStream_t st)
{
    if (n <= 0) return 0;
    if (RP::MAUX > 0 && (!auxl || !auxr)) return fail(CLAWB200_ERR_INVALID, "this Riemann solver reads aux_l / aux_r");
    if (RP::MAUX > 0 && asdq) return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise transverse solves: solvers without aux only");
    rp_point_kernel<RP, TRANS><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq,
                                                                    imp, asdq, bm, bp);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// ixy = 1 | 2 (| 3) selects the sweep direction of a 2-D (3-D) solver; auxl / auxr may be null for solvers without aux
int claw_rp_point(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                  const double *auxl, const double *auxr, double *wave, double *s, double *amdq, double *apdq, int imp, const double *asdq,
                  double *bm, double *bp, cudaStream_t st)
{
    if (p->rp_id == CLAWB200_RP_USER)
        return claw_rp_point_user(p, ixy, n, ql, qr, auxl, auxr, wave, s, amdq, apdq, imp, asdq, bm, bp, st);
    RpParams P;
    for (int i = 0; i < 8; i++) P.p[i] = p->rp_params[i];
#define GO(RPT) return rp_point_launch<RPT>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, imp, asdq, bm, bp, st)
#define GO3(RPF) return ixy == 1 ? rp_point_launch<RPF<1>, false>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr, st) \
                   : ixy == 2 ? rp_point_launch<RPF<2>, false>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr, st) \
                              : rp_point_launch<RPF<3>, false>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr, st)
    if (p->ndim == 3) { // rpn3, ixy = 1, 2, 3 (the caller has rejected transverse solves)
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS3D_VC: GO3(RpAcoustics3D);
        case CLAWB200_RP_ADVECTION3D: GO3(RpAdvection3);
        case CLAWB200_RP_EULER3D: GO3(RpEuler3);
        case CLAWB200_RP_ADVECTION3D_VC_FWAVE: GO3(RpVcAdvectionFwave3);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: no 3-D version of this solver");
        }
    }
    if (p->ndim == 1) {
        if (asdq) return fail(CLAWB200_ERR_INVALID, "1-D solvers have no transverse solve");
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: { using R = RpAcoustics<1, 1>; GO(R); }
        case CLAWB200_RP_ADVECTION: { using R = RpAdvection<1, 1>; GO(R); }
        case CLAWB200_RP_SHALLOW: GO(RpShallow1D);
        case CLAWB200_RP_BURGERS: GO(RpBurgers);
        case CLAWB200_RP_EULER1D: GO(RpEuler1D);
        case CLAWB200_RP_NEL_FWAVE: { using R = RpElasticFwave<1, 1>; GO(R); }
        case CLAWB200_RP_ADVECTION_COLOR: { using R = RpColor<1, 1>; GO(R); }
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: no 1-D version of this solver");
        }
    }
    if (ixy == 1) {
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: { using R = RpAcoustics<2, 1>; GO(R); }
        case CLAWB200_RP_ADVECTION: { using R = RpAdvection<2, 1>; GO(R); }
        case CLAWB200_RP_EULER5: GO(RpEuler5<1>);
        case CLAWB200_RP_SHALLOW: GO(RpShallow<1>);
        case CLAWB200_RP_PSYSTEM: { using R = RpElasticFwave<2, 1>; GO(R); }
        case CLAWB200_RP_VC_ACOUSTICS: GO(RpVcAcoustics<1>);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: not compiled for this solver");
        }
    }
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS: { using R = RpAcoustics<2, 2>; GO(R); }
    case CLAWB200_RP_ADVECTION: { using R = RpAdvection<2, 2>; GO(R); }
    case CLAWB200_RP_EULER5: GO(RpEuler5<2>);
    case CLAWB200_RP_SHALLOW: GO(RpShallow<2>);
    case CLAWB200_RP_PSYSTEM: { using R = RpElasticFwave<2, 2>; GO(R); }
    case CLAWB200_RP_VC_ACOUSTICS: GO(RpVcAcoustics<2>);
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: not compiled for this solver");
    }
#undef GO
#undef GO3
}
