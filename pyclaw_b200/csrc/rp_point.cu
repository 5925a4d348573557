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
// The kernel and its launcher are in rp_point.cuh.
#include "rp_point.cuh"

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
