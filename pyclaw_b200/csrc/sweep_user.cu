// sweep_user.cu -- the Riemann-solver plugin seam.
//
// The reference binds a Riemann solver at LINK time: the application's Makefile names any
// rpn2 / rpt2 Fortran file in RP_SOURCE and f2py links it into classic2.so / sharpclaw2.so
// (Makefile.rules:1-26, e.g. apps/kpp/Makefile).  Here the same seam is a header: a file that
// defines `template <int IXY> struct RpUser` with the interface of the solvers in rp.cuh is
// compiled into this translation unit (-DCLAWB200_USER_RP_HEADER="\"path\""), which
// instantiates the classic sweeps, the 1-D step, the SharpClaw stage kernels and the pointwise
// entry points for it under the reserved id CLAWB200_RP_USER:
//     python -m pyclaw_b200.build --user-rp my_rp.cuh --name mine      -> libclawb200_user_mine.so
//     solver.rp = pyclaw.riemann.from_header("my_rp.cuh", name="mine", meqn=..., mwaves=...)
// A 3-D solver is `template <int IXYZ> struct RpUser3` with the 3-D interface of rp.cuh (rpn3 / rpt3 /
// rptt3, e.g. examples/user_rp/rp_acoustics3d_user.cuh); with -DCLAWB200_USER_RP3 this unit also
// instantiates the 3-D steps (step3.cuh), the 3-D SharpClaw stage (sharpclaw3.cuh) and the 3-D
// pointwise solve for it.  A header that defines
// RpUser3 only is compiled with -DCLAWB200_USER_NO_RP as well (no 1-D / 2-D kernels).
//     solver.rp = pyclaw.riemann.from_header("my_rp3.cuh", meqn=..., mwaves=..., ndims=(3,))
// A library built without a user header answers CLAWB200_ERR_UNSUPPORTED for that id.
#include "launch.cuh"

[[maybe_unused]] static int none() { return fail(CLAWB200_ERR_UNSUPPORTED, "this build of libclawb200 has no user Riemann solver: "
                                                          "python -m pyclaw_b200.build --user-rp header.cuh"); }
[[maybe_unused]] static int none3() { return fail(CLAWB200_ERR_UNSUPPORTED, "the user Riemann solver of this build has no 3-D "
                                                                           "version (RpUser3, -DCLAWB200_USER_RP3)"); }
[[maybe_unused]] static int none12() { return fail(CLAWB200_ERR_UNSUPPORTED, "the user Riemann solver of this build is 3-D only"); }
struct ScArgs;

#ifdef CLAWB200_USER_RP_HEADER
#include CLAWB200_USER_RP_HEADER
#include "rp_point.cuh"
#include "sharpclaw3.cuh"
#include "step3.cuh"

template <class RP>
static int user_shape(int *meqn, int *mwaves, int *maux)
{
    *meqn = RP::MEQN;
    *mwaves = RP::MWAVES;
    *maux = RP::MAUX;
    return 0;
}

#ifdef CLAWB200_USER_RP3
int claw_sc3_user(bool old, const ScArgs &A, cudaStream_t st) { return sc_stage3_generic<RpUser3>(old, A, st); }

int claw_step3_user(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                    const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st)
{
    return claw_step3_generic<RpUser3>(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
}
#else
int claw_sc3_user(bool, const ScArgs &, cudaStream_t) { return none3(); }
int claw_step3_user(const clawb200_problem *, int, double, const double *, double *, const double *, double, int,
                    double *, double *, cudaStream_t) { return none3(); }
#endif

int claw_user_shape(int ndim, int *meqn, int *mwaves, int *maux)
{
    if (ndim == 3) {
#ifdef CLAWB200_USER_RP3
        return user_shape<RpUser3<1>>(meqn, mwaves, maux);
#else
        return none3();
#endif
    }
#ifdef CLAWB200_USER_NO_RP
    return none12();
#else
    return user_shape<RpUser<1>>(meqn, mwaves, maux);
#endif
}

int claw_rp_point_user(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                       const double *auxl, const double *auxr, double *wave, double *s, double *amdq,
                       double *apdq, int imp, const double *asdq, double *bm, double *bp, cudaStream_t st)
{
    RpParams P;
    for (int i = 0; i < 8; i++) P.p[i] = p->rp_params[i];
#define GO(RPT, TRANS)                                                                                      \
    return rp_point_launch<RPT, TRANS>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, imp, asdq, bm, bp, st, \
                                       "the user solver reads aux_l / aux_r")
    if (p->ndim == 3) {
#ifdef CLAWB200_USER_RP3
        if (ixy == 1) GO(RpUser3<1>, false);
        if (ixy == 2) GO(RpUser3<2>, false);
        GO(RpUser3<3>, false);
#else
        return none3();
#endif
    }
#ifdef CLAWB200_USER_NO_RP
    return none12();
#else
    if (ixy == 2) GO(RpUser<2>, true);
    GO(RpUser<1>, true);
#endif
#undef GO
}

#ifndef CLAWB200_USER_NO_RP

int claw_x_user(bool trans, const SweepArgs &A, cudaStream_t st)
{
    return A.mcapa > 0 ? launch_x<RpUser<1>, true>(trans, A, st) : launch_x<RpUser<1>>(trans, A, st);
}

int claw_y_user(bool trans, const SweepArgs &A, cudaStream_t st)
{
    return A.mcapa > 0 ? launch_y<RpUser<2>, true>(trans, A, st) : launch_y<RpUser<2>>(trans, A, st);
}

int claw_step1_user(const SweepArgs &A, cudaStream_t st) { return launch_step1<RpUser<1>, false>(A, st); }

// SharpClaw stage (WENO5, both literal readings, hand-written weno5, tvd2), 1-D and 2-D
int claw_sc_user(int ndim, bool old, const ScArgs &A, cudaStream_t st)
{
    return ndim == 1 ? sc_launch1<RpUser<1>>(old, A, st) : sc_launch2<RpUser<1>, RpUser<2>>(old, A, st);
}

#else // ---- RpUser3 only ----
int claw_x_user(bool, const SweepArgs &, cudaStream_t) { return none12(); }
int claw_y_user(bool, const SweepArgs &, cudaStream_t) { return none12(); }
int claw_step1_user(const SweepArgs &, cudaStream_t) { return none12(); }
int claw_sc_user(int, bool, const ScArgs &, cudaStream_t) { return none12(); }
#endif

#else // ---- no user solver in this build ----

int claw_user_shape(int, int *, int *, int *) { return none(); }
int claw_sc3_user(bool, const ScArgs &, cudaStream_t) { return none(); }
int claw_step3_user(const clawb200_problem *, int, double, const double *, double *, const double *, double, int,
                    double *, double *, cudaStream_t) { return none(); }
int claw_x_user(bool, const SweepArgs &, cudaStream_t) { return none(); }
int claw_y_user(bool, const SweepArgs &, cudaStream_t) { return none(); }
int claw_step1_user(const SweepArgs &, cudaStream_t) { return none(); }
int claw_sc_user(int, bool, const ScArgs &, cudaStream_t) { return none(); }
int claw_rp_point_user(const clawb200_problem *, int, long long, const double *, const double *, const double *,
                       const double *, double *, double *, double *, double *, int, const double *, double *, double *,
                       cudaStream_t) { return none(); }
#endif
