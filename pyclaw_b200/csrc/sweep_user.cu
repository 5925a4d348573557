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

template <class RP, bool TRANS>
__global__ void rp_user_point_kernel(long long n, RpParams P, const double *__restrict__ ql,
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
    for (int m = 0; m < MEQN; m++) { l[m] = ql[m * n + i]; r[m] = qr[m * n + i]; }
    const AuxCell nocell{nullptr, 0};
    const AuxCell axl = auxl ? AuxCell{auxl + i, n} : nocell, axr = auxr ? AuxCell{auxr + i, n} : nocell;
    with_arith([&](auto &ar) { RP::solve(ar, P, l, r, axl, axr, w, sp, am, ap, roe); });
    if (wave) {
        for (int m = 0; m < MEQN; m++) {
            for (int mw = 0; mw < MW; mw++) wave[(m * MW + mw) * n + i] = w[m][mw];
            amdq[m * n + i] = am[m];
            apdq[m * n + i] = ap[m];
        }
        for (int mw = 0; mw < MW; mw++) s[mw * n + i] = sp[mw];
    }
    if constexpr (TRANS) {
        if (asdq) {
            double a[MEQN], b1[MEQN], b2[MEQN];
            for (int m = 0; m < MEQN; m++) a[m] = asdq[m * n + i];
            with_arith([&](auto &ar) { RP::transverse(ar, P, roe, (imp == 1) ? l : r, nocell, nocell, nocell, a, b1, b2); });
            for (int m = 0; m < MEQN; m++) { bm[m * n + i] = b1[m]; bp[m * n + i] = b2[m]; }
        }
    }
}

int claw_rp_point_user(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                       const double *auxl, const double *auxr, double *wave, double *s, double *amdq,
                       double *apdq, int imp, const double *asdq, double *bm, double *bp, cudaStream_t st)
{
    int meqn, mwaves, maux;
    int rc = claw_user_shape(p->ndim, &meqn, &mwaves, &maux);
    if (rc) return rc;
    if (maux > 0 && (!auxl || !auxr)) return fail(CLAWB200_ERR_INVALID, "the user solver reads aux_l / aux_r");
    if (maux > 0 && asdq) return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise transverse solves: solvers without aux only");
    if (n <= 0) return 0;
    RpParams P;
    for (int i = 0; i < 8; i++) P.p[i] = p->rp_params[i];
    const unsigned nb = (unsigned)((n + 127) / 128);
#define ARGS n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, imp, asdq, bm, bp
    if (p->ndim == 3) {
#ifdef CLAWB200_USER_RP3
        if (ixy == 1) rp_user_point_kernel<RpUser3<1>, false><<<nb, 128, 0, st>>>(ARGS);
        else if (ixy == 2) rp_user_point_kernel<RpUser3<2>, false><<<nb, 128, 0, st>>>(ARGS);
        else rp_user_point_kernel<RpUser3<3>, false><<<nb, 128, 0, st>>>(ARGS);
#endif
    } else {
#ifndef CLAWB200_USER_NO_RP
        if (ixy == 2) rp_user_point_kernel<RpUser<2>, true><<<nb, 128, 0, st>>>(ARGS);
        else rp_user_point_kernel<RpUser<1>, true><<<nb, 128, 0, st>>>(ARGS);
#endif
    }
#undef ARGS
    CUDA_OK(cudaGetLastError());
    return 0;
}

#ifndef CLAWB200_USER_NO_RP

int claw_x_user(bool trans, const SweepArgs &A, cudaStream_t st)
{
    if (A.mcapa > 0)
        return trans ? launch_x<RpUser<1>, true, true>(A, st) : launch_x<RpUser<1>, false, true>(A, st);
    return trans ? launch_x<RpUser<1>, true>(A, st) : launch_x<RpUser<1>, false>(A, st);
}

int claw_y_user(bool trans, const SweepArgs &A, cudaStream_t st)
{
    if (A.mcapa > 0)
        return trans ? launch_y<RpUser<2>, true, true>(A, st) : launch_y<RpUser<2>, false, true>(A, st);
    return trans ? launch_y<RpUser<2>, true>(A, st) : launch_y<RpUser<2>, false>(A, st);
}

int claw_step1_user(const SweepArgs &A, int mx, cudaStream_t st)
{
    using RP = RpUser<1>;
    constexpr int NT = 128, NC = NT - 3;
    if (A.mcapa > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa is not compiled for the user solver in 1-D");
    size_t smem = sizeof(double) * (RP::MEQN * (NT + 1) + RP::MEQN * RP::MWAVES * NT + 2 * RP::MEQN * NT);
    step1_kernel<RP, NT><<<(mx + NC - 1) / NC, NT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// SharpClaw stage (WENO5, both literal readings, hand-written weno5, tvd2), 1-D and 2-D
int claw_sc_user(int ndim, bool old, const ScArgs &A, cudaStream_t st)
{
    constexpr int SNT = 128, NC = SNT - 2;
    using RX = RpUser<1>;
    using RY = RpUser<2>;
    if (ndim == 1) {
        size_t smem = sizeof(double) * (RX::MEQN * (SNT + 4) + 2 * RX::MEQN * SNT);
        if (old) sc1d_kernel<RX, true, SNT><<<(A.mx + NC - 1) / NC, SNT, smem, st>>>(A);
        else sc1d_kernel<RX, false, SNT><<<(A.mx + NC - 1) / NC, SNT, smem, st>>>(A);
    } else {
        size_t smem = sizeof(double) * (2 * RX::MEQN * (SNT + 4) + 2 * RX::MEQN * SNT);
        dim3 grid((A.mx + NC - 1) / NC, (A.my + A.rows_per_cta - 1) / A.rows_per_cta);
        if (old) {
            auto k = sc2d_kernel<RX, RY, true, SNT>;
            CUDA_OK(set_smem(k, smem));
            k<<<grid, SNT, smem, st>>>(A);
        } else {
            auto k = sc2d_kernel<RX, RY, false, SNT>;
            CUDA_OK(set_smem(k, smem));
            k<<<grid, SNT, smem, st>>>(A);
        }
    }
    CUDA_OK(cudaGetLastError());
    return 0;
}

#else // ---- RpUser3 only ----
int claw_x_user(bool, const SweepArgs &, cudaStream_t) { return none12(); }
int claw_y_user(bool, const SweepArgs &, cudaStream_t) { return none12(); }
int claw_step1_user(const SweepArgs &, int, cudaStream_t) { return none12(); }
int claw_sc_user(int, bool, const ScArgs &, cudaStream_t) { return none12(); }
#endif

#else // ---- no user solver in this build ----

int claw_user_shape(int, int *, int *, int *) { return none(); }
int claw_sc3_user(bool, const ScArgs &, cudaStream_t) { return none(); }
int claw_step3_user(const clawb200_problem *, int, double, const double *, double *, const double *, double, int,
                    double *, double *, cudaStream_t) { return none(); }
int claw_x_user(bool, const SweepArgs &, cudaStream_t) { return none(); }
int claw_y_user(bool, const SweepArgs &, cudaStream_t) { return none(); }
int claw_step1_user(const SweepArgs &, int, cudaStream_t) { return none(); }
int claw_sc_user(int, bool, const ScArgs &, cudaStream_t) { return none(); }
int claw_rp_point_user(const clawb200_problem *, int, long long, const double *, const double *, const double *,
                       const double *, double *, double *, double *, double *, int, const double *, double *, double *,
                       cudaStream_t) { return none(); }
#endif
