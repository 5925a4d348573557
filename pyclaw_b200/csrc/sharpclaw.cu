// sharpclaw.cu -- SharpClaw stage kernels (sharpclaw.cuh): launch dispatch and the packing of the WENO
// coefficient tables (caller-owned, no state in the library).
#include "launch.cuh"
#include "sharpclaw.cuh"

using RpColor1D = RpColor<1, 1>;

extern "C" int clawb200_weno_table_doubles(void) { return (int)(sizeof(WenoTab) / sizeof(double)); }

extern "C" int clawb200_pack_weno_tables(int k, const double *S, const double *CL, const double *CR,
                                         const double *WL, const double *WR, double eps, double *packed)
{
    if (k < 3 || k > 9) return fail(CLAWB200_ERR_INVALID, "weno_order must be an odd number between 5 and 17");
    if (!S || !CL || !CR || !WL || !WR || !packed) return fail(CLAWB200_ERR_INVALID, "null table");
    WenoTab &h = *reinterpret_cast<WenoTab *>(packed);
    memset(&h, 0, sizeof(h));
    const int npair = k * (k + 1) / 2;
    h.k = (double)k;
    h.eps = eps;
    for (int r = 0; r < k; r++) {
        for (int n = 0; n < npair; n++) h.S[r][n] = S[r * npair + n];
        for (int j = 0; j < k; j++) { h.CL[r][j] = CL[r * k + j]; h.CR[r][j] = CR[r * k + j]; }
        h.WL[r] = WL[r];
        h.WR[r] = WR[r];
    }
    return 0;
}

template <class RP>
static int sc_launch1_tab(const ScArgs &A, int weno_k, cudaStream_t st)
{
    constexpr int NC = SNT - 2;
    const int H = weno_k - 1;
    size_t smem = sizeof(double) * (RP::MEQN * (SNT + 2 * H) + 2 * RP::MEQN * SNT);
    sc1d_tab_kernel<RP, SNT><<<(A.mx + NC - 1) / NC, SNT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

template <class RPX, class RPY>
static int sc_launch2_tab(ScArgs A, int weno_k, cudaStream_t st)
{
    constexpr int NC = SNT - 2;
    const int H = weno_k - 1;
    size_t smem = sizeof(double) * (RPX::MEQN * (SNT + 2 * H) + 2 * RPX::MEQN * SNT);
    const int nxcta = (A.mx + NC - 1) / NC;
    A.rows_per_cta = pick_rows(A.my, nxcta, false);
    dim3 grid(nxcta, (A.my + A.rows_per_cta - 1) / A.rows_per_cta);
    sc2d_tab_kernel<RPX, RPY, SNT><<<grid, SNT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

static void weno_constants(ScArgs &A, int variant)
{
    const bool f32 = (variant == CLAWB200_WENO_PYWENO_F32);
#define LIT(x) (f32 ? (double)(x##f) : (double)(x))
    A.c333 = LIT(3.33333333333333); A.c1033 = LIT(10.3333333333333);
    A.c366 = LIT(3.66666666666667); A.c833 = LIT(8.33333333333333);
    A.c633 = LIT(6.33333333333333); A.c133 = LIT(1.33333333333333);
    A.c433 = LIT(4.33333333333333); A.c166 = LIT(1.66666666666667);
    A.d01 = LIT(0.1); A.d06 = LIT(0.6); A.d03 = LIT(0.3); A.eps = LIT(1.0e-36);
    A.r183 = LIT(1.83333333333333); A.r116 = LIT(1.16666666666667);
    A.r0333 = LIT(0.333333333333333); A.r0833 = LIT(0.833333333333333);
    A.r0166 = LIT(0.166666666666667);
#undef LIT
    A.epweno = (double)1.e-36f; // reconstruct.f90:7, a REAL(4) literal
}

// the stage arguments common to 1-D, 2-D and 3-D
static int sc_args(ScArgs &A, const clawb200_problem *p, const double *q, const double *qa, double *out,
                   double *dq_out, double dt, int mode, double ca, double cb, double div, double *cfl_dev,
                   const double *aux)
{
    memset(&A, 0, sizeof(A));
    A.q = q; A.qa = qa; A.out = out; A.dq_out = dq_out;
    A.mstride = p->mstride; A.pitch = p->pitch;
    A.mx = p->mx; A.my = p->my; A.mbc = p->mbc;
    A.dtdx = dt / p->dx;
    A.dtdy = (p->ndim > 1) ? dt / p->dy : 0.0;
    for (int i = 0; i < 8; i++) A.rp.p[i] = p->rp_params[i];
    weno_constants(A, p->weno_variant);
    A.aux = aux;
    A.amstride = p->mstride;
    A.mode = mode; A.ca = ca; A.cb = cb; A.div = div;
    A.cfl_bits = (unsigned long long *)cfl_dev;
    if (p->weno_variant == CLAWB200_RECON_TVD2) {
        if (p->meqn > CLAWB200_MAXWAVES) return fail(CLAWB200_ERR_INVALID, "tvd2: meqn exceeds the limiter array");
        A.tvd = 1;
        for (int m = 0; m < p->meqn; m++) A.mthlim[m] = p->mthlim[m];
    }
    return 0;
}

// 3-D (sharpclaw3.cuh): WENO5 (both literal readings), hand-written weno5 and tvd2; the caller
// (clawb200_sharpclaw_stage3) has rejected everything else
int sharpclaw_launch3(const clawb200_problem *p, int mz, double dz, const double *q, const double *qa, double *out,
                      double *dq_out, double dt, int mode, double ca, double cb, double div,
                      double *cfl_dev, cudaStream_t st, const double *aux)
{
    ScArgs A;
    int rc = sc_args(A, p, q, qa, out, dq_out, dt, mode, ca, cb, div, cfl_dev, aux);
    if (rc) return rc;
    A.plane = (long long)p->pitch * (p->my + 2 * p->mbc);
    A.mz = mz;
    A.dtdz = dt / dz;
    const bool old = (p->weno_variant == CLAWB200_WENO_OLD);
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS3D_VC: return claw_sc3_acoustics(old, A, st);
    case CLAWB200_RP_EULER3D: return claw_sc3_euler(old, A, st);
    case CLAWB200_RP_ADVECTION3D: return claw_sc3_advection(old, A, st);
    case CLAWB200_RP_ADVECTION3D_VC_FWAVE: return claw_sc3_vc_advection_fwave(old, A, st);
    default: return claw_sc3_user(old, A, st);
    }
}

int sharpclaw_launch(const clawb200_problem *p, const double *q, const double *qa, double *out,
                            double *dq_out, double dt, int mode, double ca, double cb, double div,
                            double *cfl_dev, cudaStream_t st, const double *aux)
{
    ScArgs A;
    int rc = sc_args(A, p, q, qa, out, dq_out, dt, mode, ca, cb, div, cfl_dev, aux);
    if (rc) return rc;
    const bool old = (p->weno_variant == CLAWB200_WENO_OLD);
    if (p->weno_variant == CLAWB200_WENO_TABLES) {
        const int wk = p->weno_k;
        if (wk < 3 || wk > 9 || !p->weno_tab)
            return fail(CLAWB200_ERR_INVALID, "weno_variant = tables needs problem.weno_k in 3..9 and problem.weno_tab "
                                              "(clawb200_pack_weno_tables)");
        if (p->mbc < wk) return fail(CLAWB200_ERR_INVALID, "WENO of order 2k-1 needs mbc >= k");
        A.tab = reinterpret_cast<const WenoTab *>(p->weno_tab);
        if (p->method[5] > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for WENO orders above 5");
        if (p->ndim == 2) {
            switch (p->rp_id) {
            case CLAWB200_RP_ACOUSTICS: return sc_launch2_tab<RpAcoustics<2, 1>, RpAcoustics<2, 2>>(A, wk, st);
            case CLAWB200_RP_ADVECTION: return sc_launch2_tab<RpAdvection<2, 1>, RpAdvection<2, 2>>(A, wk, st);
            case CLAWB200_RP_EULER5: return sc_launch2_tab<RpEuler5<1>, RpEuler5<2>>(A, wk, st);
            case CLAWB200_RP_SHALLOW: return sc_launch2_tab<RpShallow<1>, RpShallow<2>>(A, wk, st);
            case CLAWB200_RP_VC_ACOUSTICS: return sc_launch2_tab<RpVcAcoustics<1>, RpVcAcoustics<2>>(A, wk, st);
            default: return fail(CLAWB200_ERR_UNSUPPORTED, "WENO orders above 5 are not compiled for this solver in 2-D");
            }
        }
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: return sc_launch1_tab<RpAcoustics<1, 1>>(A, wk, st);
        case CLAWB200_RP_ADVECTION: return sc_launch1_tab<RpAdvection<1, 1>>(A, wk, st);
        case CLAWB200_RP_SHALLOW: return sc_launch1_tab<RpShallow1D>(A, wk, st);
        case CLAWB200_RP_BURGERS: return sc_launch1_tab<RpBurgers>(A, wk, st);
        case CLAWB200_RP_EULER1D: return sc_launch1_tab<RpEuler1D>(A, wk, st);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "no 1-D version of this Riemann solver");
        }
    }
    if (p->weno_variant == CLAWB200_RECON_WENO_WAVE || p->weno_variant == CLAWB200_RECON_WENO_FWAVE) {
        // char_decomp = 1 (flux1.f90:95-105).  1-D only: the reference's 2-D flux1.f90:102-106 calls
        // rpn2 with a wrong argument list and then both reconstructions, it cannot run
        if (p->ndim != 1) return fail(CLAWB200_ERR_UNSUPPORTED, "wave-based reconstruction (char_decomp = 1) exists in 1-D only");
        if (p->method[5] > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa is not compiled for the wave-based reconstruction");
        const bool fw = (p->weno_variant == CLAWB200_RECON_WENO_FWAVE);
#define WAVE1(RPT)                                                                                          \
    {                                                                                                       \
        using RP = RPT;                                                                                     \
        constexpr int NC = SNT - 6;                                                                         \
        size_t smem = sizeof(double) * (RP::MEQN * (SNT + 1) + RP::MEQN * RP::MWAVES * SNT + 2 * RP::MEQN * SNT); \
        if (fw) sc1d_wave_kernel<RP, true, SNT><<<(A.mx + NC - 1) / NC, SNT, smem, st>>>(A);               \
        else sc1d_wave_kernel<RP, false, SNT><<<(A.mx + NC - 1) / NC, SNT, smem, st>>>(A);                 \
        CUDA_OK(cudaGetLastError());                                                                        \
        return 0;                                                                                           \
    }
        using Ac1 = RpAcoustics<1, 1>;
        using Ad1 = RpAdvection<1, 1>;
        using El1 = RpElasticFwave<1, 1>;
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: WAVE1(Ac1)
        case CLAWB200_RP_ADVECTION: WAVE1(Ad1)
        case CLAWB200_RP_SHALLOW: WAVE1(RpShallow1D)
        case CLAWB200_RP_BURGERS: WAVE1(RpBurgers)
        case CLAWB200_RP_EULER1D: WAVE1(RpEuler1D)
        case CLAWB200_RP_NEL_FWAVE: WAVE1(El1)
        case CLAWB200_RP_ADVECTION_COLOR: WAVE1(RpColor1D)
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "no 1-D version of this Riemann solver");
        }
#undef WAVE1
    }
    if (p->rp_id == CLAWB200_RP_USER) {
        if (p->method[5] > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa is not compiled for the user solver in SharpClaw");
        return claw_sc_user(p->ndim, old, A, st);
    }
    if (p->method[5] > 0) {
        // capacity function (flux1.f90:59-63): compiled for the acoustics and advection solvers
        A.capa = aux + (long long)(p->method[5] - 1) * p->mstride;
        A.dt = dt; A.dx = p->dx; A.dy = (p->ndim > 1) ? p->dy : 1.0;
        if (p->ndim == 1) {
            switch (p->rp_id) {
            case CLAWB200_RP_ACOUSTICS: return sc_launch1<RpAcoustics<1, 1>, true>(old, A, st);
            case CLAWB200_RP_ADVECTION: return sc_launch1<RpAdvection<1, 1>, true>(old, A, st);
            default: return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for this solver");
            }
        }
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: return sc_launch2<RpAcoustics<2, 1>, RpAcoustics<2, 2>, true>(old, A, st);
        case CLAWB200_RP_ADVECTION: return sc_launch2<RpAdvection<2, 1>, RpAdvection<2, 2>, true>(old, A, st);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for this solver");
        }
    }
    if (p->ndim == 1) {
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: return sc_launch1<RpAcoustics<1, 1>>(old, A, st);
        case CLAWB200_RP_ADVECTION: return sc_launch1<RpAdvection<1, 1>>(old, A, st);
        case CLAWB200_RP_SHALLOW: return sc_launch1<RpShallow1D>(old, A, st);
        case CLAWB200_RP_BURGERS: return sc_launch1<RpBurgers>(old, A, st);
        case CLAWB200_RP_EULER1D: return sc_launch1<RpEuler1D>(old, A, st);
        case CLAWB200_RP_NEL_FWAVE: // with char_decomp = 0 an f-wave solver only contributes amdq / apdq
            return sc_launch1<RpElasticFwave<1, 1>>(old, A, st);
        case CLAWB200_RP_ADVECTION_COLOR: return sc_launch1<RpColor1D>(old, A, st);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "no 1-D version of this Riemann solver");
        }
    }
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS: return sc_launch2<RpAcoustics<2, 1>, RpAcoustics<2, 2>>(old, A, st);
    case CLAWB200_RP_ADVECTION: return sc_launch2<RpAdvection<2, 1>, RpAdvection<2, 2>>(old, A, st);
    case CLAWB200_RP_EULER5: return sc_launch2<RpEuler5<1>, RpEuler5<2>>(old, A, st);
    case CLAWB200_RP_SHALLOW: return sc_launch2<RpShallow<1>, RpShallow<2>>(old, A, st);
    case CLAWB200_RP_PSYSTEM: return sc_launch2<RpElasticFwave<2, 1>, RpElasticFwave<2, 2>>(old, A, st);
    case CLAWB200_RP_VC_ACOUSTICS: return sc_launch2<RpVcAcoustics<1>, RpVcAcoustics<2>>(old, A, st);
    case CLAWB200_RP_VC_ADVECTION: return sc_launch2<RpColor<2, 1>, RpColor<2, 2>>(old, A, st);
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "unknown rp_id");
    }
}
