// clawb200.cu -- C ABI (include/clawb200.h) over the sm_100a kernels in classic.cuh and
// sharpclaw.cuh (instantiated in the sweep_*.cu / step1.cu / sharpclaw.cu translation units,
// see launch.cuh).  Built in-tree with
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared ...
// -fmad=false is part of the contract: the reference's Fortran is compiled without FMA
// contraction and results must match it bit for bit (SURVEY.md section 7, "hard parts").
#include "launch.cuh"

static thread_local std::string g_err;

int fail(int code, const char *msg)
{
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *where)
{
    g_err = std::string(where) + ": " + cudaGetErrorString(e);
    return CLAWB200_ERR_CUDA;
}

extern "C" int clawb200_version(void) { return 100; }
extern "C" const char *clawb200_last_error(void) { return g_err.c_str(); }

extern "C" int clawb200_cfl_reset(double *cfl_dev, void *stream)
{
    CUDA_OK(cudaMemsetAsync(cfl_dev, 0, sizeof(double), (cudaStream_t)stream));
    return 0;
}

// ---------------------------------------------------------------------------
static int check_problem(const clawb200_problem *p, int ndim)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    if (p->ndim != ndim) return fail(CLAWB200_ERR_INVALID, "wrong ndim for this entry point");
    if (p->mx < 1 || p->my < 1) return fail(CLAWB200_ERR_INVALID, "mx, my must be positive");
    if (p->mwaves < 1 || p->mwaves > CLAWB200_MAXWAVES) return fail(CLAWB200_ERR_INVALID, "bad mwaves");
    if (p->pitch < p->mx + 2 * p->mbc) return fail(CLAWB200_ERR_INVALID, "pitch smaller than padded row");
    // a smaller component stride would make the sweeps' ghost rows of one component the first rows of the next
    if (ndim == 2 && p->mstride < (long long)p->pitch * (p->my + 2 * p->mbc))
        return fail(CLAWB200_ERR_INVALID, "mstride smaller than the padded field");
    if (p->method[5] < 0 || p->method[5] > p->maux)
        return fail(CLAWB200_ERR_INVALID, "method[5] (mcapa+1) must index an aux component");
    return 0;
}

// capacity functions / aux arrays are compiled for the 2-D classic sweeps of these solvers
static int check_aux(const clawb200_problem *p, const double *aux, bool classic2d)
{
    const bool capa = p->method[5] > 0;
    const bool bathy = p->rp_id == CLAWB200_RP_SHALLOW_BATHY_FWAVE;
    const bool fw = p->rp_id == CLAWB200_RP_NEL_FWAVE || p->rp_id == CLAWB200_RP_PSYSTEM || bathy;
    const bool vc = p->rp_id == CLAWB200_RP_VC_ACOUSTICS || p->rp_id == CLAWB200_RP_ADVECTION_COLOR ||
                    p->rp_id == CLAWB200_RP_VC_ADVECTION;
    const bool need_aux = capa || fw || vc || p->rp_id == CLAWB200_RP_SPHERE;
    if (!need_aux) return 0;
    if (!aux) return fail(CLAWB200_ERR_INVALID, "aux array required (mcapa > 0 or aux-dependent Riemann solver)");
    if (fw) { // classic step1 / step2 / step2ds only (the callers check the solver's dimension)
        if (capa) return fail(CLAWB200_ERR_UNSUPPORTED, "capacity function is not compiled for the f-wave solvers");
        if (bathy) return p->maux < 1 ? fail(CLAWB200_ERR_INVALID, "shallow water over bathymetry: aux = {b}, maux >= 1") : 0;
        if (p->rp_id == CLAWB200_RP_NEL_FWAVE ? p->maux < 2 : p->maux != 4)
            return fail(CLAWB200_ERR_INVALID, "f-wave elasticity solvers: aux = {rho, K} (1-D) or {rho, E, law, eps} (2-D)");
        return 0;
    }
    if (vc) { // variable-coefficient solvers read aux in the classic sweeps (step1 / step2 / step2ds)
        const int need = (p->rp_id == CLAWB200_RP_ADVECTION_COLOR) ? 1 : 2;
        if (p->maux < need) return fail(CLAWB200_ERR_INVALID, "this Riemann solver reads more aux components than maux");
        if (capa && p->rp_id != CLAWB200_RP_VC_ADVECTION)
            return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for this solver");
        return 0;
    }
    if (p->rp_id == CLAWB200_RP_SPHERE) {
        if (!classic2d) return fail(CLAWB200_ERR_UNSUPPORTED, "the sphere solver is compiled for the 2-D classic sweeps only");
        if (p->maux < 16 || !capa)
            return fail(CLAWB200_ERR_INVALID, "the sphere solver needs its 16 aux components and mcapa");
        return 0;
    }
    // capa: every solver in the 2-D classic sweeps; acoustics and advection in step1 and SharpClaw
    if (!classic2d && !(p->rp_id == CLAWB200_RP_ACOUSTICS || p->rp_id == CLAWB200_RP_ADVECTION))
        return fail(CLAWB200_ERR_UNSUPPORTED, "capacity function (mcapa) in 1-D / SharpClaw is compiled for the "
                                              "acoustics and advection solvers only");
    return 0;
}

static SweepArgs make_args(const clawb200_problem *p, const double *qin, double *qout, double dt,
                           double *cfl_dev, const double *aux = nullptr)
{
    SweepArgs A;
    memset(&A, 0, sizeof(A));
    A.aux = aux;
    A.amstride = p->mstride; // aux shares the padded shape (and pitch) of q
    A.mcapa = p->method[5];
    A.qin = qin; A.qbase = qin; A.qout = qout;
    A.mstride = p->mstride; A.pitch = p->pitch;
    A.mx = p->mx; A.my = p->my; A.mbc = p->mbc;
    A.dtdx = dt / p->dx;
    A.dtdy = (p->ndim > 1) ? dt / p->dy : 0.0;
    A.dt = dt;
    A.dx = p->dx;
    A.dy = (p->ndim > 1) ? p->dy : 1.0;
    A.dt_dev = p->dt_dev;
    A.order = p->method[1];
    A.trans = p->method[2];
    for (int i = 0; i < CLAW_MAXWAVES; i++) A.mthlim[i] = (i < p->mwaves) ? p->mthlim[i] : 0;
    for (int i = 0; i < 8; i++) A.rp.p[i] = p->rp_params[i];
    if (p->rp_id == CLAWB200_RP_SPHERE) { // common /comxyt/ dxcom, dycom
        if (A.rp.p[1] == 0.0) A.rp.p[1] = p->dx;
        if (A.rp.p[2] == 0.0) A.rp.p[2] = p->dy;
    }
    A.cfl_bits = (unsigned long long *)cfl_dev;
    return A;
}

// dispatch on the Riemann-solver family (one translation unit each, launch.cuh)
template <bool TRANS>
static int dispatch_x(int rp_id, const SweepArgs &A, cudaStream_t st)
{
    if (rp_id == CLAWB200_RP_EULER5) return claw_x_euler(TRANS, A, st);
    if (rp_id == CLAWB200_RP_SPHERE) return claw_x_sphere(TRANS, A, st);
    if (rp_id == CLAWB200_RP_USER) return claw_x_user(TRANS, A, st);
    return claw_x_misc(rp_id, TRANS, A, st);
}
template <bool TRANS>
static int dispatch_y(int rp_id, const SweepArgs &A, cudaStream_t st)
{
    if (rp_id == CLAWB200_RP_EULER5) return claw_y_euler(TRANS, A, st);
    if (rp_id == CLAWB200_RP_SPHERE) return claw_y_sphere(TRANS, A, st);
    if (rp_id == CLAWB200_RP_USER) return claw_y_user(TRANS, A, st);
    return claw_y_misc(rp_id, TRANS, A, st);
}

static int check_rp_shape(const clawb200_problem *p)
{
    int meqn = 0, mwaves = 0;
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS: meqn = p->ndim + 1; mwaves = 2; break;
    case CLAWB200_RP_ADVECTION: meqn = 1; mwaves = 1; break;
    case CLAWB200_RP_EULER5: meqn = 5; mwaves = 5; break;
    case CLAWB200_RP_SHALLOW: meqn = p->ndim + 1; mwaves = p->ndim + 1; break;
    case CLAWB200_RP_SPHERE: meqn = 4; mwaves = 3; break;
    case CLAWB200_RP_NEL_FWAVE: meqn = 2; mwaves = 2; break;
    case CLAWB200_RP_PSYSTEM: meqn = 3; mwaves = 2; break;
    case CLAWB200_RP_VC_ACOUSTICS: meqn = 3; mwaves = 2; break;
    case CLAWB200_RP_BURGERS: meqn = 1; mwaves = 1; break;
    case CLAWB200_RP_ADVECTION_COLOR: meqn = 1; mwaves = 1; break;
    case CLAWB200_RP_VC_ADVECTION: meqn = 1; mwaves = 1; break;
    case CLAWB200_RP_EULER1D: meqn = 3; mwaves = 3; break;
    case CLAWB200_RP_SHALLOW_BATHY_FWAVE:
        if (p->ndim != 1 && p->ndim != 2) return fail(CLAWB200_ERR_UNSUPPORTED, "this Riemann solver is 1-D / 2-D only");
        if (!(p->rp_params[1] >= 0.0)) return fail(CLAWB200_ERR_INVALID, "dry_tolerance (rp_params[1]) must be >= 0");
        meqn = p->ndim + 1; mwaves = p->ndim + 1; break;
    case CLAWB200_RP_USER: {
        int maux = 0;
        int rc = claw_user_shape(p->ndim, &meqn, &mwaves, &maux);
        if (rc) return rc;
        if (p->maux < maux) return fail(CLAWB200_ERR_INVALID, "the user Riemann solver reads more aux components than maux");
    } break;
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "unknown rp_id");
    }
    if (p->meqn != meqn || p->mwaves != mwaves)
        return fail(CLAWB200_ERR_INVALID, "meqn/mwaves do not match the Riemann solver");
    if ((p->rp_id == CLAWB200_RP_EULER5 || p->rp_id == CLAWB200_RP_SPHERE || p->rp_id == CLAWB200_RP_PSYSTEM ||
         p->rp_id == CLAWB200_RP_VC_ACOUSTICS || p->rp_id == CLAWB200_RP_VC_ADVECTION) && p->ndim != 2)
        return fail(CLAWB200_ERR_UNSUPPORTED, "this Riemann solver is 2-D only");
    if ((p->rp_id == CLAWB200_RP_NEL_FWAVE || p->rp_id == CLAWB200_RP_BURGERS ||
         p->rp_id == CLAWB200_RP_ADVECTION_COLOR || p->rp_id == CLAWB200_RP_EULER1D) && p->ndim != 1)
        return fail(CLAWB200_ERR_UNSUPPORTED, "this Riemann solver is 1-D only");
    return 0;
}

extern "C" int clawb200_step1(const clawb200_problem *p, const double *q_in, double *q_out,
                              const double *aux, double dt, double *cfl_dev, void *stream)
{
    int rc = check_problem(p, 1);
    if (rc) return rc;
    if ((rc = check_rp_shape(p))) return rc;
    if (p->mbc < 2) return fail(CLAWB200_ERR_INVALID, "classic solvers need mbc >= 2");
    if (q_in == q_out) return fail(CLAWB200_ERR_INVALID, "q_in and q_out must differ");
    if ((rc = check_aux(p, aux, false))) return rc;
    SweepArgs A = make_args(p, q_in, q_out, dt, cfl_dev, aux);
    cudaStream_t st = (cudaStream_t)stream;
    if (p->rp_id == CLAWB200_RP_USER) return claw_step1_user(A, st);
    return claw_step1(p->rp_id, A, st);
}

extern "C" int clawb200_step2ds(const clawb200_problem *p, const double *q_in, double *q_out,
                                const double *aux, double dt, int ids, double *cfl_dev,
                                void *stream)
{
    int rc = check_problem(p, 2);
    if (rc) return rc;
    if ((rc = check_rp_shape(p))) return rc;
    if (p->mbc < 2) return fail(CLAWB200_ERR_INVALID, "classic solvers need mbc >= 2");
    if (q_in == q_out) return fail(CLAWB200_ERR_INVALID, "q_in and q_out must differ");
    if ((rc = check_aux(p, aux, true))) return rc;
    SweepArgs A = make_args(p, q_in, q_out, dt, cfl_dev, aux);
    A.trans = -1;
    cudaStream_t st = (cudaStream_t)stream;
    if (ids == 1) {
        A.ilo = 1; A.ihi = p->mx;
        A.jlo = 1 - p->mbc; A.jhi = p->my + p->mbc;
        A.rows_per_cta = pick_rows(A.jhi - A.jlo + 1, (p->mx + XNT - 4) / (XNT - 3));
        return dispatch_x<false>(p->rp_id, A, st);
    } else if (ids == 2) {
        A.ilo = 1 - p->mbc; A.ihi = p->mx + p->mbc;
        A.jlo = 1; A.jhi = p->my;
        A.rows_per_cta = pick_rows(p->my, (p->mx + 2 * p->mbc + YNT - 1) / YNT);
        return dispatch_y<false>(p->rp_id, A, st);
    } else
        return fail(CLAWB200_ERR_INVALID, "ids must be 1 or 2");
    return 0;
}

// ---------------------------------------------------------------------------
// 3-D, dimensional splitting (step3ds.f:2-376; clawpack.py:656-676) and the unsplit step.  A 3-D
// field is q[m][k][j][i].  Both run the kernels of step3.cuh for every 3-D solver.
// ---------------------------------------------------------------------------
// The Riemann solver of a 3-D step: the shape it is compiled for and the aux data it reads.
static int check_rp3(const clawb200_problem *p, bool have_aux)
{
    int meqn = 0, mwaves = 0, maux = 0;
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS3D_VC: meqn = 4; mwaves = 2; maux = 2; break;
    case CLAWB200_RP_ADVECTION3D: meqn = 1; mwaves = 1; break;
    case CLAWB200_RP_EULER3D: meqn = 5; mwaves = 3; break;
    case CLAWB200_RP_ADVECTION3D_VC_FWAVE: meqn = 1; mwaves = 1; maux = 3; break;
    case CLAWB200_RP_USER: {
        int rc = claw_user_shape(3, &meqn, &mwaves, &maux);
        if (rc) return rc;
    } break;
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "no 3-D version of this Riemann solver");
    }
    if (p->meqn != meqn || p->mwaves != mwaves) return fail(CLAWB200_ERR_INVALID, "meqn/mwaves do not match the Riemann solver");
    if (maux > 0 && (p->maux < maux || !have_aux))
        return fail(CLAWB200_ERR_INVALID, p->rp_id == CLAWB200_RP_ACOUSTICS3D_VC
                                              ? "aux array required: {impedance, sound speed}"
                                              : p->rp_id == CLAWB200_RP_ADVECTION3D_VC_FWAVE
                                              ? "aux array required: {u, v, w}"
                                              : "aux array required: the Riemann solver reads more aux components than maux");
    return 0;
}

// the 3-D steps (step3.cuh), one translation unit per solver: idir = 1, 2, 3 one split sweep, 0 unsplit
static int step3_dispatch(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                          const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st)
{
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS3D_VC: return claw_step3_acoustics(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
    case CLAWB200_RP_EULER3D: return claw_step3_euler(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
    case CLAWB200_RP_ADVECTION3D: return claw_step3_advection(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
    case CLAWB200_RP_ADVECTION3D_VC_FWAVE:
        return claw_step3_vc_advection_fwave(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
    default: return claw_step3_user(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
    }
}

extern "C" int clawb200_step3ds(const clawb200_problem *p, int mz, double dz, const double *q_in,
                                double *q_out, const double *aux, double dt, int idir,
                                double *cfl_dev, void *stream)
{
    int rc = check_problem(p, 3);
    if (rc) return rc;
    if ((rc = check_rp3(p, aux != nullptr))) return rc;
    if (p->method[5] > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for the 3-D sweeps");
    if (p->mbc < 2) return fail(CLAWB200_ERR_INVALID, "classic solvers need mbc >= 2");
    if (mz < 1 || !(dz > 0.0)) return fail(CLAWB200_ERR_INVALID, "mz, dz must be positive");
    if (q_in == q_out) return fail(CLAWB200_ERR_INVALID, "q_in and q_out must differ");
    if (idir < 1 || idir > 3) return fail(CLAWB200_ERR_INVALID, "idir must be 1, 2 or 3");
    const long long plane = (long long)p->pitch * (p->my + 2 * p->mbc);
    if (p->mstride < plane * (mz + 2 * p->mbc)) return fail(CLAWB200_ERR_INVALID, "mstride smaller than the padded field");
    // one launch over the whole padded field (step3.cuh): swept cells are updated, all others copied
    return step3_dispatch(p, mz, dz, q_in, q_out, aux, dt, idir, nullptr, cfl_dev, (cudaStream_t)stream);
}

// classic3.step3 (step3.f:2-594 + flux3.f:5-595; clawpack.py:680-682): the unsplit 3-D step.
// method[2] = 0 | 10 | 11 | 20 | 21 | 22 (ClawSolver3D.no_trans / trans_inc / trans_cor and the
// intermediate settings of flux3.f:42-68).  `scratch` holds clawb200_step3_scratch_doubles() doubles.
static int check_step3(const clawb200_problem *p, int mz, double dz, const double *aux)
{
    int rc = check_problem(p, 3);
    if (rc) return rc;
    if ((rc = check_rp3(p, aux != nullptr))) return rc;
    if (p->method[5] > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for the 3-D sweeps");
    if (p->mbc < 2) return fail(CLAWB200_ERR_INVALID, "classic solvers need mbc >= 2");
    if (mz < 1 || !(dz > 0.0)) return fail(CLAWB200_ERR_INVALID, "mz, dz must be positive");
    const int t = p->method[2];
    if (t < 0) return fail(CLAWB200_ERR_INVALID, "method[2] < 0 means dimensional splitting: call step3ds");
    if (t != 0 && t != 10 && t != 11 && t != 20 && t != 21 && t != 22)
        return fail(CLAWB200_ERR_INVALID, "method[2] must be one of 0, 10, 11, 20, 21, 22 (flux3.f:42-68)");
    if (t >= 20 && p->method[1] != 2)
        return fail(CLAWB200_ERR_INVALID, "method[2] = 20, 21, 22 propagate the correction waves: method[1] must be 2 (flux3.f:57-63)");
    const long long plane = (long long)p->pitch * (p->my + 2 * p->mbc);
    if (p->mstride < plane * (mz + 2 * p->mbc)) return fail(CLAWB200_ERR_INVALID, "mstride smaller than the padded field");
    return 0;
}

extern "C" long long clawb200_step3_scratch_doubles(const clawb200_problem *p)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    return claw_step3_scratch_doubles(p->meqn, p->mstride);
}

extern "C" int clawb200_step3(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                              const double *aux, double dt, double *scratch, double *cfl_dev, void *stream)
{
    int rc = check_step3(p, mz, dz, aux);
    if (rc) return rc;
    if (!qold || !qnew || !scratch) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (qold == qnew) return fail(CLAWB200_ERR_INVALID, "qold and qnew must differ");
    return step3_dispatch(p, mz, dz, qold, qnew, aux, dt, 0, scratch, cfl_dev, (cudaStream_t)stream);
}

__global__ void bc_kernel(double *q, long long mstride, int pitch, int narr, int nx, int ny,
                          int mbc, int idim, int side, int bctype, int negate);

// Ghost cells of a 3-D field, one side of one dimension (solver.py:384-452 in 3-D).
extern "C" int clawb200_bc_fill3(const clawb200_problem *p, int mz, double *q, int narr, int idim,
                                 int side, int bctype, int negate, void *stream)
{
    if (!p || !q) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (p->ndim != 3 || idim < 0 || idim > 2 || side < 0 || side > 1)
        return fail(CLAWB200_ERR_INVALID, "bad ndim/idim/side");
    if (bctype < CLAWB200_BC_OUTFLOW || bctype > CLAWB200_BC_REFLECTING)
        return fail(CLAWB200_ERR_INVALID, "bc_fill handles outflow, periodic and reflecting");
    const int mbc = p->mbc, nx = p->pitch, ny = p->my + 2 * mbc, nz = mz + 2 * mbc;
    const long long plane = (long long)nx * ny;
    cudaStream_t st = (cudaStream_t)stream;
    auto launch = [&](double *base, int pitch, int ex, int ey, int dim2) {
        const long long total = (long long)((dim2 == 0) ? ey : ex) * mbc * narr;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        if (blocks < 1) blocks = 1;
        bc_kernel<<<blocks, 256, 0, st>>>(base, p->mstride, pitch, narr, ex, ey, mbc, dim2, side, bctype, negate);
    };
    if (idim == 0) launch(q, nx, nx, ny * nz, 0);             // ghost columns of every (j, k) row
    else if (idim == 2) launch(q, (int)plane, (int)plane, nz, 1); // ghost planes: "rows" of nx*ny cells
    else
        for (int k = 0; k < nz; k++) launch(q + plane * k, nx, nx, ny, 1);
    CUDA_OK(cudaGetLastError());
    return 0;
}

static int step2_impl(const clawb200_problem *p, const double *qold, double *qnew, const double *aux,
                      double dt, int parts, int jlo, int jhi, double *cfl_dev, void *stream)
{
    int rc = check_problem(p, 2);
    if (rc) return rc;
    if ((rc = check_rp_shape(p))) return rc;
    if (p->mbc < 2) return fail(CLAWB200_ERR_INVALID, "classic solvers need mbc >= 2");
    if (qold == qnew) return fail(CLAWB200_ERR_INVALID, "qold and qnew must differ");
    if (p->method[2] < 0) return fail(CLAWB200_ERR_INVALID, "method[2] < 0 means dimensional splitting: call step2ds");
    if (parts < 1 || parts > 3) return fail(CLAWB200_ERR_INVALID, "parts must be 1, 2 or 3");
    if (jlo < 1 || jhi > p->my) return fail(CLAWB200_ERR_INVALID, "row range outside 1..my");
    if (jlo > jhi) return 0; // empty range
    if ((rc = check_aux(p, aux, true))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    SweepArgs A = make_args(p, qold, qnew, dt, cfl_dev, aux);
    A.ilo = 1; A.ihi = p->mx; A.jlo = jlo; A.jhi = jhi;
    const int nrows = jhi - jlo + 1;
    // both sweeps in one walk over q where a single-pass kernel exists (fused.cuh): q read once,
    // written once.  problem.step2_mode = 1 keeps the two sweep kernels.
    if (p->step2_mode < 0 || p->step2_mode > 2) return fail(CLAWB200_ERR_INVALID, "step2_mode must be 0, 1 or 2");
    if (parts == 3 && p->step2_mode != 1) {
        if (claw_fused_available(p->rp_id, A)) return claw_fused(p->rp_id, A, st);
        if (p->step2_mode == 2) return fail(CLAWB200_ERR_UNSUPPORTED, "no single-pass kernel for this solver / problem (step2_mode = 2)");
    }
    if (parts & 1) {
        A.rows_per_cta = pick_rows(nrows, (p->mx + XNT - 4) / (XNT - 3));
        if ((rc = dispatch_x<true>(p->rp_id, A, st))) return rc;
    }
    if (parts & 2) {
        A.rows_per_cta = pick_rows(nrows, (p->mx + YNT - 3) / (YNT - 2));
        if ((rc = dispatch_y<true>(p->rp_id, A, st))) return rc;
    }
    return 0;
}

extern "C" int clawb200_step2_parts(const clawb200_problem *p, const double *qold, double *qnew,
                                    const double *aux, double dt, int parts, double *cfl_dev,
                                    void *stream)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    return step2_impl(p, qold, qnew, aux, dt, parts, 1, p->my, cfl_dev, stream);
}

extern "C" int clawb200_step2_launches(const clawb200_problem *p)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    int rc = check_problem(p, 2);
    if (rc) return rc;
    if (p->step2_mode == 1) return 2;
    SweepArgs A = make_args(p, nullptr, nullptr, 0.0, nullptr, nullptr);
    return claw_fused_available(p->rp_id, A) ? 1 : 2;
}

extern "C" int clawb200_step2_rows(const clawb200_problem *p, const double *qold, double *qnew,
                                   const double *aux, double dt, int jlo, int jhi, double *cfl_dev,
                                   void *stream)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    return step2_impl(p, qold, qnew, aux, dt, 3, jlo, jhi, cfl_dev, stream);
}

extern "C" int clawb200_step2(const clawb200_problem *p, const double *qold, double *qnew,
                              const double *aux, double dt, double *cfl_dev, void *stream)
{
    return clawb200_step2_parts(p, qold, qnew, aux, dt, 3, cfl_dev, stream);
}

// ---------------------------------------------------------------------------
// Boundary conditions (solver.py:384-452).  One launch per side; the ordering over
// sides (dim 0 lower, dim 0 upper, dim 1 lower, dim 1 upper) is the caller's, so
// that custom (user) conditions can be interleaved exactly like the reference does.
// ---------------------------------------------------------------------------
__global__ void bc_kernel(double *q, long long mstride, int pitch, int narr, int nx, int ny,
                          int mbc, int idim, int side, int bctype, int negate)
{
    // ghost layer g = 0..mbc-1 counted from the outside for `lower`, from the inside..
    const int len = (idim == 0) ? ny : nx; // extent along the boundary
    const long long total = (long long)len * mbc * narr;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < total;
         id += (long long)gridDim.x * blockDim.x) {
        int a, g, m;
        if (idim == 0) { // ghost columns: vary j fastest is uncoalesced either way; keep g fastest
            g = (int)(id % mbc);
            a = (int)((id / mbc) % len);
            m = (int)(id / ((long long)mbc * len));
        } else { // ghost rows: i fastest (coalesced)
            a = (int)(id % len);
            g = (int)((id / len) % mbc);
            m = (int)(id / ((long long)mbc * len));
        }
        const int n = (idim == 0) ? nx : ny; // extent across the boundary (padded)
        int dst, src;
        double sign = 1.0;
        if (side == 0) {
            dst = g;
            if (bctype == CLAWB200_BC_OUTFLOW) src = mbc;
            else if (bctype == CLAWB200_BC_PERIODIC) src = n - 2 * mbc + g;
            else { src = 2 * mbc - 1 - g; if (m == negate) sign = -1.0; }
        } else {
            dst = n - 1 - g;
            if (bctype == CLAWB200_BC_OUTFLOW) src = n - mbc - 1;
            else if (bctype == CLAWB200_BC_PERIODIC) src = mbc + (mbc - 1 - g);
            else { src = n - 2 * mbc + g; if (m == negate) sign = -1.0; }
        }
        long long od, os;
        if (idim == 0) { od = (long long)a * pitch + dst; os = (long long)a * pitch + src; }
        else { od = (long long)dst * pitch + a; os = (long long)src * pitch + a; }
        double v = q[m * mstride + os];
        q[m * mstride + od] = (sign < 0.0) ? -v : v;
    }
}

extern "C" int clawb200_bc_fill(const clawb200_problem *p, double *q, int narr, int idim,
                                int side, int bctype, int negate, void *stream)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    if (idim < 0 || idim >= p->ndim || side < 0 || side > 1)
        return fail(CLAWB200_ERR_INVALID, "bad idim/side");
    if (bctype < CLAWB200_BC_OUTFLOW || bctype > CLAWB200_BC_REFLECTING)
        return fail(CLAWB200_ERR_INVALID, "bc_fill handles outflow, periodic and reflecting only");
    int nx = p->mx + 2 * p->mbc;
    int ny = (p->ndim > 1) ? p->my + 2 * p->mbc : 1;
    long long total = (long long)((idim == 0) ? ny : nx) * p->mbc * narr;
    int threads = 256;
    int blocks = (int)((total + threads - 1) / threads);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    bc_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(q, p->mstride, p->pitch, narr, nx, ny,
                                                            p->mbc, idim, side, bctype, negate);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------
// Layout converters (tiled transposes through shared memory): the reference's host
// layout has the component index fastest, the device layout has i fastest.
// ---------------------------------------------------------------------------
template <bool TO_SOA>
__global__ void layout_kernel(const double *src, double *dst, int ncomp, int nx, int ny,
                              long long mstride, int pitch)
{
    // one CTA converts 128 consecutive cells of one row
    extern __shared__ double tile[]; // [ncomp][129]
    const int j = blockIdx.y;
    const int ibase = blockIdx.x * 128;
    const int ncell = min(128, nx - ibase);
    const long long aos0 = ((long long)j * nx + ibase) * ncomp;
    if (TO_SOA) {
        for (int e = threadIdx.x; e < ncell * ncomp; e += blockDim.x)
            tile[(e % ncomp) * 129 + e / ncomp] = src[aos0 + e];
        __syncthreads();
        for (int e = threadIdx.x; e < ncell * ncomp; e += blockDim.x) {
            int m = e / ncell, c = e % ncell;
            dst[m * mstride + (long long)j * pitch + ibase + c] = tile[m * 129 + c];
        }
    } else {
        for (int e = threadIdx.x; e < ncell * ncomp; e += blockDim.x) {
            int m = e / ncell, c = e % ncell;
            tile[m * 129 + c] = src[m * mstride + (long long)j * pitch + ibase + c];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < ncell * ncomp; e += blockDim.x)
            dst[aos0 + e] = tile[(e % ncomp) * 129 + e / ncomp];
    }
}

extern "C" int clawb200_aos_to_soa(const double *aos, double *soa, int ncomp, int nx, int ny,
                                   long long mstride, int pitch, void *stream)
{
    if (ncomp < 1 || ncomp > 32) return fail(CLAWB200_ERR_INVALID, "ncomp out of range");
    dim3 grid((nx + 127) / 128, ny);
    layout_kernel<true><<<grid, 128, sizeof(double) * ncomp * 129, (cudaStream_t)stream>>>(
        aos, soa, ncomp, nx, ny, mstride, pitch);
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int clawb200_soa_to_aos(const double *soa, double *aos, int ncomp, int nx, int ny,
                                   long long mstride, int pitch, void *stream)
{
    if (ncomp < 1 || ncomp > 32) return fail(CLAWB200_ERR_INVALID, "ncomp out of range");
    dim3 grid((nx + 127) / 128, ny);
    layout_kernel<false><<<grid, 128, sizeof(double) * ncomp * 129, (cudaStream_t)stream>>>(
        soa, aos, ncomp, nx, ny, mstride, pitch);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------
// Halo pack / unpack for the y-slab partition
// ---------------------------------------------------------------------------
template <bool PACK>
__global__ void halo_kernel(double *q, double *buf, long long mstride, int pitch, int nx, int narr,
                            int row0, int nrows)
{
    const long long total = (long long)narr * nrows * nx;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < total;
         id += (long long)gridDim.x * blockDim.x) {
        int i = (int)(id % nx);
        int r = (int)((id / nx) % nrows);
        int m = (int)(id / ((long long)nx * nrows));
        long long qi = m * mstride + (long long)(row0 + r) * pitch + i;
        if (PACK) buf[id] = q[qi];
        else q[qi] = buf[id];
    }
}

extern "C" int clawb200_halo_pack(const clawb200_problem *p, const double *q, int narr, int row0,
                                  int nrows, double *buf, void *stream)
{
    int nx = p->mx + 2 * p->mbc;
    long long total = (long long)narr * nrows * nx;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 4) blocks = 148 * 4;
    halo_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>((double *)q, buf, p->mstride, p->pitch,
                                                                nx, narr, row0, nrows);
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int clawb200_halo_unpack(const clawb200_problem *p, double *q, int narr, int row0,
                                    int nrows, const double *buf, void *stream)
{
    int nx = p->mx + 2 * p->mbc;
    long long total = (long long)narr * nrows * nx;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 4) blocks = 148 * 4;
    halo_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(q, (double *)buf, p->mstride, p->pitch,
                                                                 nx, narr, row0, nrows);
    CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int clawb200_sharpclaw_stage(const clawb200_problem *p, const double *q, const double *qa,
                                        double *out, double *dq_out, const double *aux, double dt,
                                        int mode, double ca, double cb, double div,
                                        double *cfl_dev, void *stream)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    if (p->ndim == 3) return fail(CLAWB200_ERR_INVALID, "3-D problem: the 3-D SharpClaw stage is clawb200_sharpclaw_stage3");
    int rc = check_problem(p, p->ndim);
    if (rc) return rc;
    if ((rc = check_rp_shape(p))) return rc;
    if (p->mbc < 3) return fail(CLAWB200_ERR_INVALID, "WENO5 needs mbc >= 3");
    if (mode < 0 || mode > 3) return fail(CLAWB200_ERR_INVALID, "bad stage mode");
    if ((mode == 1 || mode == 2) && !qa) return fail(CLAWB200_ERR_INVALID, "this stage mode needs qa");
    if (out == q) return fail(CLAWB200_ERR_INVALID, "out must not alias q");
    if ((rc = check_aux(p, aux, false))) return rc;
    return sharpclaw_launch(p, q, qa, out, dq_out, dt, mode, ca, cb, div, cfl_dev, (cudaStream_t)stream, aux);
}

extern "C" int clawb200_sharpclaw_stage3(const clawb200_problem *p, int mz, double dz, const double *q,
                                         const double *qa, double *out, double *dq_out, const double *aux,
                                         double dt, int mode, double ca, double cb, double div,
                                         double *cfl_dev, void *stream)
{
    int rc = check_problem(p, 3);
    if (rc) return rc;
    if ((rc = check_rp3(p, aux != nullptr))) return rc;
    if (p->method[5] > 0) return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa (capacity function) is not compiled for the 3-D SharpClaw stage");
    const int wv = p->weno_variant;
    if (wv == CLAWB200_WENO_TABLES) return fail(CLAWB200_ERR_UNSUPPORTED, "WENO orders above 5 are not compiled in 3-D");
    if (wv != CLAWB200_WENO_PYWENO_F32 && wv != CLAWB200_WENO_PYWENO_F64 && wv != CLAWB200_WENO_OLD && wv != CLAWB200_RECON_TVD2)
        return fail(CLAWB200_ERR_UNSUPPORTED, "3-D SharpClaw: weno_variant must be PyWENO (f32 / f64), the hand-written weno5 or tvd2");
    if (p->mbc < 3) return fail(CLAWB200_ERR_INVALID, "WENO5 needs mbc >= 3");
    if (mz < 1 || !(dz > 0.0)) return fail(CLAWB200_ERR_INVALID, "mz, dz must be positive");
    if (mode < 0 || mode > 3) return fail(CLAWB200_ERR_INVALID, "bad stage mode");
    if ((mode == 1 || mode == 2) && !qa) return fail(CLAWB200_ERR_INVALID, "this stage mode needs qa");
    if (mode == 3 && !dq_out) return fail(CLAWB200_ERR_INVALID, "stage mode 3 needs dq_out in 3-D");
    if (mode != 3 && !out) return fail(CLAWB200_ERR_INVALID, "this stage mode needs out");
    if (!q || out == q || dq_out == q) return fail(CLAWB200_ERR_INVALID, "out and dq_out must not alias q");
    if ((qa && (qa == out || qa == dq_out)) || (out && out == dq_out))
        return fail(CLAWB200_ERR_INVALID, "out, dq_out and qa must be different buffers (the x/y partial of dq is held in one of them)");
    const long long plane = (long long)p->pitch * (p->my + 2 * p->mbc);
    if (p->mstride < plane * (mz + 2 * p->mbc)) return fail(CLAWB200_ERR_INVALID, "mstride smaller than the padded field");
    if (mz + 2 > 65535) return fail(CLAWB200_ERR_UNSUPPORTED, "mz must be below 65534");
    return sharpclaw_launch3(p, mz, dz, q, qa, out, dq_out, dt, mode, ca, cb, div, cfl_dev, (cudaStream_t)stream, aux);
}

// ---------------------------------------------------------------------------
// apps/shallow-sphere/src2.f:2-147 as one pointwise kernel: tangent-plane projection,
// 4-stage Runge-Kutta on the Coriolis term, projection again.  The radial unit vector that
// src2.f recomputes with mapc2p at every call is aux(14:16) (same function of the same
// arguments, bit for bit).  Interior cells only.
// ---------------------------------------------------------------------------
__global__ void sphere_src2_kernel(double *__restrict__ q, const double *__restrict__ aux,
                                   long long mstride, int pitch, int mx, int my, int mbc, double dt, double df)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    if (i >= mx || j >= my) return;
    const long long o = (long long)(j + mbc) * pitch + (i + mbc);
    const double erx = aux[13 * mstride + o], ery = aux[14 * mstride + o], erz = aux[15 * mstride + o];
    double q2 = q[1 * mstride + o], q3 = q[2 * mstride + o], q4 = q[3 * mstride + o];
    double qn = erx * q2 + ery * q3 + erz * q4;
    q2 = q2 - qn * erx;
    q3 = q3 - qn * ery;
    q4 = q4 - qn * erz;
    const double fcor = df * erz;
    double RK[4][3];
    double hu = q2, hv = q3, hw = q4;
#pragma unroll
    for (int st = 0; st < 4; st++) {
        if (st > 0) {
            hu = q2 + 0.5 * RK[st - 1][0];
            hv = q3 + 0.5 * RK[st - 1][1];
            hw = q4 + 0.5 * RK[st - 1][2];
        }
        RK[st][0] = fcor * dt * (erz * hv - ery * hw);
        RK[st][1] = dt * fcor * (erx * hw - erz * hu);
        RK[st][2] = dt * fcor * (ery * hu - erx * hv);
    }
    q2 = q2 + (RK[0][0] + 2.0 * RK[1][0] + 2.0 * RK[2][0] + RK[3][0]) / 6.0;
    q3 = q3 + (RK[0][1] + 2.0 * RK[1][1] + 2.0 * RK[2][1] + RK[3][1]) / 6.0;
    q4 = q4 + (RK[0][2] + 2.0 * RK[1][2] + 2.0 * RK[2][2] + RK[3][2]) / 6.0;
    qn = erx * q2 + ery * q3 + erz * q4;
    q[1 * mstride + o] = q2 - qn * erx;
    q[2 * mstride + o] = q3 - qn * ery;
    q[3 * mstride + o] = q4 - qn * erz;
}

extern "C" int clawb200_sphere_src2(const clawb200_problem *p, double *q, const double *aux, double dt,
                                    void *stream)
{
    if (!p || !q || !aux) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (p->ndim != 2 || p->meqn != 4 || p->maux < 16)
        return fail(CLAWB200_ERR_INVALID, "sphere_src2 needs the 4-equation, 16-aux sphere problem");
    dim3 grid((p->mx + 127) / 128, p->my);
    sphere_src2_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(q, aux, p->mstride, p->pitch, p->mx, p->my,
                                                               p->mbc, dt, (double)12.600576e0f);
    CUDA_OK(cudaGetLastError());
    return 0;
}

__global__ void ssp104_combine_kernel(const double *__restrict__ q, double *__restrict__ s1,
                                      double *__restrict__ s2, long long n, double c925)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        double a = s1[i];
        double b = q[i] / 25. + c925 * a;
        s2[i] = b;
        s1[i] = 15. * b - 5. * a;
    }
}

extern "C" int clawb200_ssp104_combine(const double *q, double *s1, double *s2, long long n, void *stream)
{
    if (!q || !s1 || !s2 || n < 0) return fail(CLAWB200_ERR_INVALID, "bad argument");
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    ssp104_combine_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(q, s1, s2, n, 9. / 25);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------
// Host-pointer entry points: same kernels behind the reference's f2py signatures.
// ---------------------------------------------------------------------------
struct HostScratch {
    double *d_aos = nullptr, *d_a = nullptr, *d_b = nullptr, *d_c = nullptr, *d_cfl = nullptr;
    double *d_aux = nullptr;
    double *d_tab = nullptr; // WENO coefficient table of the current host call
    size_t aux_cap = 0;
    int ensure_aux(size_t n)
    {
        if (n > aux_cap) {
            cudaFree(d_aux);
            d_aux = nullptr; aux_cap = 0;
            CUDA_OK(cudaMalloc(&d_aux, n * sizeof(double)));
            aux_cap = n;
        }
        return 0;
    }
    double *h_cfl = nullptr;
    size_t cap = 0;
    cudaStream_t st = nullptr;
    int ensure(size_t n)
    {
        if (!st) {
            CUDA_OK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
            CUDA_OK(cudaMalloc(&d_cfl, 16 * sizeof(double)));
            CUDA_OK(cudaMallocHost(&h_cfl, 16 * sizeof(double)));
        }
        if (n > cap) {
            cudaFree(d_aos); cudaFree(d_a); cudaFree(d_b); cudaFree(d_c);
            d_aos = d_a = d_b = d_c = nullptr; cap = 0;
            CUDA_OK(cudaMalloc(&d_aos, n * sizeof(double)));
            CUDA_OK(cudaMalloc(&d_a, n * sizeof(double)));
            CUDA_OK(cudaMalloc(&d_b, n * sizeof(double)));
            CUDA_OK(cudaMalloc(&d_c, n * sizeof(double)));
            cap = n;
        }
        return 0;
    }
};
static thread_local HostScratch g_hs;

static clawb200_problem host_layout(const clawb200_problem *p)
{
    clawb200_problem P = *p;
    P.dt_dev = nullptr;
    int nx = p->mx + 2 * p->mbc;
    int ny = (p->ndim > 1) ? p->my + 2 * p->mbc : 1;
    P.pitch = nx;
    P.mstride = (long long)nx * ny;
    if (p->ndim == 1) P.my = 1;
    return P;
}

static int check_problem_host(const clawb200_problem *p)
{
    clawb200_problem P = host_layout(p);
    int rc = check_problem(&P, 2);
    if (rc) return rc;
    return check_rp_shape(&P);
}

static int host_upload(const clawb200_problem &P, const double *h, double *d_soa)
{
    int nx = P.pitch, ny = (int)(P.mstride / P.pitch);
    size_t n = (size_t)P.meqn * nx * ny;
    CUDA_OK(cudaMemcpyAsync(g_hs.d_aos, h, n * sizeof(double), cudaMemcpyHostToDevice, g_hs.st));
    return clawb200_aos_to_soa(g_hs.d_aos, d_soa, P.meqn, nx, ny, P.mstride, P.pitch, g_hs.st);
}
// aux(maux, nx, ny) host array -> device SoA with the component stride of q
static int host_upload_aux(const clawb200_problem &P, const double *h_aux, const double **d_aux)
{
    *d_aux = nullptr;
    if (!h_aux || P.maux <= 0) return 0;
    int nx = P.pitch, ny = (int)(P.mstride / P.pitch);
    size_t n = (size_t)P.maux * nx * ny;
    if (n > g_hs.cap) return fail(CLAWB200_ERR_INVALID, "internal: scratch not sized for aux");
    int rc;
    if ((rc = g_hs.ensure_aux(n))) return rc;
    CUDA_OK(cudaMemcpyAsync(g_hs.d_aos, h_aux, n * sizeof(double), cudaMemcpyHostToDevice, g_hs.st));
    if ((rc = clawb200_aos_to_soa(g_hs.d_aos, g_hs.d_aux, P.maux, nx, ny, P.mstride, P.pitch, g_hs.st))) return rc;
    *d_aux = g_hs.d_aux;
    return 0;
}

static int host_download(const clawb200_problem &P, const double *d_soa, double *h)
{
    int nx = P.pitch, ny = (int)(P.mstride / P.pitch);
    size_t n = (size_t)P.meqn * nx * ny;
    int rc = clawb200_soa_to_aos(d_soa, g_hs.d_aos, P.meqn, nx, ny, P.mstride, P.pitch, g_hs.st);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(h, g_hs.d_aos, n * sizeof(double), cudaMemcpyDeviceToHost, g_hs.st));
    return 0;
}
static int host_finish(double *cfl, int slot = 0)
{
    CUDA_OK(cudaMemcpyAsync(g_hs.h_cfl, g_hs.d_cfl, 16 * sizeof(double), cudaMemcpyDeviceToHost, g_hs.st));
    CUDA_OK(cudaStreamSynchronize(g_hs.st));
    if (cfl) *cfl = g_hs.h_cfl[slot];
    return 0;
}

// ---------------------------------------------------------------------------
// Slab pipeline for the host-pointer entry points.  A full-field H2D copy, the sweeps and a
// full-field D2H copy in sequence leave both PCIe directions idle two thirds of the time.
// The grid is cut into row slabs (the reference's arrays have j slowest, so a slab of rows
// is one contiguous chunk of the host array); slab k is uploaded while slab k-1 is computed
// and slab k-2 is downloaded, on three streams.  Each slab is an independent sub-problem
// with its own mbc ghost rows taken from the caller's qold -- exactly the slab partition of
// the multi-GPU path, so results are bit-identical to the single-pass call.
// ---------------------------------------------------------------------------
struct SlabPipe {
    static constexpr int NBUF = 3;
    double *d_in_aos[NBUF] = {}, *d_in[NBUF] = {}, *d_out[NBUF] = {}, *d_out_aos[NBUF] = {};
    size_t cap = 0;
    cudaStream_t s_in = nullptr, s_cmp = nullptr, s_out = nullptr;
    cudaEvent_t e_in[NBUF] = {}, e_cmp[NBUF] = {}, e_out[NBUF] = {};
    int ensure(size_t n)
    {
        if (!s_in) {
            CUDA_OK(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
            CUDA_OK(cudaStreamCreateWithFlags(&s_cmp, cudaStreamNonBlocking));
            CUDA_OK(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
            for (int b = 0; b < NBUF; b++) {
                CUDA_OK(cudaEventCreateWithFlags(&e_in[b], cudaEventDisableTiming));
                CUDA_OK(cudaEventCreateWithFlags(&e_cmp[b], cudaEventDisableTiming));
                CUDA_OK(cudaEventCreateWithFlags(&e_out[b], cudaEventDisableTiming));
            }
        }
        if (n > cap) {
            for (int b = 0; b < NBUF; b++) {
                cudaFree(d_in_aos[b]); cudaFree(d_in[b]); cudaFree(d_out[b]); cudaFree(d_out_aos[b]);
                d_in_aos[b] = d_in[b] = d_out[b] = d_out_aos[b] = nullptr;
            }
            cap = 0;
            for (int b = 0; b < NBUF; b++) {
                CUDA_OK(cudaMalloc(&d_in_aos[b], n * sizeof(double)));
                CUDA_OK(cudaMalloc(&d_in[b], n * sizeof(double)));
                CUDA_OK(cudaMalloc(&d_out[b], n * sizeof(double)));
                CUDA_OK(cudaMalloc(&d_out_aos[b], n * sizeof(double)));
            }
            cap = n;
        }
        return 0;
    }
};
static thread_local SlabPipe g_pipe;

// mode 0: unsplit step2 ; mode 1: step2ds x-sweeps (ids = 1) ; mode 2: step2ds y-sweeps (ids = 2).
// `p` is the full problem (host layout).  qnew_init: the caller's qnew (cells the sweep does not
// touch keep these values); it may alias qold.
static int host_pipeline(const clawb200_problem *p, const double *qold, double *qnew, double dt,
                         int mode, double *cfl)
{
    const int mbc = p->mbc, meqn = p->meqn;
    const int nx = p->mx + 2 * mbc;
    const int ny_tot = p->my + 2 * mbc;
    const size_t rowd = (size_t)nx * meqn; // doubles per padded row of the host array
    // rows this call produces, in padded (0-based) row numbers
    const int out0 = (mode == 1) ? 0 : mbc;
    const int out1 = (mode == 1) ? ny_tot : mbc + p->my;
    const int halo = (mode == 1) ? 0 : mbc; // input rows needed beyond the output rows
    // slab height: PCIe time is the bound, the first upload and the last download are the only
    // transfers that do not overlap, so slabs are kept small
    constexpr int slab_rows = 128;
    const int nout = out1 - out0;
    int nslab = (nout + slab_rows - 1) / slab_rows;
    if (nslab < 1) nslab = 1;
    // Slab k produces rows out0 + [k nout / nslab, (k + 1) nout / nslab): every slab has
    // floor(nout / nslab) or ceil(nout / nslab) rows, at least 64 for the grids sent here: a
    // mode-1 slab presents its first and last mbc rows as ghost rows and needs interior rows besides.
    const int rows_min = nout / nslab, rows_max = (nout + nslab - 1) / nslab;
    if ((mode == 1 ? rows_min - 2 * mbc : rows_min) < 1)
        return fail(CLAWB200_ERR_INVALID, "internal: host pipeline slab without interior rows");
    const size_t nmax = rowd * (size_t)(rows_max + 2 * mbc);
    int rc = g_hs.ensure(16);
    if (rc) return rc;
    if ((rc = g_pipe.ensure(nmax))) return rc;
    SlabPipe &S = g_pipe;
    CUDA_OK(cudaMemsetAsync(g_hs.d_cfl, 0, sizeof(double), S.s_cmp));
    int prev_r0 = 0, prev_off = 0, prev_n = 0, last = -1;
    for (int k = 0; k < nslab; k++) {
        const int b = k % SlabPipe::NBUF;
        const int r0 = out0 + (int)((long long)k * nout / nslab);
        const int r1 = out0 + (int)((long long)(k + 1) * nout / nslab);
        const int in0 = r0 - halo, in1 = r1 + halo; // input rows [in0, in1)
        const int nrow_in = in1 - in0;
        // the slab as a stand-alone problem in device layout
        clawb200_problem P = *p;
        P.dt_dev = nullptr;
        P.pitch = nx;
        P.my = (mode == 1) ? nrow_in - 2 * mbc : r1 - r0;
        P.mstride = (long long)nx * nrow_in;
        const size_t nd = rowd * (size_t)nrow_in;
        // buffer b is free once the download of slab k-NBUF has completed
        if (k >= SlabPipe::NBUF) {
            CUDA_OK(cudaStreamWaitEvent(S.s_in, S.e_out[b], 0));
            CUDA_OK(cudaStreamWaitEvent(S.s_cmp, S.e_out[b], 0));
        }
        CUDA_OK(cudaMemcpyAsync(S.d_in_aos[b], qold + rowd * (size_t)in0, nd * sizeof(double),
                                cudaMemcpyHostToDevice, S.s_in));
        CUDA_OK(cudaEventRecord(S.e_in[b], S.s_in));
        CUDA_OK(cudaStreamWaitEvent(S.s_cmp, S.e_in[b], 0));
        if ((rc = clawb200_aos_to_soa(S.d_in_aos[b], S.d_in[b], meqn, nx, nrow_in, P.mstride, nx, S.s_cmp))) return rc;
        // step2.f:8-9 / step2ds.f: "on entry, qold and qnew should be identical": cells the
        // sweep does not touch are taken from qold
        CUDA_OK(cudaMemcpyAsync(S.d_out[b], S.d_in[b], nd * sizeof(double), cudaMemcpyDeviceToDevice, S.s_cmp));
        if (mode == 0) {
            rc = clawb200_step2(&P, S.d_in[b], S.d_out[b], nullptr, dt, g_hs.d_cfl, S.s_cmp);
        } else if (mode == 2) {
            rc = clawb200_step2ds(&P, S.d_in[b], S.d_out[b], nullptr, dt, 2, g_hs.d_cfl, S.s_cmp);
        } else {
            // x-sweeps over every row of the slab: present the rows as ghost + interior rows
            // of a problem whose padded height is the slab height
            rc = clawb200_step2ds(&P, S.d_in[b], S.d_out[b], nullptr, dt, 1, g_hs.d_cfl, S.s_cmp);
        }
        if (rc) return rc;
        if ((rc = clawb200_soa_to_aos(S.d_out[b], S.d_out_aos[b], meqn, nx, nrow_in, P.mstride, nx, S.s_cmp))) return rc;
        CUDA_OK(cudaEventRecord(S.e_cmp[b], S.s_cmp));
        // Download the output rows of the PREVIOUS slab now, after this slab's upload has been
        // issued: with qold == qnew (the reference's aliased step2ds call) the upload of slab
        // k reads rows that the download of slab k-1 overwrites.
        if (k > 0) {
            const int pb = (k - 1) % SlabPipe::NBUF;
            CUDA_OK(cudaStreamWaitEvent(S.s_out, S.e_in[b], 0));
            CUDA_OK(cudaStreamWaitEvent(S.s_out, S.e_cmp[pb], 0));
            CUDA_OK(cudaMemcpyAsync(qnew + rowd * (size_t)prev_r0, S.d_out_aos[pb] + rowd * (size_t)prev_off,
                                    rowd * (size_t)prev_n * sizeof(double), cudaMemcpyDeviceToHost, S.s_out));
            CUDA_OK(cudaEventRecord(S.e_out[pb], S.s_out));
        }
        prev_r0 = r0; prev_off = r0 - in0; prev_n = r1 - r0; last = k;
    }
    if (last >= 0) {
        const int pb = last % SlabPipe::NBUF;
        CUDA_OK(cudaStreamWaitEvent(S.s_out, S.e_cmp[pb], 0));
        CUDA_OK(cudaMemcpyAsync(qnew + rowd * (size_t)prev_r0, S.d_out_aos[pb] + rowd * (size_t)prev_off,
                                rowd * (size_t)prev_n * sizeof(double), cudaMemcpyDeviceToHost, S.s_out));
        CUDA_OK(cudaEventRecord(S.e_out[pb], S.s_out));
    }
    CUDA_OK(cudaMemcpyAsync(g_hs.h_cfl, g_hs.d_cfl, sizeof(double), cudaMemcpyDeviceToHost, S.s_cmp));
    CUDA_OK(cudaStreamSynchronize(S.s_cmp));
    CUDA_OK(cudaStreamSynchronize(S.s_out));
    CUDA_OK(cudaStreamSynchronize(S.s_in));
    if (cfl) *cfl = g_hs.h_cfl[0];
    return 0;
}

// The host entry points keep device scratch (buffers, streams, events) per calling thread and
// reuse it from call to call; this releases all of it (the next host call allocates afresh).
extern "C" int clawb200_release_host_scratch(void)
{
    HostScratch &h = g_hs;
    if (h.st) cudaStreamSynchronize(h.st);
    cudaFree(h.d_aos); cudaFree(h.d_a); cudaFree(h.d_b); cudaFree(h.d_c); cudaFree(h.d_cfl);
    cudaFree(h.d_aux); cudaFree(h.d_tab);
    if (h.h_cfl) cudaFreeHost(h.h_cfl);
    if (h.st) cudaStreamDestroy(h.st);
    h = HostScratch();
    SlabPipe &S = g_pipe;
    if (S.s_in) {
        cudaStreamSynchronize(S.s_in); cudaStreamSynchronize(S.s_cmp); cudaStreamSynchronize(S.s_out);
        for (int b = 0; b < SlabPipe::NBUF; b++) {
            cudaFree(S.d_in_aos[b]); cudaFree(S.d_in[b]); cudaFree(S.d_out[b]); cudaFree(S.d_out_aos[b]);
            cudaEventDestroy(S.e_in[b]); cudaEventDestroy(S.e_cmp[b]); cudaEventDestroy(S.e_out[b]);
        }
        cudaStreamDestroy(S.s_in); cudaStreamDestroy(S.s_cmp); cudaStreamDestroy(S.s_out);
    }
    S = SlabPipe();
    return 0;
}

extern "C" int clawb200_step1_host(const clawb200_problem *p, double *q, const double *aux,
                                   double dt, double *cfl)
{
    if (!p || !q) return fail(CLAWB200_ERR_INVALID, "null argument");
    clawb200_problem P = host_layout(p);
    size_t n = (size_t)P.meqn * P.mstride;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, q, g_hs.d_a))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    // cells outside 1..mx keep their input values (the Fortran also updates cells 0 and
    // mx+1, which no caller reads: clawpack.py:406 keeps q[:, mbc:-mbc] only)
    CUDA_OK(cudaMemcpyAsync(g_hs.d_b, g_hs.d_a, n * sizeof(double), cudaMemcpyDeviceToDevice, g_hs.st));
    if ((rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = clawb200_step1(&P, g_hs.d_a, g_hs.d_b, d_aux, dt, g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = host_download(P, g_hs.d_b, q))) return rc;
    return host_finish(cfl);
}

extern "C" int clawb200_step2ds_host(const clawb200_problem *p, const double *qold, double *qnew,
                                     const double *aux, double dt, int ids, double *cfl)
{
    if (!p || !qold || !qnew) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (!aux && p->ndim == 2 && p->method[5] == 0 && p->rp_id != CLAWB200_RP_SPHERE && p->my >= 1024 &&
        (ids == 1 || ids == 2)) {
        int rc0 = check_problem_host(p);
        if (rc0) return rc0;
        return host_pipeline(p, qold, qnew, dt, ids, cfl);
    }
    clawb200_problem P = host_layout(p);
    size_t n = (size_t)P.meqn * P.mstride;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, qold, g_hs.d_a))) return rc;
    // step2ds.f:9-10: "on entry, qold and qnew should be identical" -- cells the sweep does
    // not touch are taken from qold (qnew is not uploaded)
    CUDA_OK(cudaMemcpyAsync(g_hs.d_b, g_hs.d_a, n * sizeof(double), cudaMemcpyDeviceToDevice, g_hs.st));
    if ((rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    if ((rc = clawb200_step2ds(&P, g_hs.d_a, g_hs.d_b, d_aux, dt, ids, g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = host_download(P, g_hs.d_b, qnew))) return rc;
    return host_finish(cfl);
}

extern "C" int clawb200_step2_host(const clawb200_problem *p, const double *qold, double *qnew,
                                   const double *aux, double dt, double *cfl)
{
    if (!p || !qold || !qnew) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (!aux && p->ndim == 2 && p->method[5] == 0 && p->rp_id != CLAWB200_RP_SPHERE && p->my >= 1024) {
        int rc0 = check_problem_host(p);
        if (rc0) return rc0;
        return host_pipeline(p, qold, qnew, dt, 0, cfl);
    }
    clawb200_problem P = host_layout(p);
    size_t n = (size_t)P.meqn * P.mstride;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, qold, g_hs.d_a))) return rc;
    CUDA_OK(cudaMemcpyAsync(g_hs.d_b, g_hs.d_a, n * sizeof(double), cudaMemcpyDeviceToDevice, g_hs.st));
    if ((rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    if ((rc = clawb200_step2(&P, g_hs.d_a, g_hs.d_b, d_aux, dt, g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = host_download(P, g_hs.d_b, qnew))) return rc;
    return host_finish(cfl);
}

extern "C" int clawb200_sharpclaw_dq_host(const clawb200_problem *p, const double *q, double *dq,
                                          const double *aux, double dt, double *cfl)
{
    if (!p || !q || !dq) return fail(CLAWB200_ERR_INVALID, "null argument");
    clawb200_problem P = host_layout(p);
    size_t n = (size_t)P.meqn * P.mstride;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, q, g_hs.d_a))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    CUDA_OK(cudaMemsetAsync(g_hs.d_b, 0, n * sizeof(double), g_hs.st));
    if ((rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st))) return rc;
    if (P.weno_variant == CLAWB200_WENO_TABLES && P.weno_tab) { // host table -> device scratch
        const size_t nb = (size_t)clawb200_weno_table_doubles() * sizeof(double);
        if (!g_hs.d_tab) CUDA_OK(cudaMalloc(&g_hs.d_tab, nb));
        CUDA_OK(cudaMemcpyAsync(g_hs.d_tab, P.weno_tab, nb, cudaMemcpyHostToDevice, g_hs.st));
        P.weno_tab = g_hs.d_tab;
    }
    if ((rc = clawb200_sharpclaw_stage(&P, g_hs.d_a, nullptr, nullptr, g_hs.d_b, d_aux, dt,
                                       CLAWB200_STAGE_DQ_ONLY, 0.0, 0.0, 1.0, g_hs.d_cfl, g_hs.st)))
        return rc;
    if ((rc = host_download(P, g_hs.d_b, dq))) return rc;
    return host_finish(cfl);
}

// ---------------------------------------------------------------------------
// Riemann solvers as pointwise operators (rp_point.cu)
// ---------------------------------------------------------------------------
static int check_rp_point(const clawb200_problem *p, int ixy, long long n)
{
    if (!p) return fail(CLAWB200_ERR_INVALID, "null problem");
    if (n < 0) return fail(CLAWB200_ERR_INVALID, "negative n");
    if (p->ndim == 2 && ixy != 1 && ixy != 2) return fail(CLAWB200_ERR_INVALID, "ixy must be 1 or 2");
    if (p->ndim == 3) {
        if (ixy < 1 || ixy > 3) return fail(CLAWB200_ERR_INVALID, "ixy must be 1, 2 or 3");
        return check_rp3(p, true); // rp_point.cu checks auxl / auxr
    }
    if (p->ndim != 1 && p->ndim != 2) return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: 1-D, 2-D and 3-D solvers");
    return check_rp_shape(p);
}

extern "C" int clawb200_rp_solve(const clawb200_problem *p, int ixy, long long n, const double *ql,
                                 const double *qr, const double *auxl, const double *auxr, double *wave,
                                 double *s, double *amdq, double *apdq, void *stream)
{
    int rc = check_rp_point(p, ixy, n);
    if (rc) return rc;
    if (!ql || !qr || !wave || !s || !amdq || !apdq) return fail(CLAWB200_ERR_INVALID, "null argument");
    return claw_rp_point(p, ixy, n, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr,
                         (cudaStream_t)stream);
}

extern "C" int clawb200_rp_transverse(const clawb200_problem *p, int ixy, long long n, const double *ql,
                                      const double *qr, int imp, const double *asdq, double *bmasdq,
                                      double *bpasdq, void *stream)
{
    int rc = check_rp_point(p, ixy, n);
    if (rc) return rc;
    if (!ql || !qr || !asdq || !bmasdq || !bpasdq) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (imp != 1 && imp != 2) return fail(CLAWB200_ERR_INVALID, "imp must be 1 or 2");
    if (p->ndim != 2) return fail(CLAWB200_ERR_INVALID, "transverse solves exist in 2-D only");
    return claw_rp_point(p, ixy, n, ql, qr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, imp, asdq, bmasdq,
                         bpasdq, (cudaStream_t)stream);
}

static int rp_point_host(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                         const double *auxl, const double *auxr, double *wave, double *s, double *amdq, double *apdq, int imp, const double *asdq,
                         double *bm, double *bp)
{
    int rc = check_rp_point(p, ixy, n);
    if (rc) return rc;
    if (n == 0) return 0;
    const size_t me = (size_t)p->meqn * n, mw = (size_t)p->mwaves * n;
    const size_t ma = (auxl && auxr && p->maux > 0) ? (size_t)p->maux * n : 0;
    // one device block: ql, qr, asdq | wave, s, amdq, apdq, bm, bp | auxl, auxr
    const size_t total = 3 * me + me * p->mwaves + mw + 4 * me + 2 * ma;
    if ((rc = g_hs.ensure(16))) return rc;
    double *d = nullptr;
    CUDA_OK(cudaMalloc(&d, total * sizeof(double)));
    double *d_ql = d, *d_qr = d + me, *d_as = d + 2 * me, *d_w = d + 3 * me, *d_s = d_w + me * p->mwaves,
           *d_am = d_s + mw, *d_ap = d_am + me, *d_bm = d_ap + me, *d_bp = d_bm + me;
    double *d_al = ma ? d_bp + me : nullptr, *d_ar = ma ? d_bp + me + ma : nullptr;
    cudaStream_t st = g_hs.st;
    auto done = [&](int code) { cudaStreamSynchronize(st); cudaFree(d); return code; };
    cudaError_t e;
    if ((e = cudaMemcpyAsync(d_ql, ql, me * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_qr, qr, me * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess)
        return done(cuda_fail(e, "upload"));
    if (ma && ((e = cudaMemcpyAsync(d_al, auxl, ma * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
               (e = cudaMemcpyAsync(d_ar, auxr, ma * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess))
        return done(cuda_fail(e, "upload"));
    if (asdq) {
        if ((e = cudaMemcpyAsync(d_as, asdq, me * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess)
            return done(cuda_fail(e, "upload"));
        if ((rc = claw_rp_point(p, ixy, n, d_ql, d_qr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, imp, d_as,
                                d_bm, d_bp, st)))
            return done(rc);
        if ((e = cudaMemcpyAsync(bm, d_bm, me * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
            (e = cudaMemcpyAsync(bp, d_bp, me * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess)
            return done(cuda_fail(e, "download"));
    } else {
        if ((rc = claw_rp_point(p, ixy, n, d_ql, d_qr, d_al, d_ar, d_w, d_s, d_am, d_ap, 0, nullptr, nullptr, nullptr, st)))
            return done(rc);
        if ((e = cudaMemcpyAsync(wave, d_w, me * p->mwaves * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
            (e = cudaMemcpyAsync(s, d_s, mw * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
            (e = cudaMemcpyAsync(amdq, d_am, me * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
            (e = cudaMemcpyAsync(apdq, d_ap, me * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess)
            return done(cuda_fail(e, "download"));
    }
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return done(cuda_fail(e, "sync"));
    cudaFree(d);
    return 0;
}

extern "C" int clawb200_rp_solve_host(const clawb200_problem *p, int ixy, long long n, const double *ql,
                                      const double *qr, const double *auxl, const double *auxr, double *wave,
                                      double *s, double *amdq, double *apdq)
{
    if (!ql || !qr || !wave || !s || !amdq || !apdq) return fail(CLAWB200_ERR_INVALID, "null argument");
    return rp_point_host(p, ixy, n, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr);
}

extern "C" int clawb200_rp_transverse_host(const clawb200_problem *p, int ixy, long long n, const double *ql,
                                           const double *qr, int imp, const double *asdq, double *bmasdq,
                                           double *bpasdq)
{
    if (!ql || !qr || !asdq || !bmasdq || !bpasdq) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (imp != 1 && imp != 2) return fail(CLAWB200_ERR_INVALID, "imp must be 1 or 2");
    if (p && p->ndim != 2) return fail(CLAWB200_ERR_INVALID, "transverse solves exist in 2-D only");
    return rp_point_host(p, ixy, n, ql, qr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, imp, asdq, bmasdq, bpasdq);
}

// classic3.step3 with host arrays (clawpack.py:680-682); qnew receives the whole padded array
extern "C" int clawb200_step3_host(const clawb200_problem *p, int mz, double dz, const double *qold,
                                   double *qnew, const double *aux, double dt, double *cfl)
{
    if (!p || !qold || !qnew) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (p->ndim != 3 || mz < 1) return fail(CLAWB200_ERR_INVALID, "3-D problem expected");
    clawb200_problem P = *p;
    P.dt_dev = nullptr;
    const int nx = p->mx + 2 * p->mbc, ny = p->my + 2 * p->mbc, nz = mz + 2 * p->mbc;
    P.pitch = nx;
    P.mstride = (long long)nx * ny * nz;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, qold, g_hs.d_a))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    double *scratch = nullptr;
    CUDA_OK(cudaMalloc(&scratch, sizeof(double) * (size_t)claw_step3_scratch_doubles(P.meqn, P.mstride)));
    if (!(rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st)))
        rc = clawb200_step3(&P, mz, dz, g_hs.d_a, g_hs.d_b, d_aux, dt, scratch, g_hs.d_cfl, g_hs.st);
    if (!rc) rc = host_download(P, g_hs.d_b, qnew);
    if (!rc) rc = host_finish(cfl);
    else cudaStreamSynchronize(g_hs.st);
    cudaFree(scratch);
    return rc;
}

// flux3 of the 3-D SharpClaw stage with host arrays q(meqn, mx+2mbc, my+2mbc, mz+2mbc)
extern "C" int clawb200_sharpclaw_dq3_host(const clawb200_problem *p, int mz, double dz, const double *q,
                                           double *dq, const double *aux, double dt, double *cfl)
{
    if (!p || !q || !dq) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (p->ndim != 3 || mz < 1) return fail(CLAWB200_ERR_INVALID, "3-D problem expected");
    clawb200_problem P = *p;
    P.dt_dev = nullptr;
    const int nx = p->mx + 2 * p->mbc, ny = p->my + 2 * p->mbc, nz = mz + 2 * p->mbc;
    P.pitch = nx;
    P.mstride = (long long)nx * ny * nz;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, q, g_hs.d_a))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    CUDA_OK(cudaMemsetAsync(g_hs.d_b, 0, (size_t)P.meqn * P.mstride * sizeof(double), g_hs.st));
    if ((rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = clawb200_sharpclaw_stage3(&P, mz, dz, g_hs.d_a, nullptr, nullptr, g_hs.d_b, d_aux, dt,
                                        CLAWB200_STAGE_DQ_ONLY, 0.0, 0.0, 1.0, g_hs.d_cfl, g_hs.st)))
        return rc;
    if ((rc = host_download(P, g_hs.d_b, dq))) return rc;
    return host_finish(cfl);
}

// classic3.step3ds with host arrays q(meqn, mx+2mbc, my+2mbc, mz+2mbc) (clawpack.py:656-676)
extern "C" int clawb200_step3ds_host(const clawb200_problem *p, int mz, double dz, const double *qold,
                                     double *qnew, const double *aux, double dt, int idir, double *cfl)
{
    if (!p || !qold || !qnew) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (p->ndim != 3 || mz < 1) return fail(CLAWB200_ERR_INVALID, "3-D problem expected");
    clawb200_problem P = *p;
    P.dt_dev = nullptr;
    const int nx = p->mx + 2 * p->mbc, ny = p->my + 2 * p->mbc, nz = mz + 2 * p->mbc;
    P.pitch = nx;
    P.mstride = (long long)nx * ny * nz;
    int rc = g_hs.ensure((size_t)(P.meqn > P.maux ? P.meqn : P.maux) * P.mstride);
    if (rc) return rc;
    if ((rc = host_upload(P, qold, g_hs.d_a))) return rc;
    const double *d_aux;
    if ((rc = host_upload_aux(P, aux, &d_aux))) return rc;
    if ((rc = clawb200_cfl_reset(g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = clawb200_step3ds(&P, mz, dz, g_hs.d_a, g_hs.d_b, d_aux, dt, idir, g_hs.d_cfl, g_hs.st))) return rc;
    if ((rc = host_download(P, g_hs.d_b, qnew))) return rc;
    return host_finish(cfl);
}
