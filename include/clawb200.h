/*
 * clawb200.h -- C ABI of libclawb200.so: PyClaw's finite-volume time-step hot path as
 * hand-written sm_100a CUDA kernels.
 *
 * This is the drop-in boundary.  Every entry point replaces one routine of the
 * reference's f2py extension modules (classic1 / classic2 / sharpclaw1 / sharpclaw2,
 * built per application by /root/reference/Makefile.rules:1-26 and called from
 * src/pyclaw/clawpack.py and src/pyclaw/sharpclaw.py).  Signatures use plain pointers
 * and sizes only.  Two families:
 *
 *   *_device entry points  take DEVICE pointers in the library's native layout
 *       (structure of arrays, q[m][j][i], i fastest, ghost cells in place) plus a
 *       cudaStream_t passed as void*.  They are asynchronous and never synchronise.
 *       The Courant number is max-accumulated into a device double (`cfl_dev`) that
 *       the caller clears with clawb200_cfl_reset() at the start of a step.
 *
 *   *_host entry points    take HOST pointers in the reference's own layout
 *       (Fortran order q(meqn, 1-mbc:mx+mbc, 1-mbc:my+mbc), what f2py hands to the
 *       Fortran) and return the Courant number by value; they copy in, run the same
 *       kernels, copy out and synchronise.  They are what a maintainer binds in place
 *       of `classic2.step2(...)` etc. (see INTEGRATION.md).
 *
 * Ownership: the caller owns every q / aux buffer; the library never frees or
 * reallocates them.  Scratch for the *_host calls is owned by the library and cached
 * per calling thread.  All functions return 0 on success and a negative code on
 * error (clawb200_last_error() gives the message); nothing aborts the process --
 * the Fortran `stop` statements (step2.f:58-63, rpn2_euler_5wave.f:54-58) have no
 * equivalent here.
 */
#ifndef CLAWB200_H
#define CLAWB200_H

#ifdef __cplusplus
extern "C" {
#endif

#define CLAWB200_MAXWAVES 8

/* Riemann solver ids (the reference selects the solver at link time through RP_SOURCE
 * in each application's Makefile, e.g. apps/euler/2d/shockbubble/Makefile:3). */
#define CLAWB200_RP_ACOUSTICS 1 /* rp1/rpn2/rpt2_acoustics ; params {rho,bulk,cc,zz}   */
#define CLAWB200_RP_ADVECTION 2 /* rp1/rpn2/rpt2_advection ; params {u,v}              */
#define CLAWB200_RP_EULER5 3    /* rpn2/rpt2_euler_5wave   ; params {gamma,gamma1}     */
#define CLAWB200_RP_SHALLOW 4   /* rpn2/rpt2_shallow_roe_with_efix ; params {grav}     */
#define CLAWB200_RP_SPHERE 5    /* rpn2/rpt2_shallow_sphere + step2qcor/qcor (apps/shallow-sphere);
                                   params {g, dxcom, dycom} (0 = take dx, dy); 16 aux, mcapa = 1 */
/* f-wave solvers: the sweeps use the second-order correction of step1fw.f:135-136 /
 * flux2fw.f:151-152 (the reference's classic1fw / classic2fw modules, clawpack.py:222). */
#define CLAWB200_RP_NEL_FWAVE 6 /* rp1_nonlinear_elasticity_fwave (apps/elasticity/1d/stegoton);
                                   aux {rho, K}; params {stress law: 1 linear, 2 exponential} */
#define CLAWB200_RP_PSYSTEM 7   /* rpn2/rpt2_psystem (test/psystem); aux {rho, E, law, eps} */
#define CLAWB200_RP_SHALLOW_BATHY_FWAVE 17 /* shallow water over bathymetry, well-balanced f-waves (1-D, 2-D);
                                              aux {b}; params {grav, dry_tolerance} */
/* further solvers of the reference's applications (external clawpack/riemann sources) */
#define CLAWB200_RP_VC_ACOUSTICS 9    /* rpn2/rpt2_vc_acoustics (apps/acoustics/2d/variable); aux {rho, c} */
#define CLAWB200_RP_BURGERS 10        /* rp1_burgers with entropy fix (apps/burgers/1d)                   */
#define CLAWB200_RP_ADVECTION_COLOR 11 /* rp1_advection_color (apps/advection/1d/variable); aux {u}        */
#define CLAWB200_RP_VC_ADVECTION 12   /* rpn2/rpt2_vc_advection (apps/advection/2d/annulus); aux {u, v[, capa]} */
#define CLAWB200_RP_EULER1D 13        /* rp1_euler_with_efix (apps/euler/1d/wcblast); params {gamma,gamma1} */
/* A Riemann solver supplied by the user as a header and compiled into a variant of the library
 * (pyclaw_b200/csrc/sweep_user.cu, `python -m pyclaw_b200.build --user-rp header.cuh`): the
 * reference's link-time RP_SOURCE seam (Makefile.rules:1-26).  meqn / mwaves / maux come from it.
 * The header defines `template <int IXY> struct RpUser` (1-D / 2-D) and / or `template <int IXYZ>
 * struct RpUser3` (3-D: solve = rpn3, transverse<ICOOR> = rpt3, double_transverse<ICOOR> = rptt3; the
 * interface is documented in pyclaw_b200/csrc/rp.cuh and examples/user_rp/rp_acoustics3d_user.cuh). */
#define CLAWB200_RP_USER 100
/* 3-D solvers (clawb200_step3ds / clawb200_step3, both with rpn3 / rpt3 / rptt3) */
#define CLAWB200_RP_ACOUSTICS3D_VC 8 /* rpn3/rpt3/rptt3_vc_acoustics (test/acoustics/3d); aux {impedance, c} */
#define CLAWB200_RP_ADVECTION3D 14   /* rpn3/rpt3/rptt3_advection; params {u, v, w}; meqn = mwaves = 1 */
#define CLAWB200_RP_EULER3D 15       /* rpn3/rpt3/rptt3_euler, Roe + Harten-Hyman entropy fix; params {gamma,
                                        gamma1}; q = (rho, rho u, rho v, rho w, E), meqn 5, mwaves 3 */
#define CLAWB200_RP_ADVECTION3D_VC_FWAVE 16 /* conservative transport q_t + div(u q) = 0, f-waves (the 3-D
                                               f-wave step, sign(s) correction); aux {u, v, w} per cell,
                                               maux >= 3; meqn = mwaves = 1 */

/* Boundary condition ids = pyclaw.BC (src/pyclaw/solver.py:17-23) */
#define CLAWB200_BC_CUSTOM 0
#define CLAWB200_BC_OUTFLOW 1
#define CLAWB200_BC_PERIODIC 2
#define CLAWB200_BC_REFLECTING 3

/* SharpClaw reconstruction variants */
#define CLAWB200_WENO_PYWENO_F32 0 /* weno.f90:35-98 with its kind-less literals read as REAL(4) */
#define CLAWB200_WENO_PYWENO_F64 1 /* same formulas, literals read as doubles                    */
#define CLAWB200_WENO_OLD 2        /* reconstruct.f90:120-185 (lim_type = 3)                     */
#define CLAWB200_WENO_TABLES 3     /* weno.f90:104-2425, orders 7..17 (1-D): coefficient tables in
                                      problem.weno_tab (clawb200_pack_weno_tables)                               */
#define CLAWB200_RECON_TVD2 4      /* reconstruct.f90:568-625 (lim_type = 1, char_decomp = 0): second-
                                      order TVD reconstruction; problem.mthlim[m] is the limiter of
                                      COMPONENT m (1 minmod, 2 superbee, 3 van Leer, 4 MC, 5 Cada-
                                      Torrilhon).  First cell of a slice: see DESIGN.md            */
#define CLAWB200_RECON_WENO_WAVE 5  /* reconstruct.f90:393-471 weno5_wave (lim_type 2, char_decomp 1), 1-D */
#define CLAWB200_RECON_WENO_FWAVE 6 /* reconstruct.f90:474-565 weno5_fwave (the same with solver.fwave), 1-D */

#define CLAWB200_ERR_INVALID (-1)
#define CLAWB200_ERR_UNSUPPORTED (-2)
#define CLAWB200_ERR_CUDA (-3)

/* Problem description: what the reference spreads over the f2py argument lists, the
 * `method` array (clawpack.py:192-212) and the cparam / ClawParams module state. */
typedef struct clawb200_problem {
    int ndim;                      /* 1, 2 or 3 */
    int meqn, mwaves, maux, mbc;
    int mx, my;                    /* interior cells (my = 1 in 1-D) */
    double dx, dy;
    int method[7];                 /* [dt_variable, order, trans(-1 = dim split), verbosity, 0, mcapa+1, maux] */
    int mthlim[CLAWB200_MAXWAVES]; /* limiter per wave family (limiter.f / philim.f ids 0-5) */
    int rp_id;
    double rp_params[8];
    /* device layout of q: element (m, i, j) (0-based, ghost cells included) is at
       m*mstride + j*pitch + i.  Unused by the *_host entry points. */
    long long mstride;
    int pitch;
    int weno_variant;              /* SharpClaw only */
    /* Optional: device address of a double holding dt.  When non-NULL the classic sweeps read
       the time step from there and ignore their `dt` argument, so that the launch sequence of
       a step does not depend on dt and can be replayed as a CUDA graph. */
    const double *dt_dev;
    /* weno_variant = CLAWB200_WENO_TABLES only: k = (weno_order+1)/2 and the coefficient table
       packed by clawb200_pack_weno_tables -- caller-owned, DEVICE memory for the device entry
       points, host memory for the *_host entry points.  The library keeps no table state. */
    int weno_k;
    const double *weno_tab;
    /* Unsplit classic step (clawb200_step2 / _rows / _host) only: which kernels run it.
       0 = the single-pass kernel (x- and y-sweeps in one walk over q: read once, written once)
           where one is compiled for the solver, otherwise the two sweep kernels;
       1 = always the two sweep kernels (one launch per family, qnew re-read by the second);
       2 = the single-pass kernel or CLAWB200_ERR_UNSUPPORTED.
       Results are bit-identical in every mode. */
    int step2_mode;
} clawb200_problem;

int clawb200_version(void);
const char *clawb200_last_error(void);

/* ---- device-pointer entry points ------------------------------------------------ */

/* cfl_dev <- 0 (stream ordered). */
int clawb200_cfl_reset(double *cfl_dev, void *stream);

/* classic1.step1 (src/fortran/1d/classic/step1.f:4-142; called at clawpack.py:323).
 * q_in has its ghost cells filled; q_out receives cells 1..mx. q_in != q_out. */
int clawb200_step1(const clawb200_problem *p, const double *q_in, double *q_out,
                   const double *aux, double dt, double *cfl_dev, void *stream);

/* classic2.step2ds (src/fortran/2d/classic/step2ds.f:2-248; clawpack.py:538-544).
 * ids = 1: x-sweeps over every row including ghost rows; ids = 2: y-sweeps.
 * q_in != q_out (the Fortran's aliased second call becomes a ping-pong). */
int clawb200_step2ds(const clawb200_problem *p, const double *q_in, double *q_out,
                     const double *aux, double dt, int ids, double *cfl_dev, void *stream);

/* classic2.step2 (src/fortran/2d/classic/step2.f:2-241; clawpack.py:550-552), unsplit
 * with transverse propagation.  qold has ghost cells filled; the interior of qnew is
 * written (qnew need not be initialised). qold != qnew. */
int clawb200_step2(const clawb200_problem *p, const double *qold, double *qnew,
                   const double *aux, double dt, double *cfl_dev, void *stream);

/* The same step restricted to one family of sweeps, for per-kernel timing (bench.py):
 * parts = 1 x-sweeps only (qnew <- qold + x contributions), 2 y-sweeps only (qnew updated
 * in place), 3 both (= clawb200_step2). */
int clawb200_step2_parts(const clawb200_problem *p, const double *qold, double *qnew,
                         const double *aux, double dt, int parts, double *cfl_dev, void *stream);

/* Number of sweep kernels one clawb200_step2 call launches for this problem: 1 when the
 * single-pass kernel runs it (problem.step2_mode, solver, capa), otherwise 2; negative on error. */
int clawb200_step2_launches(const clawb200_problem *p);

/* The same step for output rows jlo..jhi only (1-based interior rows, inclusive).  Lets the
 * caller update the rows that do not depend on a neighbour's halo while the halo exchange is
 * still in flight, and the `mbc` boundary rows afterwards; launching disjoint ranges that
 * cover 1..my gives the same result as one clawb200_step2 call (the Courant number is
 * max-accumulated). */
int clawb200_step2_rows(const clawb200_problem *p, const double *qold, double *qnew,
                        const double *aux, double dt, int jlo, int jhi, double *cfl_dev,
                        void *stream);

/* sharpclaw1.flux1 / sharpclaw2.flux2 (src/fortran/1d/sharpclaw/flux1.f90:2-195,
 * src/fortran/2d/sharpclaw/flux2.f90:2-96; sharpclaw.py:385,558) fused with the
 * Runge-Kutta stage update that sharpclaw.py:172-206 performs in numpy.  q is the
 * stage state with ghost cells filled; dq = dq_hyperbolic(q).  Interior cells of `out`:
 *   mode 0:  out = q + dq/div                (Euler; SSP33 stage 1; SSP104 stages)
 *   mode 1:  out = ca*qa + cb*(q + dq)       (SSP33 stages 2 and 3)
 *   mode 2:  out = (qa + ca*q) + cb*dq       (SSP104 final combination)
 *   mode 3:  out is not written
 * If dq_out != NULL the raw dq is stored there as well (used when a dq_src hook is set
 * and by clawb200_sharpclaw_dq_host).  `cfl_dev` receives this stage's Courant number. */
#define CLAWB200_STAGE_AXPY 0
#define CLAWB200_STAGE_CONVEX 1
#define CLAWB200_STAGE_FINAL104 2
#define CLAWB200_STAGE_DQ_ONLY 3
int clawb200_sharpclaw_stage(const clawb200_problem *p, const double *q, const double *qa,
                             double *out, double *dq_out, const double *aux, double dt,
                             int mode, double ca, double cb, double div, double *cfl_dev,
                             void *stream);
/* The same stage in 3-D (p->ndim = 3; clawb200_sharpclaw_stage fails with CLAWB200_ERR_INVALID on
 * a 3-D problem).  Field layout of clawb200_step3ds; p->rp_id any 3-D solver.  dq is flux1 summed
 * over the x-, y- and z-slices of the grid (DESIGN.md §1): ((0 + dq_x) + dq_y) + dq_z per cell.  The
 * x/y partial of dq is held in dq_out if given, otherwise in out: out, dq_out and qa must be three
 * different buffers, none of them q; mode 3 needs dq_out.  CLAWB200_ERR_UNSUPPORTED for a capacity
 * function (method[5] > 0), WENO orders above 5 (CLAWB200_WENO_TABLES) and the wave-based
 * reconstructions. */
int clawb200_sharpclaw_stage3(const clawb200_problem *p, int mz, double dz, const double *q,
                              const double *qa, double *out, double *dq_out, const double *aux,
                              double dt, int mode, double ca, double cb, double div,
                              double *cfl_dev, void *stream);

/* The stage-free combination in the middle of SSP104 (sharpclaw.py:195-196), fused:
 *     s2 = q/25. + (9./25)*s1 ;  s1 = 15.*s2 - 5.*s1
 * over n contiguous doubles (whole padded buffers). */
int clawb200_ssp104_combine(const double *q, double *s1, double *s2, long long n, void *stream);

/* Coefficient tables for weno_variant = CLAWB200_WENO_TABLES: k = (weno_order+1)/2 in 3..9
 * stencils; S[k][k(k+1)/2] smoothness quadratic forms (pairs a <= b in stencil order),
 * CL/CR[k][k] left / right edge reconstruction, WL/WR[k] ideal weights, eps (the 1e-36 of the
 * generated code).  Replaces the literals of weno7 .. weno17 (weno.f90:104-2425), selected
 * at reconstruct.f90:96-113.  clawb200_pack_weno_tables lays them out in a caller-provided HOST
 * buffer of clawb200_weno_table_doubles() doubles; the caller copies that buffer to the device
 * and points problem.weno_tab at it (no state is kept in the library, any number of solvers
 * with different orders can be alive at once). */
int clawb200_weno_table_doubles(void);
int clawb200_pack_weno_tables(int k, const double *S, const double *CL, const double *CR,
                              const double *WL, const double *WR, double eps, double *packed);

/* apps/shallow-sphere/src2.f:2-147 (the f2py `problem.src2` the reference script wraps as
 * solver.step_src): Coriolis source term with tangent-plane projection, in place on the
 * interior cells of q; aux is the 16-component sphere array. */
int clawb200_sphere_src2(const clawb200_problem *p, double *q, const double *aux, double dt, void *stream);

/* Solver.qbc_lower / qbc_upper (src/pyclaw/solver.py:384-452) for one side of one
 * dimension.  narr = number of components of the array (meqn or maux); `negate` is the
 * component whose sign flips for a reflecting wall (idim+1), or -1 for none (aux). */
int clawb200_bc_fill(const clawb200_problem *p, double *q, int narr, int idim, int side,
                     int bctype, int negate, void *stream);

/* classic3.step3ds (src/fortran/3d/classic/step3ds.f:2-376 with flux3.f:176-237, method(3) < 0;
 * called at clawpack.py:656-676): one directional sweep of the dimensionally split 3-D
 * algorithm, idir = 1, 2, 3.  p->ndim = 3; p->mx, my, dx, dy as usual, the third dimension
 * travels as (mz, dz); the field is q[m][k][j][i] with p->pitch = padded row length and
 * p->mstride >= pitch*(my+2mbc)*(mz+2mbc).  q_out receives qold in cells the sweep does not
 * touch; q_in != q_out.  p->rp_id: any 3-D solver above (meqn / mwaves / maux checked per solver). */
int clawb200_step3ds(const clawb200_problem *p, int mz, double dz, const double *q_in, double *q_out,
                     const double *aux, double dt, int idir, double *cfl_dev, void *stream);
/* classic3.step3 (src/fortran/3d/classic/step3.f:2-594 with flux3.f:5-595 and the rpt3 / rptt3
 * transverse solvers; called at clawpack.py:680-682): the unsplit 3-D step, same layout as
 * clawb200_step3ds.  p->method[2] = 0, 10, 11, 20, 21 or 22 (flux3.f:42-68; ClawSolver3D.no_trans
 * = 0, trans_inc = 11, trans_cor = 22).  qold has its ghost cells filled; the interior of qnew is
 * the result (qnew receives qold elsewhere); qold != qnew.  `scratch` is caller-owned device memory
 * of clawb200_step3_scratch_doubles(p) = 14 * meqn * mstride doubles (the per-cell flux increments of
 * one sweep family). */
long long clawb200_step3_scratch_doubles(const clawb200_problem *p);
int clawb200_step3(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                   const double *aux, double dt, double *scratch, double *cfl_dev, void *stream);
/* qbc_lower / qbc_upper for a 3-D field (idim = 0, 1, 2). */
int clawb200_bc_fill3(const clawb200_problem *p, int mz, double *q, int narr, int idim, int side,
                      int bctype, int negate, void *stream);

/* Layout converters between the reference's host layout (component fastest) and the
 * device layout, both on DEVICE memory; nx, ny include ghost cells. */
int clawb200_aos_to_soa(const double *aos, double *soa, int ncomp, int nx, int ny,
                        long long mstride, int pitch, void *stream);
int clawb200_soa_to_aos(const double *soa, double *aos, int ncomp, int nx, int ny,
                        long long mstride, int pitch, void *stream);

/* Halo pack / unpack for the slab partition (replaces DMDA globalToLocal,
 * src/petclaw/state.py:254-269): copy `nrows` full padded rows starting at array row
 * `row0` of every component to / from a contiguous buffer [m][row][i]. */
int clawb200_halo_pack(const clawb200_problem *p, const double *q, int narr, int row0,
                       int nrows, double *buf, void *stream);
int clawb200_halo_unpack(const clawb200_problem *p, double *q, int narr, int row0,
                         int nrows, const double *buf, void *stream);

/* ---- Riemann solvers as pointwise operators --------------------------------------------
 * The reference's plugin contract for a Riemann solver (doc/rp.rst:7-62, src/pyclaw/clawpack.py:349
 * `wave,s,amdq,apdq = self.rp(q_l,q_r,aux_l,aux_r,aux_global)`; Fortran rpn2 / rpt2,
 * src/fortran/2d/classic/flux2.f:99-100,167-168,180-181) on arrays of n interfaces, evaluated by
 * the very device functions that are inlined into the sweeps.
 * Structure of arrays: ql[m][n], qr[m][n] (left / right state of each interface), auxl[ma][n],
 * auxr[ma][n] (aux of the cell on either side; NULL for solvers that read none),
 * wave[m*mwaves+mw][n], s[mw][n], amdq[m][n], apdq[m][n].  ixy = 1 | 2 (ignored in 1-D), 1 | 2 | 3
 * for the 3-D solvers (p->ndim = 3: rpn3; transverse solves are 2-D only).
 * clawb200_rp_transverse: rpt2 with the Roe data of the interface (ql, qr); imp = 1 splits asdq
 * moving into the left cell, imp = 2 into the right cell. */
int clawb200_rp_solve(const clawb200_problem *p, int ixy, long long n, const double *ql,
                      const double *qr, const double *auxl, const double *auxr, double *wave, double *s,
                      double *amdq, double *apdq, void *stream);
int clawb200_rp_transverse(const clawb200_problem *p, int ixy, long long n, const double *ql,
                           const double *qr, int imp, const double *asdq, double *bmasdq,
                           double *bpasdq, void *stream);
/* the same on HOST arrays */
int clawb200_rp_solve_host(const clawb200_problem *p, int ixy, long long n, const double *ql,
                           const double *qr, const double *auxl, const double *auxr, double *wave,
                           double *s, double *amdq, double *apdq);
int clawb200_rp_transverse_host(const clawb200_problem *p, int ixy, long long n, const double *ql,
                                const double *qr, int imp, const double *asdq, double *bmasdq,
                                double *bpasdq);

/* ---- the library's division / square-root arithmetic on HOST arrays (a test entry point) -----
 * out3[k][n] receives, per element, the results of `op` under `policy`; bad[n] the fast path's
 * sticky flag (1 where it would fall back to the IEEE operators; 0 for EXACT).
 *   policy: FAST      the build's FastArith (integer zero test of a numerator)
 *           FAST_FZ   its floating-point zero-test twin (what with_arith_fz runs first)
 *           EXACT     the IEEE operators
 *           GUARDED   with_arith: FAST, repeated with EXACT if the flag is set (what kernels compute)
 *           GUARDED_FZ with_arith_fz
 *   op (a: numerator / radicand, b: denominator): out3[0] =
 *           RCP 1/b   RCP_NC 1/b (unchecked)   DIV_RCP div(a, rcp(b))   DIV div(a, b)
 *           DIV_NZ div_nz(a, rcp_nc(b))   SQRT sqrt(a)
 *           SQRT_RCP    sqrt(a); out3[1] = 1/sqrt(a)
 *           SQRT_RCPS   sqrt(a); out3[1] = 1/sqrt(a), out3[2] = 1/a
 *           SQRT_RCP2S  sqrt(a); out3[1] = 1/(2 sqrt(a)), out3[2] = 1/a */
#define CLAWB200_ARITH_FAST 0
#define CLAWB200_ARITH_FAST_FZ 1
#define CLAWB200_ARITH_EXACT 2
#define CLAWB200_ARITH_GUARDED 3
#define CLAWB200_ARITH_GUARDED_FZ 4
#define CLAWB200_ARITH_RCP 0
#define CLAWB200_ARITH_RCP_NC 1
#define CLAWB200_ARITH_DIV_RCP 2
#define CLAWB200_ARITH_DIV 3
#define CLAWB200_ARITH_DIV_NZ 4
#define CLAWB200_ARITH_SQRT 5
#define CLAWB200_ARITH_SQRT_RCP 6
#define CLAWB200_ARITH_SQRT_RCPS 7
#define CLAWB200_ARITH_SQRT_RCP2S 8
int clawb200_arith_probe(int policy, int op, long long n, const double *a, const double *b, double *out3, int *bad);

/* ---- host-pointer entry points (the f2py signatures) -----------------------------
 * As the Fortran documents (step2.f:8-9), qold and qnew are taken to be identical on entry:
 * only qold is uploaded, qnew receives the result (untouched cells = qold).  Large 2-D
 * problems are processed as a pipeline of row slabs so that the upload of one slab, the
 * sweeps of the previous one and the download of the one before overlap. */

/* The *_host entry points keep device scratch (staging buffers, three streams, events) per
 * calling thread between calls -- the f2py modules' module-level work arrays, which the
 * reference frees with dealloc_workspace at teardown (sharpclaw.py:328-340).  This frees it;
 * the device entry points hold no state at all (q, aux, WENO tables, the CFL word and the
 * stream are the caller's). */
int clawb200_release_host_scratch(void);

/* (q, cfl) = classic1.step1(mbc, mx, qbc, auxbc, dx, dt, method, mthlim); q updated in place */
int clawb200_step1_host(const clawb200_problem *p, double *q, const double *aux, double dt,
                        double *cfl);
/* (qnew, cfl) = classic2.step2ds(maxm, mbc, mx, my, qold, qnew, auxbc, dx, dy, dt, method,
 *                                mthlim, aux1, aux2, aux3, work, ids); qold may equal qnew */
int clawb200_step2ds_host(const clawb200_problem *p, const double *qold, double *qnew,
                          const double *aux, double dt, int ids, double *cfl);
/* (qnew, cfl) = classic2.step2(maxm, mbc, mx, my, qold, qnew, auxbc, dx, dy, dt, method,
 *                              mthlim, aux1, aux2, aux3, work) */
int clawb200_step2_host(const clawb200_problem *p, const double *qold, double *qnew,
                        const double *aux, double dt, double *cfl);
/* (dq, cfl) = sharpclaw1.flux1(q, auxbc, dt, t, ixy, mx, mbc, maxnx)   (ndim = 1)
 * (dq, cfl) = sharpclaw2.flux2(q, auxbc, dt, t, mbc, maxm, mx, my)     (ndim = 2) */
int clawb200_sharpclaw_dq_host(const clawb200_problem *p, const double *q, double *dq,
                               const double *aux, double dt, double *cfl);
/* (dq, cfl) = flux3 of clawb200_sharpclaw_stage3 on host arrays q(meqn, mx+2mbc, my+2mbc, mz+2mbc)
 * (Fortran order); dq is zero outside the interior.  The reference has no 3-D SharpClaw module. */
int clawb200_sharpclaw_dq3_host(const clawb200_problem *p, int mz, double dz, const double *q,
                                double *dq, const double *aux, double dt, double *cfl);

/* (qnew, cfl) = classic3.step3ds(maxm, mbc, mx, my, mz, qold, qnew, auxbc, dx, dy, dz, dt, method,
 *                                mthlim, aux1, aux2, aux3, work, idir) */
int clawb200_step3ds_host(const clawb200_problem *p, int mz, double dz, const double *qold,
                          double *qnew, const double *aux, double dt, int idir, double *cfl);
/* (qnew, cfl) = classic3.step3(maxm, mbc, mx, my, mz, qold, qnew, auxbc, dx, dy, dz, dt, method, mthlim,
 *                              aux1, aux2, aux3, work)                      (clawpack.py:680-682) */
int clawb200_step3_host(const clawb200_problem *p, int mz, double dz, const double *qold,
                        double *qnew, const double *aux, double dt, double *cfl);

#ifdef __cplusplus
}
#endif
#endif /* CLAWB200_H */
