// launch.cuh -- shared by the translation units of libclawb200.so: error reporting, shared-
// memory opt-in and the launchers of the classic kernels (classic.cuh): the two sweep engines and
// the 1-D step.  The built-in solvers and the user solver (sweep_user.cu) launch through them.
//
// The library is built from several translation units (pyclaw_b200/build.py compiles them in
// parallel): clawb200.cu (C ABI, boundary fills, layout / halo kernels, host entry points),
// sweep_euler_x.cu / sweep_euler_y.cu, sweep_sphere.cu, sweep_misc.cu (instantiations of the
// classic sweeps per Riemann-solver family), sweep_user.cu (the user-supplied solver), step1.cu,
// step3.cu / step3_euler.cu / step3_misc.cu (the 3-D steps), rp_point.cu, sharpclaw.cu,
// sharpclaw3.cu / sharpclaw3_euler.cu / sharpclaw3_misc.cu (the 3-D SharpClaw stage).
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>

#include "../../include/clawb200.h"
#include "classic.cuh"

int fail(int code, const char *msg);
int cuda_fail(cudaError_t e, const char *where);
#define CUDA_OK(call)                                             \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);     \
    } while (0)

// opt in to > 48 KB of dynamic shared memory, once per kernel
template <class K>
static cudaError_t set_smem(K kernel, size_t bytes)
{
    static std::mutex mu;
    static std::unordered_map<const void *, size_t> granted;
    if (bytes <= 48 * 1024) return cudaSuccess;
    std::lock_guard<std::mutex> lock(mu);
    size_t &g = granted[(const void *)kernel];
    if (bytes > g) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        g = bytes;
    }
    return cudaSuccess;
}

// Kernels that read many aux components per interface (the sphere) live on L1 hits: ask for
// the smallest shared-memory carve-out that still holds the resident CTAs, the rest is L1.
template <class K>
static void hint_carveout(K kernel, size_t smem_per_cta, int ctas)
{
    static std::mutex mu;
    static std::unordered_map<const void *, int> done;
    std::lock_guard<std::mutex> lock(mu);
    int &d = done[(const void *)kernel];
    if (d) return;
    int pct = (int)((smem_per_cta + 1024) * ctas * 100 / (228 * 1024)) + 1;
    if (pct > 100) pct = 100;
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    d = 1;
}

constexpr int XNT = 128; // threads per CTA of the x-engine
constexpr int YNT = 128; // threads per CTA of the y-engine

// the classic sweeps: trans selects the unsplit (transverse) form, CAPA the capacity-function form
template <class RP, bool CAPA = false>
static int launch_x(bool trans, const SweepArgs &A, cudaStream_t st)
{
    constexpr int NC = XNT - 3;
    size_t smem = sizeof(double) * (2 * RP::MEQN * (XNT + 1) + RP::MEQN * RP::MWAVES * XNT + 4 * RP::MEQN * XNT +
                                    ((rp_x_aux_smem<RP>::value && trans) ? 4 * RP::MAUX * (XNT + 2) : 0));
    auto k = trans ? xsweep_kernel<RP, true, CAPA, XNT> : xsweep_kernel<RP, false, CAPA, XNT>;
    CUDA_OK(set_smem(k, smem));
    if (RP::MAUX >= 8) hint_carveout(k, smem, RP::X_MINB);
    int ncols = A.ihi - A.ilo + 1, nrows = A.jhi - A.jlo + 1;
    dim3 grid((ncols + NC - 1) / NC, (nrows + A.rows_per_cta - 1) / A.rows_per_cta);
    k<<<grid, XNT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

template <class RP, bool CAPA = false>
static int launch_y(bool trans, const SweepArgs &A, cudaStream_t st)
{
    const int NC = trans ? YNT - 2 : YNT;
    size_t smem = sizeof(double) * YNT * (trans ? 4 * RP::MEQN + YSlots<RP, true>::COUNT : YSlots<RP, false>::COUNT);
    auto k = trans ? ysweep_kernel<RP, true, CAPA, YNT> : ysweep_kernel<RP, false, CAPA, YNT>;
    CUDA_OK(set_smem(k, smem));
    if (RP::MAUX >= 8) hint_carveout(k, smem, RP::Y_MINB);
    int ncols = A.ihi - A.ilo + 1, nrows = A.jhi - A.jlo + 1;
    dim3 grid((ncols + NC - 1) / NC, (nrows + A.rows_per_cta - 1) / A.rows_per_cta);
    k<<<grid, YNT, smem, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

// the 1-D step; CAPA: the solver has a capacity-function form, the others refuse mcapa
template <class RP, bool CAPA>
static int launch_step1(const SweepArgs &A, cudaStream_t st)
{
    constexpr int NT = 128, NC = NT - 3;
    size_t smem = sizeof(double) * (RP::MEQN * (NT + 1) + RP::MEQN * RP::MWAVES * NT + 2 * RP::MEQN * NT);
    dim3 grid((A.mx + NC - 1) / NC);
    if (A.mcapa <= 0) step1_kernel<RP, NT><<<grid, NT, smem, st>>>(A);
    else if constexpr (CAPA) step1_kernel<RP, NT, true><<<grid, NT, smem, st>>>(A);
    else return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for this solver");
    CUDA_OK(cudaGetLastError());
    return 0;
}

static inline int pick_rows(int nrows, int ncol_ctas, bool tall = true)
{
    // enough CTAs to fill 148 SMs a few times over, but strips tall enough that the
    // start-up rows of the streaming engines stay a small fraction of the work
    // very large grids: 128-row strips halve the start-up rows again and still leave ~10 waves of
    // CTAs (Euler 8192^2: 9.10 -> 8.89 ms per step; 4096^2 and the sphere are flat or worse, the
    // SharpClaw stage kernel too: tall = false)
    if (tall && (long long)ncol_ctas * ((nrows + 127) / 128) >= 148 * 28) return 128;
    int h = 64;
    while (h > 8 && (long long)ncol_ctas * ((nrows + h - 1) / h) < 148 * 4) h /= 2;
    return h;
}


// ---- per-family entry points (one translation unit each) ----
int claw_x_euler(bool trans, const SweepArgs &A, cudaStream_t st);
int claw_y_euler(bool trans, const SweepArgs &A, cudaStream_t st);
int claw_x_sphere(bool trans, const SweepArgs &A, cudaStream_t st);
int claw_y_sphere(bool trans, const SweepArgs &A, cudaStream_t st);
int claw_x_misc(int rp_id, bool trans, const SweepArgs &A, cudaStream_t st);
int claw_y_misc(int rp_id, bool trans, const SweepArgs &A, cudaStream_t st);
// single-pass unsplit step (sweep_fused.cu): solvers without aux / capa whose windows fit in registers
bool claw_fused_available(int rp_id, const SweepArgs &A);
int claw_fused(int rp_id, const SweepArgs &A, cudaStream_t st);
// 3-D steps (step3.cuh), one translation unit per solver family (step3.cu, step3_euler.cu,
// step3_misc.cu, sweep_user.cu): idir = 1, 2, 3 one dimensionally split sweep, idir = 0 the unsplit step
long long claw_step3_scratch_doubles(int meqn, long long mstride);
int claw_step3_acoustics(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                         const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st);
int claw_step3_euler(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                     const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st);
int claw_step3_advection(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                         const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st);
int claw_step3_vc_advection_fwave(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                                  const double *aux, double dt, int idir, double *scratch, double *cfl_dev,
                                  cudaStream_t st);
int claw_step3_user(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                    const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st);
// the user-supplied solver (sweep_user.cu), id CLAWB200_RP_USER
struct ScArgs;
int claw_user_shape(int ndim, int *meqn, int *mwaves, int *maux); // ndim = 3: RpUser3
int claw_x_user(bool trans, const SweepArgs &A, cudaStream_t st);
int claw_y_user(bool trans, const SweepArgs &A, cudaStream_t st);
int claw_step1_user(const SweepArgs &A, cudaStream_t st);
int claw_sc_user(int ndim, bool old, const ScArgs &A, cudaStream_t st);
// 3-D SharpClaw stage (sharpclaw3.cuh), one translation unit per solver family (sharpclaw3.cu,
// sharpclaw3_euler.cu, sharpclaw3_misc.cu, sweep_user.cu)
int claw_sc3_acoustics(bool old, const ScArgs &A, cudaStream_t st);
int claw_sc3_euler(bool old, const ScArgs &A, cudaStream_t st);
int claw_sc3_advection(bool old, const ScArgs &A, cudaStream_t st);
int claw_sc3_vc_advection_fwave(bool old, const ScArgs &A, cudaStream_t st);
int claw_sc3_user(bool old, const ScArgs &A, cudaStream_t st);
int claw_rp_point_user(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                       const double *auxl, const double *auxr, double *wave, double *s, double *amdq,
                       double *apdq, int imp, const double *asdq, double *bm, double *bp, cudaStream_t st);
int claw_rp_point(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                  const double *auxl, const double *auxr, double *wave, double *s, double *amdq, double *apdq,
                  int imp, const double *asdq, double *bm, double *bp, cudaStream_t st);
int claw_step1(int rp_id, const SweepArgs &A, cudaStream_t st);
int sharpclaw_launch(const clawb200_problem *p, const double *q, const double *qa, double *out,
                     double *dq_out, double dt, int mode, double ca, double cb, double div,
                     double *cfl_dev, cudaStream_t st, const double *aux);
int sharpclaw_launch3(const clawb200_problem *p, int mz, double dz, const double *q, const double *qa, double *out,
                      double *dq_out, double dt, int mode, double ca, double cb, double div,
                      double *cfl_dev, cudaStream_t st, const double *aux);
