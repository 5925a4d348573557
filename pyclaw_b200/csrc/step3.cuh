// step3.cuh -- the 3-D classic steps for any Riemann solver with the 3-D interface of rp.cuh
// (RpAcoustics3D, RpAdvection3, RpEuler3, a user's RpUser3): the unsplit step (step3.f:2-594 +
// flux3.f:5-595) and one sweep of the dimensionally split step (step3ds.f:2-376).
//
// The Fortran walks the grid slice by slice: flux3 turns one 1-D slice into increments qadd,
// fadd, gadd(2,-1:1), hadd(2,-1:1) per cell, and step3 scatters them at once into the nine
// cells around every cell of the slice, x-sweeps first, then y, then z.  A cell therefore
// receives 27 contributions in a fixed order (slices in the order of the Fortran loops: the
// higher dimension is the outer loop).  Here each sweep direction D is two launches:
//
//   flux3g_kernel<RPF, D>   one thread per cell of every slice (one ghost layer of slices around the
//                           grid, as the Fortran's "do k = 0, mz+1"): rpn3 at the interfaces
//                           c-1 .. c+2, the limiter and correction fluxes of the interfaces c and
//                           c+1, and the transverse (rpt3) and double-transverse (rptt3) splits of
//                           the plus side of interface c and the minus side of interface c+1 -- both
//                           enter cell c, so they read the aux data around cell c only -- end in 14
//                           increments per component in a scratch array S[14][meqn][cell];
//   apply3g_kernel<MEQN, D> one thread per interior cell: gathers the increments of the nine
//                           slices around it and applies them in the Fortran's order, in place.
//
// sweep3dsg_kernel<RPF, D> is one sweep of the dimensionally split step in one launch over the
// whole padded field.  RPF is the solver template, instantiated as RPF<D + 1>; one translation
// unit per solver family (step3.cu, step3_euler.cu, step3_misc.cu, sweep_user.cu).
//
// Thread <-> x index in all three directions, so every global access of a warp is a unit-stride
// run.  Parity first: all arithmetic is the plain IEEE operators in the Fortran's order of
// evaluation (the oracle's step3 reproduces the reference's golden test/pressure_3D.txt to the
// last printed digit, and this path equals the oracle bit for bit).  Traffic per cell and sweep:
// flux3 reads q along 5 cells and aux on 13 (cached), writes 14*meqn doubles; apply3 reads
// 9 * up to 6 increments per component.
#pragma once
#include "launch.cuh"

struct Step3Args {
    const double *qold;
    double *qnew;
    const double *aux;
    double *S;           // [14][meqn][mstride]
    long long mstride;   // doubles per component (>= nx*ny*nz)
    int nx, ny;          // padded extents (pitch, rows per plane)
    int mbc;
    int n[3];            // interior cells
    double dtd[3];       // dt/dx, dt/dy, dt/dz
    const double *dt_dev; // graph replay: dt is read from here (clawb200_problem.dt_dev)
    double d[3];         // dx, dy, dz
    int order, m3, m4;
    int mthlim[CLAW_MAXWAVES];
    unsigned long long *cfl_bits;
    RpParams rp;
};

// dt/dx of direction dir: the host's quotient or, for graph replay, the same IEEE division on the device
__device__ __forceinline__ double dtd_of(const Step3Args &A, int dir)
{
    return A.dt_dev ? __ldg(A.dt_dev) / A.d[dir] : A.dtd[dir];
}

constexpr int NV3 = 14; // qadd, fdiff, g(1..2, -1..1), h(1..2, -1..1)
// slot of gadd(k, j) / hadd(k, j), k = 1..2, j = -1..1
__host__ __device__ constexpr int gslot(int k, int j) { return 2 + (k - 1) + 2 * (j + 1); }
__host__ __device__ constexpr int hslot(int k, int j) { return 8 + (k - 1) + 2 * (j + 1); }

// Fortran index (i, j, k) of this thread for a launch that covers [lo, lo + n) per dimension
template <int D>
__device__ __forceinline__ bool thread_cell(const Step3Args &A, int &i, int &j, int &k)
{
    // slices run over 0..n+1 in the two transverse directions, cells 1..n along the sweep
    i = ((D == 0) ? 1 : 0) + blockIdx.x * blockDim.x + threadIdx.x;
    j = ((D == 1) ? 1 : 0) + blockIdx.y;
    k = ((D == 2) ? 1 : 0) + blockIdx.z;
    return i <= ((D == 0) ? A.n[0] : A.n[0] + 1);
}

static inline Step3Args make_args3(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                                   const double *aux, double dt, double *scratch, double *cfl_dev)
{
    Step3Args A;
    memset(&A, 0, sizeof(A));
    A.qold = qold; A.qnew = qnew; A.aux = aux; A.S = scratch;
    A.mstride = p->mstride;
    A.nx = p->pitch; A.ny = p->my + 2 * p->mbc;
    A.mbc = p->mbc;
    A.n[0] = p->mx; A.n[1] = p->my; A.n[2] = mz;
    A.dtd[0] = dt / p->dx; A.dtd[1] = dt / p->dy; A.dtd[2] = dt / dz;
    A.dt_dev = p->dt_dev;
    A.d[0] = p->dx; A.d[1] = p->dy; A.d[2] = dz;
    A.order = p->method[1];
    A.m3 = (p->method[2] < 0) ? -1 : p->method[2] / 10;
    A.m4 = (p->method[2] < 0) ? 0 : p->method[2] - 10 * A.m3;
    for (int i = 0; i < CLAW_MAXWAVES; i++) A.mthlim[i] = (i < p->mwaves) ? p->mthlim[i] : 0;
    A.cfl_bits = (unsigned long long *)cfl_dev;
    for (int i = 0; i < 8; i++) A.rp.p[i] = p->rp_params[i];
    return A;
}

namespace step3g {

// The normal part of flux3.f:176-241 for cell c of a slice: rpn3 at the interfaces c-1 .. c+2
// (local index n <-> interface c-1+n between q[n] and q[n+1]), the limiter and the correction
// fluxes of the interfaces c and c+1.  Returns A+ dq of interface c, A- dq of interface c+1, cqxx of
// both, the Roe data of both and the largest wave speed.
template <class RP, class AR>
__device__ __forceinline__ void normal3(AR &ar, const Step3Args &A, const double (&q)[5][RP::MEQN],
                                        const AuxCell (&ax)[5], double dtdx, double (&apdq_c)[RP::MEQN],
                                        double (&amdq_n)[RP::MEQN], double (&cqxx)[2][RP::MEQN],
                                        double (&roe)[2][RP::NROE], unsigned long long &smax)
{
    constexpr int M = RP::MEQN, MW = RP::MWAVES;
    double wave[4][M][MW], s[4][MW], amdq[4][M], apdq[4][M], rr[4][RP::NROE];
#pragma unroll
    for (int n = 0; n < 4; n++) RP::solve(ar, A.rp, q[n], q[n + 1], ax[n], ax[n + 1], wave[n], s[n], amdq[n], apdq[n], rr[n]);
    // Courant number: interfaces c and c+1 (every interface 1..n+1 of a slice is interface c or
    // c+1 of one of its cells)
#pragma unroll
    for (int mw = 0; mw < MW; mw++) { smax_update(smax, s[1][mw]); smax_update(smax, s[2][mw]); }

    // limiter (limiter.f:29-55) and correction flux (flux3.f:226-241) of the interfaces c (n = 1)
    // and c+1 (n = 2); the dot products use the unlimited waves of the neighbours.  An f-wave solver
    // leads with sign(s) instead of |s| (flux2fw.f:151-152, classic.cuh lead_factor): the 3-D f-wave step
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
        for (int m = 0; m < M; m++) cqxx[a][m] = 0.0;
    if (A.order != 1) {
#pragma unroll
        for (int a = 0; a < 2; a++) {
            const int n = 1 + a;
            double wl[M][MW];
#pragma unroll
            for (int mw = 0; mw < MW; mw++) {
                double wnorm2 = 0.0, dotl = 0.0, dotr = 0.0;
#pragma unroll
                for (int m = 0; m < M; m++) {
                    wnorm2 = wnorm2 + wave[n][m][mw] * wave[n][m][mw];
                    dotl = dotl + wave[n - 1][m][mw] * wave[n][m][mw];
                    dotr = dotr + wave[n][m][mw] * wave[n + 1][m][mw];
                }
                double wlimitr = 1.0;
                const bool lim = (A.mthlim[mw] != 0) && (wnorm2 != 0.0);
                if (lim) wlimitr = philim(ar, wnorm2, (s[n][mw] > 0.0) ? dotl : dotr, A.mthlim[mw]);
#pragma unroll
                for (int m = 0; m < M; m++) wl[m][mw] = lim ? wlimitr * wave[n][m][mw] : wave[n][m][mw];
            }
            const double dtdxave = 0.5 * (dtdx + dtdx);
#pragma unroll
            for (int mw = 0; mw < MW; mw++)
#pragma unroll
                for (int m = 0; m < M; m++)
                    cqxx[a][m] = cqxx[a][m] + 0.5 * lead_factor<RP>(s[n][mw]) * (1.0 - fabs(s[n][mw]) * dtdxave) * wl[m][mw];
        }
    }
#pragma unroll
    for (int m = 0; m < M; m++) { apdq_c[m] = apdq[1][m]; amdq_n[m] = amdq[2][m]; }
#pragma unroll
    for (int k = 0; k < RP::NROE; k++) { roe[0][k] = rr[1][k]; roe[1][k] = rr[2][k]; }
}

// One side (SIDE = +1: A+ dq of interface c with the correction cqxx(c), imp = 2; SIDE = -1: A- dq of
// interface c+1 with cqxx(c+1), imp = 1) of the transverse part of flux3.f:239-594 for cell c.
// g / h accumulate in the order of the Fortran's statements.
template <class RP, int SIDE, class AR>
__device__ __forceinline__ void transverse_side(AR &ar, const Step3Args &A, const double (&roe)[RP::NROE],
                                                const double (&ql)[RP::MEQN], const double (&qr)[RP::MEQN],
                                                const AuxNbhd<RP::MAUX> &X, const double (&asdq)[RP::MEQN],
                                                const double (&cq)[RP::MEQN], double dtdx, double dtdy, double dtdz,
                                                double (&g)[2][3][RP::MEQN], double (&h)[2][3][RP::MEQN])
{
    constexpr int M = RP::MEQN, IMP = (SIDE > 0) ? 2 : 1;
    const int m3 = A.m3, m4 = A.m4;
    const RpParams &P = A.rp;
    double bm[M], bp[M], cm[M], cp[M];           // B-+ A* dq, C-+ A* dq
    double bmq[M], bpq[M], cmq[M], cpq[M];       // the same splits of cqxx
    RP::template transverse<2>(ar, P, roe, ql, qr, X, IMP, asdq, bm, bp);
    RP::template transverse<3>(ar, P, roe, ql, qr, X, IMP, asdq, cm, cp);
    if (m3 == 2) {
        RP::template transverse<2>(ar, P, roe, ql, qr, X, IMP, cq, bmq, bpq);
        RP::template transverse<3>(ar, P, roe, ql, qr, X, IMP, cq, cmq, cpq);
    } else {
#pragma unroll
        for (int m = 0; m < M; m++) bmq[m] = bpq[m] = cmq[m] = cpq[m] = 0.0;
    }
    const double sixth = 1.0 / 6.0;
    // ---- G fluxes: the z-like splits are split again in the y-like direction (flux3.f:306-335)
    double bmcp[M], bpcp[M], bmcm[M], bpcm[M];
    if (m4 > 0) {
        double cp2[M], cm2[M];
#pragma unroll
        for (int m = 0; m < M; m++) {
            if (m4 == 2) {
                cp2[m] = (SIDE > 0) ? cp[m] - 3.0 * cpq[m] : cp[m] + 3.0 * cpq[m];
                cm2[m] = (SIDE > 0) ? cm[m] - 3.0 * cmq[m] : cm[m] + 3.0 * cmq[m];
            } else {
                cp2[m] = cp[m]; cm2[m] = cm[m];
            }
        }
        RP::template double_transverse<2>(ar, P, roe, ql, qr, X, IMP, 2, cp2, bmcp, bpcp);
        RP::template double_transverse<2>(ar, P, roe, ql, qr, X, IMP, 1, cm2, bmcm, bpcm);
    }
#pragma unroll
    for (int m = 0; m < M; m++) {
        g[0][1][m] = g[0][1][m] - 0.5 * dtdx * bm[m];
        g[1][1][m] = g[1][1][m] - 0.5 * dtdx * bp[m];
        if (m4 > 0) {
            g[1][1][m] = g[1][1][m] + sixth * dtdx * dtdz * (bpcp[m] - bpcm[m]);
            g[0][1][m] = g[0][1][m] + sixth * dtdx * dtdz * (bmcp[m] - bmcm[m]);
            g[1][2][m] = g[1][2][m] - sixth * dtdx * dtdz * bpcp[m];
            g[0][2][m] = g[0][2][m] - sixth * dtdx * dtdz * bmcp[m];
            g[1][0][m] = g[1][0][m] + sixth * dtdx * dtdz * bpcm[m];
            g[0][0][m] = g[0][0][m] + sixth * dtdx * dtdz * bmcm[m];
        }
        if (m3 >= 2) {
            if (SIDE > 0) {
                g[1][1][m] = g[1][1][m] + dtdx * bpq[m];
                g[0][1][m] = g[0][1][m] + dtdx * bmq[m];
            } else {
                g[1][1][m] = g[1][1][m] - dtdx * bpq[m];
                g[0][1][m] = g[0][1][m] - dtdx * bmq[m];
            }
        }
    }
    // ---- H fluxes: the y-like splits are split again in the z-like direction (flux3.f:449-479)
    if (m4 > 0) {
        double bp2[M], bm2[M];
#pragma unroll
        for (int m = 0; m < M; m++) {
            if (m4 == 2) {
                bp2[m] = (SIDE > 0) ? bp[m] - 3.0 * bpq[m] : bp[m] + 3.0 * bpq[m];
                bm2[m] = (SIDE > 0) ? bm[m] - 3.0 * bmq[m] : bm[m] + 3.0 * bmq[m];
            } else {
                bp2[m] = bp[m]; bm2[m] = bm[m];
            }
        }
        RP::template double_transverse<3>(ar, P, roe, ql, qr, X, IMP, 2, bp2, bmcp, bpcp);
        RP::template double_transverse<3>(ar, P, roe, ql, qr, X, IMP, 1, bm2, bmcm, bpcm);
    }
#pragma unroll
    for (int m = 0; m < M; m++) {
        h[0][1][m] = h[0][1][m] - 0.5 * dtdx * cm[m];
        h[1][1][m] = h[1][1][m] - 0.5 * dtdx * cp[m];
        if (m4 > 0) {
            h[1][1][m] = h[1][1][m] + sixth * dtdx * dtdy * (bpcp[m] - bpcm[m]);
            h[0][1][m] = h[0][1][m] + sixth * dtdx * dtdy * (bmcp[m] - bmcm[m]);
            h[1][2][m] = h[1][2][m] - sixth * dtdx * dtdy * bpcp[m];
            h[0][2][m] = h[0][2][m] - sixth * dtdx * dtdy * bmcp[m];
            h[1][0][m] = h[1][0][m] + sixth * dtdx * dtdy * bpcm[m];
            h[0][0][m] = h[0][0][m] + sixth * dtdx * dtdy * bmcm[m];
        }
        if (m3 >= 2) {
            if (SIDE > 0) {
                h[1][1][m] = h[1][1][m] + dtdx * cpq[m];
                h[0][1][m] = h[0][1][m] + dtdx * cmq[m];
            } else {
                h[1][1][m] = h[1][1][m] - dtdx * cpq[m];
                h[0][1][m] = h[0][1][m] - dtdx * cmq[m];
            }
        }
    }
}

// q and the aux cells along the slice of direction D, cells c-2 .. c+2
template <class RP>
__device__ __forceinline__ void load_slice(const Step3Args &A, long long pos, long long sd, double (&q)[5][RP::MEQN],
                                           AuxCell (&ax)[5])
{
#pragma unroll
    for (int o = 0; o < 5; o++) {
#pragma unroll
        for (int m = 0; m < RP::MEQN; m++) q[o][m] = A.qold[m * A.mstride + pos + (o - 2) * sd];
        ax[o] = AuxCell{RP::MAUX > 0 ? A.aux + pos + (o - 2) * sd : nullptr, A.mstride};
    }
}

template <template <int> class RPF, int D>
__global__ void __launch_bounds__(128) flux3g_kernel(const Step3Args A)
{
    using RP = RPF<D + 1>;
    constexpr int M = RP::MEQN;
    constexpr int E = (D + 1) % 3, F = (D + 2) % 3;
    int i, j, k;
    const bool active = thread_cell<D>(A, i, j, k);
    // a warp with no cell at all leaves (a warp-uniform exit); the idle lanes of the last partly
    // filled warp redo cell 1 so that every lane reaches the warp reduction of the Courant number
    if (!__any_sync(0xffffffffu, active)) return;
    if (!active) i = 1;
    const long long plane = (long long)A.nx * A.ny;
    const long long stride[3] = {1, A.nx, plane};
    const long long sd = stride[D], se = stride[E], sf = stride[F];
    const long long pos = (i + A.mbc - 1) + (long long)A.nx * (j + A.mbc - 1) + plane * (k + A.mbc - 1);
    const double dtdx = dtd_of(A, D), dtdy = dtd_of(A, E), dtdz = dtd_of(A, F);

    double q[5][M];
    AuxCell ax[5];
    load_slice<RP>(A, pos, sd, q, ax);
    AuxNbhd<RP::MAUX> X;
    if (RP::MAUX > 0 && A.m3 > 0) {
#pragma unroll
        for (int ma = 0; ma < RP::MAUX; ma++)
#pragma unroll
            for (int eo = -1; eo <= 1; eo++)
#pragma unroll
                for (int fo = -1; fo <= 1; fo++) X.v[ma][eo + 1][fo + 1] = __ldg(A.aux + ma * A.mstride + pos + eo * se + fo * sf);
    }
    unsigned long long smax = 0ULL;
    double out[NV3][M];
    with_arith([&](auto &ar) {
        double apdq_c[M], amdq_n[M], cqxx[2][M], roe[2][RP::NROE];
        normal3<RP>(ar, A, q, ax, dtdx, apdq_c, amdq_n, cqxx, roe, smax);
#pragma unroll
        for (int m = 0; m < M; m++) {
            out[0][m] = (0.0 - dtdx * apdq_c[m]) - dtdx * amdq_n[m];         // qadd(c)
            out[1][m] = (0.0 + cqxx[1][m]) - (0.0 + cqxx[0][m]);             // fadd(c+1) - fadd(c)
        }
        double g[2][3][M], h[2][3][M];
#pragma unroll
        for (int kk = 0; kk < 2; kk++)
#pragma unroll
            for (int jj = 0; jj < 3; jj++)
#pragma unroll
                for (int m = 0; m < M; m++) { g[kk][jj][m] = 0.0; h[kk][jj][m] = 0.0; }
        if (A.m3 > 0) {
            // iteration i = c of the Fortran's loops 180 / 200 (plus side), then i = c+1 (minus side)
            transverse_side<RP, +1>(ar, A, roe[0], q[1], q[2], X, apdq_c, cqxx[0], dtdx, dtdy, dtdz, g, h);
            transverse_side<RP, -1>(ar, A, roe[1], q[2], q[3], X, amdq_n, cqxx[1], dtdx, dtdy, dtdz, g, h);
        }
#pragma unroll
        for (int kk = 0; kk < 2; kk++)
#pragma unroll
            for (int jj = 0; jj < 3; jj++)
#pragma unroll
                for (int m = 0; m < M; m++) {
                    out[gslot(kk + 1, jj - 1)][m] = g[kk][jj][m];
                    out[hslot(kk + 1, jj - 1)][m] = h[kk][jj][m];
                }
    });
    if (active) {
#pragma unroll
        for (int v = 0; v < NV3; v++)
#pragma unroll
            for (int m = 0; m < M; m++) A.S[(long long)(v * M + m) * A.mstride + pos] = out[v][m];
    }
    cfl_commit(active ? dtdx * __longlong_as_double((long long)smax) : 0.0, A.cfl_bits);
}

// step3.f:185-220 / 340-377 / 497-534 as a gather: the statement of the slice at offset (so_e, so_f)
// that targets this cell is the one written for the offset (-so_e, -so_f).
template <int M, int D>
__global__ void __launch_bounds__(128) apply3g_kernel(const Step3Args A)
{
    constexpr int E = (D + 1) % 3, F = (D + 2) % 3;
    const int i = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    const int j = 1 + blockIdx.y, k = 1 + blockIdx.z;
    if (i > A.n[0]) return;
    const long long plane = (long long)A.nx * A.ny;
    const long long stride[3] = {1, A.nx, plane};
    const long long se = stride[E], sf = stride[F];
    const long long pos = (i + A.mbc - 1) + (long long)A.nx * (j + A.mbc - 1) + plane * (k + A.mbc - 1);
    const double dtd = dtd_of(A, D), dte = dtd_of(A, E), dtf = dtd_of(A, F);
#define SV(slot, m, p) A.S[(long long)((slot) * M + (m)) * A.mstride + (p)]
#pragma unroll
    for (int m = 0; m < M; m++) {
        double q = A.qnew[m * A.mstride + pos];
        // slices in the order of the Fortran loops: the higher physical dimension is the outer loop
#pragma unroll
        for (int a = -1; a <= 1; a++)
#pragma unroll
            for (int b = -1; b <= 1; b++) {
                // (outer, inner) = (f, e) when f is the higher dimension (D = 0, 2), else (e, f)
                const int so_e = (F > E) ? b : a, so_f = (F > E) ? a : b;
                const long long p = pos + so_e * se + so_f * sf;
                const int eo = -so_e, fo = -so_f;
                if (eo == 0 && fo == 0) {
                    q = q + SV(0, m, p) - dtd * SV(1, m, p) - dte * (SV(gslot(2, 0), m, p) - SV(gslot(1, 0), m, p)) -
                        dtf * (SV(hslot(2, 0), m, p) - SV(hslot(1, 0), m, p));
                } else if (eo == -1 && fo == 0) {
                    q = q - dte * SV(gslot(1, 0), m, p) - dtf * (SV(hslot(2, -1), m, p) - SV(hslot(1, -1), m, p));
                } else if (eo == -1 && fo == -1) {
                    q = q - dte * SV(gslot(1, -1), m, p) - dtf * SV(hslot(1, -1), m, p);
                } else if (eo == 0 && fo == -1) {
                    q = q - dte * (SV(gslot(2, -1), m, p) - SV(gslot(1, -1), m, p)) - dtf * SV(hslot(1, 0), m, p);
                } else if (eo == 1 && fo == -1) {
                    q = q + dte * SV(gslot(2, -1), m, p) - dtf * SV(hslot(1, 1), m, p);
                } else if (eo == 1 && fo == 0) {
                    q = q + dte * SV(gslot(2, 0), m, p) - dtf * (SV(hslot(2, 1), m, p) - SV(hslot(1, 1), m, p));
                } else if (eo == 1 && fo == 1) {
                    q = q + dte * SV(gslot(2, 1), m, p) + dtf * SV(hslot(2, 1), m, p);
                } else if (eo == 0 && fo == 1) {
                    q = q - dte * (SV(gslot(2, 1), m, p) - SV(gslot(1, 1), m, p)) + dtf * SV(hslot(2, 0), m, p);
                } else { // (-1, 1)
                    q = q - dte * SV(gslot(1, 1), m, p) + dtf * SV(hslot(2, -1), m, p);
                }
            }
        A.qnew[m * A.mstride + pos] = q;
    }
#undef SV
}

// step3ds.f:2-376: cells of the swept slices (1..n along D, one ghost layer of slices in the other
// two directions) get q + qadd - dtdx (fadd(c+1) - fadd(c)), every other cell a copy of q_in.
template <template <int> class RPF, int D>
__global__ void __launch_bounds__(128) sweep3dsg_kernel(const Step3Args A)
{
    using RP = RPF<D + 1>;
    constexpr int M = RP::MEQN;
    const int ip = blockIdx.x * blockDim.x + threadIdx.x; // padded indices, 0-based
    const int jp = blockIdx.y, kp = blockIdx.z;
    const bool inside = ip < A.nx;
    if (!__any_sync(0xffffffffu, inside)) return;
    const int mbc = A.mbc;
    const int c[3] = {ip - mbc + 1, jp - mbc + 1, kp - mbc + 1}; // Fortran indices
    constexpr int E = (D + 1) % 3, F = (D + 2) % 3;
    const bool swept = inside && c[D] >= 1 && c[D] <= A.n[D] && c[E] >= 0 && c[E] <= A.n[E] + 1 &&
                       c[F] >= 0 && c[F] <= A.n[F] + 1;
    const long long plane = (long long)A.nx * A.ny;
    const long long stride[3] = {1, A.nx, plane};
    const long long pos = (long long)min(ip, A.nx - 1) + (long long)A.nx * jp + plane * kp;
    const double dtdx = dtd_of(A, D);
    unsigned long long smax = 0ULL;
    double res[M];
#pragma unroll
    for (int m = 0; m < M; m++) res[m] = A.qold[m * A.mstride + pos];
    if (swept) {
        double q[5][M];
        AuxCell ax[5];
        load_slice<RP>(A, pos, stride[D], q, ax);
        with_arith([&](auto &ar) {
            double apdq_c[M], amdq_n[M], cqxx[2][M], roe[2][RP::NROE];
            normal3<RP>(ar, A, q, ax, dtdx, apdq_c, amdq_n, cqxx, roe, smax);
#pragma unroll
            for (int m = 0; m < M; m++) {
                const double qadd = (0.0 - dtdx * apdq_c[m]) - dtdx * amdq_n[m];
                const double fdiff = (0.0 + cqxx[1][m]) - (0.0 + cqxx[0][m]);
                res[m] = (q[2][m] + qadd) - dtdx * fdiff;
            }
        });
    }
    if (inside) {
#pragma unroll
        for (int m = 0; m < M; m++) A.qnew[m * A.mstride + pos] = res[m];
    }
    cfl_commit(swept ? dtdx * __longlong_as_double((long long)smax) : 0.0, A.cfl_bits);
}

template <template <int> class RPF, int D>
int sweep3(const Step3Args &A, cudaStream_t st)
{
    const int ni = (D == 0) ? A.n[0] : A.n[0] + 2;
    const int nj = (D == 1) ? A.n[1] : A.n[1] + 2;
    const int nk = (D == 2) ? A.n[2] : A.n[2] + 2;
    dim3 gf((ni + 127) / 128, nj, nk);
    flux3g_kernel<RPF, D><<<gf, 128, 0, st>>>(A);
    CUDA_OK(cudaGetLastError());
    dim3 ga((A.n[0] + 127) / 128, A.n[1], A.n[2]);
    apply3g_kernel<RPF<1>::MEQN, D><<<ga, 128, 0, st>>>(A);
    CUDA_OK(cudaGetLastError());
    return 0;
}

} // namespace step3g

// One 3-D step for the solver family RPF: idir = 1, 2, 3 is one sweep of the dimensionally split
// step (q_out receives the whole field), idir = 0 the unsplit step (`scratch`: 14 * meqn * mstride
// doubles).  The caller (clawb200.cu) has validated the problem.
template <template <int> class RPF>
int claw_step3_generic(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                       const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st)
{
    using namespace step3g;
    const Step3Args A = make_args3(p, mz, dz, qold, qnew, aux, dt, scratch, cfl_dev);
    if (idir > 0) {
        const int nzpad = mz + 2 * p->mbc;
        if (A.ny > 65535 || nzpad > 65535) return fail(CLAWB200_ERR_UNSUPPORTED, "my, mz must be below 65532");
        dim3 grid((A.nx + 127) / 128, A.ny, nzpad);
        if (idir == 1) sweep3dsg_kernel<RPF, 0><<<grid, 128, 0, st>>>(A);
        else if (idir == 2) sweep3dsg_kernel<RPF, 1><<<grid, 128, 0, st>>>(A);
        else sweep3dsg_kernel<RPF, 2><<<grid, 128, 0, st>>>(A);
        CUDA_OK(cudaGetLastError());
        return 0;
    }
    if (A.n[1] + 2 > 65535 || A.n[2] + 2 > 65535) return fail(CLAWB200_ERR_UNSUPPORTED, "my, mz must be below 65534");
    // step3.f: qnew holds qold on entry and accumulates the three families of sweeps
    CUDA_OK(cudaMemcpyAsync(qnew, qold, sizeof(double) * (size_t)p->meqn * p->mstride, cudaMemcpyDeviceToDevice, st));
    int rc;
    if ((rc = sweep3<RPF, 0>(A, st))) return rc;
    if ((rc = sweep3<RPF, 1>(A, st))) return rc;
    if ((rc = sweep3<RPF, 2>(A, st))) return rc;
    return 0;
}
