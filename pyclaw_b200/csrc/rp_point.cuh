// rp_point.cuh -- the Riemann solvers as stand-alone pointwise operators, one thread per
// interface: the kernel and its launcher, for the built-in solvers (rp_point.cu) and the user
// solver (sweep_user.cu).
//
// Layout: structure of arrays, ql[m][n], wave[(m * mwaves + mw)][n], s[mw][n].
#pragma once
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
                           double *bp, cudaStream_t st, const char *noaux = "this Riemann solver reads aux_l / aux_r")
{
    if (n <= 0) return 0;
    if (RP::MAUX > 0 && (!auxl || !auxr)) return fail(CLAWB200_ERR_INVALID, noaux);
    if (RP::MAUX > 0 && asdq) return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise transverse solves: solvers without aux only");
    rp_point_kernel<RP, TRANS><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq,
                                                                    imp, asdq, bm, bp);
    CUDA_OK(cudaGetLastError());
    return 0;
}
