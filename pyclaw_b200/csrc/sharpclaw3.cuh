// sharpclaw3.cuh -- SharpClaw in 3-D: WENO5 reconstruction + interface / in-cell Riemann solves +
// fluctuation sum in x, y and z, fused with the SSP Runge-Kutta stage update (sm_100a).
//
// The reference has no 3-D SharpClaw.  dq is its flux2.f90:2-96 pattern extended by one dimension
// (DESIGN.md §1): flux1 over every x-slice (j, k) in [0, my+1] x [0, mz+1], every y-slice (i, k) in
// [0, mx+1] x [0, mz+1] and every z-slice (i, j) in [0, mx+1] x [0, my+1], each adding its dq1d to the
// interior cells, so that a cell gets ((0 + dq_x) + dq_y) + dq_z.  The Courant number is the largest
// interface Courant number of all these slices (the ghost slices add to it, never to dq).
//
// A stage is two launches, both on the engines of sharpclaw.cuh:
//   sc2d_kernel<RPF<1>, RPF<2>, OLD, SNT, false, true>   one z-plane k = 0 .. mz+1 per blockIdx.z: x
//       through shared memory, y through the rolling 5-row register window, exactly as in 2-D.  It
//       writes the partial (0 + dq_x) + dq_y of the interior cells into dq_out if the caller gave
//       one, into out otherwise.  In the ghost planes 0 and mz+1 every slice adds to the Courant
//       number only.
//   sc3d_z_kernel<RPF<3>, OLD>   one thread per (i, j) column of [0, mx+1] x [0, my+1] (threads run
//       along i, so every warp access is a unit-stride run), walking k with the rolling 5-cell window
//       of the y-engine and the plane as its stride.  Interior columns add dq_z to the partial and
//       store the stage combination; ghost columns add to the Courant number only.  k is cut into
//       chunks of rows_per_cta cells, as the rows of the 2-D kernel.
// No scratch field: the partial lives in the stage's own output buffer.
#pragma once
#include "launch.cuh"
#include "sharpclaw.cuh"

template <class RPZ, bool OLD, int NT>
__global__ void __launch_bounds__(NT, (RPZ::MEQN <= 3) ? CLAW_SC_MINB : 2) sc3d_z_kernel(const ScArgs A)
{
    constexpr int MEQN = RPZ::MEQN, MW = RPZ::MWAVES, NROE = RPZ::NROE;
    constexpr bool AUXRP = (RPZ::MAUX > 0);
    const int mbc = A.mbc;
    const int nxc = A.mx + 2; // columns i = 0 .. mx+1
    const long long ncol = (long long)nxc * (A.my + 2);
    const long long col = (long long)blockIdx.x * NT + threadIdx.x;
    const bool live = col < ncol;
    const long long cc = live ? col : ncol - 1; // idle lanes walk the last column and store nothing
    const int i = (int)(cc % nxc), j = (int)(cc / nxc);
    const bool interior = live && i >= 1 && i <= A.mx && j >= 1 && j <= A.my;
    const long long base = (long long)A.pitch * (j + mbc - 1) + (i + mbc - 1);
    const long long P = A.plane;
    const int k0 = 1 + blockIdx.y * A.rows_per_cta;
    const int k1 = min(k0 + A.rows_per_cta, A.mz + 1);
    const double *partial = A.dq_out ? A.dq_out : A.out;
    const double dtdz = A.dtdz;

    double cfl = 0.0;
    double w0[MEQN], w1[MEQN], w2[MEQN], w3[MEQN], w4[MEQN];
    double qr_prev[MEQN], apdq_prev[MEQN], amdq2_prev[MEQN], apdq2_prev[MEQN];
#pragma unroll
    for (int m = 0; m < MEQN; m++) {
        w0[m] = w1[m] = w2[m] = w3[m] = w4[m] = 1.0;
        qr_prev[m] = 1.0; apdq_prev[m] = amdq2_prev[m] = apdq2_prev[m] = 0.0;
    }
    const AuxCell nocell{nullptr, 0};
    for (int k = k0 - 3; k <= k1 + 2; k++) {
        const long long off = base + P * (k + mbc - 1);
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            w0[m] = w1[m]; w1[m] = w2[m]; w2[m] = w3[m]; w3[m] = w4[m];
            w4[m] = __ldg(&A.q[m * A.mstride + off]);
        }
        // reconstruct cell c = k-2 from cells k-4 .. k
        const int c = k - 2;
        if (c < k0 - 1) continue;
        double ql[MEQN], qr[MEQN];
        with_arith_fz([&](auto &ar) {
#pragma unroll
            for (int m = 0; m < MEQN; m++) weno5<OLD>(ar, A, w0[m], w1[m], w2[m], w3[m], w4[m], ql[m], qr[m], m);
        });
        double wave[MEQN][MW], s[MW], amdq[MEQN], apdq[MEQN], roe[NROE];
        double amdq2[MEQN], apdq2[MEQN];
#pragma unroll
        for (int m = 0; m < MEQN; m++) { amdq[m] = apdq[m] = amdq2[m] = apdq2[m] = 0.0; }
        if (c >= k0) {
            const long long offc = base + P * (c + mbc - 1);
            const AuxCell azc = AUXRP ? sc_aux(A, offc) : nocell;
            const AuxCell azm = AUXRP ? sc_aux(A, offc - P) : nocell;
            // interface c between cells c-1 and c
            with_arith_fz([&](auto &ar) { RPZ::solve(ar, A.rp, qr_prev, ql, azm, azc, wave, s, amdq, apdq, roe); });
            if (live && c >= 1 && c <= A.mz + 1) {
#pragma unroll
                for (int mw = 0; mw < MW; mw++) cfl = dmax2(dmax2(cfl, dtdz * s[mw]), -dtdz * s[mw]);
            }
            if (c < k1 && interior)
                with_arith_fz([&](auto &ar) { RPZ::solve(ar, A.rp, ql, qr, azc, azc, wave, s, amdq2, apdq2, roe); });
            // cell c-1 = k-3 is complete
            const int kc = c - 1;
            if (kc >= k0 && kc < k1 && interior) {
                const long long o = base + P * (kc + mbc - 1);
                double dq[MEQN];
#pragma unroll
                for (int m = 0; m < MEQN; m++) {
                    const double dqz = 0.0 - dtdz * (amdq[m] + apdq_prev[m] + amdq2_prev[m] + apdq2_prev[m]);
                    dq[m] = partial[m * A.mstride + o] + dqz;
                }
                stage_store<MEQN>(A, o, w1, dq);
            }
        }
#pragma unroll
        for (int m = 0; m < MEQN; m++) {
            qr_prev[m] = qr[m]; apdq_prev[m] = apdq[m];
            amdq2_prev[m] = amdq2[m]; apdq2_prev[m] = apdq2[m];
        }
    }
    sc_cfl_commit(cfl, A.cfl_bits);
}

// One 3-D stage for the solver family RPF (sharpclaw3*.cu, sweep_user.cu).  The caller
// (clawb200_sharpclaw_stage3) has validated the problem and filled A for the stage; A.rows_per_cta
// is set here for each launch.
template <template <int> class RPF, bool OLD>
int sc_launch3(ScArgs A, cudaStream_t st)
{
    constexpr int NT = SNT, NC = NT - 2;
    using RX = RPF<1>;
    // x and y, plane by plane: the partial goes to dq_out (or out) through stage mode 3
    {
        ScArgs B = A;
        B.mode = CLAWB200_STAGE_DQ_ONLY;
        B.dq_out = A.dq_out ? A.dq_out : A.out;
        const int nxcta = (A.mx + NC - 1) / NC;
        B.rows_per_cta = pick_rows(A.my, nxcta * (A.mz + 2), false);
        constexpr size_t smem = sc2d_smem<RX>();
        auto k = sc2d_kernel<RX, RPF<2>, OLD, NT, false, true>;
        CUDA_OK(set_smem(k, smem));
        dim3 grid(nxcta, (A.my + B.rows_per_cta - 1) / B.rows_per_cta, A.mz + 2);
        k<<<grid, NT, smem, st>>>(B);
        CUDA_OK(cudaGetLastError());
    }
    // z: adds dq_z to the partial and stores the stage combination
    {
        const long long ncol = (long long)(A.mx + 2) * (A.my + 2);
        const long long ncta = (ncol + NT - 1) / NT;
        if (ncta > 0x7fffffffLL) return fail(CLAWB200_ERR_UNSUPPORTED, "too many (i, j) columns for one launch");
        A.rows_per_cta = pick_rows(A.mz, (int)(ncta < (1 << 24) ? ncta : (1 << 24)), false);
        dim3 grid((unsigned)ncta, (A.mz + A.rows_per_cta - 1) / A.rows_per_cta);
        sc3d_z_kernel<RPF<3>, OLD, NT><<<grid, NT, 0, st>>>(A);
        CUDA_OK(cudaGetLastError());
    }
    return 0;
}

template <template <int> class RPF>
int sc_stage3_generic(bool old, const ScArgs &A, cudaStream_t st)
{
    return old ? sc_launch3<RPF, true>(A, st) : sc_launch3<RPF, false>(A, st);
}
