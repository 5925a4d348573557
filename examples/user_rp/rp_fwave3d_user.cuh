// rp_fwave3d_user.cuh -- the built-in 3-D f-wave transport solver (pyclaw.riemann.vc_advection_fwave_3d)
// written as a user plugin through the public 3-D interface (documented in rp_acoustics3d_user.cuh).
// tests/test_gpu_3d_fwave.py checks that runs on this header are bit for bit the runs on the built-in
// solver, split, unsplit and SharpClaw.
//
//     rs = pyclaw.riemann.from_header("rp_fwave3d_user.cuh", meqn=1, mwaves=1, maux=3, ndims=(3,), fwave=True)
//
// An f-wave solver returns waves that sum to the flux difference f(q_r) - f(q_l) and declares
//     static constexpr bool FWAVE = true;
// The 3-D steps then lead the second-order correction of each wave with sign(s) instead of |s|
// (flux2fw.f:151-152); nothing else changes, and the header needs no code of its own for it.
//
// Here: q_t + (u q)_x + (v q)_y + (w q)_z = 0; aux = {u, v, w} of each cell.
//   rpn3:  fwave = (ur*qr) - (ul*ql) with the velocity component of the sweep, s = 0.5*(ul + ur); the
//          whole f-wave goes to the side s points to (half to each when s == 0).
//   rpt3:  bm = min(0.5*(vt(-1) + vt(0)), 0) * asdq, bp = max(0.5*(vt(0) + vt(+1)), 0) * asdq, vt the
//          transverse velocity of the line of three cells through the cell asdq enters.
//   rptt3: the same along the line through the cell the first split moved bsasdq into.
#pragma once

template <int IXYZ>
struct RpUser3 {
    static constexpr int MEQN = 1, MWAVES = 1, NROE = 1, MAUX = 3;
    static constexpr bool FWAVE = true;

    template <class AR>
    __device__ __forceinline__ static void solve(AR &, const RpParams &, const double (&l)[1], const double (&r)[1],
                                                 const AuxCell &axl, const AuxCell &axr, double (&wave)[1][1],
                                                 double (&s)[1], double (&amdq)[1], double (&apdq)[1],
                                                 double (&roe)[NROE])
    {
        const double ul = axl(IXYZ - 1), ur = axr(IXYZ - 1);
        // __dmul_rn / __dsub_rn: the same bits with and without FMA contraction
        const double fwave = __dsub_rn(__dmul_rn(ur, r[0]), __dmul_rn(ul, l[0]));
        const double sp = 0.5 * (ul + ur);
        wave[0][0] = fwave;
        s[0] = sp;
        if (sp > 0.0) { amdq[0] = 0.0; apdq[0] = fwave; }
        else if (sp < 0.0) { amdq[0] = fwave; apdq[0] = 0.0; }
        else { amdq[0] = 0.5 * fwave; apdq[0] = 0.5 * fwave; }
        roe[0] = 0.0;
    }

    // asdq split along the line of three cells through (e0, f0) in direction ICOOR
    template <int ICOOR>
    __device__ __forceinline__ static void split(const AuxNbhd<MAUX> &aux, int e0, int f0, const double (&asdq)[1],
                                                 double (&bm)[1], double (&bp)[1])
    {
        constexpr int MA = rp3_dir(IXYZ, ICOOR) - 1;
        constexpr int de = (ICOOR == 2) ? 1 : 0, df = (ICOOR == 3) ? 1 : 0;
        const double vm = aux(MA, e0 - de, f0 - df), v0 = aux(MA, e0, f0), vp = aux(MA, e0 + de, f0 + df);
        bm[0] = dmin2(0.5 * (vm + v0), 0.0) * asdq[0];
        bp[0] = dmax2(0.5 * (v0 + vp), 0.0) * asdq[0];
    }

    template <int ICOOR, class AR>
    __device__ __forceinline__ static void transverse(AR &, const RpParams &, const double (&)[NROE],
                                                      const double (&)[1], const double (&)[1],
                                                      const AuxNbhd<MAUX> &aux, int, const double (&asdq)[1],
                                                      double (&bm)[1], double (&bp)[1])
    {
        split<ICOOR>(aux, 0, 0, asdq, bm, bp);
    }

    // the velocity of the plane (ICOOR = 2) or row (ICOOR = 3) the first split moved into
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void double_transverse(AR &, const RpParams &, const double (&)[NROE],
                                                             const double (&)[1], const double (&)[1],
                                                             const AuxNbhd<MAUX> &aux, int, int impt,
                                                             const double (&bsasdq)[1], double (&cm)[1], double (&cp)[1])
    {
        const int off = (impt == 1) ? -1 : 1;
        if (ICOOR == 2) split<ICOOR>(aux, 0, off, bsasdq, cm, cp);
        else split<ICOOR>(aux, off, 0, bsasdq, cm, cp);
    }
};
