// rp_acoustics3d_user.cuh -- the built-in 3-D variable-coefficient acoustics solver
// (rpn3 / rpt3 / rptt3_vc_acoustics, test/acoustics/3d) written as a user plugin through the public
// 3-D interface.  tests/test_gpu_3d_solvers.py checks that runs on this header are bit for bit the
// runs on pyclaw.riemann.vc_acoustics_3d, i.e. the user seam adds nothing of its own.
//
//     rs = pyclaw.riemann.from_header("rp_acoustics3d_user.cuh", meqn=4, mwaves=2, maux=2, ndims=(3,))
//
// The 3-D interface (see also pyclaw_b200/csrc/rp.cuh, RpAdvection3 / RpEuler3):
//   template <int IXYZ> struct RpUser3     IXYZ = 1, 2, 3: the sweep direction
//     MEQN, MWAVES, MAUX                   sizes; NROE: doubles solve() hands to the transverse solves
//     solve(ar, P, l, r, axl, axr, wave, s, amdq, apdq, roe)
//         rpn3 at one interface: l / r the states left / right of it, axl / axr their aux cells
//         (axl(ma) = component ma), wave[MEQN][MWAVES], s[MWAVES], the fluctuations amdq / apdq.
//     transverse<ICOOR>(ar, P, roe, ql, qr, aux, imp, asdq, bm, bp)
//         rpt3: asdq split in the y-like (ICOOR = 2) or z-like (ICOOR = 3) direction of the sweep
//         into its down- / up-going parts bm / bp.  imp = 1: asdq = A- dq (it enters the cell left
//         of the interface), 2: A+ dq.  aux(ma, e, f) is the aux data of the 3x3 cells around the
//         cell it enters, e / f = -1..1 the offset in the y-like / z-like direction.
//     double_transverse<ICOOR>(ar, P, roe, ql, qr, aux, imp, impt, bsasdq, cm, cp)
//         rptt3: bsasdq, already split in the OTHER transverse direction (impt = 1 / 2: its down- /
//         up-going part), split again in direction ICOOR.
//   The y-like direction is IXYZ % 3 + 1; rp3_dir(IXYZ, ICOOR) gives the velocity component of ICOOR.
//   Every division and square root goes through `ar` (ar.div, ar.rcp, ar.sqrt).  P.p[0..7] are the
//   parameters (from aux_global through from_header(param_names=...)).
//
// Here: q = (p, u, v, w); aux = {impedance Z, sound speed c} of each cell.
#pragma once

template <int IXYZ>
struct RpUser3 {
    static constexpr int MEQN = 4, MWAVES = 2, NROE = 1, MAUX = 2;

    template <class AR>
    __device__ __forceinline__ static void solve(AR &ar, const RpParams &, const double (&l)[4], const double (&r)[4],
                                                 const AuxCell &axl, const AuxCell &axr, double (&wave)[4][2],
                                                 double (&s)[2], double (&amdq)[4], double (&apdq)[4],
                                                 double (&roe)[NROE])
    {
        const double zi = axr(0), zim = axl(0);
        const double delta1 = r[0] - l[0];
        const double delta2 = r[IXYZ] - l[IXYZ];
        const Recip rz = ar.rcp(zim + zi);
        const double a1 = ar.div(-delta1 + zi * delta2, rz);
        const double a2 = ar.div(delta1 + zim * delta2, rz);
        for (int m = 0; m < 4; m++) { wave[m][0] = 0.0; wave[m][1] = 0.0; }
        wave[0][0] = -a1 * zim;
        wave[IXYZ][0] = a1;
        s[0] = -axl(1);
        wave[0][1] = a2 * zi;
        wave[IXYZ][1] = a2;
        s[1] = axr(1);
        for (int m = 0; m < 4; m++) {
            amdq[m] = s[0] * wave[m][0];
            apdq[m] = s[1] * wave[m][1];
        }
        roe[0] = 0.0;
    }

    // asdq split along the line of three cells through (e0, f0) in direction ICOOR
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void split(AR &ar, const AuxNbhd<MAUX> &aux, int e0, int f0,
                                                 const double (&asdq)[4], double (&bm)[4], double (&bp)[4])
    {
        constexpr int IU = rp3_dir(IXYZ, ICOOR);
        constexpr int de = (ICOOR == 2) ? 1 : 0, df = (ICOOR == 3) ? 1 : 0;
        const double zm = aux(0, e0 - de, f0 - df), zz = aux(0, e0, f0), zp = aux(0, e0 + de, f0 + df);
        const double cm = aux(1, e0 - de, f0 - df), cp = aux(1, e0 + de, f0 + df);
        const double a1 = ar.div(-asdq[0] + asdq[IU] * zz, zm + zz);
        const double a2 = ar.div(asdq[0] + asdq[IU] * zz, zz + zp);
        for (int m = 0; m < 4; m++) { bm[m] = 0.0; bp[m] = 0.0; }
        bm[0] = cm * a1 * zm;
        bp[0] = cp * a2 * zp;
        bm[IU] = -cm * a1;
        bp[IU] = cp * a2;
    }

    template <int ICOOR, class AR>
    __device__ __forceinline__ static void transverse(AR &ar, const RpParams &, const double (&)[NROE],
                                                      const double (&)[4], const double (&)[4],
                                                      const AuxNbhd<MAUX> &aux, int, const double (&asdq)[4],
                                                      double (&bm)[4], double (&bp)[4])
    {
        split<ICOOR>(ar, aux, 0, 0, asdq, bm, bp);
    }

    // the material of the row (ICOOR = 3) or plane (ICOOR = 2) the first split moved into
    template <int ICOOR, class AR>
    __device__ __forceinline__ static void double_transverse(AR &ar, const RpParams &, const double (&)[NROE],
                                                             const double (&)[4], const double (&)[4],
                                                             const AuxNbhd<MAUX> &aux, int, int impt,
                                                             const double (&bsasdq)[4], double (&cm)[4], double (&cp)[4])
    {
        const int off = (impt == 1) ? -1 : 1;
        if (ICOOR == 2) split<ICOOR>(ar, aux, 0, off, bsasdq, cm, cp);
        else split<ICOOR>(ar, aux, off, 0, bsasdq, cm, cp);
    }
};
