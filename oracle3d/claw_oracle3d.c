/*
 * claw_oracle3d.c -- CPU restatement of the 3-D classic steps for the 3-D Riemann solvers other
 * than vc-acoustics (TEST INFRASTRUCTURE ONLY, never linked into the product), next to oracle/claw_oracle.c,
 * which holds the same steps for the variable-coefficient acoustics solver:
 *   src/fortran/3d/classic/step3ds.f:2-376 with flux3.f:176-237 (dimensional splitting)
 *   src/fortran/3d/classic/step3.f:2-594 with flux3.f:5-595 (unsplit, method(3) = 0, 10, 11, 20, 21, 22)
 *   limiter.f / philim.f
 * in the statement order of oracle/claw_oracle.c (flux3_ds, oracle_step3ds, flux3, oracle_step3,
 * limiter, philim), with the rp_id switch of this file's solvers.  The solvers live in the external
 * clawpack/riemann repository (un-vendored): rpn3 / rpt3 / rptt3_advection and rpn3 / rpt3 /
 * rptt3_euler (Roe + Harten-Hyman entropy fix), restated from the published algorithm (LeVeque 2002,
 * sec. 15.3 and 18.8), parity unpinned.  The f-wave transport solver (aux = {u, v, w} per cell) runs the
 * 3-D f-wave step: flux3.f with the delta of flux2fw.f (sign(s) leads the correction flux), DESIGN.md §1.
 * Strict IEEE double: compiled without FMA contraction (oracle3d/Makefile).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define RP_ADVECTION3D 14 /* p[0..2] = u, v, w          */
#define RP_EULER3D 15     /* p[0] = gamma, p[1] = gamma1 */
#define RP_ADVECTION3D_VC_FWAVE 16 /* aux = u, v, w of each cell; f-waves */
#define RP_IS_FWAVE3(id) ((id) == RP_ADVECTION3D_VC_FWAVE)

/* aux1d (maux, slice): the aux data of the slice's cells; aux9 (maux, 3, 3, slice): the 3x3 cells
   around each cell of the slice in the plane normal to it, aux9[ma + maux * ((e+1) + 3 * (f+1))] at the
   offset e / f in the y-like / z-like direction.  Both NULL for the solvers without aux data. */
typedef struct {
    int rp_id;
    double p[8];
    int maux;
    const double *aux1d, *aux9;
} rp_ctx3;

static inline double dmax2(double a, double b) { return (a > b) ? a : b; }
static inline double dmin2(double a, double b) { return (a < b) ? a : b; }

/* slice indexing: Fortran index i in [1-mbc, maxm+mbc] -> offset i+mbc-1 */
#define IX(i) ((i) + mbc - 1)
#define Q2(arr, m, i) arr[(m) + meqn * IX(i)]
#define WV(m, mw, i) wave[(m) + meqn * ((mw) + mwaves * IX(i))]
#define SP(mw, i) s[(mw) + mwaves * IX(i)]

/* ixyz = 1, 2, 3 is the sweep direction; the transverse direction icoor = 2 (y-like) / 3 (z-like)
   has velocity component rp3_dir(ixyz, icoor) */
static inline int rp3_dir(int ixyz, int icoor) { return (ixyz - 1 + icoor - 1) % 3 + 1; }

/* ---- rpn3 / rpt3 / rptt3_advection ---- */
static void rpn3_advection(const rp_ctx3 *c, int ixyz, int mbc, int mx, const double *ql, const double *qr,
                           double *wave, double *s, double *amdq, double *apdq)
{
    const int meqn = 1, mwaves = 1;
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        WV(0, 0, i) = Q2(ql, 0, i) - Q2(qr, 0, i - 1);
        SP(0, i) = c->p[ixyz - 1];
        Q2(amdq, 0, i) = dmin2(SP(0, i), 0.0) * WV(0, 0, i);
        Q2(apdq, 0, i) = dmax2(SP(0, i), 0.0) * WV(0, 0, i);
    }
}

/* rpt3_advection (and rptt3_advection, the same split of an already split fluctuation) */
static void rpt3_advection(const rp_ctx3 *c, int ixyz, int icoor, int mbc, int mx, const double *asdq,
                           double *bmasdq, double *bpasdq)
{
    const int meqn = 1;
    const double st = c->p[rp3_dir(ixyz, icoor) - 1];
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        Q2(bmasdq, 0, i) = dmin2(st, 0.0) * Q2(asdq, 0, i);
        Q2(bpasdq, 0, i) = dmax2(st, 0.0) * Q2(asdq, 0, i);
    }
}

/* ---- the f-wave transport solver (rpn3 / rpt3 / rptt3; rp.cuh RpVcAdvectionFwave3) ---- */
/* interface i between cell i-1 (qr, auxr) and cell i (ql, auxl): ul = u_d(i-1), ur = u_d(i);
   fwave = ur q(i) - ul q(i-1), s = (ul + ur) / 2, the whole f-wave to the side s points to */
static void rpn3_vc_fwave(int ixyz, int mbc, int mx, int maux, const double *ql, const double *qr,
                          const double *auxl, const double *auxr, double *wave, double *s, double *amdq,
                          double *apdq)
{
    const int meqn = 1, mwaves = 1, d = rp3_dir(ixyz, 1) - 1;
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        double ul = auxr[d + maux * IX(i - 1)], ur = auxl[d + maux * IX(i)];
        double fwave = (ur * Q2(ql, 0, i)) - (ul * Q2(qr, 0, i - 1));
        double sp = 0.5 * (ul + ur);
        WV(0, 0, i) = fwave;
        SP(0, i) = sp;
        if (sp > 0.0) { Q2(amdq, 0, i) = 0.0; Q2(apdq, 0, i) = fwave; }
        else if (sp < 0.0) { Q2(amdq, 0, i) = fwave; Q2(apdq, 0, i) = 0.0; }
        else { Q2(amdq, 0, i) = 0.5 * fwave; Q2(apdq, 0, i) = 0.5 * fwave; }
    }
}

/* rpt3 (impt = 0) / rptt3 (impt = 1, 2): asdq of interface i enters cell i-1 (imp = 1) or i (imp = 2); split
   along the line of three cells in direction icoor through that cell (rpt3) or through the cell one step
   down (impt = 1) / up (impt = 2) in the other transverse direction (rptt3) */
static void rpt3_vc_fwave(const rp_ctx3 *c, int ixyz, int icoor, int imp, int impt, int mbc, int mx,
                          const double *asdq, double *bmasdq, double *bpasdq)
{
    const int meqn = 1, maux = c->maux, ma = rp3_dir(ixyz, icoor) - 1;
    const int de = (icoor == 2) ? 1 : 0, df = (icoor == 3) ? 1 : 0;
    const int off = (impt == 1) ? -1 : 1;
    const int e0 = (impt != 0 && icoor == 3) ? off : 0, f0 = (impt != 0 && icoor == 2) ? off : 0;
#define A9(cell, e, f) c->aux9[ma + maux * (((e) + 1) + 3 * ((f) + 1)) + (size_t)9 * maux * IX(cell)]
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        const int cell = (imp == 1) ? i - 1 : i;
        double vm = A9(cell, e0 - de, f0 - df), v0 = A9(cell, e0, f0), vp = A9(cell, e0 + de, f0 + df);
        Q2(bmasdq, 0, i) = dmin2(0.5 * (vm + v0), 0.0) * Q2(asdq, 0, i);
        Q2(bpasdq, 0, i) = dmax2(0.5 * (v0 + vp), 0.0) * Q2(asdq, 0, i);
    }
#undef A9
}

/* ---- rpn3 / rpt3 / rptt3_euler ---- */
/* Roe averages of the interface between l and r: roe = {u, v, w, enth, a, u^2 + v^2 + w^2} */
static void euler3_roe(double gamma1, const double *l, const double *r, double *roe)
{
    double rhsqrtl = sqrt(l[0]), rhsqrtr = sqrt(r[0]);
    double pl = gamma1 * (l[4] - 0.5 * (l[1] * l[1] + l[2] * l[2] + l[3] * l[3]) / l[0]);
    double pr = gamma1 * (r[4] - 0.5 * (r[1] * r[1] + r[2] * r[2] + r[3] * r[3]) / r[0]);
    double rhsq2 = rhsqrtl + rhsqrtr;
    for (int k = 0; k < 3; k++) roe[k] = (l[1 + k] / rhsqrtl + r[1 + k] / rhsqrtr) / rhsq2;
    double enth = (((l[4] + pl) / rhsqrtl + (r[4] + pr) / rhsqrtr)) / rhsq2;
    double uvw2 = roe[0] * roe[0] + roe[1] * roe[1] + roe[2] * roe[2];
    roe[3] = enth;
    roe[4] = sqrt(gamma1 * (enth - 0.5 * uvw2));
    roe[5] = uvw2;
}

/* d split into the eigenvectors of the Roe matrix of direction mt (velocity component 1..3):
   wave 0 at un - a, wave 1 at un (entropy and both shear jumps), wave 2 at un + a */
static void euler3_waves(int mt, double gamma1, const double *roe, const double *d, double wv[5][3], double *sp)
{
    const int m1 = mt % 3 + 1, m2 = (mt + 1) % 3 + 1;
    double un = roe[mt - 1], u1 = roe[m1 - 1], u2 = roe[m2 - 1];
    double enth = roe[3], a = roe[4], uvw2 = roe[5];
    double a3 = gamma1 / (a * a) * ((enth - uvw2) * d[0] + roe[0] * d[1] + roe[1] * d[2] + roe[2] * d[3] - d[4]);
    double b1 = d[m1] - u1 * d[0], b2 = d[m2] - u2 * d[0];
    double a5 = (d[mt] + (a - un) * d[0] - a * a3) / (2.0 * a);
    double a1 = d[0] - a3 - a5;
    wv[0][0] = a1; wv[mt][0] = a1 * (un - a); wv[m1][0] = a1 * u1; wv[m2][0] = a1 * u2;
    wv[4][0] = a1 * (enth - un * a); sp[0] = un - a;
    wv[0][1] = a3; wv[mt][1] = a3 * un; wv[m1][1] = a3 * u1 + b1; wv[m2][1] = a3 * u2 + b2;
    wv[4][1] = a3 * 0.5 * uvw2 + b1 * u1 + b2 * u2; sp[1] = un;
    wv[0][2] = a5; wv[mt][2] = a5 * (un + a); wv[m1][2] = a5 * u1; wv[m2][2] = a5 * u2;
    wv[4][2] = a5 * (enth + un * a); sp[2] = un + a;
}

/* rpn3_euler: the operations of rp1_euler_with_efix (oracle/claw_oracle.c, rpn_euler1d) with the
   full kinetic energy; with v = w = 0 they are the same operations on the same values */
static void rpn3_euler(const rp_ctx3 *c, int ixyz, int mbc, int mx, const double *ql, const double *qr,
                       double *wave, double *s, double *amdq, double *apdq)
{
    const int meqn = 5, mwaves = 3, mu = ixyz;
    const double gamma1 = c->p[1];
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        const double *l = &Q2(qr, 0, i - 1), *r = &Q2(ql, 0, i);
        double roe[6], d[5], wv[5][3], sp[3], am[5];
        euler3_roe(gamma1, l, r, roe);
        for (int m = 0; m < 5; m++) d[m] = r[m] - l[m];
        euler3_waves(mu, gamma1, roe, d, wv, sp);
        /* Harten-Hyman entropy fix on the acoustic waves, left-going fluctuation first */
        int done = 0;
        double ulx = l[1] / l[0], uly = l[2] / l[0], ulz = l[3] / l[0];
        double cl = sqrt(gamma1 * (gamma1 + 1.0) * (l[4] / l[0] - 0.5 * (ulx * ulx + uly * uly + ulz * ulz)));
        double s0 = l[mu] / l[0] - cl;
        if (s0 >= 0.0 && sp[0] > 0.0) {
            for (int m = 0; m < 5; m++) am[m] = 0.0;
            done = 1;
        }
        if (!done) {
            double q1[5];
            for (int m = 0; m < 5; m++) q1[m] = l[m] + wv[m][0];
            double p1 = gamma1 * (q1[4] - 0.5 * (q1[1] * q1[1] + q1[2] * q1[2] + q1[3] * q1[3]) / q1[0]);
            double c1 = sqrt((gamma1 + 1.0) * p1 / q1[0]);
            double s1 = q1[mu] / q1[0] - c1;
            double sfract;
            if (s0 < 0.0 && s1 > 0.0) sfract = s0 * (s1 - sp[0]) / (s1 - s0);
            else if (sp[0] < 0.0) sfract = sp[0];
            else sfract = 0.0;
            for (int m = 0; m < 5; m++) am[m] = sfract * wv[m][0];
            if (sp[1] >= 0.0) done = 1;
        }
        if (!done) {
            for (int m = 0; m < 5; m++) am[m] = am[m] + sp[1] * wv[m][1];
            double urx = r[1] / r[0], ury = r[2] / r[0], urz = r[3] / r[0];
            double cr = sqrt(gamma1 * (gamma1 + 1.0) * (r[4] / r[0] - 0.5 * (urx * urx + ury * ury + urz * urz)));
            double s3 = r[mu] / r[0] + cr;
            double q2[5];
            for (int m = 0; m < 5; m++) q2[m] = r[m] - wv[m][2];
            double p2 = gamma1 * (q2[4] - 0.5 * (q2[1] * q2[1] + q2[2] * q2[2] + q2[3] * q2[3]) / q2[0]);
            double c2 = sqrt((gamma1 + 1.0) * p2 / q2[0]);
            double s2 = q2[mu] / q2[0] + c2;
            double sfract = 0.0;
            int add = 1;
            if (s2 < 0.0 && s3 > 0.0) sfract = s2 * (s3 - sp[2]) / (s3 - s2);
            else if (sp[2] < 0.0) sfract = sp[2];
            else add = 0;
            if (add) for (int m = 0; m < 5; m++) am[m] = am[m] + sfract * wv[m][2];
        }
        for (int m = 0; m < 5; m++) {
            double df = 0.0;
            for (int mw = 0; mw < 3; mw++) df = df + sp[mw] * wv[m][mw];
            Q2(amdq, m, i) = am[m];
            Q2(apdq, m, i) = df - am[m];
            for (int mw = 0; mw < 3; mw++) WV(m, mw, i) = wv[m][mw];
        }
        for (int mw = 0; mw < 3; mw++) SP(mw, i) = sp[mw];
    }
}

/* rpt3_euler (and rptt3_euler, the same split of an already split fluctuation): asdq split with the
   eigenvectors of the Roe matrix of direction icoor at the Roe averages of interface i, q(:, i-1) | q(:, i) */
static void rpt3_euler(const rp_ctx3 *c, int ixyz, int icoor, int mbc, int mx, const double *q1d,
                       const double *asdq, double *bmasdq, double *bpasdq)
{
    const int meqn = 5;
    const double gamma1 = c->p[1];
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        double roe[6], wv[5][3], sp[3];
        euler3_roe(gamma1, &Q2(q1d, 0, i - 1), &Q2(q1d, 0, i), roe);
        euler3_waves(rp3_dir(ixyz, icoor), gamma1, roe, &Q2(asdq, 0, i), wv, sp);
        for (int m = 0; m < 5; m++) {
            Q2(bmasdq, m, i) = dmin2(sp[0], 0.0) * wv[m][0] + dmin2(sp[1], 0.0) * wv[m][1] + dmin2(sp[2], 0.0) * wv[m][2];
            Q2(bpasdq, m, i) = dmax2(sp[0], 0.0) * wv[m][0] + dmax2(sp[1], 0.0) * wv[m][1] + dmax2(sp[2], 0.0) * wv[m][2];
        }
    }
}

/* ---- the rp_id switches ---- */
static void rpn3(const rp_ctx3 *c, int ixyz, int mbc, int mx, const double *ql, const double *qr, double *wave,
                 double *s, double *amdq, double *apdq)
{
    if (c->rp_id == RP_EULER3D) rpn3_euler(c, ixyz, mbc, mx, ql, qr, wave, s, amdq, apdq);
    else if (c->rp_id == RP_ADVECTION3D_VC_FWAVE)
        rpn3_vc_fwave(ixyz, mbc, mx, c->maux, ql, qr, c->aux1d, c->aux1d, wave, s, amdq, apdq);
    else rpn3_advection(c, ixyz, mbc, mx, ql, qr, wave, s, amdq, apdq);
}
/* rpt3 (impt = 0) and rptt3 (impt = 1, 2): advection and Euler read no aux data, so they depend on
   neither imp nor impt */
static void rpt3(const rp_ctx3 *c, int ixyz, int icoor, int imp, int impt, int mbc, int mx, const double *q1d,
                 const double *asdq, double *bmasdq, double *bpasdq)
{
    if (c->rp_id == RP_EULER3D) rpt3_euler(c, ixyz, icoor, mbc, mx, q1d, asdq, bmasdq, bpasdq);
    else if (c->rp_id == RP_ADVECTION3D_VC_FWAVE) rpt3_vc_fwave(c, ixyz, icoor, imp, impt, mbc, mx, asdq, bmasdq, bpasdq);
    else rpt3_advection(c, ixyz, icoor, mbc, mx, asdq, bmasdq, bpasdq);
}
static int known(int rp_id) { return rp_id == RP_ADVECTION3D || rp_id == RP_EULER3D || rp_id == RP_ADVECTION3D_VC_FWAVE; }
/* the f-wave transport solver reads aux {u, v, w}, the 3x3 neighbourhood of each cell included */
static int aux_ok(int rp_id, const double *aux, int maux, int mbc)
{
    if (rp_id != RP_ADVECTION3D_VC_FWAVE) return 1;
    return aux != NULL && maux >= 3 && mbc >= 2;
}

/* ---- limiter.f / philim.f (as oracle/claw_oracle.c) ---- */
static double philim(double a, double b, int meth)
{
    double r = b / a;
    switch (meth) {
    case 2: return dmax2(dmax2(0.0, dmin2(1.0, 2.0 * r)), dmin2(2.0, r));
    case 3: return (r + fabs(r)) / (1.0 + fabs(r));
    case 4: {
        double c = (1.0 + r) / 2.0;
        return dmax2(0.0, dmin2(dmin2(c, 2.0), 2.0 * r));
    }
    case 5: return r;
    default: return dmax2(0.0, dmin2(1.0, r)); /* philim.f:19: out-of-range ids fall through to minmod */
    }
}

static void limiter(int meqn, int mwaves, int mbc, int mx, double *wave, const double *s, const int *mthlim)
{
    for (int mw = 0; mw < mwaves; mw++) {
        if (mthlim[mw] == 0) continue;
        double dotr = 0.0;
        for (int i = 0; i <= mx + 1; i++) {
            double wnorm2 = 0.0;
            double dotl = dotr;
            dotr = 0.0;
            for (int m = 0; m < meqn; m++) {
                wnorm2 = wnorm2 + WV(m, mw, i) * WV(m, mw, i);
                dotr = dotr + WV(m, mw, i) * WV(m, mw, i + 1);
            }
            if (i == 0) continue;
            if (wnorm2 == 0.0) continue;
            double wlimitr;
            if (SP(mw, i) > 0.0)
                wlimitr = philim(wnorm2, dotl, mthlim[mw]);
            else
                wlimitr = philim(wnorm2, dotr, mthlim[mw]);
            for (int m = 0; m < meqn; m++) WV(m, mw, i) = wlimitr * WV(m, mw, i);
        }
    }
}

/* the normal part of flux3.f:176-241 on one slice (q1d, uniform dtdx): qadd, fadd and cqxx; returns cfl */
static double flux3_normal(const rp_ctx3 *c, int ixyz, int meqn, int mwaves, int mbc, int mx, const double *q1d,
                           double dtdx, int order, const int *mthlim, double *wave, double *s, double *amdq,
                           double *apdq, double *cqxx, double *qadd, double *fadd)
{
    int limit = 0;
    for (int mw = 0; mw < mwaves; mw++) if (mthlim[mw] > 0) limit = 1;
    for (int i = 1 - mbc; i <= mx + mbc; i++)
        for (int m = 0; m < meqn; m++) { Q2(qadd, m, i) = 0.0; Q2(fadd, m, i) = 0.0; Q2(cqxx, m, i) = 0.0; }
    rpn3(c, ixyz, mbc, mx, q1d, q1d, wave, s, amdq, apdq);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++) Q2(qadd, m, i) = Q2(qadd, m, i) - dtdx * Q2(apdq, m, i);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++) Q2(qadd, m, i - 1) = Q2(qadd, m, i - 1) - dtdx * Q2(amdq, m, i);
    double cfl1d = 0.0;
    for (int i = 1; i <= mx + 1; i++)
        for (int mw = 0; mw < mwaves; mw++)
            cfl1d = dmax2(dmax2(cfl1d, dtdx * SP(mw, i)), -dtdx * SP(mw, i));
    if (order == 1) return cfl1d;
    if (limit) limiter(meqn, mwaves, mbc, mx, wave, s, mthlim);
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        double dtdxave = 0.5 * (dtdx + dtdx);
        for (int m = 0; m < meqn; m++) Q2(cqxx, m, i) = 0.0;
        for (int mw = 0; mw < mwaves; mw++) {
            /* flux2fw.f:151-152: an f-wave solver leads with sign(s) */
            double lead = RP_IS_FWAVE3(c->rp_id) ? copysign(1.0, SP(mw, i)) : fabs(SP(mw, i));
            for (int m = 0; m < meqn; m++)
                Q2(cqxx, m, i) = Q2(cqxx, m, i) + 0.5 * lead * (1.0 - fabs(SP(mw, i)) * dtdxave) * WV(m, mw, i);
        }
        for (int m = 0; m < meqn; m++) Q2(fadd, m, i) = Q2(fadd, m, i) + Q2(cqxx, m, i);
    }
    return cfl1d;
}

/* the aux data of one slice in direction d (cells l = 1-mbc .. len[d]+mbc at the transverse position idx):
   aux1d (maux, n) and, where the neighbours exist, the 3x3 neighbourhood aux9 (maux, 3, 3, n) */
static void slice_aux(const double *aux, int maux, int mbc, int mx, int my, int mz, int d, const int *idx,
                      double *aux1d, double *aux9)
{
    const size_t NXs = mx + 2 * mbc, NYs = my + 2 * mbc;
    const int len[3] = {mx, my, mz}, e = (d + 1) % 3, f = (d + 2) % 3;
    for (int l = 1 - mbc; l <= len[d] + mbc; l++)
        for (int fo = -1; fo <= 1; fo++)
            for (int eo = -1; eo <= 1; eo++) {
                int p[3] = {idx[0], idx[1], idx[2]};
                p[d] = l; p[e] += eo; p[f] += fo;
                if (p[e] < 1 - mbc || p[e] > len[e] + mbc || p[f] < 1 - mbc || p[f] > len[f] + mbc) continue;
                const size_t off = ((p[0] + mbc - 1) + NXs * ((p[1] + mbc - 1) + NYs * (p[2] + mbc - 1)));
                for (int ma = 0; ma < maux; ma++) {
                    double v = aux[ma + (size_t)maux * off];
                    aux9[ma + maux * ((eo + 1) + 3 * (fo + 1)) + (size_t)9 * maux * IX(l)] = v;
                    if (eo == 0 && fo == 0) aux1d[ma + maux * IX(l)] = v;
                }
            }
}

/* ------------------------------------------------------------------------- */
/* step3ds.f:2-376 (method(3) < 0), idir = 1, 2, 3; sweeps cover one ghost     */
/* layer of the other two directions.  q(meqn, 1-mbc:mx+mbc, ..., 1-mbc:mz+mbc) */
/* ------------------------------------------------------------------------- */
/* aux (maux, 1-mbc:mx+mbc, ...) or NULL: the f-wave transport solver needs it */
double oracle3d_step3ds_aux(int rp_id, const double *rp_params, int meqn, int mwaves, int mbc, int mx, int my, int mz,
                            const double *qold, double *qnew, const double *aux, int maux, double dx, double dy,
                            double dz, double dt, const int *method, const int *mthlim, int idir)
{
    if (!known(rp_id) || method[5] > 0 || !aux_ok(rp_id, aux, maux, mbc)) return -1.0;
    rp_ctx3 c = {0};
    c.rp_id = rp_id;
    memcpy(c.p, rp_params, 8 * sizeof(double));
    int maxm = mx > my ? mx : my;
    if (mz > maxm) maxm = mz;
    const int n = maxm + 2 * mbc;
    const int ma = aux ? maux : 0;
    double *aux1d = (double *)calloc((size_t)n * (ma > 0 ? ma : 1), sizeof(double));
    double *aux9 = (double *)calloc((size_t)n * 9 * (ma > 0 ? ma : 1), sizeof(double));
    c.maux = ma;
    c.aux1d = aux1d;
    c.aux9 = aux9;
    double *v[7];
    for (int a = 0; a < 7; a++) v[a] = (double *)calloc((size_t)n * meqn * mwaves, sizeof(double));
    double *q1d = v[0], *wave = v[1], *s = v[2], *amdq = v[3], *apdq = v[4], *qadd = v[5], *fadd = v[6];
    double *cqxx = (double *)calloc((size_t)n * meqn, sizeof(double));
    const size_t NXs = mx + 2 * mbc, NYs = my + 2 * mbc;
#define Q4(arr, m, i, j, k) arr[(m) + (size_t)meqn * (((i) + mbc - 1) + NXs * (((j) + mbc - 1) + NYs * ((k) + mbc - 1)))]
    const double dtd[3] = {dt / dx, dt / dy, dt / dz};
    const int len[3] = {mx, my, mz};
    double cfl = 0.0;
    const int d = idir - 1;
    const int o1 = (d == 0) ? 1 : 0, o2 = (d == 2) ? 1 : 2;
    int idx[3];
    for (idx[o2] = 0; idx[o2] <= len[o2] + 1; idx[o2]++)
        for (idx[o1] = 0; idx[o1] <= len[o1] + 1; idx[o1]++) {
            for (int l = 1 - mbc; l <= len[d] + mbc; l++) {
                idx[d] = l;
                for (int m = 0; m < meqn; m++) Q2(q1d, m, l) = Q4(qold, m, idx[0], idx[1], idx[2]);
            }
            if (ma > 0) slice_aux(aux, ma, mbc, mx, my, mz, d, idx, aux1d, aux9);
            double cfl1d = flux3_normal(&c, idir, meqn, mwaves, mbc, len[d], q1d, dtd[d], method[1], mthlim, wave, s,
                                        amdq, apdq, cqxx, qadd, fadd);
            cfl = dmax2(cfl, cfl1d);
            for (int l = 1; l <= len[d]; l++) {
                idx[d] = l;
                for (int m = 0; m < meqn; m++) {
                    double upd = dtd[d] * (Q2(fadd, m, l + 1) - Q2(fadd, m, l));
                    Q4(qnew, m, idx[0], idx[1], idx[2]) = Q4(qnew, m, idx[0], idx[1], idx[2]) + Q2(qadd, m, l) - upd;
                }
            }
        }
    for (int a = 0; a < 7; a++) free(v[a]);
    free(cqxx); free(aux1d); free(aux9);
    return cfl;
}

double oracle3d_step3ds(int rp_id, const double *rp_params, int meqn, int mwaves, int mbc, int mx, int my, int mz,
                        const double *qold, double *qnew, double dx, double dy, double dz, double dt,
                        const int *method, const int *mthlim, int idir)
{
    return oracle3d_step3ds_aux(rp_id, rp_params, meqn, mwaves, mbc, mx, my, mz, qold, qnew, NULL, 0, dx, dy, dz, dt,
                                method, mthlim, idir);
}

/* gadd / hadd (meqn, 2, -1:1, 1-mbc:maxm+mbc): k = 1..2, j = -1..1 */
#define GH(arr, m, k, j, i) arr[(m) + meqn * (((k) - 1) + 2 * (((j) + 1) + 3 * IX(i)))]

/* flux3.f:5-595 for a slice without aux data; qadd, fadd, gadd, hadd */
static double flux3(const rp_ctx3 *c, int ixyz, int meqn, int mwaves, int mbc, int mx, int n1d, const double *q1d,
                    double dtdx, double dtdy, double dtdz, const int *method, const int *mthlim, double *wave,
                    double *s, double *qadd, double *fadd, double *gadd, double *hadd, double **v)
{
    double *amdq = v[0], *apdq = v[1], *cqxx = v[2];
    double *bmamdq = v[3], *bmapdq = v[4], *bpamdq = v[5], *bpapdq = v[6];
    double *cmamdq = v[7], *cmapdq = v[8], *cpamdq = v[9], *cpapdq = v[10];
    double *cmamdq2 = v[11], *cmapdq2 = v[12], *cpamdq2 = v[13], *cpapdq2 = v[14];
    double *bmcqxxp = v[15], *bpcqxxp = v[16], *bmcqxxm = v[17], *bpcqxxm = v[18];
    double *cmcqxxp = v[19], *cpcqxxp = v[20], *cmcqxxm = v[21], *cpcqxxm = v[22];
    double *bmcmamdq = v[23], *bmcmapdq = v[24], *bpcmamdq = v[25], *bpcmapdq = v[26];
    double *bmcpamdq = v[27], *bmcpapdq = v[28], *bpcpamdq = v[29], *bpcpapdq = v[30];
    (void)n1d;
    for (int i = 1 - mbc; i <= mx + mbc; i++)
        for (int m = 0; m < meqn; m++)
            for (int k = 1; k <= 2; k++)
                for (int j = -1; j <= 1; j++) { GH(gadd, m, k, j, i) = 0.0; GH(hadd, m, k, j, i) = 0.0; }
    int m3, m4;
    if (method[2] < 0) { m3 = -1; m4 = 0; }
    else { m3 = method[2] / 10; m4 = method[2] - 10 * m3; }
    double cfl1d = flux3_normal(c, ixyz, meqn, mwaves, mbc, mx, q1d, dtdx, method[1], mthlim, wave, s, amdq, apdq,
                                cqxx, qadd, fadd);
    if (m3 <= 0) return cfl1d;

#define RPT3(icoor, imp, impt, as, bm, bp) rpt3(c, ixyz, icoor, imp, impt, mbc, mx, q1d, as, bm, bp)
    RPT3(2, 1, 0, amdq, bmamdq, bpamdq);
    RPT3(2, 2, 0, apdq, bmapdq, bpapdq);
    RPT3(3, 1, 0, amdq, cmamdq, cpamdq);
    RPT3(3, 2, 0, apdq, cmapdq, cpapdq);
    if (m3 == 2) { /* cqxx split with imp = 1 and imp = 2 (flux3.f:262-283) */
        RPT3(2, 1, 0, cqxx, bmcqxxm, bpcqxxm);
        RPT3(2, 2, 0, cqxx, bmcqxxp, bpcqxxp);
        RPT3(3, 1, 0, cqxx, cmcqxxm, cpcqxxm);
        RPT3(3, 2, 0, cqxx, cmcqxxp, cpcqxxp);
    }
    /* ---- G fluxes (y-like direction) ---- */
    if (m4 == 1) {
        for (int i = 0; i <= mx + 2; i++)
            for (int m = 0; m < meqn; m++) {
                Q2(cpapdq2, m, i) = Q2(cpapdq, m, i); Q2(cpamdq2, m, i) = Q2(cpamdq, m, i);
                Q2(cmapdq2, m, i) = Q2(cmapdq, m, i); Q2(cmamdq2, m, i) = Q2(cmamdq, m, i);
            }
    } else if (m4 == 2) {
        for (int i = 0; i <= mx + 2; i++)
            for (int m = 0; m < meqn; m++) {
                Q2(cpapdq2, m, i) = Q2(cpapdq, m, i) - 3.0 * Q2(cpcqxxp, m, i);
                Q2(cpamdq2, m, i) = Q2(cpamdq, m, i) + 3.0 * Q2(cpcqxxm, m, i);
                Q2(cmapdq2, m, i) = Q2(cmapdq, m, i) - 3.0 * Q2(cmcqxxp, m, i);
                Q2(cmamdq2, m, i) = Q2(cmamdq, m, i) + 3.0 * Q2(cmcqxxm, m, i);
            }
    }
    if (m4 > 0) { /* rptt3 */
        RPT3(2, 2, 2, cpapdq2, bmcpapdq, bpcpapdq);
        RPT3(2, 1, 2, cpamdq2, bmcpamdq, bpcpamdq);
        RPT3(2, 2, 1, cmapdq2, bmcmapdq, bpcmapdq);
        RPT3(2, 1, 1, cmamdq2, bmcmamdq, bpcmamdq);
    }
    const double sixth = 1.0 / 6.0;
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++) {
            const double dl = dtdx, dr = dtdx;
            GH(gadd, m, 1, 0, i - 1) = GH(gadd, m, 1, 0, i - 1) - 0.5 * dl * Q2(bmamdq, m, i);
            GH(gadd, m, 2, 0, i - 1) = GH(gadd, m, 2, 0, i - 1) - 0.5 * dl * Q2(bpamdq, m, i);
            GH(gadd, m, 1, 0, i) = GH(gadd, m, 1, 0, i) - 0.5 * dr * Q2(bmapdq, m, i);
            GH(gadd, m, 2, 0, i) = GH(gadd, m, 2, 0, i) - 0.5 * dr * Q2(bpapdq, m, i);
            if (m4 > 0) {
                GH(gadd, m, 2, 0, i) = GH(gadd, m, 2, 0, i) + sixth * dr * dtdz * (Q2(bpcpapdq, m, i) - Q2(bpcmapdq, m, i));
                GH(gadd, m, 1, 0, i) = GH(gadd, m, 1, 0, i) + sixth * dr * dtdz * (Q2(bmcpapdq, m, i) - Q2(bmcmapdq, m, i));
                GH(gadd, m, 2, 1, i) = GH(gadd, m, 2, 1, i) - sixth * dr * dtdz * Q2(bpcpapdq, m, i);
                GH(gadd, m, 1, 1, i) = GH(gadd, m, 1, 1, i) - sixth * dr * dtdz * Q2(bmcpapdq, m, i);
                GH(gadd, m, 2, -1, i) = GH(gadd, m, 2, -1, i) + sixth * dr * dtdz * Q2(bpcmapdq, m, i);
                GH(gadd, m, 1, -1, i) = GH(gadd, m, 1, -1, i) + sixth * dr * dtdz * Q2(bmcmapdq, m, i);
                GH(gadd, m, 2, 0, i - 1) = GH(gadd, m, 2, 0, i - 1) + sixth * dl * dtdz * (Q2(bpcpamdq, m, i) - Q2(bpcmamdq, m, i));
                GH(gadd, m, 1, 0, i - 1) = GH(gadd, m, 1, 0, i - 1) + sixth * dl * dtdz * (Q2(bmcpamdq, m, i) - Q2(bmcmamdq, m, i));
                GH(gadd, m, 2, 1, i - 1) = GH(gadd, m, 2, 1, i - 1) - sixth * dl * dtdz * Q2(bpcpamdq, m, i);
                GH(gadd, m, 1, 1, i - 1) = GH(gadd, m, 1, 1, i - 1) - sixth * dl * dtdz * Q2(bmcpamdq, m, i);
                GH(gadd, m, 2, -1, i - 1) = GH(gadd, m, 2, -1, i - 1) + sixth * dl * dtdz * Q2(bpcmamdq, m, i);
                GH(gadd, m, 1, -1, i - 1) = GH(gadd, m, 1, -1, i - 1) + sixth * dl * dtdz * Q2(bmcmamdq, m, i);
            }
            if (m3 >= 2) {
                GH(gadd, m, 2, 0, i) = GH(gadd, m, 2, 0, i) + dr * Q2(bpcqxxp, m, i);
                GH(gadd, m, 1, 0, i) = GH(gadd, m, 1, 0, i) + dr * Q2(bmcqxxp, m, i);
                GH(gadd, m, 2, 0, i - 1) = GH(gadd, m, 2, 0, i - 1) - dl * Q2(bpcqxxm, m, i);
                GH(gadd, m, 1, 0, i - 1) = GH(gadd, m, 1, 0, i - 1) - dl * Q2(bmcqxxm, m, i);
            }
        }
    /* ---- H fluxes (z-like direction) ---- */
    if (m4 == 2) {
        for (int i = 0; i <= mx + 2; i++)
            for (int m = 0; m < meqn; m++) {
                Q2(bpapdq, m, i) = Q2(bpapdq, m, i) - 3.0 * Q2(bpcqxxp, m, i);
                Q2(bpamdq, m, i) = Q2(bpamdq, m, i) + 3.0 * Q2(bpcqxxm, m, i);
                Q2(bmapdq, m, i) = Q2(bmapdq, m, i) - 3.0 * Q2(bmcqxxp, m, i);
                Q2(bmamdq, m, i) = Q2(bmamdq, m, i) + 3.0 * Q2(bmcqxxm, m, i);
            }
    }
    if (m4 > 0) { /* rptt3 */
        RPT3(3, 2, 2, bpapdq, bmcpapdq, bpcpapdq);
        RPT3(3, 1, 2, bpamdq, bmcpamdq, bpcpamdq);
        RPT3(3, 2, 1, bmapdq, bmcmapdq, bpcmapdq);
        RPT3(3, 1, 1, bmamdq, bmcmamdq, bpcmamdq);
    }
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++) {
            const double dl = dtdx, dr = dtdx;
            GH(hadd, m, 1, 0, i - 1) = GH(hadd, m, 1, 0, i - 1) - 0.5 * dl * Q2(cmamdq, m, i);
            GH(hadd, m, 2, 0, i - 1) = GH(hadd, m, 2, 0, i - 1) - 0.5 * dl * Q2(cpamdq, m, i);
            GH(hadd, m, 1, 0, i) = GH(hadd, m, 1, 0, i) - 0.5 * dr * Q2(cmapdq, m, i);
            GH(hadd, m, 2, 0, i) = GH(hadd, m, 2, 0, i) - 0.5 * dr * Q2(cpapdq, m, i);
            if (m4 > 0) {
                GH(hadd, m, 2, 0, i) = GH(hadd, m, 2, 0, i) + sixth * dr * dtdy * (Q2(bpcpapdq, m, i) - Q2(bpcmapdq, m, i));
                GH(hadd, m, 1, 0, i) = GH(hadd, m, 1, 0, i) + sixth * dr * dtdy * (Q2(bmcpapdq, m, i) - Q2(bmcmapdq, m, i));
                GH(hadd, m, 2, 1, i) = GH(hadd, m, 2, 1, i) - sixth * dr * dtdy * Q2(bpcpapdq, m, i);
                GH(hadd, m, 1, 1, i) = GH(hadd, m, 1, 1, i) - sixth * dr * dtdy * Q2(bmcpapdq, m, i);
                GH(hadd, m, 2, -1, i) = GH(hadd, m, 2, -1, i) + sixth * dr * dtdy * Q2(bpcmapdq, m, i);
                GH(hadd, m, 1, -1, i) = GH(hadd, m, 1, -1, i) + sixth * dr * dtdy * Q2(bmcmapdq, m, i);
                GH(hadd, m, 2, 0, i - 1) = GH(hadd, m, 2, 0, i - 1) + sixth * dl * dtdy * (Q2(bpcpamdq, m, i) - Q2(bpcmamdq, m, i));
                GH(hadd, m, 1, 0, i - 1) = GH(hadd, m, 1, 0, i - 1) + sixth * dl * dtdy * (Q2(bmcpamdq, m, i) - Q2(bmcmamdq, m, i));
                GH(hadd, m, 2, 1, i - 1) = GH(hadd, m, 2, 1, i - 1) - sixth * dl * dtdy * Q2(bpcpamdq, m, i);
                GH(hadd, m, 1, 1, i - 1) = GH(hadd, m, 1, 1, i - 1) - sixth * dl * dtdy * Q2(bmcpamdq, m, i);
                GH(hadd, m, 2, -1, i - 1) = GH(hadd, m, 2, -1, i - 1) + sixth * dl * dtdy * Q2(bpcmamdq, m, i);
                GH(hadd, m, 1, -1, i - 1) = GH(hadd, m, 1, -1, i - 1) + sixth * dl * dtdy * Q2(bmcmamdq, m, i);
            }
            if (m3 >= 2) {
                GH(hadd, m, 2, 0, i) = GH(hadd, m, 2, 0, i) + dr * Q2(cpcqxxp, m, i);
                GH(hadd, m, 1, 0, i) = GH(hadd, m, 1, 0, i) + dr * Q2(cmcqxxp, m, i);
                GH(hadd, m, 2, 0, i - 1) = GH(hadd, m, 2, 0, i - 1) - dl * Q2(cpcqxxm, m, i);
                GH(hadd, m, 1, 0, i - 1) = GH(hadd, m, 1, 0, i - 1) - dl * Q2(cmcqxxm, m, i);
            }
        }
#undef RPT3
    return cfl1d;
}

/* step3.f:2-594.  qnew == qold on entry; q(meqn, 1-mbc:mx+mbc, ...). */
double oracle3d_step3_aux(int rp_id, const double *rp_params, int meqn, int mwaves, int mbc, int mx, int my, int mz,
                          const double *qold, double *qnew, const double *aux, int maux, double dx, double dy,
                          double dz, double dt, const int *method, const int *mthlim)
{
    if (!known(rp_id) || method[5] > 0 || !aux_ok(rp_id, aux, maux, mbc)) return -1.0;
    rp_ctx3 c = {0};
    c.rp_id = rp_id;
    memcpy(c.p, rp_params, 8 * sizeof(double));
    int maxm = mx > my ? mx : my;
    if (mz > maxm) maxm = mz;
    const int n1d = maxm + 2 * mbc;
    const int ma = aux ? maux : 0;
    double *aux1d = (double *)calloc((size_t)n1d * (ma > 0 ? ma : 1), sizeof(double));
    double *aux9 = (double *)calloc((size_t)n1d * 9 * (ma > 0 ? ma : 1), sizeof(double));
    c.maux = ma;
    c.aux1d = aux1d;
    c.aux9 = aux9;
    const size_t nm = (size_t)n1d * meqn;
    double *q1d = (double *)calloc(nm, sizeof(double)), *qadd = (double *)calloc(nm, sizeof(double));
    double *fadd = (double *)calloc(nm, sizeof(double));
    double *gadd = (double *)calloc(nm * 6, sizeof(double)), *hadd = (double *)calloc(nm * 6, sizeof(double));
    double *wave = (double *)calloc(nm * mwaves, sizeof(double)), *s = (double *)calloc((size_t)n1d * mwaves, sizeof(double));
    double *v[31];
    for (int a = 0; a < 31; a++) v[a] = (double *)calloc(nm, sizeof(double));
    const size_t NXs = mx + 2 * mbc, NYs = my + 2 * mbc;
    const double dtd[3] = {dt / dx, dt / dy, dt / dz};
    const int len[3] = {mx, my, mz};
    double cfl = 0.0;
    for (int d = 0; d < 3; d++) {
        const int e = (d + 1) % 3, f = (d + 2) % 3; /* y-like, z-like directions of this sweep */
        const int o1 = (d == 0) ? 1 : 0;            /* the two other directions: lower one is the inner loop */
        const int o2 = (d == 2) ? 1 : 2;
        const double dtde = dtd[e], dtdf = dtd[f];
        int idx[3];
        for (idx[o2] = 0; idx[o2] <= len[o2] + 1; idx[o2]++)
            for (idx[o1] = 0; idx[o1] <= len[o1] + 1; idx[o1]++) {
                for (int l = 1 - mbc; l <= len[d] + mbc; l++) {
                    idx[d] = l;
                    for (int m = 0; m < meqn; m++) Q2(q1d, m, l) = Q4(qold, m, idx[0], idx[1], idx[2]);
                }
                if (ma > 0) slice_aux(aux, ma, mbc, mx, my, mz, d, idx, aux1d, aux9);
                double cfl1d = flux3(&c, d + 1, meqn, mwaves, mbc, len[d], n1d, q1d, dtd[d], dtde, dtdf, method, mthlim,
                                     wave, s, qadd, fadd, gadd, hadd, v);
                cfl = dmax2(cfl, cfl1d);
                /* step3.f:185-220 (x), 340-377 (y), 497-534 (z); (eo, fo) = offset in the y-like / z-like direction */
                for (int l = 1; l <= len[d]; l++)
                    for (int m = 0; m < meqn; m++) {
                        int p[3];
#define QN(eo, fo) (p[0] = idx[0], p[1] = idx[1], p[2] = idx[2], p[d] = l, p[e] += (eo), p[f] += (fo), &Q4(qnew, m, p[0], p[1], p[2]))
                        double *t;
                        t = QN(0, 0);
                        *t = *t + Q2(qadd, m, l) - dtd[d] * (Q2(fadd, m, l + 1) - Q2(fadd, m, l))
                             - dtde * (GH(gadd, m, 2, 0, l) - GH(gadd, m, 1, 0, l))
                             - dtdf * (GH(hadd, m, 2, 0, l) - GH(hadd, m, 1, 0, l));
                        t = QN(-1, 0);
                        *t = *t - dtde * GH(gadd, m, 1, 0, l) - dtdf * (GH(hadd, m, 2, -1, l) - GH(hadd, m, 1, -1, l));
                        t = QN(-1, -1);
                        *t = *t - dtde * GH(gadd, m, 1, -1, l) - dtdf * GH(hadd, m, 1, -1, l);
                        t = QN(0, -1);
                        *t = *t - dtde * (GH(gadd, m, 2, -1, l) - GH(gadd, m, 1, -1, l)) - dtdf * GH(hadd, m, 1, 0, l);
                        t = QN(1, -1);
                        *t = *t + dtde * GH(gadd, m, 2, -1, l) - dtdf * GH(hadd, m, 1, 1, l);
                        t = QN(1, 0);
                        *t = *t + dtde * GH(gadd, m, 2, 0, l) - dtdf * (GH(hadd, m, 2, 1, l) - GH(hadd, m, 1, 1, l));
                        t = QN(1, 1);
                        *t = *t + dtde * GH(gadd, m, 2, 1, l) + dtdf * GH(hadd, m, 2, 1, l);
                        t = QN(0, 1);
                        *t = *t - dtde * (GH(gadd, m, 2, 1, l) - GH(gadd, m, 1, 1, l)) + dtdf * GH(hadd, m, 2, 0, l);
                        t = QN(-1, 1);
                        *t = *t - dtde * GH(gadd, m, 1, 1, l) + dtdf * GH(hadd, m, 2, -1, l);
#undef QN
                    }
            }
    }
    free(q1d); free(qadd); free(fadd); free(gadd); free(hadd); free(wave); free(s); free(aux1d); free(aux9);
    for (int a = 0; a < 31; a++) free(v[a]);
    return cfl;
}

double oracle3d_step3(int rp_id, const double *rp_params, int meqn, int mwaves, int mbc, int mx, int my, int mz,
                      const double *qold, double *qnew, double dx, double dy, double dz, double dt,
                      const int *method, const int *mthlim)
{
    return oracle3d_step3_aux(rp_id, rp_params, meqn, mwaves, mbc, mx, my, mz, qold, qnew, NULL, 0, dx, dy, dz, dt,
                              method, mthlim);
}
#undef Q4

/* ------------------------------------------------------------------------- */
/* Pointwise rpn3 / rpt3 (property tests): n interfaces ql | qr (structure of */
/* arrays [m][n]), presented as a 3-cell slice left | right | right (mbc = 1,  */
/* mx = 1, interface i = 1).  asdq == NULL: rpn3 into wave, s, amdq, apdq;     */
/* otherwise rpt3 / rptt3 of asdq in direction icoor into bm, bp.              */
/* ------------------------------------------------------------------------- */
/* With aux data (maux > 0): auxl / auxr [maux][n] are the cells left / right of each interface (rpn3),
   aux9 [maux][3][3][n] the 3x3 cells around the cell the fluctuation enters, [ma][e+1][f+1] at the
   offset e / f in the y-like / z-like direction (rpt3; rptt3 with impt = 1, 2). */
void oracle3d_rp_point_aux(int rp_id, const double *rp_params, int ixyz, int meqn, int mwaves, int maux, long long n,
                           const double *ql, const double *qr, const double *auxl_i, const double *auxr_i,
                           double *wave_o, double *s_o, double *amdq_o, double *apdq_o, int icoor, int imp,
                           int impt, const double *aux9_i, const double *asdq_i, double *bm_o, double *bp_o)
{
    const int mbc = 1, mx = 1, nc = 3;
    rp_ctx3 c = {0};
    c.rp_id = rp_id;
    memcpy(c.p, rp_params, 8 * sizeof(double));
    const int ma = maux > 0 ? maux : 1;
    double *aux1d = (double *)calloc((size_t)ma * nc, sizeof(double));
    double *aux9 = (double *)calloc((size_t)ma * 9 * nc, sizeof(double));
    c.maux = maux;
    c.aux1d = aux1d;
    c.aux9 = aux9;
    double *q = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *wave = (double *)calloc((size_t)meqn * mwaves * nc, sizeof(double));
    double *s = (double *)calloc((size_t)mwaves * nc, sizeof(double));
    double *amdq = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *apdq = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *asdq = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *bm = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *bp = (double *)calloc((size_t)meqn * nc, sizeof(double));
    for (long long k = 0; k < n; k++) {
        for (int m = 0; m < meqn; m++) {
            Q2(q, m, 0) = ql[m * n + k];
            Q2(q, m, 1) = qr[m * n + k];
            Q2(q, m, 2) = qr[m * n + k];
        }
        for (int a = 0; a < maux; a++) {
            if (auxl_i) {
                aux1d[a + maux * 0] = auxl_i[a * n + k];
                aux1d[a + maux * 1] = auxr_i[a * n + k];
                aux1d[a + maux * 2] = auxr_i[a * n + k];
            }
            if (aux9_i)
                for (int e = 0; e < 3; e++)
                    for (int f = 0; f < 3; f++)
                        for (int i = 0; i <= 2; i++)
                            aux9[a + maux * (e + 3 * f) + (size_t)9 * maux * i] = aux9_i[(((size_t)a * 3 + e) * 3 + f) * n + k];
        }
        if (!asdq_i) {
            rpn3(&c, ixyz, mbc, mx, q, q, wave, s, amdq, apdq);
            for (int m = 0; m < meqn; m++) {
                for (int mw = 0; mw < mwaves; mw++) wave_o[(m * mwaves + mw) * n + k] = WV(m, mw, 1);
                amdq_o[m * n + k] = Q2(amdq, m, 1);
                apdq_o[m * n + k] = Q2(apdq, m, 1);
            }
            for (int mw = 0; mw < mwaves; mw++) s_o[mw * n + k] = SP(mw, 1);
        } else {
            for (int m = 0; m < meqn; m++)
                for (int i = 0; i <= 2; i++) Q2(asdq, m, i) = asdq_i[m * n + k];
            rpt3(&c, ixyz, icoor, imp, impt, mbc, mx, q, asdq, bm, bp);
            for (int m = 0; m < meqn; m++) {
                bm_o[m * n + k] = Q2(bm, m, 1);
                bp_o[m * n + k] = Q2(bp, m, 1);
            }
        }
    }
    free(q); free(wave); free(s); free(amdq); free(apdq); free(asdq); free(bm); free(bp); free(aux1d); free(aux9);
}

void oracle3d_rp_point(int rp_id, const double *rp_params, int ixyz, int meqn, int mwaves, long long n,
                       const double *ql, const double *qr, double *wave_o, double *s_o, double *amdq_o,
                       double *apdq_o, int icoor, const double *asdq_i, double *bm_o, double *bp_o)
{
    oracle3d_rp_point_aux(rp_id, rp_params, ixyz, meqn, mwaves, 0, n, ql, qr, NULL, NULL, wave_o, s_o, amdq_o, apdq_o,
                          icoor, 2, 0, NULL, asdq_i, bm_o, bp_o);
}

/* =========================================================================================== */
/* SharpClaw in 3-D (the reference has none): flux1 (src/fortran/1d/sharpclaw/flux1.f90:2-195)  */
/* over the x-, y- and z-slices of the grid, flux2.f90:2-96 extended by one dimension            */
/* (DESIGN.md §1).  The reconstructions, flux1 and rpn3_vc_acoustics are copied from             */
/* oracle/claw_oracle.c (weno5_pyweno, weno5_old, tvd2, sc_flux1_capa without a capacity         */
/* function, rpn3_vc_acoustics) and pinned against it bit for bit by tests/test_sc3_oracle.py.    */
/* =========================================================================================== */
#define RP_ACOUSTICS3D_VC 8 /* aux = impedance, sound speed */
#define WENO_PYWENO_F32 0
#define WENO_PYWENO_F64 1
#define WENO_OLD 2
#define RECON_TVD2 4

/* rpn3_vc_acoustics.f (oracle/claw_oracle.c) */
static void rpn3_vc_acoustics(int ixyz, int meqn, int mwaves, int mbc, int mx, int maux,
                              const double *ql, const double *qr, const double *auxl,
                              const double *auxr, double *wave, double *s, double *amdq,
                              double *apdq)
{
    const int mu = ixyz;
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        double delta1 = Q2(ql, 0, i) - Q2(qr, 0, i - 1);
        double delta2 = Q2(ql, mu, i) - Q2(qr, mu, i - 1);
        double zi = auxl[0 + maux * IX(i)], zim = auxr[0 + maux * IX(i - 1)];
        double a1 = (-delta1 + zi * delta2) / (zim + zi);
        double a2 = (delta1 + zim * delta2) / (zim + zi);
        for (int m = 0; m < meqn; m++) { WV(m, 0, i) = 0.0; WV(m, 1, i) = 0.0; }
        WV(0, 0, i) = -a1 * zim;
        WV(mu, 0, i) = a1;
        SP(0, i) = -auxr[1 + maux * IX(i - 1)];
        WV(0, 1, i) = a2 * zi;
        WV(mu, 1, i) = a2;
        SP(1, i) = auxl[1 + maux * IX(i)];
        for (int m = 0; m < meqn; m++) {
            Q2(amdq, m, i) = SP(0, i) * WV(m, 0, i);
            Q2(apdq, m, i) = SP(1, i) * WV(m, 1, i);
        }
    }
    (void)mwaves;
}

/* the normal solve of a SharpClaw slice: every 3-D solver of this file */
static void rpn3_sc(const rp_ctx3 *c, int ixyz, int meqn, int mwaves, int mbc, int mx, int maux, const double *ql,
                    const double *qr, const double *auxl, const double *auxr, double *wave, double *s, double *amdq,
                    double *apdq)
{
    if (c->rp_id == RP_ACOUSTICS3D_VC)
        rpn3_vc_acoustics(ixyz, meqn, mwaves, mbc, mx, maux, ql, qr, auxl, auxr, wave, s, amdq, apdq);
    else if (c->rp_id == RP_ADVECTION3D_VC_FWAVE)
        rpn3_vc_fwave(ixyz, mbc, mx, maux, ql, qr, auxl, auxr, wave, s, amdq, apdq);
    else rpn3(c, ixyz, mbc, mx, ql, qr, wave, s, amdq, apdq);
}

#define QP(arr, m, p) arr[(m) + meqn * ((p)-1)]

/* weno.f90:5-102 (PyWENO generated), as oracle/claw_oracle.c weno5_pyweno */
static void weno5_pyweno(const double *q, double *ql, double *qr, int meqn, int mx, int mbc,
                         int f32lit)
{
#define LIT(x) (f32lit ? (double)(x##f) : (double)(x))
    const double c333 = LIT(3.33333333333333), c1033 = LIT(10.3333333333333),
                 c366 = LIT(3.66666666666667), c833 = LIT(8.33333333333333),
                 c633 = LIT(6.33333333333333), c133 = LIT(1.33333333333333),
                 c433 = LIT(4.33333333333333), c166 = LIT(1.66666666666667);
    const double d01 = LIT(0.1), d06 = LIT(0.6), d03 = LIT(0.3), eps = LIT(1.0e-36);
    const double r183 = LIT(1.83333333333333), r116 = LIT(1.16666666666667),
                 r0333 = LIT(0.333333333333333), r0833 = LIT(0.833333333333333),
                 r0166 = LIT(0.166666666666667);
#undef LIT
    for (int p = mbc; p <= mx + mbc + 1; p++) {
        for (int m = 0; m < meqn; m++) {
            double qm2 = QP(q, m, p - 2), qm1 = QP(q, m, p - 1), q0 = QP(q, m, p),
                   qp1 = QP(q, m, p + 1), qp2 = QP(q, m, p + 2);
            double sigma0 = ((c333)*q0) * q0 + ((-c1033) * q0) * qp1 + ((c366)*q0) * qp2 +
                            ((c833)*qp1) * qp1 + ((-c633) * qp1) * qp2 + ((c133)*qp2) * qp2;
            double sigma1 = ((c133)*qm1) * qm1 + ((-c433) * qm1) * q0 + ((c166)*qm1) * qp1 +
                            ((c433)*q0) * q0 + ((-c433) * q0) * qp1 + ((c133)*qp1) * qp1;
            double sigma2 = ((c133)*qm2) * qm2 + ((-c633) * qm2) * qm1 + ((c366)*qm2) * q0 +
                            ((c833)*qm1) * qm1 + ((-c1033) * qm1) * q0 + ((c333)*q0) * q0;
            double acc = 0.0;
            double omega0 = d01 / ((sigma0 + eps) * (sigma0 + eps));
            acc = acc + omega0;
            double omega1 = d06 / ((sigma1 + eps) * (sigma1 + eps));
            acc = acc + omega1;
            double omega2 = d03 / ((sigma2 + eps) * (sigma2 + eps));
            acc = acc + omega2;
            omega0 = omega0 / acc;
            omega1 = omega1 / acc;
            omega2 = omega2 / acc;
            acc = 0.0;
            double omega3 = d03 / ((sigma0 + eps) * (sigma0 + eps));
            acc = acc + omega3;
            double omega4 = d06 / ((sigma1 + eps) * (sigma1 + eps));
            acc = acc + omega4;
            double omega5 = d01 / ((sigma2 + eps) * (sigma2 + eps));
            acc = acc + omega5;
            omega3 = omega3 / acc;
            omega4 = omega4 / acc;
            omega5 = omega5 / acc;
            double fr0 = (r183)*q0 + (-r116) * qp1 + (r0333)*qp2;
            double fr1 = (r0333)*qm1 + (r0833)*q0 + (-r0166) * qp1;
            double fr2 = (-r0166) * qm2 + (r0833)*qm1 + (r0333)*q0;
            double fr3 = (r0333)*q0 + (r0833)*qp1 + (-r0166) * qp2;
            double fr4 = (-r0166) * qm1 + (r0833)*q0 + (r0333)*qp1;
            double fr5 = (r0333)*qm2 + (-r116) * qm1 + (r183)*q0;
            QP(ql, m, p) = omega0 * fr0 + omega1 * fr1 + omega2 * fr2;
            QP(qr, m, p) = omega3 * fr3 + omega4 * fr4 + omega5 * fr5;
        }
    }
}

/* reconstruct.f90:120-185 (hand-written weno5, lim_type = 3), as oracle/claw_oracle.c weno5_old */
static void weno5_old(const double *q, double *ql, double *qr, int meqn, int mx, int mbc,
                      double *dq1m, double *uu)
{
    const double epweno = (double)1.e-36f; /* "1.e-36" is a REAL(4) literal, reconstruct.f90:7 */
    int mx2 = mx + 2 * mbc;
    for (int m = 0; m < meqn; m++) {
        for (int p = 2; p <= mx2; p++) dq1m[p] = QP(q, m, p) - QP(q, m, p - 1);
        for (int m1 = 1; m1 <= 2; m1++) {
            int im = (m1 == 1) ? 1 : -1;
            int ione = im, inone = -im, intwo = -2 * im;
            for (int p = mbc; p <= mx2 - mbc + 1; p++) {
                double t1 = im * (dq1m[p + intwo] - dq1m[p + inone]);
                double t2 = im * (dq1m[p + inone] - dq1m[p]);
                double t3 = im * (dq1m[p] - dq1m[p + ione]);
                double e1 = dq1m[p + intwo] - 3. * dq1m[p + inone];
                double e2 = dq1m[p + inone] + dq1m[p];
                double e3 = 3. * dq1m[p] - dq1m[p + ione];
                double tt1 = 13. * (t1 * t1) + 3. * (e1 * e1);
                double tt2 = 13. * (t2 * t2) + 3. * (e2 * e2);
                double tt3 = 13. * (t3 * t3) + 3. * (e3 * e3);
                tt1 = (epweno + tt1) * (epweno + tt1);
                tt2 = (epweno + tt2) * (epweno + tt2);
                tt3 = (epweno + tt3) * (epweno + tt3);
                double s1 = tt2 * tt3;
                double s2 = 6. * tt1 * tt3;
                double s3 = 3. * tt1 * tt2;
                double t0 = 1. / (s1 + s2 + s3);
                s1 = s1 * t0;
                s3 = s3 * t0;
                uu[(m1 - 1) + 2 * p] =
                    (s1 * (t2 - t1) + (0.5 * s3 - 0.25) * (t3 - t2)) / 3. +
                    (-QP(q, m, p - 2) + 7. * (QP(q, m, p - 1) + QP(q, m, p)) - QP(q, m, p + 1)) / 12.;
            }
        }
        for (int p = mbc; p <= mx2 - mbc + 1; p++) {
            QP(qr, m, p - 1) = uu[0 + 2 * p];
            QP(ql, m, p) = uu[1 + 2 * p];
        }
    }
}

/* gfortran's MIN / MAX: a NaN argument loses (oracle/claw_oracle.c) */
static inline double fmin_g(double a1, double a2) { return (a2 < a1 || a1 != a1) ? a2 : a1; }
static inline double fmax_g(double a1, double a2) { return (a2 > a1 || a1 != a1) ? a2 : a1; }

/* reconstruct.f90:568-625 (tvd2), as oracle/claw_oracle.c tvd2 with the limiter per component
   passed in (mthlim[m]) instead of set beforehand; the first cell uses its own backward difference */
static void tvd2(const double *q, double *ql, double *qr, int meqn, int mx, int mbc, const int *mthlim)
{
    const int mx2 = mx + 2 * mbc;
    for (int m = 0; m < meqn; m++) {
        double dqp = QP(q, m, 3) - QP(q, m, 2);
        for (int p = 3; p <= mx2 - 2; p++) {
            double dqm = dqp;
            dqp = QP(q, m, p + 1) - QP(q, m, p);
            double r = dqp / dqm;
            double qlimitr = 0.0;
            switch (mthlim[m]) {
            case 1: qlimitr = fmax_g(0.0, fmin_g(1.0, r)); break;
            case 2: qlimitr = fmax_g(fmax_g(0.0, fmin_g(1.0, 2.0 * r)), fmin_g(2.0, r)); break;
            case 3: qlimitr = (r + fabs(r)) / (1.0 + fabs(r)); break;
            case 4: {
                double c = (1.0 + r) / 2.0;
                qlimitr = fmax_g(0.0, fmin_g(fmin_g(c, 2.0), 2.0 * r));
            } break;
            case 5: {
                const double beta = 2.0, xgamma = 2.0, alpha = 1.0 / 3.0;
                double pp = (2.0 + r) / 3.0;
                double amax = fmax_g(fmax_g(-alpha * r, 0.0), fmin_g(fmin_g(beta * r, pp), xgamma));
                qlimitr = fmax_g(0.0, fmin_g(pp, amax));
            } break;
            default: qlimitr = 0.0;
            }
            QP(qr, m, p) = QP(q, m, p) + 0.5 * qlimitr * dqm;
            QP(ql, m, p) = QP(q, m, p) - 0.5 * qlimitr * dqm;
        }
    }
}

typedef struct {
    double *ql, *qr, *wave, *s, *amdq, *apdq, *amdq2, *apdq2, *dq1m, *uu, *auxl2, *auxr2;
} sc_work;

/* flux1.f90:2-195 on one slice (sc_flux1_capa of oracle/claw_oracle.c without a capacity function):
   dq1d = 0 - dtdx (amdq(i+1) + apdq(i) + amdq2(i) + apdq2(i)) for i = 1..mx; returns the Courant number
   of the interfaces 1..mx+1.  aux1d (maux, n) or NULL. */
static double sc_flux1(const rp_ctx3 *c, const double *q1d, const double *aux1d, int maux, double *dq1d, double dt,
                       double dxv, int ixyz, int meqn, int mwaves, int mx, int mbc, int weno_variant,
                       const int *mthlim, sc_work *w)
{
    int n = mx + 2 * mbc;
    double *ql = w->ql, *qr = w->qr, *wave = w->wave, *s = w->s;
    double *amdq = w->amdq, *apdq = w->apdq, *amdq2 = w->amdq2, *apdq2 = w->apdq2;
    const double dtdx = dt / dxv;
    for (int k = 0; k < n * meqn; k++) dq1d[k] = 0.0;
    memcpy(ql, q1d, sizeof(double) * n * meqn);
    memcpy(qr, q1d, sizeof(double) * n * meqn);
    if (weno_variant == RECON_TVD2) tvd2(q1d, ql, qr, meqn, mx, mbc, mthlim);
    else if (weno_variant == WENO_OLD) weno5_old(q1d, ql, qr, meqn, mx, mbc, w->dq1m, w->uu);
    else weno5_pyweno(q1d, ql, qr, meqn, mx, mbc, weno_variant == WENO_PYWENO_F32);
    /* :128 rp(ql, qr, aux, aux) */
    rpn3_sc(c, ixyz, meqn, mwaves, mbc, mx, maux, ql, qr, aux1d, aux1d, wave, s, amdq, apdq);
    double cfl = 0.0;
    for (int mw = 0; mw < mwaves; mw++)
        for (int i = 1; i <= mx + 1; i++) cfl = dmax2(dmax2(cfl, dtdx * SP(mw, i)), -dtdx * SP(mw, i));
    /* :170-175 swap so that interface i of the second solve is the in-cell problem */
    for (int i = 1 - mbc + 1; i <= mx + mbc; i++)
        for (int m = 0; m < meqn; m++) {
            Q2(qr, m, i - 1) = Q2(ql, m, i);
            Q2(ql, m, i) = Q2(qr, m, i);
        }
    const double *auxl2 = NULL, *auxr2 = NULL;
    if (aux1d && maux > 0) { /* :177-184 auxr(i-1) = aux(i), auxl(i) = aux(i) */
        memcpy(w->auxl2, aux1d, sizeof(double) * n * maux);
        memcpy(w->auxr2, aux1d, sizeof(double) * n * maux);
        for (int i = 1 - mbc + 1; i <= mx + mbc; i++)
            for (int ma = 0; ma < maux; ma++) {
                w->auxr2[ma + maux * IX(i - 1)] = aux1d[ma + maux * IX(i)];
                w->auxl2[ma + maux * IX(i)] = aux1d[ma + maux * IX(i)];
            }
        auxl2 = w->auxl2;
        auxr2 = w->auxr2;
    }
    rpn3_sc(c, ixyz, meqn, mwaves, mbc, mx, maux, ql, qr, auxl2, auxr2, wave, s, amdq2, apdq2);
    for (int i = 1; i <= mx; i++)
        for (int m = 0; m < meqn; m++)
            Q2(dq1d, m, i) = Q2(dq1d, m, i) -
                             dtdx * (Q2(amdq, m, i + 1) + Q2(apdq, m, i) + Q2(amdq2, m, i) + Q2(apdq2, m, i));
    return cfl;
}

static int sc_known(int rp_id, int weno_variant)
{
    return (known(rp_id) || rp_id == RP_ACOUSTICS3D_VC) &&
           (weno_variant == WENO_PYWENO_F32 || weno_variant == WENO_PYWENO_F64 || weno_variant == WENO_OLD ||
            weno_variant == RECON_TVD2);
}

static void sc_work_alloc(sc_work *w, int n, int meqn, int mwaves, int maux)
{
    double **a[] = {&w->ql, &w->qr, &w->amdq, &w->apdq, &w->amdq2, &w->apdq2};
    for (int k = 0; k < 6; k++) *a[k] = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->wave = (double *)calloc((size_t)n * meqn * mwaves, sizeof(double));
    w->s = (double *)calloc((size_t)n * mwaves, sizeof(double));
    w->dq1m = (double *)calloc(n + 2, sizeof(double));
    w->uu = (double *)calloc(2 * (size_t)(n + 2), sizeof(double));
    w->auxl2 = (double *)calloc((size_t)n * (maux > 0 ? maux : 1), sizeof(double));
    w->auxr2 = (double *)calloc((size_t)n * (maux > 0 ? maux : 1), sizeof(double));
}
static void sc_work_free(sc_work *w)
{
    free(w->ql); free(w->qr); free(w->amdq); free(w->apdq); free(w->amdq2); free(w->apdq2);
    free(w->wave); free(w->s); free(w->dq1m); free(w->uu); free(w->auxl2); free(w->auxr2);
}

/* One slice (flux1) on its own: q1d (meqn, mx+2mbc), aux1d (maux, mx+2mbc) or NULL, dq1d out.
   ixyz = 1, 2, 3 is the direction of the slice.  Returns the Courant number, -1 if unsupported. */
double oracle3d_sc_flux1(int rp_id, const double *rp_params, int meqn, int mwaves, int maux, int mbc, int mx,
                         const double *q1d, const double *aux1d, double *dq1d, double dx, double dt, int ixyz,
                         int weno_variant, const int *mthlim)
{
    if (!sc_known(rp_id, weno_variant)) return -1.0;
    rp_ctx3 c = {0};
    c.rp_id = rp_id;
    memcpy(c.p, rp_params, 8 * sizeof(double));
    sc_work w;
    sc_work_alloc(&w, mx + 2 * mbc, meqn, mwaves, maux);
    double cfl = sc_flux1(&c, q1d, aux1d, maux, dq1d, dt, dx, ixyz, meqn, mwaves, mx, mbc, weno_variant, mthlim, &w);
    sc_work_free(&w);
    return cfl;
}

/* flux3 of SharpClaw in 3-D: q (meqn, NX, NY, NZ) Fortran order with ghost cells filled, aux (maux, ...)
   or NULL, dq zero on entry; dq(:, i, j, k) = ((0 + dq_x) + dq_y) + dq_z on the interior.  Slices: x over
   (j, k) in [0, my+1] x [0, mz+1], y over (i, k) in [0, mx+1] x [0, mz+1], z over (i, j) in [0, mx+1] x
   [0, my+1].  Returns the largest Courant number of all slices, -1 if unsupported. */
double oracle3d_sc_flux3(int rp_id, const double *rp_params, int meqn, int mwaves, int maux, int mbc, int mx,
                         int my, int mz, const double *q, const double *aux, double *dq, double dx, double dy,
                         double dz, double dt, int weno_variant, const int *mthlim)
{
    if (!sc_known(rp_id, weno_variant)) return -1.0;
    if (rp_id == RP_ACOUSTICS3D_VC && (!aux || maux < 2)) return -1.0;
    if (rp_id == RP_ADVECTION3D_VC_FWAVE && (!aux || maux < 3)) return -1.0;
    rp_ctx3 c = {0};
    c.rp_id = rp_id;
    memcpy(c.p, rp_params, 8 * sizeof(double));
    int maxm = mx > my ? mx : my;
    if (mz > maxm) maxm = mz;
    const int n = maxm + 2 * mbc;
    const int ma = aux ? maux : 0;
    sc_work w;
    sc_work_alloc(&w, n, meqn, mwaves, ma);
    double *q1d = (double *)calloc((size_t)n * meqn, sizeof(double));
    double *dq1d = (double *)calloc((size_t)n * meqn, sizeof(double));
    double *aux1d = (double *)calloc((size_t)n * (ma > 0 ? ma : 1), sizeof(double));
    const size_t NXs = mx + 2 * mbc, NYs = my + 2 * mbc;
#define OFF4(i, j, k) (((i) + mbc - 1) + NXs * (((j) + mbc - 1) + NYs * ((k) + mbc - 1)))
#define Q4(arr, m, i, j, k) arr[(m) + (size_t)meqn * OFF4(i, j, k)]
#define AUX4(a, i, j, k) aux[(a) + (size_t)ma * OFF4(i, j, k)]
    const double dd[3] = {dx, dy, dz};
    const int len[3] = {mx, my, mz};
    double cfl = 0.0;
    for (int d = 0; d < 3; d++) {
        const int o1 = (d == 0) ? 1 : 0, o2 = (d == 2) ? 1 : 2;
        int idx[3];
        for (idx[o2] = 0; idx[o2] <= len[o2] + 1; idx[o2]++)
            for (idx[o1] = 0; idx[o1] <= len[o1] + 1; idx[o1]++) {
                for (int l = 1 - mbc; l <= len[d] + mbc; l++) {
                    idx[d] = l;
                    for (int m = 0; m < meqn; m++) Q2(q1d, m, l) = Q4(q, m, idx[0], idx[1], idx[2]);
                    for (int a = 0; a < ma; a++) aux1d[a + ma * IX(l)] = AUX4(a, idx[0], idx[1], idx[2]);
                }
                double cfl1d = sc_flux1(&c, q1d, ma > 0 ? aux1d : NULL, ma, dq1d, dt, dd[d], d + 1, meqn, mwaves,
                                        len[d], mbc, weno_variant, mthlim, &w);
                cfl = dmax2(cfl, cfl1d);
                const int interior = idx[o1] >= 1 && idx[o1] <= len[o1] && idx[o2] >= 1 && idx[o2] <= len[o2];
                if (!interior) continue; /* ghost slices: Courant number only */
                for (int l = 1; l <= len[d]; l++) {
                    idx[d] = l;
                    for (int m = 0; m < meqn; m++)
                        Q4(dq, m, idx[0], idx[1], idx[2]) = Q4(dq, m, idx[0], idx[1], idx[2]) + Q2(dq1d, m, l);
                }
            }
    }
#undef AUX4
#undef Q4
#undef OFF4
    free(q1d); free(dq1d); free(aux1d);
    sc_work_free(&w);
    return cfl;
}
