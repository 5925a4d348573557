/*
 * claw_oracle_bathy.c -- CPU restatement of the classic steps with the shallow-water-over-bathymetry
 * f-wave solver (shallow_bathymetry_fwave) -- TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * The solver is restated from its published algorithm (Bale, LeVeque, Mitran & Rossmanith 2002, SIAM J.
 * Sci. Comput. 24; LeVeque 2002 sec. 15.5) in the operation order of RpShallowBathyFwave
 * (pyclaw_b200/csrc/rp.cuh), where its definition is written out; PARITY UNPINNED (the reference has no such
 * solver), pinned by properties (tests/test_rp_bathymetry_properties.py).  The steps around it -- step1
 * (step1.f + step1fw.f), flux2 (flux2.f + flux2fw.f), step2ds and step2 without a capacity function -- are
 * oracle/claw_oracle.c's, statement by statement, with this one solver in place of its dispatch.
 *
 * Layout as in oracle/claw_oracle.c: Fortran order q(meqn, 1-mbc:mx+mbc[, 1-mbc:my+mbc]), component
 * fastest; aux(1) = b.  Strict IEEE double: compile with -ffp-contract=off.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    double grav, dry; /* params {grav, dry_tolerance} */
    int maux;
    double *u, *v, *a; /* Roe averages of each interface of the slice, for the transverse solve */
} bctx;

static void bctx_init(bctx *c, const double *p, int maux, int n)
{
    c->grav = p[0]; c->dry = p[1]; c->maux = maux;
    c->u = (double *)calloc(n, sizeof(double));
    c->v = (double *)calloc(n, sizeof(double));
    c->a = (double *)calloc(n, sizeof(double));
}
static void bctx_free(bctx *c) { free(c->u); free(c->v); free(c->a); }

static inline double dmax2(double a, double b) { return (a > b) ? a : b; }
static inline double dmin2(double a, double b) { return (a < b) ? a : b; }

#define IX(i) ((i) + mbc - 1)
#define Q2(arr, m, i) arr[(m) + meqn * IX(i)]
#define WV(m, mw, i) wave[(m) + meqn * ((mw) + mwaves * IX(i))]
#define SP(mw, i) s[(mw) + mwaves * IX(i)]

/* rpn: interface i has left state qr(:,i-1), right state ql(:,i); b from auxr(i-1), auxl(i).
   ixy = 0: the 1-D solver (q = h, hu; two waves), ixy = 1, 2: rpn2 (q = h, hu, hv; three waves). */
static void rpn_bathy(bctx *c, int ixy, int meqn, int mwaves, int mbc, int mx, const double *ql, const double *qr,
                      const double *auxl, const double *auxr, double *wave, double *s, double *amdq, double *apdq)
{
    const double grav = c->grav, dry = c->dry;
    const int maux = c->maux;
    const int two = (ixy != 0);
    int mu = (ixy <= 1) ? 1 : 2, mv = (ixy <= 1) ? 2 : 1;
    const int nw = two ? 3 : 2;
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        int k = IX(i);
        double hl = Q2(qr, 0, i - 1), hr = Q2(ql, 0, i);
        for (int m = 0; m < meqn; m++) {
            for (int mw = 0; mw < mwaves; mw++) WV(m, mw, i) = 0.0;
            Q2(amdq, m, i) = 0.0;
            Q2(apdq, m, i) = 0.0;
        }
        for (int mw = 0; mw < mwaves; mw++) SP(mw, i) = 0.0;
        c->u[k] = 0.0; c->v[k] = 0.0; c->a[k] = 0.0;
        int wetl = hl > dry, wetr = hr > dry;
        if (!wetl && !wetr) continue;
        double hul = Q2(qr, mu, i - 1), hur = Q2(ql, mu, i);
        double ul = wetl ? hul / hl : 0.0, ur = wetr ? hur / hr : 0.0;
        double vl = 0.0, vr = 0.0;
        if (two) {
            vl = wetl ? Q2(qr, mv, i - 1) / hl : 0.0;
            vr = wetr ? Q2(ql, mv, i) / hr : 0.0;
        }
        double phil = hul * ul + 0.5 * grav * (hl * hl);
        double phir = hur * ur + 0.5 * grav * (hr * hr);
        double hl0 = dmax2(hl, 0.0), hr0 = dmax2(hr, 0.0);
        double sql = sqrt(hl0), sqr = sqrt(hr0);
        double ubar = (sql * ul + sqr * ur) / (sql + sqr);
        double vbar = two ? (sql * vl + sqr * vr) / (sql + sqr) : 0.0;
        double cbar = sqrt(0.5 * grav * (hl0 + hr0));
        double s1 = dmin2(ul - sqrt(grav * hl0), ubar - cbar);
        double s3 = dmax2(ur + sqrt(grav * hr0), ubar + cbar);
        double bl = auxr[0 + maux * IX(i - 1)], br = auxl[0 + maux * IX(i)];
        double d1 = hur - hul;
        double d2 = phir - phil + 0.5 * grav * (hl + hr) * (br - bl);
        double b1 = (s3 * d1 - d2) / (s3 - s1);
        double b3 = (d2 - s1 * d1) / (s3 - s1);
        WV(0, 0, i) = b1;
        WV(mu, 0, i) = b1 * s1;
        SP(0, i) = s1;
        WV(0, nw - 1, i) = b3;
        WV(mu, nw - 1, i) = b3 * s3;
        SP(nw - 1, i) = s3;
        if (two) {
            double d3 = hur * vr - hul * vl;
            WV(mv, 0, i) = b1 * vl;
            WV(mv, 1, i) = d3 - b1 * vl - b3 * vr;
            SP(1, i) = ubar;
            WV(mv, 2, i) = b3 * vr;
        }
        for (int m = 0; m < meqn; m++)
            for (int mw = 0; mw < nw; mw++) {
                double z = WV(m, mw, i);
                if (SP(mw, i) < 0.0) Q2(amdq, m, i) = Q2(amdq, m, i) + z;
                else if (SP(mw, i) > 0.0) Q2(apdq, m, i) = Q2(apdq, m, i) + z;
                else {
                    Q2(amdq, m, i) = Q2(amdq, m, i) + 0.5 * z;
                    Q2(apdq, m, i) = Q2(apdq, m, i) + 0.5 * z;
                }
            }
        c->u[k] = ubar; c->v[k] = vbar; c->a[k] = cbar;
    }
}

/* rpt2: clawpack/riemann rpt2_shallow_roe_with_efix.f (as in oracle/claw_oracle.c) at the Roe averages of
   rpn_bathy; nothing is split at a dry interface (a = 0).  Reads no aux. */
static void rpt_bathy(bctx *c, int ixy, int meqn, int mbc, int mx, const double *asdq, double *bmasdq,
                      double *bpasdq)
{
    int mu = (ixy == 1) ? 1 : 2, mv = (ixy == 1) ? 2 : 1;
    double *u = c->u, *v = c->v, *a = c->a;
    double waveb[3][3], sb[3];
    for (int i = 2 - mbc; i <= mx + mbc; i++) {
        int k = IX(i);
        if (a[k] == 0.0) {
            for (int m = 0; m < meqn; m++) { Q2(bmasdq, m, i) = 0.0; Q2(bpasdq, m, i) = 0.0; }
            continue;
        }
        double a1 = (0.50 / a[k]) * ((v[k] + a[k]) * Q2(asdq, 0, i) - Q2(asdq, mv, i));
        double a2 = Q2(asdq, mu, i) - u[k] * Q2(asdq, 0, i);
        double a3 = (0.50 / a[k]) * (-(v[k] - a[k]) * Q2(asdq, 0, i) + Q2(asdq, mv, i));
        waveb[0][0] = a1;
        waveb[mu][0] = a1 * u[k];
        waveb[mv][0] = a1 * (v[k] - a[k]);
        sb[0] = v[k] - a[k];
        waveb[0][1] = 0.0;
        waveb[mu][1] = a2;
        waveb[mv][1] = 0.0;
        sb[1] = v[k];
        waveb[0][2] = a3;
        waveb[mu][2] = a3 * u[k];
        waveb[mv][2] = a3 * (v[k] + a[k]);
        sb[2] = v[k] + a[k];
        for (int m = 0; m < meqn; m++) {
            Q2(bmasdq, m, i) = 0.0;
            Q2(bpasdq, m, i) = 0.0;
            for (int mw = 0; mw < 3; mw++) {
                Q2(bmasdq, m, i) = Q2(bmasdq, m, i) + dmin2(sb[mw], 0.0) * waveb[m][mw];
                Q2(bpasdq, m, i) = Q2(bpasdq, m, i) + dmax2(sb[mw], 0.0) * waveb[m][mw];
            }
        }
    }
}

/* philim.f:4-58 and limiter.f:4-60 */
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
    default: return dmax2(0.0, dmin2(1.0, r));
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

/* step1.f:4-142 with the step1fw.f:135-136 correction (sign(s)); q updated in place; returns cfl.
   method = {dt_variable, order, trans, verbosity, 0, mcapa (must be 0), maux} */
double oracle_bathy_step1(const double *rp_params, int meqn, int mwaves, int mbc, int maux, int mx, double *q,
                          const double *aux, double dx, double dt, const int *method, const int *mthlim)
{
    bctx c;
    int n = mx + 2 * mbc;
    bctx_init(&c, rp_params, maux, n);
    double *f = (double *)calloc((size_t)meqn * n, sizeof(double));
    double *s = (double *)calloc((size_t)mwaves * n, sizeof(double));
    double *wave = (double *)calloc((size_t)meqn * mwaves * n, sizeof(double));
    double *amdq = (double *)calloc((size_t)meqn * n, sizeof(double));
    double *apdq = (double *)calloc((size_t)meqn * n, sizeof(double));
    double *dtdx = (double *)calloc(n, sizeof(double));
    int limit = 0;
    for (int mw = 0; mw < mwaves; mw++) if (mthlim[mw] > 0) limit = 1;
    for (int i = 1 - mbc; i <= mx + mbc; i++) dtdx[IX(i)] = dt / dx;
    rpn_bathy(&c, 0, meqn, mwaves, mbc, mx, q, q, aux, aux, wave, s, amdq, apdq);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++)
            Q2(q, m, i) = Q2(q, m, i) - dtdx[IX(i)] * Q2(apdq, m, i);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++)
            Q2(q, m, i - 1) = Q2(q, m, i - 1) - dtdx[IX(i - 1)] * Q2(amdq, m, i);
    double cfl = 0.0;
    for (int mw = 0; mw < mwaves; mw++)
        for (int i = 1; i <= mx + 1; i++)
            cfl = dmax2(dmax2(cfl, dtdx[IX(i)] * SP(mw, i)), -dtdx[IX(i - 1)] * SP(mw, i));
    if (method[1] != 1) {
        for (int k = 0; k < meqn * n; k++) f[k] = 0.0;
        if (limit) limiter(meqn, mwaves, mbc, mx, wave, s, mthlim);
        for (int i = 1; i <= mx + 1; i++)
            for (int m = 0; m < meqn; m++)
                for (int mw = 0; mw < mwaves; mw++) {
                    double dtdxave = 0.5 * (dtdx[IX(i - 1)] + dtdx[IX(i)]);
                    double lead = copysign(1.0, SP(mw, i));
                    Q2(f, m, i) = Q2(f, m, i) + 0.5 * lead * (1.0 - fabs(SP(mw, i)) * dtdxave) * WV(m, mw, i);
                }
        for (int i = 1; i <= mx + 1; i++)
            for (int m = 0; m < meqn; m++)
                Q2(q, m, i) = Q2(q, m, i) - dtdx[IX(i)] * (Q2(f, m, i + 1) - Q2(f, m, i));
    }
    free(f); free(s); free(wave); free(amdq); free(apdq); free(dtdx);
    bctx_free(&c);
    return cfl;
}

/* flux2.f:5-193 with the flux2fw.f:151-152 correction */
typedef struct {
    double *wave, *s, *amdq, *apdq, *cqxx, *bmasdq, *bpasdq;
    double *q1d, *qadd, *fadd, *gadd, *dtdx1d, *aux2;
} work2;

static void work2_alloc(work2 *w, int n, int meqn, int mwaves, int maux)
{
    w->wave = (double *)calloc((size_t)n * meqn * mwaves, sizeof(double));
    w->s = (double *)calloc((size_t)n * mwaves, sizeof(double));
    w->amdq = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->apdq = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->cqxx = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->bmasdq = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->bpasdq = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->q1d = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->qadd = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->fadd = (double *)calloc((size_t)n * meqn, sizeof(double));
    w->gadd = (double *)calloc((size_t)n * meqn * 2, sizeof(double));
    w->dtdx1d = (double *)calloc(n, sizeof(double));
    w->aux2 = (double *)calloc((size_t)n * maux, sizeof(double));
}
static void work2_free(work2 *w)
{
    free(w->wave); free(w->s); free(w->amdq); free(w->apdq); free(w->cqxx); free(w->bmasdq); free(w->bpasdq);
    free(w->q1d); free(w->qadd); free(w->fadd); free(w->gadd); free(w->dtdx1d); free(w->aux2);
}

#define GADD(m, k, i) gadd[(m) + meqn * ((k) + 2 * IX(i))]

static double flux2(bctx *c, int ixy, int meqn, int mwaves, int mbc, int mx, const int *method, const int *mthlim,
                    work2 *w)
{
    double *wave = w->wave, *s = w->s, *amdq = w->amdq, *apdq = w->apdq, *cqxx = w->cqxx;
    double *bmasdq = w->bmasdq, *bpasdq = w->bpasdq;
    double *qadd = w->qadd, *fadd = w->fadd, *gadd = w->gadd;
    const double *q1d = w->q1d, *dtdx1d = w->dtdx1d;
    int limit = 0;
    for (int mw = 0; mw < mwaves; mw++) if (mthlim[mw] > 0) limit = 1;
    for (int i = 1 - mbc; i <= mx + mbc; i++)
        for (int m = 0; m < meqn; m++) {
            Q2(qadd, m, i) = 0.0;
            Q2(fadd, m, i) = 0.0;
            GADD(m, 0, i) = 0.0;
            GADD(m, 1, i) = 0.0;
        }
    rpn_bathy(c, ixy, meqn, mwaves, mbc, mx, q1d, q1d, w->aux2, w->aux2, wave, s, amdq, apdq);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++)
            Q2(qadd, m, i) = Q2(qadd, m, i) - dtdx1d[IX(i)] * Q2(apdq, m, i);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++)
            Q2(qadd, m, i - 1) = Q2(qadd, m, i - 1) - dtdx1d[IX(i - 1)] * Q2(amdq, m, i);
    double cfl1d = 0.0;
    for (int mw = 0; mw < mwaves; mw++)
        for (int i = 1; i <= mx + 1; i++)
            cfl1d = dmax2(dmax2(cfl1d, dtdx1d[IX(i)] * SP(mw, i)), -dtdx1d[IX(i - 1)] * SP(mw, i));
    if (method[1] != 1) {
        if (limit) limiter(meqn, mwaves, mbc, mx, wave, s, mthlim);
        for (int i = 2 - mbc; i <= mx + mbc; i++) {
            double dtdxave = 0.5 * (dtdx1d[IX(i - 1)] + dtdx1d[IX(i)]);
            for (int m = 0; m < meqn; m++) {
                Q2(cqxx, m, i) = 0.0;
                for (int mw = 0; mw < mwaves; mw++) {
                    double lead = copysign(1.0, SP(mw, i));
                    Q2(cqxx, m, i) = Q2(cqxx, m, i) + lead * (1.0 - fabs(SP(mw, i)) * dtdxave) * WV(m, mw, i);
                }
                Q2(fadd, m, i) = Q2(fadd, m, i) + 0.5 * Q2(cqxx, m, i);
            }
        }
    }
    if (method[2] <= 0) return cfl1d;
    if (method[1] > 1 && method[2] == 2) {
        for (int i = 1; i <= mx + 1; i++)
            for (int m = 0; m < meqn; m++) {
                Q2(amdq, m, i) = Q2(amdq, m, i) + Q2(cqxx, m, i);
                Q2(apdq, m, i) = Q2(apdq, m, i) - Q2(cqxx, m, i);
            }
    }
    rpt_bathy(c, ixy, meqn, mbc, mx, amdq, bmasdq, bpasdq);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++) {
            GADD(m, 0, i - 1) = GADD(m, 0, i - 1) - 0.5 * dtdx1d[IX(i - 1)] * Q2(bmasdq, m, i);
            GADD(m, 1, i - 1) = GADD(m, 1, i - 1) - 0.5 * dtdx1d[IX(i - 1)] * Q2(bpasdq, m, i);
        }
    rpt_bathy(c, ixy, meqn, mbc, mx, apdq, bmasdq, bpasdq);
    for (int i = 1; i <= mx + 1; i++)
        for (int m = 0; m < meqn; m++) {
            GADD(m, 0, i) = GADD(m, 0, i) - 0.5 * dtdx1d[IX(i)] * Q2(bmasdq, m, i);
            GADD(m, 1, i) = GADD(m, 1, i) - 0.5 * dtdx1d[IX(i)] * Q2(bpasdq, m, i);
        }
    return cfl1d;
}

#define NX (mx + 2 * mbc)
#define Q3(arr, m, i, j) arr[(m) + (size_t)meqn * (((i) + mbc - 1) + (size_t)NX * ((j) + mbc - 1))]
#define AUX3(ma, i, j) aux[(ma) + (size_t)maux * (((i) + mbc - 1) + (size_t)NX * ((j) + mbc - 1))]
#define AUXS(arr, ma, i) arr[(ma) + maux * IX(i)]

/* step2ds.f:2-248 without a capacity function: one directional sweep, ids = 1 | 2 */
double oracle_bathy_step2ds(const double *rp_params, int maxm, int meqn, int mwaves, int maux, int mbc, int mx,
                            int my, const double *qold, double *qnew, const double *aux, double dx, double dy,
                            double dt, const int *method, const int *mthlim, int ids)
{
    int n = maxm + 2 * mbc;
    bctx c;
    bctx_init(&c, rp_params, maux, n);
    work2 w;
    work2_alloc(&w, n, meqn, mwaves, maux);
    double cfl = 0.0;
    double dtdx = dt / dx, dtdy = dt / dy;
    double *q1d = w.q1d, *qadd = w.qadd, *fadd = w.fadd;
    if (ids == 1) {
        for (int k = 0; k < n; k++) w.dtdx1d[k] = dtdx;
        for (int j = 1 - mbc; j <= my + mbc; j++) {
            for (int i = 1 - mbc; i <= mx + mbc; i++)
                for (int m = 0; m < meqn; m++) Q2(q1d, m, i) = Q3(qold, m, i, j);
            for (int ma = 0; ma < maux; ma++)
                for (int i = 1 - mbc; i <= mx + mbc; i++) AUXS(w.aux2, ma, i) = AUX3(ma, i, j);
            cfl = dmax2(cfl, flux2(&c, 1, meqn, mwaves, mbc, mx, method, mthlim, &w));
            for (int i = 1; i <= mx; i++)
                for (int m = 0; m < meqn; m++)
                    Q3(qnew, m, i, j) = Q3(qnew, m, i, j) + Q2(qadd, m, i) - dtdx * (Q2(fadd, m, i + 1) - Q2(fadd, m, i));
        }
    }
    if (ids == 2) {
        for (int k = 0; k < n; k++) w.dtdx1d[k] = dtdy;
        for (int i = 1 - mbc; i <= mx + mbc; i++) {
            for (int j = 1 - mbc; j <= my + mbc; j++)
                for (int m = 0; m < meqn; m++) Q2(q1d, m, j) = Q3(qold, m, i, j);
            for (int ma = 0; ma < maux; ma++)
                for (int j = 1 - mbc; j <= my + mbc; j++) AUXS(w.aux2, ma, j) = AUX3(ma, i, j);
            cfl = dmax2(cfl, flux2(&c, 2, meqn, mwaves, mbc, my, method, mthlim, &w));
            for (int j = 1; j <= my; j++)
                for (int m = 0; m < meqn; m++)
                    Q3(qnew, m, i, j) = Q3(qnew, m, i, j) + Q2(qadd, m, j) - dtdy * (Q2(fadd, m, j + 1) - Q2(fadd, m, j));
        }
    }
    work2_free(&w);
    bctx_free(&c);
    return cfl;
}

/* step2.f:2-241 without a capacity function: the unsplit step, qnew (== qold on entry) updated in place */
double oracle_bathy_step2(const double *rp_params, int maxm, int meqn, int mwaves, int maux, int mbc, int mx,
                          int my, const double *qold, double *qnew, const double *aux, double dx, double dy,
                          double dt, const int *method, const int *mthlim)
{
    int n = maxm + 2 * mbc;
    bctx c;
    bctx_init(&c, rp_params, maux, n);
    work2 w;
    work2_alloc(&w, n, meqn, mwaves, maux);
    double cfl = 0.0;
    double dtdx = dt / dx, dtdy = dt / dy;
    double *q1d = w.q1d, *qadd = w.qadd, *fadd = w.fadd, *gadd = w.gadd;
    for (int k = 0; k < n; k++) w.dtdx1d[k] = dtdx;
    for (int j = 0; j <= my + 1; j++) {
        for (int m = 0; m < meqn; m++)
            for (int i = 1 - mbc; i <= mx + mbc; i++) Q2(q1d, m, i) = Q3(qold, m, i, j);
        for (int ma = 0; ma < maux; ma++)
            for (int i = 1 - mbc; i <= mx + mbc; i++) AUXS(w.aux2, ma, i) = AUX3(ma, i, j);
        cfl = dmax2(cfl, flux2(&c, 1, meqn, mwaves, mbc, mx, method, mthlim, &w));
        for (int m = 0; m < meqn; m++)
            for (int i = 1; i <= mx; i++) {
                Q3(qnew, m, i, j) = Q3(qnew, m, i, j) + Q2(qadd, m, i) - dtdx * (Q2(fadd, m, i + 1) - Q2(fadd, m, i)) -
                                    dtdy * (GADD(m, 1, i) - GADD(m, 0, i));
                Q3(qnew, m, i, j - 1) = Q3(qnew, m, i, j - 1) - dtdy * GADD(m, 0, i);
                Q3(qnew, m, i, j + 1) = Q3(qnew, m, i, j + 1) + dtdy * GADD(m, 1, i);
            }
    }
    for (int k = 0; k < n; k++) w.dtdx1d[k] = dtdy;
    for (int i = 0; i <= mx + 1; i++) {
        for (int m = 0; m < meqn; m++)
            for (int j = 1 - mbc; j <= my + mbc; j++) Q2(q1d, m, j) = Q3(qold, m, i, j);
        for (int ma = 0; ma < maux; ma++)
            for (int j = 1 - mbc; j <= my + mbc; j++) AUXS(w.aux2, ma, j) = AUX3(ma, i, j);
        cfl = dmax2(cfl, flux2(&c, 2, meqn, mwaves, mbc, my, method, mthlim, &w));
        for (int m = 0; m < meqn; m++)
            for (int j = 1; j <= my; j++) {
                Q3(qnew, m, i, j) = Q3(qnew, m, i, j) + (Q2(qadd, m, j) - dtdy * (Q2(fadd, m, j + 1) - Q2(fadd, m, j)) -
                                                         dtdx * (GADD(m, 1, j) - GADD(m, 0, j)));
                Q3(qnew, m, i - 1, j) = Q3(qnew, m, i - 1, j) - dtdx * GADD(m, 0, j);
                Q3(qnew, m, i + 1, j) = Q3(qnew, m, i + 1, j) + dtdx * GADD(m, 1, j);
            }
    }
    work2_free(&w);
    bctx_free(&c);
    return cfl;
}

/* The solver on n independent interfaces: ql, qr [meqn][n] (left / right state), aux_l, aux_r [maux][n];
   normal solve into wave / s / amdq / apdq, or, with asdq given, the transverse split of asdq (imp = 1, 2)
   at the Roe averages of the same interfaces.  Each pair is a 3-cell slice (mbc = 1, mx = 1), cells
   0 | 1 | 2 = left | right | right; ixy = 0 for the 1-D solver. */
void oracle_bathy_rp_point(const double *rp_params, int ixy, int meqn, int mwaves, long long n, const double *ql,
                           const double *qr, int maux, const double *auxl_i, const double *auxr_i, double *wave_o,
                           double *s_o, double *amdq_o, double *apdq_o, int imp, const double *asdq_i, double *bm_o,
                           double *bp_o)
{
    const int mbc = 1, mx = 1, nc = 3;
    bctx c;
    bctx_init(&c, rp_params, maux, nc);
    double *q = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *wave = (double *)calloc((size_t)meqn * mwaves * nc, sizeof(double));
    double *s = (double *)calloc((size_t)mwaves * nc, sizeof(double));
    double *amdq = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *apdq = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *asdq = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *bm = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *bp = (double *)calloc((size_t)meqn * nc, sizeof(double));
    double *aux = (double *)calloc((size_t)maux * nc, sizeof(double));
    (void)imp; /* the split does not depend on the side asdq enters (it reads no aux) */
    for (long long k = 0; k < n; k++) {
        for (int m = 0; m < meqn; m++) {
            Q2(q, m, 0) = ql[m * n + k];
            Q2(q, m, 1) = qr[m * n + k];
            Q2(q, m, 2) = qr[m * n + k];
        }
        for (int ma = 0; ma < maux; ma++) {
            aux[ma + maux * 0] = auxl_i[ma * n + k];
            aux[ma + maux * 1] = auxr_i[ma * n + k];
            aux[ma + maux * 2] = auxr_i[ma * n + k];
        }
        rpn_bathy(&c, ixy, meqn, mwaves, mbc, mx, q, q, aux, aux, wave, s, amdq, apdq);
        if (wave_o) {
            for (int m = 0; m < meqn; m++) {
                for (int mw = 0; mw < mwaves; mw++) wave_o[(m * mwaves + mw) * n + k] = WV(m, mw, 1);
                amdq_o[m * n + k] = Q2(amdq, m, 1);
                apdq_o[m * n + k] = Q2(apdq, m, 1);
            }
            for (int mw = 0; mw < mwaves; mw++) s_o[mw * n + k] = SP(mw, 1);
        }
        if (asdq_i) {
            for (int m = 0; m < meqn; m++)
                for (int i = 0; i <= 2; i++) Q2(asdq, m, i) = asdq_i[m * n + k];
            rpt_bathy(&c, ixy, meqn, mbc, mx, asdq, bm, bp);
            for (int m = 0; m < meqn; m++) {
                bm_o[m * n + k] = Q2(bm, m, 1);
                bp_o[m * n + k] = Q2(bp, m, 1);
            }
        }
    }
    free(q); free(wave); free(s); free(amdq); free(apdq); free(asdq); free(bm); free(bp); free(aux);
    bctx_free(&c);
}
