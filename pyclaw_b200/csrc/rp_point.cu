// rp_point.cu -- the Riemann solvers as stand-alone pointwise operators.
//
// The reference's plugin seam for a Riemann solver is
//     rp(q_l, q_r, aux_l, aux_r, aux_global) -> (wave, s, amdq, apdq)          (doc/rp.rst:7-62,
//     src/pyclaw/clawpack.py:349) and, in Fortran, rpn2 / rpt2 (flux2.f:99-100, 167-168, 180-181).
// These entry points evaluate exactly the device functions that are inlined into the sweeps
// (rp.cuh) on arrays of left / right states, one thread per interface, so that the solvers can
// be checked on their own -- against the oracle, and against properties that do not depend on
// any restatement (sum of waves = jump, conservation, B(q^) asdq = bm + bp).
//
// The kernel and its launcher are in rp_point.cuh.
#include "rp_point.cuh"

// ixy = 1 | 2 (| 3) selects the sweep direction of a 2-D (3-D) solver; auxl / auxr may be null for solvers without aux
int claw_rp_point(const clawb200_problem *p, int ixy, long long n, const double *ql, const double *qr,
                  const double *auxl, const double *auxr, double *wave, double *s, double *amdq, double *apdq, int imp, const double *asdq,
                  double *bm, double *bp, cudaStream_t st)
{
    if (p->rp_id == CLAWB200_RP_USER)
        return claw_rp_point_user(p, ixy, n, ql, qr, auxl, auxr, wave, s, amdq, apdq, imp, asdq, bm, bp, st);
    RpParams P;
    for (int i = 0; i < 8; i++) P.p[i] = p->rp_params[i];
#define GO(RPT) return rp_point_launch<RPT>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, imp, asdq, bm, bp, st)
#define GO3(RPF) return ixy == 1 ? rp_point_launch<RPF<1>, false>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr, st) \
                   : ixy == 2 ? rp_point_launch<RPF<2>, false>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr, st) \
                              : rp_point_launch<RPF<3>, false>(n, P, ql, qr, auxl, auxr, wave, s, amdq, apdq, 0, nullptr, nullptr, nullptr, st)
    if (p->ndim == 3) { // rpn3, ixy = 1, 2, 3 (the caller has rejected transverse solves)
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS3D_VC: GO3(RpAcoustics3D);
        case CLAWB200_RP_ADVECTION3D: GO3(RpAdvection3);
        case CLAWB200_RP_EULER3D: GO3(RpEuler3);
        case CLAWB200_RP_ADVECTION3D_VC_FWAVE: GO3(RpVcAdvectionFwave3);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: no 3-D version of this solver");
        }
    }
    if (p->ndim == 1) {
        if (asdq) return fail(CLAWB200_ERR_INVALID, "1-D solvers have no transverse solve");
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: { using R = RpAcoustics<1, 1>; GO(R); }
        case CLAWB200_RP_ADVECTION: { using R = RpAdvection<1, 1>; GO(R); }
        case CLAWB200_RP_SHALLOW: GO(RpShallow1D);
        case CLAWB200_RP_BURGERS: GO(RpBurgers);
        case CLAWB200_RP_EULER1D: GO(RpEuler1D);
        case CLAWB200_RP_NEL_FWAVE: { using R = RpElasticFwave<1, 1>; GO(R); }
        case CLAWB200_RP_ADVECTION_COLOR: { using R = RpColor<1, 1>; GO(R); }
        case CLAWB200_RP_SHALLOW_BATHY_FWAVE: { using R = RpShallowBathyFwave<1, 1>; GO(R); }
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: no 1-D version of this solver");
        }
    }
    if (ixy == 1) {
        switch (p->rp_id) {
        case CLAWB200_RP_ACOUSTICS: { using R = RpAcoustics<2, 1>; GO(R); }
        case CLAWB200_RP_ADVECTION: { using R = RpAdvection<2, 1>; GO(R); }
        case CLAWB200_RP_EULER5: GO(RpEuler5<1>);
        case CLAWB200_RP_SHALLOW: GO(RpShallow<1>);
        case CLAWB200_RP_PSYSTEM: { using R = RpElasticFwave<2, 1>; GO(R); }
        case CLAWB200_RP_VC_ACOUSTICS: GO(RpVcAcoustics<1>);
        case CLAWB200_RP_SHALLOW_BATHY_FWAVE: { using R = RpShallowBathyFwave<2, 1>; GO(R); }
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: not compiled for this solver");
        }
    }
    switch (p->rp_id) {
    case CLAWB200_RP_ACOUSTICS: { using R = RpAcoustics<2, 2>; GO(R); }
    case CLAWB200_RP_ADVECTION: { using R = RpAdvection<2, 2>; GO(R); }
    case CLAWB200_RP_EULER5: GO(RpEuler5<2>);
    case CLAWB200_RP_SHALLOW: GO(RpShallow<2>);
    case CLAWB200_RP_PSYSTEM: { using R = RpElasticFwave<2, 2>; GO(R); }
    case CLAWB200_RP_VC_ACOUSTICS: GO(RpVcAcoustics<2>);
    case CLAWB200_RP_SHALLOW_BATHY_FWAVE: { using R = RpShallowBathyFwave<2, 2>; GO(R); }
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "pointwise entry: not compiled for this solver");
    }
#undef GO
#undef GO3
}

// ---------------------------------------------------------------------------
// The division / square-root operators of arith.cuh on arrays (clawb200_arith_probe).  This unit is
// compiled with each build's flags, so the strict and the fma library each probe their own FastArith.
// ---------------------------------------------------------------------------
template <class A>
__device__ __forceinline__ void arith_probe_op(A &ar, int op, double a, double b, double &o0, double &o1, double &o2)
{
    Recip r, rx;
    switch (op) {
    case CLAWB200_ARITH_RCP: o0 = ar.rcp(b).r; break;
    case CLAWB200_ARITH_RCP_NC: o0 = ar.rcp_nc(b).r; break;
    case CLAWB200_ARITH_DIV_RCP: o0 = ar.div(a, ar.rcp(b)); break;
    case CLAWB200_ARITH_DIV: o0 = ar.div(a, b); break;
    case CLAWB200_ARITH_DIV_NZ: o0 = ar.div_nz(a, ar.rcp_nc(b)); break; // as the WENO weights use it
    case CLAWB200_ARITH_SQRT: o0 = ar.sqrt(a); break;
    case CLAWB200_ARITH_SQRT_RCP: ar.sqrt_rcp(a, o0, r); o1 = r.r; break;
    case CLAWB200_ARITH_SQRT_RCPS: ar.sqrt_rcps(a, o0, r, rx); o1 = r.r; o2 = rx.r; break;
    case CLAWB200_ARITH_SQRT_RCP2S: ar.sqrt_rcp2s(a, o0, r, rx); o1 = r.r; o2 = rx.r; break;
    }
}

#ifdef CLAWB200_FMA
using FastArithFz = FmaArithT<false>; // what with_arith_fz runs first
#else
using FastArithFz = FastArithT<false>;
#endif

template <class A>
__device__ __forceinline__ int arith_probe_fast(int op, double a, double b, double &o0, double &o1, double &o2)
{
    A fa;
    arith_probe_op(fa, op, a, b, o0, o1, o2);
    return fa.bad();
}

__global__ void arith_probe_kernel(int policy, int op, long long n, const double *__restrict__ a,
                                   const double *__restrict__ b, double *__restrict__ out, int *__restrict__ bad)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double x = a[i], y = b[i];
    double o0 = 0.0, o1 = 0.0, o2 = 0.0, u0, u1, u2;
    int flag = 0;
    switch (policy) {
    case CLAWB200_ARITH_FAST: flag = arith_probe_fast<FastArith>(op, x, y, o0, o1, o2); break;
    case CLAWB200_ARITH_FAST_FZ: flag = arith_probe_fast<FastArithFz>(op, x, y, o0, o1, o2); break;
    case CLAWB200_ARITH_EXACT: { ExactArith ea; arith_probe_op(ea, op, x, y, o0, o1, o2); break; }
    // what the kernels compute: the values of with_arith(_fz), the flag of its fast attempt
    case CLAWB200_ARITH_GUARDED:
        flag = arith_probe_fast<FastArith>(op, x, y, u0, u1, u2);
        with_arith([&](auto &ar) { arith_probe_op(ar, op, x, y, o0, o1, o2); });
        break;
    case CLAWB200_ARITH_GUARDED_FZ:
        flag = arith_probe_fast<FastArithFz>(op, x, y, u0, u1, u2);
        with_arith_fz([&](auto &ar) { arith_probe_op(ar, op, x, y, o0, o1, o2); });
        break;
    }
    out[i] = o0;
    out[n + i] = o1;
    out[2 * n + i] = o2;
    bad[i] = flag;
}

extern "C" int clawb200_arith_probe(int policy, int op, long long n, const double *a, const double *b, double *out3,
                                    int *bad)
{
    if (policy < CLAWB200_ARITH_FAST || policy > CLAWB200_ARITH_GUARDED_FZ)
        return fail(CLAWB200_ERR_INVALID, "arith probe: unknown policy");
    if (op < CLAWB200_ARITH_RCP || op > CLAWB200_ARITH_SQRT_RCP2S) return fail(CLAWB200_ERR_INVALID, "arith probe: unknown op");
    if (n < 0 || !a || !b || !out3 || !bad) return fail(CLAWB200_ERR_INVALID, "null argument");
    if (n == 0) return 0;
    const size_t nb = (size_t)n * sizeof(double);
    char *d = nullptr;
    CUDA_OK(cudaMalloc(&d, 5 * nb + (size_t)n * sizeof(int)));
    double *d_a = (double *)d, *d_b = d_a + n, *d_o = d_b + n;
    int *d_bad = (int *)(d_o + 3 * n);
    const cudaStream_t st = 0;
    cudaError_t e;
    if ((e = cudaMemcpyAsync(d_a, a, nb, cudaMemcpyHostToDevice, st)) == cudaSuccess &&
        (e = cudaMemcpyAsync(d_b, b, nb, cudaMemcpyHostToDevice, st)) == cudaSuccess) {
        arith_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(policy, op, n, d_a, d_b, d_o, d_bad);
        if ((e = cudaGetLastError()) == cudaSuccess &&
            (e = cudaMemcpyAsync(out3, d_o, 3 * nb, cudaMemcpyDeviceToHost, st)) == cudaSuccess &&
            (e = cudaMemcpyAsync(bad, d_bad, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st)) == cudaSuccess)
            e = cudaStreamSynchronize(st);
    }
    cudaStreamSynchronize(st);
    cudaFree(d);
    return e == cudaSuccess ? 0 : cuda_fail(e, "arith probe");
}
