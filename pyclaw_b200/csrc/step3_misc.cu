// step3_misc.cu -- the 3-D steps (step3.cuh) instantiated for the 3-D advection solver (RpAdvection3) and the
// 3-D f-wave transport solver (RpVcAdvectionFwave3).
#include "step3.cuh"

int claw_step3_advection(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                         const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st)
{
    return claw_step3_generic<RpAdvection3>(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
}

int claw_step3_vc_advection_fwave(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                                  const double *aux, double dt, int idir, double *scratch, double *cfl_dev,
                                  cudaStream_t st)
{
    return claw_step3_generic<RpVcAdvectionFwave3>(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
}
