// step3_euler.cu -- the 3-D steps (step3.cuh) instantiated for the 3-D Euler solver (RpEuler3).
#include "step3.cuh"

int claw_step3_euler(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                     const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st)
{
    return claw_step3_generic<RpEuler3>(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
}
