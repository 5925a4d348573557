// step3.cu -- the 3-D classic steps (step3.cuh) instantiated for the 3-D variable-coefficient
// acoustics solver (rpn3 / rpt3 / rptt3_vc_acoustics, test/acoustics/3d; RpAcoustics3D), and the
// scratch size of the unsplit step.
#include "step3.cuh"

int claw_step3_acoustics(const clawb200_problem *p, int mz, double dz, const double *qold, double *qnew,
                         const double *aux, double dt, int idir, double *scratch, double *cfl_dev, cudaStream_t st)
{
    return claw_step3_generic<RpAcoustics3D>(p, mz, dz, qold, qnew, aux, dt, idir, scratch, cfl_dev, st);
}

long long claw_step3_scratch_doubles(int meqn, long long mstride) { return (long long)NV3 * meqn * mstride; }
