// sweep_euler_x.cu -- x-engine instantiations for the Euler 5-wave Roe solver.
#include "launch.cuh"

int claw_x_euler(bool trans, const SweepArgs &A, cudaStream_t st)
{
    return A.mcapa > 0 ? launch_x<RpEuler5<1>, true>(trans, A, st) : launch_x<RpEuler5<1>>(trans, A, st);
}
