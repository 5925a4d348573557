// sweep_euler_y.cu -- y-engine instantiations for the Euler 5-wave Roe solver.
#include "launch.cuh"

int claw_y_euler(bool trans, const SweepArgs &A, cudaStream_t st)
{
    return A.mcapa > 0 ? launch_y<RpEuler5<2>, true>(trans, A, st) : launch_y<RpEuler5<2>>(trans, A, st);
}
