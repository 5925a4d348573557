// sweep_sphere.cu -- classic sweeps for shallow water on the sphere (16 aux, capacity function,
// step2qcor correction).
#include "launch.cuh"

int claw_x_sphere(bool trans, const SweepArgs &A, cudaStream_t st) { return launch_x<RpSphere<1>, true>(trans, A, st); }
int claw_y_sphere(bool trans, const SweepArgs &A, cudaStream_t st) { return launch_y<RpSphere<2>, true>(trans, A, st); }
