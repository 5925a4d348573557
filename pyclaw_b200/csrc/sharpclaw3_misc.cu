// sharpclaw3_misc.cu -- the 3-D SharpClaw stage (sharpclaw3.cuh) instantiated for the 3-D advection solver
// (RpAdvection3).
#include "sharpclaw3.cuh"

int claw_sc3_advection(bool old, const ScArgs &A, cudaStream_t st) { return sc_stage3_generic<RpAdvection3>(old, A, st); }
