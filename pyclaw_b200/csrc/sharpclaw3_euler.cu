// sharpclaw3_euler.cu -- the 3-D SharpClaw stage (sharpclaw3.cuh) instantiated for the 3-D Euler solver (RpEuler3).
#include "sharpclaw3.cuh"

int claw_sc3_euler(bool old, const ScArgs &A, cudaStream_t st) { return sc_stage3_generic<RpEuler3>(old, A, st); }
