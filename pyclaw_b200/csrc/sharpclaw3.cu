// sharpclaw3.cu -- the 3-D SharpClaw stage (sharpclaw3.cuh) instantiated for the 3-D variable-coefficient
// acoustics solver (RpAcoustics3D).
#include "sharpclaw3.cuh"

int claw_sc3_acoustics(bool old, const ScArgs &A, cudaStream_t st) { return sc_stage3_generic<RpAcoustics3D>(old, A, st); }
