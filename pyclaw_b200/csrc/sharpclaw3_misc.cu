// sharpclaw3_misc.cu -- the 3-D SharpClaw stage (sharpclaw3.cuh) instantiated for the 3-D advection solver
// (RpAdvection3) and the 3-D f-wave transport solver (RpVcAdvectionFwave3: with char_decomp = 0 the stage
// reads amdq / apdq only, so an f-wave solver runs unchanged).
#include "sharpclaw3.cuh"

int claw_sc3_advection(bool old, const ScArgs &A, cudaStream_t st) { return sc_stage3_generic<RpAdvection3>(old, A, st); }
int claw_sc3_vc_advection_fwave(bool old, const ScArgs &A, cudaStream_t st)
{
    return sc_stage3_generic<RpVcAdvectionFwave3>(old, A, st);
}
