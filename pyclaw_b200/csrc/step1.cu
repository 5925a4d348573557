// step1.cu -- the 1-D classic step (step1.f) for every 1-D Riemann solver.
#include "launch.cuh"

int claw_step1(int rp_id, const SweepArgs &A, cudaStream_t st)
{
    switch (rp_id) {
    case CLAWB200_RP_ACOUSTICS: return launch_step1<RpAcoustics<1, 1>, true>(A, st);
    case CLAWB200_RP_ADVECTION: return launch_step1<RpAdvection<1, 1>, true>(A, st);
    case CLAWB200_RP_SHALLOW: return launch_step1<RpShallow1D, false>(A, st);
    case CLAWB200_RP_NEL_FWAVE: return launch_step1<RpElasticFwave<1, 1>, false>(A, st);
    case CLAWB200_RP_BURGERS: return launch_step1<RpBurgers, false>(A, st);
    case CLAWB200_RP_ADVECTION_COLOR: return launch_step1<RpColor<1, 1>, false>(A, st);
    case CLAWB200_RP_EULER1D: return launch_step1<RpEuler1D, false>(A, st);
    case CLAWB200_RP_SHALLOW_BATHY_FWAVE: return launch_step1<RpShallowBathyFwave<1, 1>, false>(A, st);
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "no 1-D version of this Riemann solver");
    }
}
