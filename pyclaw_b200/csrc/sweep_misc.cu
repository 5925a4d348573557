// sweep_misc.cu -- classic sweeps for the light solvers: acoustics, advection, shallow water
// (Roe + entropy fix), p-system f-waves, variable-coefficient acoustics / advection, shallow water over
// bathymetry (f-waves).
#include "launch.cuh"

int claw_x_misc(int rp_id, bool trans, const SweepArgs &A, cudaStream_t st)
{
    if (A.mcapa > 0) {
        switch (rp_id) {
        case CLAWB200_RP_ACOUSTICS: return launch_x<RpAcoustics<2, 1>, true>(trans, A, st);
        case CLAWB200_RP_ADVECTION: return launch_x<RpAdvection<2, 1>, true>(trans, A, st);
        case CLAWB200_RP_SHALLOW: return launch_x<RpShallow<1>, true>(trans, A, st);
        case CLAWB200_RP_VC_ADVECTION: return launch_x<RpColor<2, 1>, true>(trans, A, st);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for this solver");
        }
    }
    switch (rp_id) {
    case CLAWB200_RP_ACOUSTICS: return launch_x<RpAcoustics<2, 1>>(trans, A, st);
    case CLAWB200_RP_ADVECTION: return launch_x<RpAdvection<2, 1>>(trans, A, st);
    case CLAWB200_RP_SHALLOW: return launch_x<RpShallow<1>>(trans, A, st);
    case CLAWB200_RP_PSYSTEM: return launch_x<RpElasticFwave<2, 1>>(trans, A, st);
    case CLAWB200_RP_VC_ACOUSTICS: return launch_x<RpVcAcoustics<1>>(trans, A, st);
    case CLAWB200_RP_VC_ADVECTION: return launch_x<RpColor<2, 1>>(trans, A, st);
    case CLAWB200_RP_SHALLOW_BATHY_FWAVE: return launch_x<RpShallowBathyFwave<2, 1>>(trans, A, st);
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "unknown rp_id");
    }
}

int claw_y_misc(int rp_id, bool trans, const SweepArgs &A, cudaStream_t st)
{
    if (A.mcapa > 0) {
        switch (rp_id) {
        case CLAWB200_RP_ACOUSTICS: return launch_y<RpAcoustics<2, 2>, true>(trans, A, st);
        case CLAWB200_RP_ADVECTION: return launch_y<RpAdvection<2, 2>, true>(trans, A, st);
        case CLAWB200_RP_SHALLOW: return launch_y<RpShallow<2>, true>(trans, A, st);
        case CLAWB200_RP_VC_ADVECTION: return launch_y<RpColor<2, 2>, true>(trans, A, st);
        default: return fail(CLAWB200_ERR_UNSUPPORTED, "mcapa not compiled for this solver");
        }
    }
    switch (rp_id) {
    case CLAWB200_RP_ACOUSTICS: return launch_y<RpAcoustics<2, 2>>(trans, A, st);
    case CLAWB200_RP_ADVECTION: return launch_y<RpAdvection<2, 2>>(trans, A, st);
    case CLAWB200_RP_SHALLOW: return launch_y<RpShallow<2>>(trans, A, st);
    case CLAWB200_RP_PSYSTEM: return launch_y<RpElasticFwave<2, 2>>(trans, A, st);
    case CLAWB200_RP_VC_ACOUSTICS: return launch_y<RpVcAcoustics<2>>(trans, A, st);
    case CLAWB200_RP_VC_ADVECTION: return launch_y<RpColor<2, 2>>(trans, A, st);
    case CLAWB200_RP_SHALLOW_BATHY_FWAVE: return launch_y<RpShallowBathyFwave<2, 2>>(trans, A, st);
    default: return fail(CLAWB200_ERR_UNSUPPORTED, "unknown rp_id");
    }
}
