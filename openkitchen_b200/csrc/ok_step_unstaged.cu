// ok_step_unstaged.cu -- the UNSTAGED shape of the beam kernel (ok_step.cuh: several 256-thread CTAs per SM, the track
// read from global memory) in a translation unit of its own.
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::unstaged, StepVariant::plain>::unit = beam_step_unit<false, false, StepVariant::plain>();
} // namespace ok
