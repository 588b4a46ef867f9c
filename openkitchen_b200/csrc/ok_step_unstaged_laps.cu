// ok_step_unstaged_laps.cu -- the kernel of ok_step_unstaged.cu with lap accounting (StepVariant::laps).
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::unstaged, StepVariant::laps>::unit = beam_step_unit<false, false, StepVariant::laps>();
} // namespace ok
