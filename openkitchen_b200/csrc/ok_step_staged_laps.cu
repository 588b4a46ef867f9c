// ok_step_staged_laps.cu -- the kernel of ok_step_staged.cu with lap accounting (StepVariant::laps).
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::staged, StepVariant::laps>::unit = beam_step_unit<true, false, StepVariant::laps>();
} // namespace ok
