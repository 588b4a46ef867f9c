// ok_step_staged_drawn.cu -- the kernel of ok_step_staged.cu with the drawn auto-reset (StepVariant::drawn).
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::staged, StepVariant::drawn>::unit = beam_step_unit<true, false, StepVariant::drawn>();
} // namespace ok
