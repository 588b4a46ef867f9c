// ok_step_unstaged_drawn.cu -- the kernel of ok_step_unstaged.cu with the drawn auto-reset (StepVariant::drawn).
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::unstaged, StepVariant::drawn>::unit = beam_step_unit<false, false, StepVariant::drawn>();
} // namespace ok
