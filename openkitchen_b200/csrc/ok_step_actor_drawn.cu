// ok_step_actor_drawn.cu -- the kernel of ok_step_actor.cu with the drawn auto-reset (StepVariant::drawn).
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::actor, StepVariant::drawn>::unit = beam_step_unit<false, true, StepVariant::drawn>();
} // namespace ok
