// ok_step_actor_laps.cu -- the kernel of ok_step_actor.cu with lap accounting (StepVariant::laps).
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::actor, StepVariant::laps>::unit = beam_step_unit<false, true, StepVariant::laps>();
} // namespace ok
