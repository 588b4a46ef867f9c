// ok_step_actor.cu -- the unstaged beam kernel (the shape of small populations) with the PPO racers' policy step fused in
// as phase 0 of every tile (ok_step.cuh, kActor; ok_ppo_actor_step), in a translation unit of its own like the other
// shapes.  (The staged shape has no fused instantiation: its shared memory is sized to the last kilobyte, and it is the
// shape of populations whose tick is not launch latency.)
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::actor, StepVariant::plain>::unit = beam_step_unit<false, true, StepVariant::plain>();
} // namespace ok
