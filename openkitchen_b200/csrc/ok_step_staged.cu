// ok_step_staged.cu -- the STAGED shape of the beam kernel (ok_step.cuh: one 1,024-thread CTA per SM behind the track staged
// in shared memory), the throughput path, in a translation unit of its own.
#include "ok_step.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::staged, StepVariant::plain>::unit = beam_step_unit<true, false, StepVariant::plain>();
} // namespace ok
