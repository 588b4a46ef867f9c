// ok_step_grid_laps.cu -- the kernel of ok_step_grid.cu with lap accounting (StepVariant::laps).
#include "ok_step_grid.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::grid, StepVariant::laps>::unit = grid_step_unit<StepVariant::laps>();
} // namespace ok
