// ok_step_grid_drawn.cu -- the kernel of ok_step_grid.cu with the drawn auto-reset (StepVariant::drawn).
#include "ok_step_grid.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::grid, StepVariant::drawn>::unit = grid_step_unit<StepVariant::drawn>();
} // namespace ok
