// ok_step_grid.cu -- the grid / brute-force step kernel (OK_RAYCAST_GRID, OK_RAYCAST_BRUTE; body in ok_step_grid.cuh) in a
// translation unit of its own.
#include "ok_step_grid.cuh"

namespace ok
{
template <> const StepUnit StepUnitOf<StepShape::grid, StepVariant::plain>::unit = grid_step_unit<StepVariant::plain>();
} // namespace ok
