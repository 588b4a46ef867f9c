// ok_step_grid.cu -- the grid / brute-force step kernel (OK_RAYCAST_GRID, OK_RAYCAST_BRUTE; body in ok_step_grid.cuh) in a
// translation unit of its own.
#include "ok_step_grid.cuh"

namespace ok
{
__global__ void __launch_bounds__(kGridBlock, 1) grid_step_kernel(const StepParams p)
{
    grid_tick<false>(p);
}

cudaError_t launch_step_grid(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    grid_step_kernel<<<grid, kGridBlock, smem_bytes, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t arm_step_grid(int smem_optin, int *max_dynamic)
{
    return arm_dynamic_smem(reinterpret_cast<const void *>(grid_step_kernel), smem_optin, max_dynamic);
}

cudaError_t violations_step_grid(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
