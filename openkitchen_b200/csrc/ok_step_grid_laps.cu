// ok_step_grid_laps.cu -- the grid / brute-force kernel (ok_step_grid.cu) with lap accounting (OkLaps; agent_pre /
// agent_post with kLaps), in a translation unit of its own like every step kernel.  The host launches it instead of the
// kernels without accounting for every moving tick while accounting is on; its auto-reset draws when p.reset_flags says so.
#include "ok_step_grid.cuh"

namespace ok
{
__global__ void __launch_bounds__(kGridBlock, 1) grid_step_laps_kernel(const StepParams p)
{
    grid_tick<false, true>(p);
}

cudaError_t launch_step_grid_laps(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    grid_step_laps_kernel<<<grid, kGridBlock, smem_bytes, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t arm_step_grid_laps(int smem_optin, int *max_dynamic)
{
    return arm_dynamic_smem(reinterpret_cast<const void *>(grid_step_laps_kernel), smem_optin, max_dynamic);
}

cudaError_t violations_step_grid_laps(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
