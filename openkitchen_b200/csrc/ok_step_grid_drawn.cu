// ok_step_grid_drawn.cu -- the grid / brute-force kernel (ok_step_grid.cu) with the drawn auto-reset (OkResetDraws;
// agent_pre<true>), in a translation unit of its own like every step kernel.  The host launches it instead of the
// kernel without draws for a tick whose auto-reset draws.
#include "ok_step_grid.cuh"

namespace ok
{
__global__ void __launch_bounds__(kGridBlock, 1) grid_step_drawn_kernel(const StepParams p)
{
    grid_tick<true>(p);
}

cudaError_t launch_step_grid_drawn(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    grid_step_drawn_kernel<<<grid, kGridBlock, smem_bytes, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t arm_step_grid_drawn(int smem_optin, int *max_dynamic)
{
    return arm_dynamic_smem(reinterpret_cast<const void *>(grid_step_drawn_kernel), smem_optin, max_dynamic);
}

cudaError_t violations_step_grid_drawn(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
