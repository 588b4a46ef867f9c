// ok_step_unstaged.cu -- the UNSTAGED shape of the beam kernel (ok_step.cuh: several 256-thread CTAs per SM, the track
// read from global memory) in a translation unit of its own.
#include "ok_step.cuh"

namespace ok
{
cudaError_t launch_step_unstaged(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    beam_step_kernel<false><<<grid, kBeamBlockUnstaged, smem_bytes, stream>>>(p, NoActor{});
    return cudaGetLastError();
}

cudaError_t occupancy_step_unstaged(size_t smem_bytes, int *ctas_per_sm)
{
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, beam_step_kernel<false>, kBeamBlockUnstaged, smem_bytes);
}

cudaError_t violations_step_unstaged(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
