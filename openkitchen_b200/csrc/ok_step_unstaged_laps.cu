// ok_step_unstaged_laps.cu -- the UNSTAGED beam kernel (ok_step_unstaged.cu) with lap accounting (OkLaps; agent_pre /
// agent_post with kLaps), in a translation unit of its own like every step kernel.  The host launches it instead of the
// kernels without accounting for every moving tick while accounting is on; its auto-reset draws when p.reset_flags says so.
#include "ok_step.cuh"

namespace ok
{
cudaError_t launch_step_unstaged_laps(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    beam_step_laps_kernel<false><<<grid, kBeamBlockUnstaged, smem_bytes, stream>>>(p, NoActor{});
    return cudaGetLastError();
}

cudaError_t violations_step_unstaged_laps(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
