// ok_step_unstaged_drawn.cu -- the UNSTAGED beam kernel (ok_step_unstaged.cu) with the drawn auto-reset (OkResetDraws;
// agent_pre<true>), in a translation unit of its own like every step kernel.  The host launches it instead of the
// kernel without draws for a tick whose auto-reset draws.
#include "ok_step.cuh"

namespace ok
{
cudaError_t launch_step_unstaged_drawn(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    beam_step_drawn_kernel<false><<<grid, kBeamBlockUnstaged, smem_bytes, stream>>>(p, NoActor{});
    return cudaGetLastError();
}

cudaError_t violations_step_unstaged_drawn(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
