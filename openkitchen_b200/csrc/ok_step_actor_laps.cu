// ok_step_actor_laps.cu -- the unstaged beam kernel with the policy step fused in (ok_step_actor.cu) with lap accounting
// (OkLaps; agent_pre / agent_post with kLaps), in a translation unit of its own like every step kernel.  The host launches
// it instead of the kernels without accounting for every moving tick while accounting is on; its auto-reset draws when
// p.reset_flags says so.
#include "ok_step.cuh"

namespace ok
{
cudaError_t launch_step_actor_laps(const StepParams &p, const ActorParams &q, int grid, size_t smem_bytes, cudaStream_t stream)
{
    beam_step_laps_kernel<false, true><<<grid, kBeamBlockUnstaged, smem_bytes, stream>>>(p, q);
    return cudaGetLastError();
}

cudaError_t arm_step_actor_laps(int smem_optin, int *max_dynamic)
{
    return arm_dynamic_smem(reinterpret_cast<const void *>(beam_step_laps_kernel<false, true>), smem_optin, max_dynamic);
}

cudaError_t violations_step_actor_laps(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
