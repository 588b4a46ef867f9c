// ok_step_actor.cu -- the unstaged beam kernel (the shape of small populations) with the PPO racers' policy step fused in
// as phase 0 of every tile (ok_step.cuh, kActor; ok_ppo_actor_step), in a translation unit of its own like the other
// shapes.  (The staged shape has no fused instantiation: its shared memory is sized to the last kilobyte, and it is the
// shape of populations whose tick is not launch latency.)
#include "ok_step.cuh"

namespace ok
{
cudaError_t launch_step_actor(const StepParams &p, const ActorParams &q, int grid, size_t smem_bytes, cudaStream_t stream)
{
    beam_step_kernel<false, true><<<grid, kBeamBlockUnstaged, smem_bytes, stream>>>(p, q);
    return cudaGetLastError();
}

cudaError_t arm_step_actor(int smem_optin, int *max_dynamic)
{
    return arm_dynamic_smem(reinterpret_cast<const void *>(beam_step_kernel<false, true>), smem_optin, max_dynamic);
}

cudaError_t violations_step_actor(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
