// ok_step_actor.cu -- the unstaged beam kernel (the shape of small populations) with the PPO racers' policy step fused in as
// phase 0 of every tile (ok_kernels.cuh, kActor; ok_ppo_actor_step), in a translation unit of its own like the other shapes:
// nothing here may change the code ptxas generates for the throughput kernel in ok_capi.cu.  (The staged shape has no fused
// instantiation: its shared memory is sized to the last kilobyte, and it is the shape of populations whose tick is not
// launch latency.)
#define OK_STEP_KERNEL_ONLY 1
#include "ok_kernels.cuh"

namespace ok
{
cudaError_t launch_step_actor(const StepParams &p, const ActorParams &q, int grid, size_t smem_bytes, cudaStream_t stream)
{
    step_kernel<kBeamBlockUnstaged, true, false, true><<<grid, kBeamBlockUnstaged, smem_bytes, stream>>>(p, q);
    return cudaGetLastError();
}

// cudaFuncAttributeMaxDynamicSharedMemorySize = everything the device allows (an attribute of the function, not the env);
// *max_dynamic: what that is after the kernel's static shared memory
cudaError_t arm_step_actor(int smem_optin, int *max_dynamic)
{
    cudaFuncAttributes fa{};
    cudaError_t        rc = cudaFuncGetAttributes(&fa, step_kernel<kBeamBlockUnstaged, true, false, true>);
    if (rc != cudaSuccess)
        return rc;
    *max_dynamic = smem_optin - static_cast<int>(fa.sharedSizeBytes);
    return cudaFuncSetAttribute(step_kernel<kBeamBlockUnstaged, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, *max_dynamic);
}
} // namespace ok
