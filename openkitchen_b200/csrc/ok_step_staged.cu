// ok_step_staged.cu -- the STAGED shape of the beam kernel (ok_step.cuh: one 1,024-thread CTA per SM behind the track staged
// in shared memory), the throughput path, in a translation unit of its own.
#include "ok_step.cuh"

namespace ok
{
cudaError_t launch_step_staged(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream)
{
    beam_step_kernel<true><<<grid, kBeamBlockStaged, smem_bytes, stream>>>(p, NoActor{});
    return cudaGetLastError();
}

cudaError_t arm_step_staged(int smem_optin, int *max_dynamic)
{
    return arm_dynamic_smem(reinterpret_cast<const void *>(beam_step_kernel<true>), smem_optin, max_dynamic);
}

cudaError_t violations_step_staged(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
