// One translation unit per (kernel kind, NV): compiled several times by build.py with -DPHX_KIND_ADJ=0/1 and
// -DPHX_NV=1/2/4 so the template instantiations build in parallel.
#include "phx_resident.cuh"

namespace {
template <typename KernelT>
int launch_coop(KernelT kernel, const ResParams& p, const ResLaunchPlan& plan, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem_bytes);
    if (e != cudaSuccess) {
        phx_set_error("cudaFuncSetAttribute(smem=%zu): %s", plan.smem_bytes, cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    ResParams pl = p;
    void* args[] = {&pl};
    e = cudaLaunchCooperativeKernel((const void*)kernel, dim3(plan.nCTA), dim3(THREADS), args, plan.smem_bytes,
                                    stream);
    if (e != cudaSuccess) {
        phx_set_error("cudaLaunchCooperativeKernel(grid=%d, smem=%zu): %s", plan.nCTA, plan.smem_bytes,
                      cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

}  // namespace

#define PHX_CAT2(a, b) a##b
#define PHX_CAT(a, b) PHX_CAT2(a, b)
#if PHX_KIND_ADJ
#define PHX_KERNEL phx_adj_kernel
#define PHX_FN PHX_CAT(phx_launch_adj_nv, PHX_NV)
#else
#define PHX_KERNEL phx_fwd_kernel
#define PHX_FN PHX_CAT(phx_launch_fwd_nv, PHX_NV)
#endif

#if PHX_KIND_ADJ
int PHX_FN(const ResParams& p, const ResLaunchPlan& plan, cudaStream_t stream) {
    if (p.pmask & PHX_NORM_SEMINORM) {
        if (p.B > 1) return launch_coop(PHX_KERNEL<PHX_NV, 4, true>, p, plan, stream);
        return launch_coop(PHX_KERNEL<PHX_NV, 1, true>, p, plan, stream);
    }
    if (p.B > 1) return launch_coop(PHX_KERNEL<PHX_NV, 4, false>, p, plan, stream);
    return launch_coop(PHX_KERNEL<PHX_NV, 1, false>, p, plan, stream);
}
#else
int PHX_FN(const ResParams& p, const ResLaunchPlan& plan, cudaStream_t stream) {
    if (p.B > 1) return launch_coop(PHX_KERNEL<PHX_NV, 4>, p, plan, stream);
    return launch_coop(PHX_KERNEL<PHX_NV, 1>, p, plan, stream);
}
#endif
