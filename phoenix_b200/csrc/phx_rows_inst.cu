// Launchers of the rows kernels (phx_rows.cuh): compiled twice by build.py, -DPHX_KIND_ADJ=0/1.
#include "phx_rows.cuh"

namespace {
template <typename KernelT>
int launch_rows(KernelT kernel, const ResParams& p, const RowsPlan& plan, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem_bytes);
    if (e != cudaSuccess) {
        phx_set_error("cudaFuncSetAttribute(smem=%zu): %s", plan.smem_bytes, cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    ResParams pl = p;
    void* args[] = {&pl};
    e = cudaLaunchCooperativeKernel((const void*)kernel, dim3(plan.nCTA), dim3(THREADS), args, plan.smem_bytes, stream);
    if (e != cudaSuccess) {
        phx_set_error("cudaLaunchCooperativeKernel(rows, grid=%d, smem=%zu): %s", plan.nCTA, plan.smem_bytes,
                      cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}
}  // namespace

#if PHX_KIND_ADJ
int phx_launch_rows_adj(const ResParams& p, const RowsPlan& plan, cudaStream_t stream) {
    if (p.pmask & PHX_NORM_SEMINORM) return launch_rows(phx_rows_adj_kernel<true>, p, plan, stream);
    return launch_rows(phx_rows_adj_kernel<false>, p, plan, stream);
}
#else
int phx_launch_rows_fwd(const ResParams& p, const RowsPlan& plan, cudaStream_t stream) {
    return launch_rows(phx_rows_fwd_kernel, p, plan, stream);
}
#endif
