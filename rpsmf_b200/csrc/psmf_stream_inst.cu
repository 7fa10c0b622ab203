// One translation unit per latent rank for the TMA-staged kernel: compiled with -DPSMF_R=<r>.
#include "psmf_stream.cuh"

#ifndef PSMF_R
#error "compile with -DPSMF_R=<rank>"
#endif

#define PSMF_CAT2(a, b) a##b
#define PSMF_CAT(a, b) PSMF_CAT2(a, b)

namespace psmf {

template <typename T>
static cudaError_t launch_t(const KParams& p, int grid, size_t dyn, cudaStream_t st, bool coop) {
    // F_LOGLIK: one variant that also serves F_GRAD_LINEAR and the moment record (glin_on / ll_on in psmf_filter.cuh)
    auto kern = ((p.flags & F_LOGLIK) || p.mom) ? psmf_stream_kernel<PSMF_R, T, true, true>
                : (p.flags & F_GRAD_LINEAR)     ? psmf_stream_kernel<PSMF_R, T, true>
                                                : psmf_stream_kernel<PSMF_R, T>;
    constexpr int threads = s_threads();
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    if (coop) {
        KParams pc = p;
        void* args[] = {&pc};
        return cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(threads), args, dyn, st);
    }
    kern<<<grid, threads, dyn, st>>>(p);
    return cudaGetLastError();
}

// the F_GRAD_LINEAR and F_LOGLIK variants have the same launch bounds and static shared memory: its shape is this one's
template <typename T>
static cudaError_t shape_t(size_t dyn, LaunchShape* out) {
    auto kern = psmf_stream_kernel<PSMF_R, T>;
    constexpr int threads = s_threads();
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    out->threads = threads;
    out->static_smem = (int)fa.sharedSizeBytes;
    out->max_ctas_per_sm = 0;
    if (dyn > 0) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
        if (e != cudaSuccess) return e;
        int nb = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, threads, dyn);
        if (e != cudaSuccess) return e;
        out->max_ctas_per_sm = nb;
    }
    return cudaSuccess;
}

cudaError_t PSMF_CAT(launch_stream_r, PSMF_R)(const KParams& p, int dtype, int grid, size_t dyn, cudaStream_t st, bool coop) {
    return dtype == 0 ? launch_t<double>(p, grid, dyn, st, coop) : launch_t<float>(p, grid, dyn, st, coop);
}
cudaError_t PSMF_CAT(shape_stream_r, PSMF_R)(int dtype, size_t dyn, LaunchShape* out) {
    return dtype == 0 ? shape_t<double>(dyn, out) : shape_t<float>(dyn, out);
}

}  // namespace psmf
