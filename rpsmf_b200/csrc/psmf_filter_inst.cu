// One translation unit per latent rank: compiled with -DPSMF_R=<r> for r = 1..16.
#include "psmf_filter.cuh"

#ifndef PSMF_R
#error "compile with -DPSMF_R=<rank>"
#endif

#define PSMF_CAT2(a, b) a##b
#define PSMF_CAT(a, b) PSMF_CAT2(a, b)

namespace psmf {

template <typename T, bool RHOV = false>
static cudaError_t launch_t(const KParams& p, int grid, size_t dyn, cudaStream_t st, bool coop) {
    // F_LOGLIK: one variant that also serves F_GRAD_LINEAR (glin_on in psmf_filter.cuh)
    auto kern = (p.flags & F_LOGLIK)        ? psmf_filter_kernel<PSMF_R, T, RHOV, true, true>
                : (p.flags & F_GRAD_LINEAR) ? psmf_filter_kernel<PSMF_R, T, RHOV, true>
                                            : psmf_filter_kernel<PSMF_R, T, RHOV>;
    constexpr int threads = V1_WARPS * 32;
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
template <typename T, bool RHOV = false>
static cudaError_t shape_t(size_t dyn, LaunchShape* out) {
    auto kern = psmf_filter_kernel<PSMF_R, T, RHOV>;
    constexpr int threads = V1_WARPS * 32;
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, threads, dyn);
    if (e != cudaSuccess) return e;
    out->threads = threads;
    out->static_smem = (int)fa.sharedSizeBytes;
    out->max_ctas_per_sm = nb;
    return cudaSuccess;
}

cudaError_t PSMF_CAT(launch_filter_r, PSMF_R)(const KParams& p, int dtype, int grid, size_t dyn, cudaStream_t st, bool coop) {
    return dtype == 0 ? launch_t<double>(p, grid, dyn, st, coop) : launch_t<float>(p, grid, dyn, st, coop);
}
cudaError_t PSMF_CAT(shape_filter_r, PSMF_R)(int dtype, size_t dyn, LaunchShape* out) {
    return dtype == 0 ? shape_t<double>(dyn, out) : shape_t<float>(dyn, out);
}

// non-uniform diagonal R (F_RHO_VECTOR)
cudaError_t PSMF_CAT(launch_filterv_r, PSMF_R)(const KParams& p, int dtype, int grid, size_t dyn, cudaStream_t st, bool coop) {
    return dtype == 0 ? launch_t<double, true>(p, grid, dyn, st, coop) : launch_t<float, true>(p, grid, dyn, st, coop);
}
cudaError_t PSMF_CAT(shape_filterv_r, PSMF_R)(int dtype, size_t dyn, LaunchShape* out) {
    return dtype == 0 ? shape_t<double, true>(dyn, out) : shape_t<float, true>(dyn, out);
}

}  // namespace psmf
