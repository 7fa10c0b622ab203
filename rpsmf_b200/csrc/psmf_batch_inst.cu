// One translation unit per latent rank for the resident batch kernel: compiled with -DPSMF_R=<r>.
#include "psmf_batch.cuh"

#ifndef PSMF_R
#error "compile with -DPSMF_R=<rank>"
#endif

#define PSMF_CAT2(a, b) a##b
#define PSMF_CAT(a, b) PSMF_CAT2(a, b)

namespace psmf {

template <typename T, int NW>
static cudaError_t launch_t(const KParams& p, int grid, size_t dyn, cudaStream_t st) {
    // F_LOGLIK: one variant that also serves F_GRAD_LINEAR (glin_on in psmf_filter.cuh)
    auto kern = (p.flags & F_LOGLIK)        ? psmf_batch_kernel<PSMF_R, T, NW, true, true>
                : (p.flags & F_GRAD_LINEAR) ? psmf_batch_kernel<PSMF_R, T, NW, true>
                                            : psmf_batch_kernel<PSMF_R, T, NW>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    kern<<<grid, NW * 32, dyn, st>>>(p);
    return cudaGetLastError();
}

// the F_GRAD_LINEAR and F_LOGLIK variants have the same launch bounds and static shared memory: its shape is this one's
template <typename T, int NW>
static cudaError_t shape_t(size_t dyn, LaunchShape* out) {
    auto kern = psmf_batch_kernel<PSMF_R, T, NW>;
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) return e;
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, NW * 32, dyn);
    if (e != cudaSuccess) return e;
    out->threads = NW * 32;
    out->static_smem = (int)fa.sharedSizeBytes;
    out->max_ctas_per_sm = nb;
    return cudaSuccess;
}

// `coop` carries the warp count of the variant (4 or 8): the batch kernel never launches cooperatively
cudaError_t PSMF_CAT(launch_batch_r, PSMF_R)(const KParams& p, int dtype, int grid, size_t dyn, cudaStream_t st, bool eight) {
    if (eight) return dtype == 0 ? launch_t<double, 8>(p, grid, dyn, st) : launch_t<float, 8>(p, grid, dyn, st);
    return dtype == 0 ? launch_t<double, 4>(p, grid, dyn, st) : launch_t<float, 4>(p, grid, dyn, st);
}
cudaError_t PSMF_CAT(shape_batch4_r, PSMF_R)(int dtype, size_t dyn, LaunchShape* out) {
    return dtype == 0 ? shape_t<double, 4>(dyn, out) : shape_t<float, 4>(dyn, out);
}
cudaError_t PSMF_CAT(shape_batch8_r, PSMF_R)(int dtype, size_t dyn, LaunchShape* out) {
    return dtype == 0 ? shape_t<double, 8>(dyn, out) : shape_t<float, 8>(dyn, out);
}

}  // namespace psmf
