// One translation unit per latent rank: compiled with -DPSMF_R=<r> for r = 1..16.
#include <cstring>
#include "psmf_filter.cuh"

#ifndef PSMF_R
#error "compile with -DPSMF_R=<rank>"
#endif

#define PSMF_CAT2(a, b) a##b
#define PSMF_CAT(a, b) PSMF_CAT2(a, b)

namespace psmf {

template <typename T, bool RHOV = false>
static cudaError_t launch_t(const KParams& p, int grid, size_t dyn, cudaStream_t st, bool coop) {
    // F_LOGLIK: one variant that also serves F_GRAD_LINEAR and the moment record (glin_on / ll_on in psmf_filter.cuh)
    auto kern = ((p.flags & F_LOGLIK) || p.mom) ? psmf_filter_kernel<PSMF_R, T, RHOV, true, true>
                : (p.flags & F_GRAD_LINEAR)     ? psmf_filter_kernel<PSMF_R, T, RHOV, true>
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

// batched engines whose series do not fit one CTA: a thread-block cluster of `csize` CTAs per series, an ordinary launch.
// One variant per (T, RHOV) serves plain runs, F_GRAD_LINEAR and F_LOGLIK (glin_on / ll_on in psmf_filter.cuh).
template <typename T, bool RHOV>
static cudaError_t cluster_kernel(int csize, size_t dyn, void (**out)(const KParams)) {
    auto kern = psmf_filter_kernel<PSMF_R, T, RHOV, true, true, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e == cudaSuccess && csize > 8) e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    *out = kern;
    return e;
}
static void cluster_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute& attr, int grid, int csize, size_t dyn, cudaStream_t st) {
    memset(&cfg, 0, sizeof(cfg));
    memset(&attr, 0, sizeof(attr));
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = (unsigned)csize;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(V1_WARPS * 32);
    cfg.dynamicSmemBytes = dyn;
    cfg.stream = st;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
}
template <typename T, bool RHOV>
static cudaError_t launch_cluster_t(const KParams& p, int grid, size_t dyn, cudaStream_t st, int csize) {
    void (*kern)(const KParams);
    cudaError_t e = cluster_kernel<T, RHOV>(csize, dyn, &kern);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    cluster_config(cfg, attr, grid, csize, dyn, st);
    return cudaLaunchKernelEx(&cfg, kern, p);
}
// CTAs per SM and clusters of `csize` the device holds at once with `dyn` bytes of dynamic shared memory
template <typename T, bool RHOV>
static cudaError_t cluster_shape_t(size_t dyn, int csize, LaunchShape* out, int* nclusters) {
    void (*kern)(const KParams);
    cudaError_t e = cluster_kernel<T, RHOV>(csize, dyn, &kern);
    if (e != cudaSuccess) return e;
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, V1_WARPS * 32, dyn);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess) return e;
    out->threads = V1_WARPS * 32;
    out->static_smem = (int)fa.sharedSizeBytes;
    out->max_ctas_per_sm = nb;
    *nclusters = 0;
    if (nb < 1) return cudaSuccess;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    cluster_config(cfg, attr, csize, csize, dyn, nullptr);
    return cudaOccupancyMaxActiveClusters(nclusters, kern, &cfg);
}
cudaError_t PSMF_CAT(launch_filterc_r, PSMF_R)(const KParams& p, int dtype, bool rhov, int grid, size_t dyn, cudaStream_t st, int csize) {
    if (rhov) return dtype == 0 ? launch_cluster_t<double, true>(p, grid, dyn, st, csize) : launch_cluster_t<float, true>(p, grid, dyn, st, csize);
    return dtype == 0 ? launch_cluster_t<double, false>(p, grid, dyn, st, csize) : launch_cluster_t<float, false>(p, grid, dyn, st, csize);
}
cudaError_t PSMF_CAT(shape_filterc_r, PSMF_R)(int dtype, bool rhov, size_t dyn, int csize, LaunchShape* out, int* nclusters) {
    if (rhov) return dtype == 0 ? cluster_shape_t<double, true>(dyn, csize, out, nclusters) : cluster_shape_t<float, true>(dyn, csize, out, nclusters);
    return dtype == 0 ? cluster_shape_t<double, false>(dyn, csize, out, nclusters) : cluster_shape_t<float, false>(dyn, csize, out, nclusters);
}

// non-uniform diagonal R (F_RHO_VECTOR)
cudaError_t PSMF_CAT(launch_filterv_r, PSMF_R)(const KParams& p, int dtype, int grid, size_t dyn, cudaStream_t st, bool coop) {
    return dtype == 0 ? launch_t<double, true>(p, grid, dyn, st, coop) : launch_t<float, true>(p, grid, dyn, st, coop);
}
cudaError_t PSMF_CAT(shape_filterv_r, PSMF_R)(int dtype, size_t dyn, LaunchShape* out) {
    return dtype == 0 ? shape_t<double, true>(dyn, out) : shape_t<float, true>(dyn, out);
}

}  // namespace psmf
