// Fixed-interval (Rauch-Tung-Striebel) smoother over the per-step moment records of the filter kernels
// (include/psmf_b200.h psmf_set_moments / psmf_smooth).
//
// One CTA per series walks backward in chunks of SM_CHUNK steps.  The gains J_t = P_t F_{t+1}' Pbar_{t+1}^-1 depend on forward
// quantities only, so the warps solve the gains of a chunk in parallel (one r x r system with r right-hand sides each, Gauss-
// Jordan with partial pivoting on [Pbar_{t+1}' | F_{t+1} P_t']) into shared memory; the CTA then runs the sequential recursion
//   x^s_t = x_t + J_t (x^s_{t+1} - xbar_{t+1}),   P^s_t = P_t + J_t (P^s_{t+1} - Pbar_{t+1}) J_t'
// over the chunk.  Nothing in global memory grows with T besides the records and the outputs.
#pragma once
#include "psmf_common.cuh"

namespace psmf {

constexpr int SM_WARPS = 8;     // warps per CTA; each solves SM_CHUNK / SM_WARPS gains per chunk
constexpr int SM_CHUNK = 16;    // steps per chunk

// dynamic shared memory of smooth_kernel (doubles): gains [SM_CHUNK][r][r], per warp [r][2r] augmented matrix + [r] pivot column,
// carried x^s (r), P^s (r x r), and two r x r temporaries
__host__ __device__ constexpr size_t smooth_smem_bytes(int r) {
    return (size_t)(SM_CHUNK * r * r + SM_WARPS * (2 * r * r + r) + r + 3 * r * r) * sizeof(double);
}

// J' = Pbar1'^-1 (F1 P0') by one warp: rows of the augmented matrix are swapped (partial pivoting), so row k ends as row k of J'.
// A singular Pbar1 leaves non-finite entries.
__device__ __forceinline__ void smooth_gain(const double* __restrict__ m0, const double* __restrict__ m1, int r, double* A, double* colk,
                                            double* J, int lane) {
    const int ld = 2 * r;
    const double* F1 = m1 + r;
    const double* Pb1 = m1 + r + r * r;
    const double* P0 = m0 + 2 * r + 2 * r * r;
    __syncwarp();                                         // the previous gain of this warp has been read out of A
    for (int idx = lane; idx < r * r; idx += 32) {
        const int i = idx / r, j = idx % r;
        A[i * ld + j] = Pb1[j * r + i];
        double acc = 0.0;
        for (int k = 0; k < r; ++k) acc = fma(F1[i * r + k], P0[j * r + k], acc);
        A[i * ld + r + j] = acc;
    }
    __syncwarp();
    for (int k = 0; k < r; ++k) {
        double v = (lane >= k && lane < r) ? fabs(A[lane * ld + k]) : -1.0;
        int bi = (lane >= k && lane < r) ? lane : r;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > v || (ov == v && oi < bi)) { v = ov; bi = oi; }
        }
        if (bi >= r) bi = k;                              // NaN column: no swap, the NaN propagates
        if (bi != k && lane < ld) {
            const double a = A[k * ld + lane];
            A[k * ld + lane] = A[bi * ld + lane];
            A[bi * ld + lane] = a;
        }
        __syncwarp();
        const double inv = 1.0 / A[k * ld + k];
        if (lane < r) colk[lane] = A[lane * ld + k];
        __syncwarp();
        if (lane < ld) {
            const double pk = A[k * ld + lane] * inv;
            A[k * ld + lane] = pk;
            for (int i = 0; i < r; ++i)
                if (i != k) A[i * ld + lane] = fma(-colk[i], pk, A[i * ld + lane]);
        }
        __syncwarp();
    }
    for (int idx = lane; idx < r * r; idx += 32) {
        const int i = idx / r, k = idx % r;
        J[idx] = A[k * ld + r + i];                       // J[i][k] = J'[k][i]
    }
}

__global__ void __launch_bounds__(SM_WARPS * 32) smooth_kernel(const double* __restrict__ mom, int64_t sst, int64_t T, int r,
                                                               double* __restrict__ Xs, double* __restrict__ Ps) {
    extern __shared__ __align__(16) double sm_dyn[];
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nm = nmom(r), rr = r * r;
    const int oXB = 0, oPB = r + rr, oX = r + 2 * rr, oP = 2 * r + 2 * rr;
    const double* ms = mom + (int64_t)s * sst;
    double* gains = sm_dyn;
    double* A = gains + SM_CHUNK * rr + warp * (2 * rr + r);
    double* colk = A + 2 * rr;
    double* xs = gains + SM_CHUNK * rr + SM_WARPS * (2 * rr + r);
    double* Pc = xs + r;
    double* D = Pc + rr;
    double* Tm = D + rr;
    double* Xo = Xs + (int64_t)s * T * r;
    double* Po = Ps ? Ps + (int64_t)s * T * rr : nullptr;

    // t = T - 1: the filtered moments
    {
        const double* m = ms + (T - 1) * nm;
        if (tid < r) {
            xs[tid] = m[oX + tid];
            Xo[(T - 1) * r + tid] = m[oX + tid];
        }
        if (Po)
            for (int idx = tid; idx < rr; idx += blockDim.x) {
                Pc[idx] = m[oP + idx];
                Po[(T - 1) * rr + idx] = m[oP + idx];
            }
    }
    for (int64_t hi = T - 2; hi >= 0; hi -= SM_CHUNK) {
        const int64_t lo = hi - SM_CHUNK + 1 > 0 ? hi - SM_CHUNK + 1 : 0;
        __syncthreads();                                  // the gains of the previous chunk are consumed
        for (int64_t t = lo + warp; t <= hi; t += SM_WARPS)
            smooth_gain(ms + t * nm, ms + (t + 1) * nm, r, A, colk, gains + (t - lo) * rr, lane);
        __syncthreads();
        for (int64_t t = hi; t >= lo; --t) {
            const double* m0 = ms + t * nm;
            const double* m1 = ms + (t + 1) * nm;
            const double* J = gains + (t - lo) * rr;
            double xn = 0.0;
            if (tid < r) {
                xn = m0[oX + tid];
                for (int k = 0; k < r; ++k) xn = fma(J[tid * r + k], xs[k] - m1[oXB + k], xn);
            }
            if (Po)
                for (int idx = tid; idx < rr; idx += blockDim.x) D[idx] = Pc[idx] - m1[oPB + idx];
            __syncthreads();
            if (tid < r) {
                xs[tid] = xn;
                Xo[t * r + tid] = xn;
            }
            if (Po) {
                for (int idx = tid; idx < rr; idx += blockDim.x) {   // Tm = J D
                    const int i = idx / r, j = idx % r;
                    double acc = 0.0;
                    for (int k = 0; k < r; ++k) acc = fma(J[i * r + k], D[k * r + j], acc);
                    Tm[idx] = acc;
                }
                __syncthreads();
                for (int idx = tid; idx < rr; idx += blockDim.x) {   // P^s_t = P_t + Tm J'
                    const int i = idx / r, j = idx % r;
                    double acc = m0[oP + idx];
                    for (int k = 0; k < r; ++k) acc = fma(Tm[i * r + k], J[j * r + k], acc);
                    Pc[idx] = acc;
                    Po[t * rr + idx] = acc;
                }
            }
            __syncthreads();
        }
    }
}

}  // namespace psmf
