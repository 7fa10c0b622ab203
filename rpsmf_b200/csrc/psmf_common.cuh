// Shared definitions for the PSMF / rPSMF filter kernels (sm_100a).
//
// Data layout in HBM
//   C      tiled structure-of-arrays: rows are grouped in tiles of 32; inside a tile the layout is
//          [r][32] (column-major) with an XOR swizzle of the row index (tile_pos below), i.e. element
//          (i, j) lives at   tile(i) * (R*32) + j*32 + ((i & 31) ^ ((j & 7) << 2)).
//          A warp that maps lane -> row reads column j of a tile as one 256-byte coalesced request,
//          and a tile is one contiguous R*256-byte block (bulk-copy friendly).
//   Y, M   time-major (T, ld): the d values of one time step are contiguous.
//   small  per series: [x R][P R*R][V R*R][Q R*R][theta R][rho][lambda] float64.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace psmf {

constexpr int TILE = 32;
constexpr int NSCAL = 8;
constexpr int NSCAL_LL = 10;   // F_LOGLIK: the record gains [nll_k, log p_k] (include/psmf_b200.h PSMF_SCAL_NLL / PSMF_SCAL_LOGPRED)
// per-step moment record (include/psmf_b200.h PSMF_NMOM): [x_bar | F (row-major) | P_bar | x | P] float64
__host__ __device__ constexpr int nmom(int R) { return 2 * R + 3 * R * R; }
constexpr int MAXR = 16;
constexpr int MAX_PEERS = 8;

// flags (mirror include/psmf_b200.h)
constexpr int F_ROBUST = 1, F_SIMPLIFIED = 2, F_CUPDATE_VT = 4, F_FIXED_LAMBDA = 16, F_LL_STUDENT = 32, F_NAN_MASK = 64,
              F_RHO_VECTOR = 128, F_GRAD_LINEAR = 256, F_LOGLIK = 512;
constexpr int DYN_IDENTITY = 0, DYN_COS = 1, DYN_LINEAR = 2, DYN_EXTERNAL = 3;
constexpr int NEVAL = 4;     // fused evaluation record (include/psmf_b200.h PSMF_EVAL_*)
// debug-only flag bits (env PSMF_DEBUG_FLAGS; results are WRONG with them): compiled in only with -DPSMF_DEBUG,
// release builds of the library carry neither the flags nor the environment knobs
#ifdef PSMF_DEBUG
constexpr int F_DBG_NOCOMPUTE = 1 << 20, F_DBG_NOSTORE = 1 << 21;
#endif

// ---- tile layout and statistics vector ------------------------------------------------------------
// Inside a 32-row tile, element (row i, column j) lives at  j*32 + (i ^ ((j & 7) << 2)).
// The XOR swizzle keeps BOTH access patterns of the kernels at the shared-memory bank-conflict floor:
//   * lane = row (rank-1 update, y_hat, e):   a column is a permuted, contiguous 256-byte segment
//   * DMMA fragments of the Gram (lane -> (column lane/4, row 4s + lane%4)): 32 distinct 8-byte banks x2
__host__ __device__ constexpr int tile_pos(int j, int i) { return j * 32 + (i ^ ((j & 7) << 2)); }

constexpr int V1_WARPS = 8;     // direct-load kernel: warps per CTA (one tile per warp at a time)
constexpr int V3_PF = 4;        // resident batch kernel: tiles per warp whose y / m are prefetched one step ahead
// resident batch kernel: CTAs per SM the register budget is sized for (shared memory permitting)
#ifndef PSMF_BATCH_MIN_R8
#define PSMF_BATCH_MIN_R8 4
#endif
__host__ __device__ constexpr int batch_min_ctas(int R, int NW) { return NW >= 8 ? 2 : (R <= 8 ? PSMF_BATCH_MIN_R8 : (R <= 12 ? 4 : 3)); }
constexpr int V2_CWARPS = 14;   // TMA-staged kernel: pass warps (+1 reduce warp, +1 producer warp)
// TMA-staged kernel: tiles per shared-memory chunk slot.  The single-thread bulk-copy loop costs ~0.6 us per iteration
// whatever the chunk size (scratch/bulkbench.cu), so a chunk must carry ~16 KB to sustain the HBM rate: 4 tiles at
// r = 16 / fp64, 8 at fp32 or r = 8, at most 16.
__host__ __device__ constexpr int v2_ts(int R, int esize) {
    const int want = 16384 / (R * TILE * esize);
    return want < 4 ? 4 : (want > 16 ? 16 : want);
}
constexpr int MAXW = 12;        // max warps that write per-warp partial statistics in any kernel

__host__ __device__ constexpr int ngram(int R) { return R * (R + 1) / 2; }
// statistics: packed upper triangle of G, then b (R), s, q1, q0, n_obs
__host__ __device__ constexpr int nstat(int R) { return ngram(R) + R + 4; }
__host__ __device__ constexpr int nstat_pad(int R) { return (nstat(R) + 7) / 8 * 8; }
// pipelined kernel: packed upper triangle of A0, u (R), h0 (R), kappa, psi, gamma, q0, n_obs
__host__ __device__ constexpr int nstat2(int R) { return ngram(R) + 2 * R + 5; }
__host__ __device__ constexpr int nstat2_pad(int R) { return (nstat2(R) + 7) / 8 * 8; }
// non-uniform diagonal R (F_RHO_VECTOR): w_i = 1 / (rho_i + a) differs per row, so the weighted Gram no longer follows
// from the unweighted one -- both are reduced:  [G = sum m w c c' | b = sum m w e c | s q1 q0 n_obs | G0 = sum m c c' |
// bu = sum m e c | n_rho = sum m rho]
__host__ __device__ constexpr int nstat_v(int R) { return 2 * ngram(R) + 2 * R + 5; }
__host__ __device__ constexpr int nstat_v_pad(int R) { return (nstat_v(R) + 7) / 8 * 8; }
__host__ __device__ constexpr int sv_G0(int R) { return ngram(R) + R + 4; }
__host__ __device__ constexpr int sv_bu(int R) { return 2 * ngram(R) + R + 4; }
__host__ __device__ constexpr int sv_nrho(int R) { return 2 * ngram(R) + 2 * R + 4; }
// F_RHO_VECTOR with F_LOGLIK: one more entry behind them, sum m log(rho_i + a) (the diagonal part of log det S_obs).  nstat_v(R)
// is odd, so the padding always has room for it: buffers sized by nstat_v_pad hold it.
__host__ __device__ constexpr int sv_nlog(int R) { return nstat_v(R); }
// packed index of Gram entry (j, j) in row-major upper-triangular order
__host__ __device__ constexpr int gram_off(int R, int j) { return j * R - j * (j - 1) / 2; }
// tagged 16-byte cells behind KParams.gparams: [2][2 MAXR] parameter sets, then [2][nstat2_pad(MAXR)] reduced totals
constexpr size_t GPARAMS_BYTES = (size_t)(4 * MAXR + 2 * nstat2_pad(MAXR)) * 16;

// resident batch kernel: dynamic shared memory = [C tiles][residuals e (ntiles * 32 doubles)][evaluation buffers]
__host__ __device__ constexpr size_t batch_c_bytes(int64_t ntiles, int R, size_t esize) {
    return ((size_t)ntiles * R * TILE * esize + 127) / 128 * 128;
}
__host__ __device__ constexpr size_t batch_dyn_bytes(int64_t ntiles, int R, size_t esize, bool eval) {
    return batch_c_bytes(ntiles, R, esize) + (size_t)ntiles * TILE * 8 + (eval ? (size_t)ntiles * TILE * 17 + 16 : 0);
}

// small-state layout (doubles per series)
__host__ __device__ constexpr int st_x(int R) { return 0; }
__host__ __device__ constexpr int st_P(int R) { return R; }
__host__ __device__ constexpr int st_V(int R) { return R + R * R; }
__host__ __device__ constexpr int st_Q(int R) { return R + 2 * R * R; }
__host__ __device__ constexpr int st_theta(int R) { return R + 3 * R * R; }
__host__ __device__ constexpr int st_rho(int R) { return 2 * R + 3 * R * R; }
__host__ __device__ constexpr int st_lam(int R) { return 2 * R + 3 * R * R + 1; }
__host__ __device__ constexpr int st_size(int R) { return 2 * R + 3 * R * R + 2; }

struct KParams {
    void* C;                  // tiled, per series stride c_series_stride elements
    int64_t c_series_stride;
    double* state;            // n_series * st_size(R)
    const void* Y; int64_t ldy; int64_t ysst;
    const uint8_t* M; int64_t ldm; int64_t msst;
    double* X_out;
    void* Yrec; int64_t ldrec; int64_t recsst;
    double* scal_out;
    const double* xbar_ext; const double* F_ext;
    double* grad_out;         // (n_series, R) accumulated theta gradient, F_GRAD_LINEAR: (n_series, R*R + R) [G_A | G_c]; or nullptr
    double* partials;         // direct kernel: grid_reduce scratch; pipelined kernel: [2][nstat2_pad][pstr] tagged cells
    unsigned long long* bar;  // direct kernel: grid barrier counter; pipelined kernel: [0..1] arrival counters, [2] flag
    long long* status;        // [0] timeout / mismatch code, [1] first bad step; -1 = none
    int64_t d, d_global;
    int64_t n_steps, k0;
    int32_t n_series, cps;    // CTAs per series
    int32_t flags, dynamics;
    double alpha, beta;
    // multi-GPU stats exchange
    int32_t world, rank;
    double* mbox_local;                    // NVLink mailbox: [2 parities][MAX_PEERS][192] tagged 16-byte cells
    double* mbox_peer[MAX_PEERS];
    unsigned long long step_base;
    // streaming kernel
    int32_t nslot;            // shared-memory chunk slots per CTA
    int32_t npw;              // pipelined kernel: active pass warps per data CTA
    int32_t trace_cta;        // CTA whose thread 0 writes the control stamps (0: direct kernel, cps: control CTA)
    double* gparams;          // pipelined kernel: [2][2 * MAXR] parameter sets published by the control CTA
    int32_t trace_steps;      // debug: number of steps recorded in `trace`
    unsigned long long* trace; // debug: [trace_steps][8] globaltimer stamps of CTA 0 (or nullptr)
    // fused evaluation (common.py:79-94): both nullptr = off
    const void* Yorig;        // original values, same layout / strides as Y
    const uint8_t* E; int64_t lde; int64_t esst;   // 1 = evaluate here (the artificially removed entries, Mmiss)
    double sig;               // interval half-width in sigmas (rPSMF.py:121-123)
    double* eval_part;        // [n_series][cps][NEVAL] per-CTA sums of this launch: sum (yhat - yorig)^2, inside, count
    // caller-driven statistics exchange (psmf_config.exchange = external): 0 = whole step, 1 = pass + reduction only
    // (statistics -> stats_ext, residuals -> e_ext), 2 = r x r update + rank-1 update from stats_ext / e_ext
    int32_t phase;
    double* stats_ext;        // nstat_pad(R) doubles
    double* e_ext;            // d doubles
    const double* rho_vec;    // F_RHO_VECTOR: diag(R) as set by the caller, (n_series, rho_sst) padded to whole tiles; the state
    int64_t rho_sst;          // scalar `rho` is then the accumulated scale prod omega_k (rPSMF.py:134 multiplies all of R)
    const double* rho_mean;   // F_RHO_VECTOR: mean of the caller's diag(R) per series (tr(R)/d of the simplified step)
    const double* lin_A;      // DYN_LINEAR: (r, r) row-major A and (r) offset c (x_bar = A x + c, F = A), device pointers
    const double* lin_c;
    int64_t glin_off;         // F_GRAD_LINEAR, direct-load and batch kernels: byte offset in dynamic shared memory of the
                              // accumulator G_A (R * R doubles, row-major); the TMA-staged control CTA uses the start
    unsigned long long spin_ns; // a wait (tagged cell, mbarrier, grid barrier, NVLink mailbox) that makes no progress for
                                // this long gives up: status word <- STATUS_TIMEOUT | step, abort word (bar[7]) <- 1
    double* mom;              // psmf_set_moments: record of step t, series s at mom + s * mom_sst + t * nmom(R), or nullptr.
    int64_t mom_sst;          // Written by the LL variant of each kernel only: the launchers pick it when mom is set
};

// ---- tags and the status word --------------------------------------------------------------------
// Tags of the 16-byte cells: never 0 (zeroed memory must not look valid), period 2^31 steps.  A stale cell holds
// the tag of two steps earlier (two parities), so a wrapped tag can never be mistaken for a current one.
__host__ __device__ constexpr uint32_t tag_of(unsigned long long step) { return (uint32_t)step | 0x80000000u; }
// status words (KParams.status, int64[2]), both reset to -1 (all bits set) by every launch:
//   [0] STATUS_TIMEOUT | (where << 48) | step = a bounded wait expired (peer GPU or CTA gone): psmf_status -> PSMF_E_STATE;
//       STATUS_MISMATCH | step = a peer runs another kernel / statistics layout (mailbox header)
//   [1] smallest step (launch-relative, over every series) with a non-finite N / omega / phi / x or N == 0, else -1
constexpr long long STATUS_TIMEOUT = 1LL << 62;
constexpr long long STATUS_MISMATCH = 1LL << 61;
constexpr int STATUS_WORDS = 2;
// An unsigned minimum over the empty word ~0: the earliest bad step wins whatever order the series ran in (a batched engine
// runs its series in waves when they outnumber the device), and a timeout or mismatch in word 0 is never overwritten.
__device__ __forceinline__ void status_bad_step(long long* status, long long t) {
    atomicMin((unsigned long long*)status + 1, (unsigned long long)t);
}
constexpr int ABORT_WORD = 7;                          // index into KParams.bar
enum SpinSite { SPIN_CELL = 1, SPIN_PEER = 2, SPIN_MBAR = 3, SPIN_GRID = 4, SPIN_RING = 5, SPIN_PARTIALS = 6 };
// NVLink mailbox: [2 parities][MAX_PEERS] slots of MBOX_SLOT tagged cells; the last cell of a slot is the header
// {kernel id, statistics count} that every receiver checks, so the stride is the same whatever kernel a peer runs
constexpr int MBOX_SLOT = 192;

struct LaunchShape {
    int threads;
    int static_smem;
    int max_ctas_per_sm;   // with the given dynamic smem
};

// per-R entry points, one translation unit each (psmf_filter_inst.cu compiled with -DPSMF_R=n)
typedef cudaError_t (*launch_fn)(const KParams&, int dtype, int grid, size_t dyn_smem, cudaStream_t, bool cooperative);
typedef cudaError_t (*shape_fn)(int dtype, size_t dyn_smem, LaunchShape*);
// cluster variant of the direct-load kernel (batched engines): grid = n_series * csize, clusters of csize CTAs; its dynamic
// shared memory ends with the parity-double-buffered partial statistics that the peers of the cluster read
typedef cudaError_t (*launch_c_fn)(const KParams&, int dtype, bool rhov, int grid, size_t dyn_smem, cudaStream_t, int csize);
typedef cudaError_t (*shape_c_fn)(int dtype, bool rhov, size_t dyn_smem, int csize, LaunchShape*, int* max_clusters);
__host__ __device__ constexpr size_t cluster_pub_bytes(int R, bool rhov) { return (size_t)2 * (rhov ? nstat_v_pad(R) : nstat_pad(R)) * 8; }

}  // namespace psmf

#define PSMF_DECLARE_R(n)                                                                                   \
    namespace psmf {                                                                                        \
    cudaError_t launch_filter_r##n(const KParams&, int, int, size_t, cudaStream_t, bool);                   \
    cudaError_t shape_filter_r##n(int, size_t, LaunchShape*);                                               \
    cudaError_t launch_filterv_r##n(const KParams&, int, int, size_t, cudaStream_t, bool);                  \
    cudaError_t shape_filterv_r##n(int, size_t, LaunchShape*);                                              \
    cudaError_t launch_filterc_r##n(const KParams&, int, bool, int, size_t, cudaStream_t, int);             \
    cudaError_t shape_filterc_r##n(int, bool, size_t, int, LaunchShape*, int*);                             \
    cudaError_t launch_stream_r##n(const KParams&, int, int, size_t, cudaStream_t, bool);                   \
    cudaError_t shape_stream_r##n(int, size_t, LaunchShape*);                                               \
    cudaError_t launch_batch_r##n(const KParams&, int, int, size_t, cudaStream_t, bool);                    \
    cudaError_t shape_batch4_r##n(int, size_t, LaunchShape*);                                               \
    cudaError_t shape_batch8_r##n(int, size_t, LaunchShape*);                                               \
    }
