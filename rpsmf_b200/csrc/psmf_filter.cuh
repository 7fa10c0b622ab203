// PSMF / rPSMF filter on sm_100a: shared device code + the direct-load persistent kernel.
//
// Per step (SURVEY.md 3.4; reference ExperimentImpute/rPSMF.py:81-135, PSMF.py:60-84,
// pypsmf/psmf/psmf.py:90-165, rpsmf.py:116-171):
//
//   row pass   one warp per 32-row tile, all warps independent
//              phase 1 (lane = row)   c_i += e_i(t-1) g(t-1)        rank-1 update of the PREVIOUS step, fused in
//                                     yhat_i = c_i . xbar ; e_i = y_i - m_i yhat_i ; w_i in {1/(rho+a), 1/a}
//                                     b += m w e c ; s += w e^2 ; q1, q0, n_obs
//              phase 2 (fragments)    G += sum_i m_i c_i c_i'  as fp64 DMMA.8x8x4 on the updated tile in
//                                     shared memory: the k-dimension of the MMA is the row index, so the
//                                     r(r+1)/2 Gram entries need 6 accumulator registers per thread instead
//                                     of 136 (measured on B200: DMMA runs at exactly the DFMA pipe rate, so
//                                     this is a register / latency optimisation, not a FLOP one)
//   reduce     warp -> CTA (fixed order) -> grid (fixed order; one or two grid barriers)
//   small      K = (I + Pbar G)^-1 Pbar (Gauss-Jordan, partial pivoting, fp64), x, omega, P, eta, N, phi,
//              V, Q, rho, lambda, g = V xbar / N, then the predict half of the next step
//
// C is touched exactly once per step (read + write); e_i stays in shared memory between steps.
// Every CTA (and every GPU) derives the small state from bit-identical reduced statistics, so the
// replicated r x r state never diverges.
#pragma once
#include <type_traits>
#include "psmf_common.cuh"

namespace psmf {

constexpr unsigned FULL = 0xffffffffu;

template <int R>
struct Smem {
    static constexpr int NSP = nstat_pad(R);
    double x[R];        // x_{t-1}, then x_t
    double xb[R];       // x_bar = f(x_{t-1})
    double fd[R];       // diagonal of F = df/dx (identity / cos dynamics)
    double vx[R];       // V x_bar
    double vxt[R];      // V' x_bar
    double g[R];        // rank-1 direction of the previous step
    double th[R];
    double P[R * R], V[R * R], Q[R * R], Pb[R * R];
    double aug[2][R][2 * R + 2];   // double-buffered augmented matrix of the r x r solve; column 2R + 1 is padding, where
                                   // F_LOGLIK keeps the pivot of elimination step k: aug[0][k][2R + 1]
    double tot[NSP];
    double part[NSP];
    double a, rho, lam;
    double w1, w0;                 // 1/(rho + a), 1/a : the only two values of w_i (rPSMF.py:92,98,32)
    double sc[8];                  // omega, eta, N, phi, sSe, alpha*phi, beta*omega
    double grad[R];                // running sum of d ell_k / d theta over the launch
    int perm[R];                   // pivot row of elimination step k
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_f64(double* p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void red_release_gpu(unsigned long long* p, unsigned long long v) {
    asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Tagged 16-byte cells {lo, tag, hi, tag}: a double that carries its own "valid for step tag" mark in each
// 8-byte half (the layout of NCCL's LL protocol), so a reader polls the data itself -- one memory round trip,
// no separate flag, no fence on the writer side, and a torn 16-byte access can never be taken for valid.
__device__ __forceinline__ void cell_store(uint4* cell, double v, uint32_t tag) {
    const uint32_t lo = (uint32_t)__double2loint(v), hi = (uint32_t)__double2hiint(v);
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(cell), "r"(lo), "r"(tag), "r"(hi), "r"(tag) : "memory");
}
// ---- bounded waits ------------------------------------------------------------------------------------
// Every wait of the kernels (tagged cells, NVLink mailbox, mbarriers, grid barrier, chunk ring) goes through a
// Spin guard: the fast path is a counter, every 64th failed attempt looks at the abort word and the clock.  A wait
// without progress for KParams.spin_ns marks the status word (STATUS_TIMEOUT | site | step) and raises the abort
// word; every other wait of the grid then gives up as well, the launch drains (results are garbage) and
// psmf_status reports PSMF_E_STATE -- a dead peer GPU or CTA cannot hang the survivors.
__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
    return v;
}
// slow path (every 64th failed attempt); takes scalars, not KParams, so that the kernel parameters stay in the
// constant bank.  Returns the start time of the wait, or ~0 when the wait has expired / the grid is aborting.
static __device__ __noinline__ unsigned long long spin_slow(unsigned long long* bar, long long* status, unsigned long long spin_ns,
                                                            unsigned long long t0, int where, long long step) {
    if (*reinterpret_cast<volatile unsigned long long*>(bar + ABORT_WORD) != 0ULL) return ~0ULL;
    const unsigned long long now = gtimer();
    if (t0 == 0ULL) return now;
    if (now - t0 < spin_ns) return t0;
    const unsigned long long code = (unsigned long long)STATUS_TIMEOUT | ((unsigned long long)where << 48) |
                                    ((unsigned long long)step & 0xFFFFFFFFFFFFULL);
    atomicCAS((unsigned long long*)status, ~0ULL, code);
    atomicExch(bar + ABORT_WORD, 1ULL);
    return ~0ULL;
}
struct Spin {
    unsigned n = 0;
    unsigned long long t0 = 0;
    __device__ __forceinline__ bool expired(const KParams& p, int where, long long step) {
        if ((++n & 63u) != 0u) return false;
        t0 = spin_slow(p.bar, p.status, p.spin_ns, t0, where, step);
        return t0 == ~0ULL;
    }
};

// pollers share their SM with warps that do arithmetic (the solvers of the control CTA, the pass warps of a data CTA):
// a short sleep after a failed attempt keeps them out of the issue slots; it adds at most this much to the wake-up
#ifndef PSMF_POLL_BACKOFF_NS
#define PSMF_POLL_BACKOFF_NS 40
#endif
constexpr unsigned POLL_BACKOFF_NS = PSMF_POLL_BACKOFF_NS;
template <bool BACKOFF = true>
__device__ __forceinline__ double cell_poll(const KParams& p, const uint4* cell, uint32_t tag, long long step) {
    uint32_t lo, t0, hi, t1;
    Spin sp;
    for (;;) {
        asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t0), "=r"(hi), "=r"(t1) : "l"(cell) : "memory");
        if (t0 == tag && t1 == tag) break;
        if (sp.expired(p, SPIN_CELL, step)) break;
        if (BACKOFF && POLL_BACKOFF_NS > 0) __nanosleep(POLL_BACKOFF_NS);
    }
    return __hiloint2double((int)hi, (int)lo);
}
__device__ __forceinline__ void cell_store_sys(uint4* cell, double v, uint32_t tag) {      // peer GPU over NVLink
    const uint32_t lo = (uint32_t)__double2loint(v), hi = (uint32_t)__double2hiint(v);
    asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(cell), "r"(lo), "r"(tag), "r"(hi), "r"(tag) : "memory");
}
__device__ __forceinline__ double cell_poll_sys(const KParams& p, const uint4* cell, uint32_t tag, long long step) {
    uint32_t lo, t0, hi, t1;
    Spin sp;
    for (;;) {
        asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t0), "=r"(hi), "=r"(t1) : "l"(cell) : "memory");
        if (t0 == tag && t1 == tag) break;
        if (sp.expired(p, SPIN_PEER, step)) break;
    }
    return __hiloint2double((int)hi, (int)lo);
}

// barrier 0 over the first `n` threads of the CTA (n == blockDim.x: plain __syncthreads; the streaming
// kernel excludes its producer warp)
template <int BAR = 0>
__device__ __forceinline__ void sync_n(int n) { asm volatile("bar.sync %0, %1;" ::"n"(BAR), "r"(n) : "memory"); }

// All CTAs of the grid are co-resident (cooperative launch).  `target` grows monotonically.
template <int BAR = 0>
__device__ __forceinline__ void grid_barrier(const KParams& p, unsigned long long target, int nthr, int tid, long long step) {
    sync_n<BAR>(nthr);
    if (tid == 0) {
        red_release_gpu(p.bar, 1ULL);
        Spin sp;
        while (ld_acquire_gpu(p.bar) < target) {
            if (sp.expired(p, SPIN_GRID, step)) break;
        }
    }
    sync_n<BAR>(nthr);
}

// debug phase stamps (CTA 0, thread 0): enabled when KParams.trace != nullptr
__device__ __forceinline__ void stamp(const KParams& p, int64_t t, int slot, int who = 0) {
    if (p.trace != nullptr && blockIdx.x == p.trace_cta && threadIdx.x == who && t < p.trace_steps) {
        unsigned long long v;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
        p.trace[t * 16 + slot] = v;
    }
    __syncwarp();   // the single-thread branch above must not leave the warp split (shuffles would take the slow path)
}

// debug stamps of the first pass warp (psmf_stream.cuh): slot 8.. of the 16-entry trace row
__device__ __forceinline__ void stamp_pass(const KParams& p, int64_t t, int slot, unsigned long long v, bool timer) {
    if (p.trace != nullptr && blockIdx.x == 0 && t < p.trace_steps) {
        if (timer) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
        p.trace[t * 16 + slot] = v;
    }
}

// Warp index as a WARP-UNIFORM value (broadcast from lane 0): the compiler can then see that a branch on it never splits a
// warp and emits plain SHFL / REDUX in the role-specialised code below it; with `threadIdx.x >> 5` every shuffle is
// wrapped in WARPSYNC.COLLECTIVE ... ENDCOLLECTIVE (~15 extra cycles each, measured on the one-warp solver).
__device__ __forceinline__ int uniform_warp_id() { return __shfl_sync(FULL, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ double warp_allsum(double v) {
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;   // bit-identical on every lane (a+b == b+a at every stage)
}

// 1/x to ~1 ulp: MUFU.RCP64H seed + two Newton steps (the pivots of the solve are O(1) or larger)
__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(fma(-x, r, 1.0), r, r);
    r = fma(fma(-x, r, 1.0), r, r);
    return r;
}

// Transposing butterfly: reduces N per-lane accumulators over the 32 lanes with ~N shuffles instead of
// 5N.  On return lane l holds the full sums of entries [base, base + bfly_final(N)).
__host__ __device__ constexpr int bfly_final(int n) {
    for (int i = 0; i < 5; ++i) n = (n + 1) / 2;
    return n;
}
// Entries with index >= lim are padding (odd counts are rounded up at every stage) and must not be stored.
template <int N, int O, int NA>
__device__ __forceinline__ void bfly(double (&v)[NA], int lane, int& base, int& lim) {
    constexpr int H = (N + 1) / 2;
    const bool up = (lane & O) != 0;
    lim = min(lim, base + N);
#pragma unroll
    for (int i = 0; i < H; ++i) {
        const double lo = v[i];
        const double hi = (i + H < N) ? v[i + H] : 0.0;
        const double send = up ? lo : hi;
        const double keep = up ? hi : lo;
        v[i] = keep + __shfl_xor_sync(FULL, send, O);
    }
    if (up) base += H;
    if constexpr (O > 1) bfly<H, O / 2, NA>(v, lane, base, lim);
}

// ---- per-warp statistics of one pass -------------------------------------------------------------------
// D(8x8) += A(8x4) * B(4x8), fp64 (SASS: DMMA.8x8x4).  Fragments: a = A[lane/4][lane%4],
// b = B[lane%4][lane/4], d[0..1] = D[lane/4][2*(lane%4) + 0..1].
__device__ __forceinline__ void dmma884(double (&d)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d[0]), "+d"(d[1])
                 : "d"(a), "d"(b));
}

template <int R>
struct TileAcc {
    double g00[2], g01[2], g11[2];   // fragments of sum_i m_i c_i c_i' : blocks (0..7,0..7), (0..7,8..15), (8..15,8..15)
    double g00x[2];                  // r <= 8: second accumulator of block (0,0) -- two independent DMMA chains instead of one
    double v[R + 4];                 // per-lane: b (R), s, q1, q0, n_obs
    __device__ __forceinline__ void zero() {
        g00[0] = g00[1] = g01[0] = g01[1] = g11[0] = g11[1] = g00x[0] = g00x[1] = 0.0;
#pragma unroll
        for (int i = 0; i < R + 4; ++i) v[i] = 0.0;
    }
};

// phase 1 for one row (lane = row): c holds the row on entry, the updated row on exit.
template <int R>
__device__ __forceinline__ void row_stats(TileAcc<R>& A, const Smem<R>& sh, double (&c)[R], double ep, bool inb, bool mi,
                                          double yi, double w1, double w0, double& e, double& yh) {
#pragma unroll
    for (int j = 0; j < R; ++j) c[j] = fma(ep, sh.g[j], c[j]);                // rPSMF.py:111 (previous step)
    double yh4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int j = 0; j < R; ++j) yh4[j & 3] = fma(c[j], sh.xb[j], yh4[j & 3]);   // rPSMF.py:89
    yh = (yh4[0] + yh4[1]) + (yh4[2] + yh4[3]);
    e = yi - (mi ? yh : 0.0);                                                  // rPSMF.py:101
    const double w = mi ? w1 : w0;                                             // rPSMF.py:92,98,32
    const double ew = mi ? e * w1 : 0.0;
#pragma unroll
    for (int j = 0; j < R; ++j) A.v[j] = fma(ew, c[j], A.v[j]);               // b = CM' Ri diff
    const double e2 = e * e;
    // diff' Ri diff.  A missing row with a zero residual adds nothing, also when a = 0 makes w0 = 1/a infinite (x'Vx
    // vanishes exactly after a step with every row missing at r = 1): the same rule as s = w1 q1 + w0 q0 of the TMA kernel
    A.v[R + 0] = fma((inb && (mi || e2 != 0.0)) ? w : 0.0, e2, A.v[R + 0]);
    A.v[R + 1] += mi ? e2 : 0.0;                                               // rPSMF.py:112-114 (observed rows)
    A.v[R + 2] += mi ? 0.0 : e2;                                               //                  (missing rows)
    A.v[R + 3] += mi ? 1.0 : 0.0;
}

// phase 2: masked Gram of the updated tile (swizzled [R][32] layout in shared memory).  mbits = ballot of m_i.
template <int R, typename TS>
__device__ __forceinline__ void tile_gram(TileAcc<R>& A, const TS* __restrict__ tile, unsigned mbits, int lane) {
    const int kk = lane & 3, mm = lane >> 2;
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const int row = 4 * s + kk;
        const bool mrow = (mbits >> row) & 1u;
        const int pos = row ^ (mm << 2);                       // tile_pos(mm, row) - mm*32 == tile_pos(8+mm, row) - (8+mm)*32
        const double a0 = (mm < R) ? (double)tile[mm * 32 + pos] : 0.0;
        const double b0 = mrow ? a0 : 0.0;
        if constexpr (R > 8) {
            dmma884(A.g00, a0, b0);
            const double a1 = (8 + mm < R) ? (double)tile[(8 + mm) * 32 + pos] : 0.0;
            const double b1 = mrow ? a1 : 0.0;
            dmma884(A.g01, a0, b1);
            dmma884(A.g11, a1, b1);
        } else {
            // a single block: alternate between two accumulators so that consecutive DMMAs do not wait for each other
            if (s & 1) dmma884(A.g00x, a0, b0);
            else dmma884(A.g00, a0, b0);
        }
    }
}

// two tiles at once (r <= 8): tile A accumulates into g00, tile B into g00x -- two independent DMMA chains
template <int R, typename TS>
__device__ __forceinline__ void tile_gram2(TileAcc<R>& A, const TS* __restrict__ ta, unsigned mba, const TS* __restrict__ tb, unsigned mbb,
                                           int lane) {
    static_assert(R <= 8, "tile_gram2 is the single-block form");
    const int kk = lane & 3, mm = lane >> 2;
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const int row = 4 * s + kk;
        const int pos = row ^ (mm << 2);
        const double a = (mm < R) ? (double)ta[mm * 32 + pos] : 0.0;
        const double b = (mm < R) ? (double)tb[mm * 32 + pos] : 0.0;
        dmma884(A.g00, a, ((mba >> row) & 1u) ? a : 0.0);
        dmma884(A.g00x, b, ((mbb >> row) & 1u) ? b : 0.0);
    }
}

// end of pass: this warp's partial statistics -> red[0 .. nstat(R))   (G = w1 * sum m c c', rPSMF.py:35)
template <int R>
__device__ __forceinline__ void acc_writeout(TileAcc<R>& A, double* __restrict__ red, double w1, int lane) {
    const int kk = lane & 3, mm = lane >> 2;
#pragma unroll
    for (int x = 0; x < 2; ++x) {
        const int n = 2 * kk + x;
        if (mm <= n && n < R) red[gram_off(R, mm) + (n - mm)] = w1 * (R > 8 ? A.g00[x] : A.g00[x] + A.g00x[x]);
        if constexpr (R > 8) {
            if (8 + n < R) red[gram_off(R, mm) + (8 + n - mm)] = w1 * A.g01[x];
            if (mm <= n && 8 + n < R) red[gram_off(R, 8 + mm) + (n - mm)] = w1 * A.g11[x];
        }
    }
    constexpr int NV = R + 4;
    int base = 0, lim = NV;
    bfly<NV, 16, NV>(A.v, lane, base, lim);
    constexpr int NF = bfly_final(NV);
#pragma unroll
    for (int i = 0; i < NF; ++i)
        if (base + i < lim) red[ngram(R) + base + i] = A.v[i];
}

// ---- non-uniform diagonal R (F_RHO_VECTOR; psmf.py:144-152 takes the Woodbury branch for ANY diagonal R) -------------
// Per-row weights w_i = 1 / (rho_i + a): the weighted Gram G (for K) and the unweighted G0 (for eta = tr(M R M + C Pbar C')
// / d, rPSMF.py:108) are both accumulated, as fp64 DMMAs on the same fragments; sum m e c (theta gradient) rides along as
// plain FMAs on the element a lane holds anyway, like [u | h0] of the pipelined kernel.
template <int R>
struct TileAccV : TileAcc<R> {
    double h00[2], h01[2], h11[2];   // fragments of sum_i m_i w_i c_i c_i'
    double u0, u1;                   // partial sums of sum m e c for column lane/4 (u0) and 8 + lane/4 (u1)
    double nrho;                     // per-lane sum m rho
    __device__ __forceinline__ void zero_v() {
        this->zero();
        h00[0] = h00[1] = h01[0] = h01[1] = h11[0] = h11[1] = u0 = u1 = nrho = 0.0;
    }
};
template <int R, typename TS>
__device__ __forceinline__ void tile_gram_v(TileAccV<R>& A, const TS* __restrict__ tile, unsigned mbits, double wm, double me, int lane) {
    const int kk = lane & 3, mm = lane >> 2;
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const int row = 4 * s + kk;
        const bool mrow = (mbits >> row) & 1u;
        const int pos = row ^ (mm << 2);
        const double wr = __shfl_sync(FULL, wm, row), er = __shfl_sync(FULL, me, row);     // m w and m e of the row
        const double a0 = (mm < R) ? (double)tile[mm * 32 + pos] : 0.0;
        dmma884(A.g00, a0, mrow ? a0 : 0.0);
        dmma884(A.h00, a0, a0 * wr);
        A.u0 = fma(a0, er, A.u0);
        if constexpr (R > 8) {
            const double a1 = (8 + mm < R) ? (double)tile[(8 + mm) * 32 + pos] : 0.0;
            const double b1 = mrow ? a1 : 0.0, c1 = a1 * wr;
            dmma884(A.g01, a0, b1);
            dmma884(A.g11, a1, b1);
            dmma884(A.h01, a0, c1);
            dmma884(A.h11, a1, c1);
            A.u1 = fma(a1, er, A.u1);
        }
    }
}
template <int R>
__device__ __forceinline__ void acc_writeout_v(TileAccV<R>& A, double* __restrict__ red, int lane) {
    const int kk = lane & 3, mm = lane >> 2;
    double* g0 = red + sv_G0(R);
#pragma unroll
    for (int x = 0; x < 2; ++x) {
        const int n = 2 * kk + x;
        if (mm <= n && n < R) {
            red[gram_off(R, mm) + (n - mm)] = A.h00[x];
            g0[gram_off(R, mm) + (n - mm)] = A.g00[x];
        }
        if constexpr (R > 8) {
            if (8 + n < R) {
                red[gram_off(R, mm) + (8 + n - mm)] = A.h01[x];
                g0[gram_off(R, mm) + (8 + n - mm)] = A.g01[x];
            }
            if (mm <= n && 8 + n < R) {
                red[gram_off(R, 8 + mm) + (n - mm)] = A.h11[x];
                g0[gram_off(R, 8 + mm) + (n - mm)] = A.g11[x];
            }
        }
    }
    constexpr int NV = R + 4;
    int base = 0, lim = NV;
    bfly<NV, 16, NV>(A.v, lane, base, lim);
    constexpr int NF = bfly_final(NV);
#pragma unroll
    for (int i = 0; i < NF; ++i)
        if (base + i < lim) red[ngram(R) + base + i] = A.v[i];
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {                              // sum over the four row classes kk (fixed order)
        A.u0 += __shfl_xor_sync(FULL, A.u0, o);
        if constexpr (R > 8) A.u1 += __shfl_xor_sync(FULL, A.u1, o);
    }
    if (kk == 0) {
        if (mm < R) red[sv_bu(R) + mm] = A.u0;
        if constexpr (R > 8) {
            if (8 + mm < R) red[sv_bu(R) + 8 + mm] = A.u1;
        }
    }
    const double nr = warp_allsum(A.nrho);
    if (lane == 0) red[sv_nrho(R)] = nr;
}

// x_bar_i = c_i + sum_k A_ik x_k in a FIXED operation order: the pipelined kernel evaluates it in two places (the
// published x_bar of the data CTAs and the control CTA's own copy) and both must be bit-identical
template <int R>
__device__ __forceinline__ double linear_predict(const KParams& p, const double* __restrict__ x, int i) {
    double acc = p.lin_c != nullptr ? p.lin_c[i] : 0.0;
#pragma unroll
    for (int k = 0; k < R; ++k) acc = fma(p.lin_A[i * R + k], x[k], acc);
    return acc;
}

// d ell_k / d f_i of the incremental log-likelihood with f = x_bar, N, eta and V held fixed (psmf.py:57-64,167-177;
// rpsmf.py:62-71,196-200): s = f'Vf + eta = N, e = y - M C f, cte = C'Me, n = n_obs, q = q1
__device__ __forceinline__ double dll_df(int flags, double vx, double vxt, double cte, double q1, double nobs, double lam, double N) {
    const double vsf = 0.5 * (vx + vxt);
    if ((flags & F_LL_STUDENT) != 0) {
        const double gq = 1.0 + q1 / (lam * N);
        return nobs * vsf / N - (nobs + lam) / (gq * lam * N) * (cte + (q1 / N) * vsf);
    }
    return (nobs / N - q1 / (N * N)) * vsf - cte / N;
}

// F_LOGLIK: nll_k and log p_k of one step (include/psmf_b200.h PSMF_LOGLIK), by one whole warp; every lane returns both.
//   n = n_obs, N = a + eta, q1 = sum_obs e^2, lam = lambda entering the step, ldr = sum_obs log(rho_i + a),
//   d2 = Delta^2 = diff_obs' S_obs^-1 diff_obs (w1 q1 - b'Kb);
//   lane i < R holds pivot i of the elimination of I + Pbar G (1.0 on the other lanes and without an elimination):
//   log det S_obs = ldr + sum_i log|pivot_i| (matrix-determinant lemma; det(I + Pbar G) >= 1, so no sign to track).
// The transcendentals of the different terms are the same instruction on different lanes, and the pivot sum has a fixed
// order: every CTA and every rank gets the same bits.
__device__ __forceinline__ void step_loglik(int flags, double piv, double n, double N, double q1, double lam, double ldr, double d2,
                                            int lane, double& nll, double& lp) {
    constexpr double PI = 3.141592653589793;
    const double lgdet = warp_allsum(log(fabs(piv)));
    const double lg = lgamma(0.5 * (lane == 1 ? lam + n : lam));                    // lane 0: lgamma(lam/2), 1: lgamma((lam+n)/2)
    const double lv = log(((lane & 1) ? lam : 2.0) * PI * (lane < 2 ? N : 1.0));    // lane 0: log 2piN, 1: log lam pi N, 2: log 2pi,
                                                                                    // 3: log lam pi
    const double l1 = log1p(lane == 0 ? q1 / (lam * N) : d2 / lam);                 // lane 0: log(1 + q1/(lam N)), 1: log(1 + d2/lam)
    const double lg0 = __shfl_sync(FULL, lg, 0), lg1 = __shfl_sync(FULL, lg, 1);
    const double l2piN = __shfl_sync(FULL, lv, 0), llpiN = __shfl_sync(FULL, lv, 1);
    const double l2pi = __shfl_sync(FULL, lv, 2), llpi = __shfl_sync(FULL, lv, 3);
    const double lq = __shfl_sync(FULL, l1, 0), ld = __shfl_sync(FULL, l1, 1);
    const double logdet = ldr + lgdet;
    if (n == 0.0) {                                                                 // every row missing: no observation, no term
        nll = 0.0;
        lp = 0.0;
        return;
    }
    nll = (flags & F_LL_STUDENT) != 0 ? (lg0 - lg1) + 0.5 * n * llpiN + 0.5 * (lam + n) * lq : 0.5 * n * l2piN + q1 / (2.0 * N);
    lp = (flags & F_ROBUST) != 0 ? (lg1 - lg0) - 0.5 * n * llpi - 0.5 * logdet - 0.5 * (lam + n) * ld : -0.5 * (n * l2pi + logdet + d2);
}

// The F_LOGLIK variant (LL) of each kernel serves F_GRAD_LINEAR too (GL = true, the flag decides at run time): one more
// instantiation per kernel instead of the GL x LL product.  In the GL-only variant this is a constant, so it compiles as before.
template <bool GL, bool LL>
__device__ __forceinline__ bool glin_on(const KParams& p) { return GL && (!LL || (p.flags & F_GRAD_LINEAR) != 0); }

// F_GRAD_LINEAR: the accumulator G_A (R * R doubles, row-major) in dynamic shared memory at p.glin_off.  Recomputed where it
// is used (p lives in the constant bank): no pointer stays live across the row pass.
__device__ __forceinline__ double* glin_acc(const KParams& p) {
    extern __shared__ __align__(16) unsigned char psmf_dyn_smem[];
    return reinterpret_cast<double*>(psmf_dyn_smem + p.glin_off);
}

// F_GRAD_LINEAR: G_A += gf x_{k-1}' (row-major R x R in shared memory) by one whole warp; lane i < R holds gf_i and
// x_{k-1, i}.  One FMA per entry and step, in step order, so every kernel, CTA and rank forms the same sum.
template <int R>
__device__ __forceinline__ void lin_grad_accum(double* __restrict__ gA, double gf, double xo, int lane) {
#pragma unroll
    for (int b = 0; b < R * R; b += 32) {
        const int idx = b + lane;
        const double gi = __shfl_sync(FULL, gf, (idx / R) & 31), xj = __shfl_sync(FULL, xo, idx % R);
        if (idx < R * R) gA[idx] = fma(gi, xj, gA[idx]);
    }
}

// end of launch: [G_A row-major | G_c] -> out (R * R + R doubles); G_A was written by another warp
template <int R>
__device__ __forceinline__ void lin_grad_writeout(double* __restrict__ out, const double* gA, const double* gc, int tid, int nthr) {
    __syncthreads();
    for (int i = tid; i < R * R + R; i += nthr) out[i] = i < R * R ? gA[i] : gc[i - R * R];
}

// ---- fused evaluation (ExperimentImpute/common.py:79-94) -----------------------------------------------------
// Accumulated inside the row pass instead of materialising (n, d) Yrec / YrecL / YrecH arrays: over the entries
// marked in E (the artificially removed ones, Mmiss) the squared one-step prediction error (Epred, rPSMF.py:139) and
// the number of original values inside the interval yhat -+ sig sqrt(U) (rPSMF.py:121-123, common.py:87-94).  U
// needs eta of the SAME step, which only exists after the solve: the prediction, the original value and the flags of
// a row wait in shared memory and are scored at the start of the next pass (or in the flush after the last step).
struct EvalAcc {
    double se = 0.0, ne = 0.0, inside = 0.0;
};
struct EvalBuf {          // per-CTA shared-memory buffers, one entry per local row (nullptr: evaluation off)
    double* yh;           // prediction of the previous step
    double* yo;           // original value of the previous step
    unsigned char* fl;    // bit 0: evaluate, bit 1: observed (m_i)
};
__device__ __forceinline__ void eval_cover(EvalAcc& ev, const EvalBuf& eb, int rl, double a, double eta, double N, bool robust, double sig) {
    const unsigned f = eb.fl[rl];
    if (f & 1u) {
        const double U = robust ? __dadd_rn(__dmul_rn(a, (double)((f >> 1) & 1u)), eta) : N;    // rPSMF.py:112 / PSMF.py:83-84
        const double s = __dmul_rn(sig, sqrt(U));
        const double yh = eb.yh[rl], yo = eb.yo[rl];
        const double hi = __dadd_rn(yh, s), lo = __dsub_rn(yh, s);                              // rPSMF.py:122-123
        ev.inside += (yo < hi && lo < yo) ? 1.0 : 0.0;                                          // common.py:91-93
    }
}
__device__ __forceinline__ void eval_row(EvalAcc& ev, const EvalBuf& eb, int rl, bool ei, bool mi, double yh, double yo) {
    if (ei) {
        const double dlt = __dsub_rn(yh, yo);
        ev.se = __dadd_rn(ev.se, __dmul_rn(dlt, dlt));                                          // common.py:79-84
        ev.ne += 1.0;
    }
    eb.yh[rl] = yh;
    eb.yo[rl] = yo;
    eb.fl[rl] = (unsigned char)((ei ? 1u : 0u) | (mi ? 2u : 0u));
}
// end of launch: per-lane sums -> warp (butterfly, fixed order) -> shared scratch -> CTA record in p.eval_part
template <int NW>
__device__ __forceinline__ void eval_writeout(const KParams& p, EvalAcc& ev, double* scratch /* NW * 4 doubles */, int series, int part,
                                              int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    const double a = warp_allsum(ev.se), b = warp_allsum(ev.inside), c = warp_allsum(ev.ne);
    if (lane == 0) {
        scratch[warp * 4 + 0] = a;
        scratch[warp * 4 + 1] = b;
        scratch[warp * 4 + 2] = c;
    }
    __syncthreads();
    if (tid < 3) {
        double t = 0.0;
        for (int w = 0; w < NW; ++w) t += scratch[w * 4 + tid];
        p.eval_part[((int64_t)series * p.cps + part) * NEVAL + tid] = t;
    }
}

// ---- predict half: x_bar = f(x), P_bar = F P F' + Q, V x_bar, a (all `nthr` threads; ends with a barrier) ----
template <int R, int BAR = 0>
__device__ void predict_cta(const KParams& p, Smem<R>& sh, int tid, int64_t k, int series, int nthr) {
    const bool simp = (p.flags & F_SIMPLIFIED) != 0;
    const int lane = tid & 31;
    if (tid < R) {
        double xb, fd = 1.0;
        if (p.dynamics == DYN_COS) {                                          // synthetic_psmf.py:105-106
            const double arg = __dadd_rn(__dmul_rn(__dmul_rn(6.283185307179586, sh.th[tid]), (double)k), sh.x[tid]);
            xb = cos(arg);
            fd = -sin(arg);
        } else if (p.dynamics == DYN_EXTERNAL) {
            xb = p.xbar_ext[(int64_t)series * R + tid];
        } else if (p.dynamics == DYN_LINEAR) {                                // x_bar = A x + c (psmf.py:104 with a linear f;
            xb = linear_predict<R>(p, sh.x, tid);                             //  ExperimentChange/PSMF.m:29: Xp = A * X)
        } else {
            xb = sh.x[tid];                                                   // rPSMF.py:86
        }
        sh.xb[tid] = xb;
        sh.fd[tid] = fd;
    }
    sync_n<BAR>(nthr);
    if (tid >= nthr - 32) {
        // last warp: V x_bar, V' x_bar, a = x_bar' V x_bar and the two possible row weights
        double v = 0.0;
        if (lane < 2 * R) {
            const int j = lane < R ? lane : lane - R;
            double v0 = 0.0, v1 = 0.0;
#pragma unroll
            for (int k2 = 0; k2 < R; k2 += 2) {
                v0 = fma(lane < R ? sh.V[j * R + k2] : sh.V[k2 * R + j], sh.xb[k2], v0);
                if (k2 + 1 < R) v1 = fma(lane < R ? sh.V[j * R + k2 + 1] : sh.V[(k2 + 1) * R + j], sh.xb[k2 + 1], v1);
            }
            v = v0 + v1;
            if (lane < R) sh.vx[j] = v; else sh.vxt[j] = v;
        }
        double av = lane < R ? sh.xb[lane] * v : 0.0;
        av = warp_allsum(av);                                                 // rPSMF.py:93
        if (lane == 0) {
            sh.a = av;
            sh.w1 = 1.0 / (sh.rho + av);
            sh.w0 = 1.0 / av;
        }
    }
    for (int idx = tid; idx < R * R; idx += nthr) {
        const int i = idx / R, j = idx % R;
        double pb;
        if (simp) {                                                           // synthetic_psmf.py:83-84
            pb = sh.P[idx];
        } else if (p.dynamics == DYN_EXTERNAL || p.dynamics == DYN_LINEAR) {   // psmf.py:115 with a dense F (PSMF.m:30: A P A' + Q)
            const double* F = p.dynamics == DYN_LINEAR ? p.lin_A : p.F_ext + (int64_t)series * R * R;
            double acc = 0.0;
            for (int k2 = 0; k2 < R; ++k2) {
                double t2 = 0.0;
                for (int l = 0; l < R; ++l) t2 = fma(sh.P[k2 * R + l], F[j * R + l], t2);
                acc = fma(F[i * R + k2], t2, acc);
            }
            pb = acc + sh.Q[idx];
        } else {                                                              // rPSMF.py:87 / psmf.py:115
            pb = sh.fd[i] * sh.P[idx] * sh.fd[j] + sh.Q[idx];
        }
        sh.Pb[idx] = pb;
    }
    sync_n<BAR>(nthr);
}

// Gauss-Jordan with partial pivoting on the R x (2R+1) augmented matrix [I + Pbar G | Pbar | Pbar b], run by
// GJ_THREADS threads with one named barrier per elimination step.  Thread (row i, q) keeps its <= CPT
// elements of row i in registers; the matrix is double-buffered in shared memory so that everybody can read
// column k and the pivot row of the previous step.  Rows are not swapped: step k eliminates with the unused
// row of largest |a_ik| -- found redundantly by every warp (no broadcast barrier) with one warp-wide
// integer max over the high words of |a_ik| (16 mantissa bits decide, ties -> lowest row) -- and perm[k]
// remembers it, so the solution row of unknown k is aug[R & 1][perm[k]].  PIV (F_LOGLIK): the writer of perm[k] also keeps
// the pivot a_{perm[k], k} in aug[0][k][2R + 1] (a padding column) for log det(I + Pbar G).
constexpr int GJ_THREADS = 192;                         // direct-load kernel; the pipelined kernel uses its control warps
template <int R, int NGJ, int GJBAR = 1, int NC = 2 * R + 1, bool PIV = false>
__device__ void gauss_jordan_cta(Smem<R>& sh, int tid) {
    constexpr int TPR = NGJ / R;                        // threads per row
    constexpr int CPT = (NC + TPR - 1) / TPR;           // columns per thread
    const bool active = tid < R * TPR;
    const int i = active ? tid / TPR : 0;
    const int q = tid - (tid / TPR) * TPR;
    double own[CPT];
#pragma unroll
    for (int e = 0; e < CPT; ++e) {
        const int c = q + TPR * e;
        own[e] = (active && c < NC) ? sh.aug[0][i][c] : 0.0;
    }
    unsigned used = 0;
    const int r2 = tid & 15;                            // pivot search: lane -> candidate row (both half-warps)
    for (int k = 0; k < R; ++k) {
        const int cur = k & 1, nxt = cur ^ 1;
        // every warp finds the pivot row on its own: one candidate per lane, integer max over the high word
        // of |a_ik| (REDUX), and the reciprocal of every candidate is computed while the max is in flight
        const double cand = (r2 < R) ? sh.aug[cur][r2][k] : 1.0;
        const double aik = sh.aug[cur][i][k];
        const int hi = __double2hiint(fabs(cand));
        const int key = (r2 >= R || ((used >> r2) & 1u)) ? -1 : ((hi & 0x7ffffff0) | (15 - r2));
        const double cinv = fast_rcp(cand);
        const int pi = 15 - (__reduce_max_sync(FULL, key) & 15);
        const double inv = __shfl_sync(FULL, cinv, pi);
        used |= 1u << pi;
        if (tid == 0) {
            sh.perm[k] = pi;
            if constexpr (PIV) sh.aug[0][k][2 * R + 1] = sh.aug[cur][pi][k];
        }
        // all pivot-row loads first: the stores below may alias them as far as the compiler can tell, and
        // interleaving would serialise load -> multiply -> store per column
        double rp[CPT];
#pragma unroll
        for (int e = 0; e < CPT; ++e) {
            const int c = q + TPR * e;
            rp[e] = sh.aug[cur][pi][c < NC ? c : NC - 1];
        }
#pragma unroll
        for (int e = 0; e < CPT; ++e) {
            const int c = q + TPR * e;
            const double rpc = rp[e] * inv;
            own[e] = (i == pi) ? rpc : fma(-aik, rpc, own[e]);
            if (active && c < NC) sh.aug[nxt][i][c] = own[e];
        }
        named_bar_sync(GJBAR, NGJ);
    }
}

// F_GRAD_LINEAR, one whole warp of small_update, after side_half and before x_k replaces x_{k-1}: G_c += gf, G_A += gf x_{k-1}'
template <int R>
__device__ __forceinline__ void lin_grad_step(const KParams& p, Smem<R>& sh, const double* tot) {
    constexpr int NGm = ngram(R);
    const int lane = threadIdx.x & 31;
    const bool rhov = (p.flags & F_RHO_VECTOR) != 0;                           // tot is then the nstat_v vector
    __syncwarp();                                                              // N of side_half (lane 0)
    double gf = 0.0, xo = 0.0;
    if (lane < R) {
        const double cte = rhov ? tot[sv_bu(R) + lane] : tot[NGm + lane] * (sh.rho + sh.a);
        gf = dll_df(p.flags, sh.vx[lane], sh.vxt[lane], cte, tot[NGm + R + 1], tot[NGm + R + 3], sh.lam, sh.sc[2]);
        xo = sh.x[lane];
        sh.grad[lane] += gf;
    }
    lin_grad_accum<R>(glin_acc(p), gf, xo, lane);
}

// ---- r x r part of the step (rPSMF.py:102-115,133-135), identical on every CTA; all `nthr` threads ----
// Two halves.  eta, N, phi, the update of V and the rank-1 direction g need the reduced statistics but NOT the inverse:
// when the CTA has a warp outside the NGJ elimination threads (nthr >= NGJ + 32) that warp computes them WHILE the
// Gauss-Jordan elimination runs; x, omega, P, Q, rho, lambda follow the elimination.  The arithmetic is the same either
// way (bit-identical results), only the schedule differs.
// GL: F_GRAD_LINEAR is set, LL: F_LOGLIK is set (template parameters so that the kernels without them compile to the code they
// had before them; see glin_on)
template <int R, int NGJ, bool GL = false, bool LL = false, int BAR = 0, int GJBAR = 1>
__device__ void small_update(const KParams& p, Smem<R>& sh, int tid, int lane, int warp, int series, int64_t t,
                             bool writer, int nthr, const double* totv = nullptr) {
    constexpr int NGm = ngram(R);
    constexpr int FIN = R & 1;                      // buffer holding the result of the elimination
    const bool simp = (p.flags & F_SIMPLIFIED) != 0;
    const bool robust = (p.flags & F_ROBUST) != 0;
    // totv != nullptr: non-uniform diagonal R, statistics in the nstat_v layout (G, b, s, q1, q0, n_obs as usual, then
    // the unweighted Gram, sum m e c and sum m rho)
    const bool rhov = totv != nullptr;
    const double* tot = rhov ? totv : sh.tot;
    const double* G0p = rhov ? totv + sv_G0(R) : sh.tot;
    const double dg = (double)p.d_global;
    const bool side_warp = !simp && nthr >= NGJ + 32;          // a whole warp next to the elimination threads

    // the half that does not need the inverse, executed by ONE warp (all 32 lanes): eta, N, phi -> sc[1..3,5,7], V, g
    auto side_half = [&]() {
        const double a = sh.a, rho = sh.rho, lam = sh.lam;
        const double q1 = tot[NGm + R + 1], q0 = tot[NGm + R + 2], nobs = tot[NGm + R + 3];
        double trpg = 0.0;
        if (!simp && lane < R) {
            double t0 = 0.0, t1 = 0.0;
#pragma unroll
            for (int i = 0; i < R; i += 2) {
                const int lo = i < lane ? i : lane, hi = i < lane ? lane : i;
                t0 = fma(sh.Pb[i * R + lane], G0p[gram_off(R, lo) + hi - lo], t0);
                if (i + 1 < R) {
                    const int lo1 = i + 1 < lane ? i + 1 : lane, hi1 = i + 1 < lane ? lane : i + 1;
                    t1 = fma(sh.Pb[(i + 1) * R + lane], G0p[gram_off(R, lo1) + hi1 - lo1], t1);
                }
            }
            trpg = t0 + t1;
        }
        trpg = warp_allsum(trpg);
        double eta;
        if (simp) eta = rhov ? rho * p.rho_mean[series] : rho;                 // tr(R)/d, synthetic_psmf.py:86-87
        // rPSMF.py:108: trace(M R M + CM Pbar CM') / d; uniform R: sum m c c' = (rho + a) G
        else eta = rhov ? (tot[sv_nrho(R)] + trpg) / dg : (rho * nobs + (rho + a) * trpg) / dg;
        const double N = a + eta;                                              // rPSMF.py:109
        const double phi = robust ? (lam + q1 / (a + eta) + (q0 != 0.0 ? q0 / eta : 0.0)) / (lam + dg) : 1.0;
        const double aphi = p.alpha * phi;
        for (int idx = lane; idx < R * R; idx += 32) {
            const int i = idx / R, j = idx % R;
            sh.V[idx] = aphi * (sh.V[idx] - sh.vx[i] * sh.vxt[j] / N);         // rPSMF.py:115
        }
        if (lane < R) sh.g[lane] = (((p.flags & F_CUPDATE_VT) != 0) ? sh.vx[lane] : sh.vxt[lane]) / N;   // rPSMF.py:111 / PSMF.py:80
        if (lane == 0) {
            sh.sc[1] = eta; sh.sc[2] = N; sh.sc[3] = phi; sh.sc[5] = aphi;
            sh.sc[7] = a;                                  // a of THIS step (sh.a is overwritten by the next predict)
        }
    };

    if (!simp) {
        for (int idx = tid; idx < R * R; idx += nthr) {
            const int i = idx / R, j = idx % R;
            double acc = (i == j) ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < R; ++k) {
                const int lo = k < j ? k : j, hi = k < j ? j : k;
                acc = fma(sh.Pb[i * R + k], tot[gram_off(R, lo) + hi - lo], acc);
            }
            sh.aug[0][i][j] = acc;
            sh.aug[0][i][R + j] = sh.Pb[i * R + j];
        }
        if (tid >= nthr - R) {                           // right-hand side Pbar b: the solve then yields K b
            const int i = tid - (nthr - R);
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < R; ++k) acc = fma(sh.Pb[i * R + k], tot[NGm + k], acc);
            sh.aug[0][i][2 * R] = acc;
        }
        sync_n<BAR>(nthr);
        // the elimination is latency-bound: a subset of the warps runs it (less redundant pivot-search work on
        // the fp64 pipe, cheaper barrier); the first warp past them computes the inverse-free half meanwhile
        if (warp < NGJ / 32) gauss_jordan_cta<R, NGJ, GJBAR, 2 * R + 1, LL>(sh, tid);   // aug[FIN][perm[k]][R..2R) = K[k][:], [..][2R] = (K b)[k]
        else if (side_warp && warp == NGJ / 32) {
            side_half();
            // F_GRAD_LINEAR needs N from side_half and the x that entered the step, nothing from the elimination: the side
            // warp accumulates it while the elimination runs
            if constexpr (GL) if (glin_on<GL, LL>(p) && p.grad_out != nullptr) lin_grad_step<R>(p, sh, tot);
        }
        sync_n<BAR>(nthr);
    }
    stamp(p, t, 7);
    if (warp == 0) {
        if (!side_warp) {
            side_half();
            __syncwarp();
            if constexpr (GL) if (glin_on<GL, LL>(p) && p.grad_out != nullptr) lin_grad_step<R>(p, sh, tot);
        }
        const double a = sh.a, rho = sh.rho, lam = sh.lam;
        const double s = tot[NGm + R], q1 = tot[NGm + R + 1], nobs = tot[NGm + R + 3];
        const double eta = sh.sc[1], N = sh.sc[2], phi = sh.sc[3];
        double xn = 0.0, bkb = 0.0;
        if (lane < R) {
            if (simp) {
                xn = sh.xb[lane];                                              // synthetic_psmf.py:93-94
            } else {
                const double kb = sh.aug[FIN][sh.perm[lane]][2 * R];
                xn = sh.xb[lane] + kb;                                         // rPSMF.py:104
                bkb = tot[NGm + lane] * kb;
            }
        }
        bkb = warp_allsum(bkb);
        const double sSe = simp ? s : s - bkb;                                 // diff' CPinv diff (synthetic_rpsmf.py:93-98: s)
        const double omega = robust ? (lam + sSe) / (lam + dg) : 1.0;          // rPSMF.py:105
        if (lane < R) {
            sh.x[lane] = xn;
            if (writer && p.X_out != nullptr) p.X_out[((int64_t)series * p.n_steps + t) * R + lane] = xn;
            if (p.grad_out != nullptr && (p.dynamics == DYN_COS || p.dynamics == DYN_EXTERNAL)) {
                // d ell_k / d theta = J_theta' d ell_k / d f; C'Me = b (rho + a)
                const double cte = rhov ? tot[sv_bu(R) + lane] : tot[NGm + lane] * (rho + a);
                const double gf = dll_df(p.flags, sh.vx[lane], sh.vxt[lane], cte, q1, nobs, lam, N);
                const double kabs = (double)(p.k0 + t);
                // cos dynamics: J_theta = diag(-2 pi k sin(.)); external dynamics: the caller owns f and applies its own
                // J_theta' to d ell / d f (one step per launch)
                sh.grad[lane] += p.dynamics == DYN_COS ? gf * (6.283185307179586 * kabs * sh.fd[lane]) : gf;
            }
        }
        if (lane == 0) {
            sh.sc[0] = omega; sh.sc[4] = sSe; sh.sc[6] = p.beta * omega;
            if (writer) {
                if (p.scal_out != nullptr) {
                    double* so = p.scal_out + ((int64_t)series * p.n_steps + t) * (LL ? NSCAL_LL : NSCAL);
                    so[0] = a; so[1] = eta; so[2] = N; so[3] = omega; so[4] = phi; so[5] = sSe; so[6] = lam; so[7] = rho;
                }
                if (!(isfinite(N) && isfinite(omega) && isfinite(phi) && isfinite(xn)) || N == 0.0)
                    atomicCAS((unsigned long long*)p.status, ~0ULL, (unsigned long long)t);
            }
        }
        if constexpr (LL) {
            if (p.scal_out != nullptr) {
                // S_obs = C_o Pbar C_o' + diag(rho_i + a): log det from the pivots and sum_obs log(rho_i + a), Delta^2 = s over
                // the observed rows - b'Kb (s also carries w0 q0 of the missing rows; simplified: S_obs^-1 = diag(w_i), b'Kb = 0)
                const double q0 = tot[NGm + R + 2];
                const double piv = (!simp && lane < R) ? sh.aug[0][lane][2 * R + 1] : 1.0;
                const double ldr = rhov ? tot[sv_nlog(R)] : nobs * log(rho + a);
                const double d2 = (rhov ? s - (q0 != 0.0 ? sh.w0 * q0 : 0.0) : sh.w1 * q1) - bkb;
                double nll, lp;
                step_loglik(p.flags, piv, nobs, N, q1, lam, ldr, d2, lane, nll, lp);
                if (lane == 0 && writer) {
                    double* so = p.scal_out + ((int64_t)series * p.n_steps + t) * NSCAL_LL;
                    so[8] = nll; so[9] = lp;
                }
            }
        }
    }
    sync_n<BAR>(nthr);
    {
        const double omega = sh.sc[0], bom = sh.sc[6];
        for (int idx = tid; idx < R * R; idx += nthr) {
            const int i = idx / R, j = idx % R;
            sh.P[idx] = simp ? sh.Pb[idx] : bom * sh.aug[FIN][sh.perm[i]][R + j];          // rPSMF.py:106
            if (!simp) sh.Q[idx] = omega * sh.Q[idx];                                        // rPSMF.py:133
        }
        if (tid == nthr - 32) {
            const double lam = sh.lam;
            sh.rho = omega * sh.rho;                                                         // rPSMF.py:134
            sh.lam = (robust && (p.flags & F_FIXED_LAMBDA) == 0) ? lam + (double)p.d_global : lam;   // rPSMF.py:135
        }
    }
    sync_n<BAR>(nthr);
    if (t + 1 < p.n_steps) predict_cta<R, BAR>(p, sh, tid, p.k0 + t + 1, series, nthr);
}

// ---- cross-GPU exchange of the (already grid-reduced) statistics over NVLink -------------------------------
// Rows of C are sharded over `world` GPUs; V, P, Q, x, lambda are replicated.  Per step every GPU needs
// the sum over all shards of the statistics vector (1.4 kB at r = 16).  One CTA of each GPU (part == 0) stores
// its local totals as tagged cells into slot [parity][rank] of every peer's mailbox with plain peer stores
// (NVLink P2P); every CTA polls the cells of its LOCAL mailbox and adds the world slots in rank order -- the
// same order on every GPU, so the replicated state stays bit-identical.  No fence and no flag: the latency
// is one NVLink store plus one local poll.  Two parities make the mailbox safe without a handshake: a GPU
// can only be one step ahead of its slowest peer (it needs that peer's cells of the current step to proceed).
// Sum of one statistics entry over all GPUs in RANK ORDER (bit-identical on every GPU): the peers' contributions are
// tagged cells of the local mailbox, polled CONCURRENTLY -- all outstanding loads are issued before any tag is looked at, so
// the wait costs one round trip however many peers there are (a per-peer poll loop costs one round trip per peer).
// local_cell != nullptr: this GPU's own contribution is a tagged cell as well (gpu scope, tag ltag), else it is `own`.
__device__ __forceinline__ double gather_ranks(const KParams& p, const uint4* __restrict__ slots /* [MAX_PEERS][MBOX_SLOT] */, int e,
                                               uint32_t xtag, const uint4* local_cell, uint32_t ltag, double own, long long step) {
    if (p.world == 1) return local_cell != nullptr ? cell_poll(p, local_cell, ltag, step) : own;
    // every index below is a compile-time constant after unrolling (the rank only enters through bit masks and selects):
    // the values stay in registers
    double v[MAX_PEERS];
#pragma unroll
    for (int s = 0; s < MAX_PEERS; ++s) v[s] = 0.0;
    unsigned pending = ((1u << p.world) - 1u) & ~(1u << p.rank);        // peers still missing
    bool lpend = local_cell != nullptr;                                 // own contribution still missing
    Spin sp;
    while (pending != 0u || lpend) {
        uint32_t lo[MAX_PEERS], hi[MAX_PEERS], t0[MAX_PEERS], t1[MAX_PEERS];
        uint32_t llo = 0u, lhi = 0u, lt0 = 0u, lt1 = 0u;
        if (lpend)
            asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(llo), "=r"(lt0), "=r"(lhi), "=r"(lt1) : "l"(local_cell) : "memory");
#pragma unroll
        for (int s = 0; s < MAX_PEERS; ++s) {
            lo[s] = 0u; hi[s] = 0u; t0[s] = 0u; t1[s] = 0u;
            if ((pending >> s) & 1u)
                asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(lo[s]), "=r"(t0[s]), "=r"(hi[s]), "=r"(t1[s]) : "l"(slots + (size_t)s * MBOX_SLOT + e) : "memory");
        }
        if (lpend && lt0 == ltag && lt1 == ltag) {
            own = __hiloint2double((int)lhi, (int)llo);
            lpend = false;
        }
#pragma unroll
        for (int s = 0; s < MAX_PEERS; ++s) {
            if (((pending >> s) & 1u) && t0[s] == xtag && t1[s] == xtag) {
                v[s] = __hiloint2double((int)hi[s], (int)lo[s]);
                pending &= ~(1u << s);
            }
        }
        if (pending != 0u || lpend) {
            if (sp.expired(p, SPIN_PEER, step)) break;
            if (POLL_BACKOFF_NS > 0) __nanosleep(POLL_BACKOFF_NS);   // leave the issue slots to the warps that do arithmetic on this SM
        }
    }
    double sum = 0.0;
#pragma unroll
    for (int s = 0; s < MAX_PEERS; ++s)
        if (s < p.world) sum += (s == p.rank) ? own : v[s];             // rank order: the same on every GPU
    return sum;
}

// Mailbox depth.  A slot is reused MBOX_DEPTH steps later; with two filter steps in flight (pipelined kernel) a GPU can
// publish step t+2 before a slow peer has read step t, but never step t+4: that needs its own solve of t+2, hence the
// peer's statistics of t+2, hence the peer's solve of t -- which has read the cells of step t.
constexpr int MBOX_DEPTH = 4;

// header cell of a mailbox slot: {kernel id, statistics count}; exchanged once per launch (step 0) by one thread
__device__ __forceinline__ void mailbox_check_peers(const KParams& p, int kernel_id, int nst, int64_t t) {
    const unsigned long long step = p.step_base + (unsigned long long)t;
    const int slot = (int)(step % MBOX_DEPTH);
    const uint32_t tag = tag_of(step + 1ULL);
    const double header = (double)(kernel_id * 4096 + nst);
    for (int pr = 0; pr < p.world; ++pr)
        if (pr != p.rank)
            cell_store_sys(reinterpret_cast<uint4*>(p.mbox_peer[pr]) + ((size_t)slot * MAX_PEERS + p.rank) * MBOX_SLOT + MBOX_SLOT - 1, header, tag);
    const uint4* local = reinterpret_cast<const uint4*>(p.mbox_local) + (size_t)slot * MAX_PEERS * MBOX_SLOT;
    for (int src = 0; src < p.world; ++src)
        if (src != p.rank && cell_poll_sys(p, local + (size_t)src * MBOX_SLOT + MBOX_SLOT - 1, tag, t) != header) {
            // all ranks must run the same kernel with the same statistics vector (the host agrees on it in
            // psmf_mailbox_connect); a mismatch would add unrelated numbers: flag it instead
            if (*reinterpret_cast<volatile unsigned long long*>(p.bar + ABORT_WORD) == 0ULL)
                atomicCAS((unsigned long long*)p.status, ~0ULL, (unsigned long long)STATUS_MISMATCH | (unsigned long long)t);
        }
}

template <int NST, int NSP, int BAR = 0>
__device__ __forceinline__ void gpu_exchange(const KParams& p, double* __restrict__ tot, double* __restrict__ /*tmp*/, int tid,
                                             int64_t t, int part, int nthr, int kernel_id) {
    const unsigned long long step = p.step_base + (unsigned long long)t;
    const int slot = (int)(step % MBOX_DEPTH);
    const uint32_t tag = tag_of(step + 1ULL);
    if (part == 0) {
        for (int e = tid; e < NST; e += nthr) {
            const double v = tot[e];
            for (int pr = 0; pr < p.world; ++pr)
                if (pr != p.rank)
                    cell_store_sys(reinterpret_cast<uint4*>(p.mbox_peer[pr]) + ((size_t)slot * MAX_PEERS + p.rank) * MBOX_SLOT + e, v, tag);
        }
        if (t == 0 && tid == nthr - 1) mailbox_check_peers(p, kernel_id, NST, t);
    }
    const uint4* local = reinterpret_cast<const uint4*>(p.mbox_local) + (size_t)slot * MAX_PEERS * MBOX_SLOT;
    for (int e = tid; e < NST; e += nthr)
        tot[e] = gather_ranks(p, local, e, tag, nullptr, 0u, tot[e], t);      // entry e is read and written by this thread only
    sync_n<BAR>(nthr);
}

// ---- cross-CTA reduction of the statistics, deterministic (fixed summation order) ---------------------
//   cps <= 16 : every CTA reads all partials after one grid barrier
//   cps  > 16 : reduce-scatter / all-gather through L2: CTA c sums entries {c, c + cps, ..} over all CTAs
//               (coalesced reads of a transposed partial array), a second barrier publishes the totals.
// sh.part -> sh.tot; ends with a barrier over the `nthr` threads.
template <int NST, int NSP, int BAR = 0>
__device__ __forceinline__ void grid_reduce(const KParams& p, double* __restrict__ part_v, double* __restrict__ tot, int tid,
                                            int lane, int warp, int64_t t, int series, int part, int nthr) {
    if (p.cps == 1) {
        for (int e = tid; e < NST; e += nthr) tot[e] = part_v[e];
        sync_n<BAR>(nthr);
        if (p.world > 1) gpu_exchange<NST, NSP, BAR>(p, tot, part_v, tid, t, part, nthr, 1);
        return;
    }
    const int parity = (int)(t & 1);
    const int cps = p.cps;
    if (cps <= 16) {
        double* mine = p.partials + ((size_t)parity * cps + part) * NSP;
        for (int e = tid; e < NST; e += nthr) mine[e] = part_v[e];
        stamp(p, t, 3);
        grid_barrier<BAR>(p, (unsigned long long)gridDim.x * (unsigned long long)(t + 1), nthr, tid, t);
        stamp(p, t, 4);
        const double* basep = p.partials + (size_t)parity * cps * NSP;
        for (int e = tid; e < NST; e += nthr) {
            double v[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) v[c] = c < cps ? __ldcg(basep + (size_t)c * NSP + e) : 0.0;
            tot[e] = (((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]))) +
                     (((v[8] + v[9]) + (v[10] + v[11])) + ((v[12] + v[13]) + (v[14] + v[15])));
        }
    } else {
        const int pstr = (cps + 7) & ~7;
        double* pT = p.partials + (size_t)parity * NSP * (pstr + 1);
        double* totals = pT + (size_t)NSP * pstr;
        for (int e = tid; e < NST; e += nthr) pT[(size_t)e * pstr + part] = part_v[e];
        stamp(p, t, 3);
        grid_barrier<BAR>(p, (unsigned long long)gridDim.x * (unsigned long long)(2 * t + 1), nthr, tid, t);
        const int nw = nthr >> 5;
        for (int e = part + warp * cps; e < NST; e += nw * cps) {
            const double* src = pT + (size_t)e * pstr;
            double s = 0.0;
            for (int c0 = 0; c0 < cps; c0 += 256) {
                double v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = c0 + lane + 32 * j;
                    v[j] = c < cps ? __ldcg(src + c) : 0.0;
                }
                s += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
            }
            s = warp_allsum(s);
            if (lane == 0) totals[e] = s;
        }
        grid_barrier<BAR>(p, (unsigned long long)gridDim.x * (unsigned long long)(2 * t + 2), nthr, tid, t);
        stamp(p, t, 4);
        for (int e = tid; e < NST; e += nthr) tot[e] = __ldcg(totals + e);
    }
    sync_n<BAR>(nthr);
    if (p.world > 1) gpu_exchange<NST, NSP, BAR>(p, tot, part_v, tid, t, part, nthr, 1);
}

// ---- observation of one row: value and mask, whatever the encoding --------------------------------------
// bytes: y zero-filled where missing + one mask byte (rPSMF.py:198-202); F_NAN_MASK: missing entries are NaN in y (the
// raw data form, rPSMF.py:160-164) and there is no mask stream: m = !isnan(y), y := 0 where missing.
template <typename T>
__device__ __forceinline__ void observe(const KParams& p, const T* __restrict__ Yt, const uint8_t* __restrict__ Mt, int64_t row, bool inb,
                                        double& yi, bool& mi) {
    yi = inb ? (double)Yt[row] : 0.0;
    mi = inb;
    if (Mt != nullptr) {
        if (inb) mi = Mt[row] != 0;
    } else if ((p.flags & F_NAN_MASK) != 0) {
        mi = inb && !isnan(yi);
        yi = mi ? yi : 0.0;
    }
}

// ---- direct-load persistent kernel: C tiles are read from / written to global memory by the warp that
// owns them; general fallback (any alignment, any d) and the path for small problems / batched series ----
// p.phase (caller-driven statistics exchange, one step per launch): 1 = pass + grid reduction, statistics -> p.stats_ext
// and residuals -> p.e_ext; 2 = r x r update from p.stats_ext (all-reduced by the caller) + the rank-1 update of C.
template <int R, typename T, bool RHOV = false, bool GL = false, bool LL = false>
__global__ void __launch_bounds__(V1_WARPS * 32, 2) psmf_filter_kernel(const KParams p) {
    // RHOV with LL: one more statistic, sum m log(rho_i + a), inside the padding
    constexpr int NW = V1_WARPS, NSP = RHOV ? nstat_v_pad(R) : nstat_pad(R), NST = RHOV ? nstat_v(R) + (LL ? 1 : 0) : nstat(R);
    static_assert(NST <= NSP, "statistics vector longer than its padded size");
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    __shared__ Smem<R> sh;
    __shared__ double red[V1_WARPS * NSP];                                     // per-warp partial statistics
    __shared__ double totv[RHOV ? NSP : 1], partv[RHOV ? NSP : 1];             // non-uniform R: the longer statistics vector
    double* const part_p = RHOV ? partv : sh.part;
    double* const tot_p = RHOV ? totv : sh.tot;
    double* stage_all = reinterpret_cast<double*>(dyn_smem);                   // NW staging tiles [R][32] fp64
    double* ebuf = stage_all + NW * R * TILE;

    const int tid = threadIdx.x, lane = tid & 31, warp = uniform_warp_id();
    const int series = blockIdx.x / p.cps;
    const int part = blockIdx.x % p.cps;
    const int ntiles = (int)((p.d + TILE - 1) / TILE);
    const int tb = (int)((int64_t)ntiles * part / p.cps);
    const int te = (int)((int64_t)ntiles * (part + 1) / p.cps);
    const bool writer = part == 0;
    double* stage = stage_all + warp * R * TILE;
    const int nrows = (te - tb) * TILE;
    const bool evalon = p.E != nullptr;
    EvalBuf eb;                                                                // behind the residual buffer (host sizes it)
    eb.yh = ebuf + ((int64_t)ntiles + p.cps - 1) / p.cps * TILE + TILE;
    eb.yo = eb.yh + nrows;
    eb.fl = reinterpret_cast<unsigned char*>(eb.yo + nrows);
    EvalAcc ev;
    const bool robust = (p.flags & F_ROBUST) != 0;

    T* Cs = reinterpret_cast<T*>(p.C) + (int64_t)series * p.c_series_stride;
    double* stg = p.state + (int64_t)series * st_size(R);

    for (int i = tid; i < R * R; i += blockDim.x) {
        sh.P[i] = stg[st_P(R) + i];
        sh.V[i] = stg[st_V(R) + i];
        sh.Q[i] = stg[st_Q(R) + i];
        if constexpr (GL) if (glin_on<GL, LL>(p)) glin_acc(p)[i] = 0.0;
    }
    if (tid < R) {
        sh.x[tid] = stg[st_x(R) + tid];
        sh.th[tid] = stg[st_theta(R) + tid];
        sh.g[tid] = 0.0;
        sh.grad[tid] = 0.0;
    }
    if (tid == 0) {
        sh.rho = stg[st_rho(R)];
        sh.lam = stg[st_lam(R)];
    }
    for (int i = tid; i < nrows; i += blockDim.x) ebuf[i] = p.phase == 2 ? p.e_ext[(int64_t)tb * TILE + i] : 0.0;
    if (evalon)
        for (int i = tid; i < nrows; i += blockDim.x) eb.fl[i] = 0;
    __syncthreads();
    predict_cta<R>(p, sh, tid, p.k0, series, blockDim.x);

    for (int64_t t = 0; t < p.n_steps; ++t) {
        const T* __restrict__ Yt = reinterpret_cast<const T*>(p.Y) + (int64_t)series * p.ysst + t * p.ldy;
        const uint8_t* __restrict__ Mt = p.M ? p.M + (int64_t)series * p.msst + t * p.ldm : nullptr;
        T* Yrec_t = p.Yrec ? reinterpret_cast<T*>(p.Yrec) + (int64_t)series * p.recsst + t * p.ldrec : nullptr;
        const T* __restrict__ Yo_t = evalon ? reinterpret_cast<const T*>(p.Yorig) + (int64_t)series * p.ysst + t * p.ldy : nullptr;
        const uint8_t* __restrict__ Et = evalon ? p.E + (int64_t)series * p.esst + t * p.lde : nullptr;
        stamp(p, t, 0);
        const double w1 = sh.w1, w0 = sh.w0;
        if (p.phase != 2) {
            typename std::conditional<RHOV, TileAccV<R>, TileAcc<R>>::type acc;
            if constexpr (RHOV) acc.zero_v(); else acc.zero();
            const double* __restrict__ rho0 = RHOV ? p.rho_vec + (int64_t)series * p.rho_sst : nullptr;
            const double rscale = sh.rho, aa = sh.a;
            double nlog = 0.0;                                                     // RHOV && LL: sum m log(rho_i + a)
            for (int tile = tb + warp; tile < te; tile += NW) {
                const int64_t row = (int64_t)tile * TILE + lane;
                const int rl = (tile - tb) * TILE + lane;
                T* gt = Cs + (int64_t)tile * (R * TILE);
                double c[R];
#pragma unroll
                for (int j = 0; j < R; ++j) c[j] = (double)gt[tile_pos(j, lane)];
                const double ep = ebuf[rl];
                const bool inb = row < p.d;
                bool mi;
                double yi;
                observe<T>(p, Yt, Mt, row, inb, yi, mi);
                if (evalon && t > 0) eval_cover(ev, eb, rl, sh.sc[7], sh.sc[1], sh.sc[2], robust, p.sig);   // step t-1, now that eta exists
                double e, yh;
                double wi = w1;
                if constexpr (RHOV) {
                    const double rho_i = inb ? __dmul_rn(rscale, rho0[row]) : 1.0;       // R = omega-scale * diag(R0)  (rPSMF.py:134)
                    wi = 1.0 / (rho_i + aa);                                               // rPSMF.py:92,98,32
                    acc.nrho += mi ? rho_i : 0.0;
                    if constexpr (LL) if (p.scal_out != nullptr) nlog += mi ? log(rho_i + aa) : 0.0;
                }
                row_stats<R>(acc, sh, c, ep, inb, mi, yi, wi, w0, e, yh);
#pragma unroll
                for (int j = 0; j < R; ++j) {
                    gt[tile_pos(j, lane)] = (T)c[j];
                    stage[tile_pos(j, lane)] = c[j];
                }
                ebuf[rl] = e;
                if (Yrec_t != nullptr && inb) Yrec_t[row] = (T)yh;
                if (evalon) eval_row(ev, eb, rl, inb && Et[row] != 0, mi, yh, inb ? (double)Yo_t[row] : 0.0);
                const unsigned mbits = __ballot_sync(FULL, mi);
                __syncwarp();
                if constexpr (RHOV) tile_gram_v<R, double>(acc, stage, mbits, mi ? wi : 0.0, mi ? e : 0.0, lane);
                else tile_gram<R, double>(acc, stage, mbits, lane);
                __syncwarp();
            }
            if constexpr (RHOV) acc_writeout_v<R>(acc, red + warp * NSP, lane);
            else acc_writeout<R>(acc, red + warp * NSP, w1, lane);
            if constexpr (RHOV && LL) {
                const double nl = warp_allsum(nlog);
                if (lane == 0) red[warp * NSP + sv_nlog(R)] = nl;
            }
            stamp(p, t, 1);
            __syncthreads();
            stamp(p, t, 2);
            for (int e2 = tid; e2 < NST; e2 += blockDim.x) {   // CTA partial: fixed order over the warps
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < NW; ++w) s += red[w * NSP + e2];
                part_p[e2] = s;
            }
            grid_reduce<NST, NSP>(p, part_p, tot_p, tid, lane, warp, t, series, part, blockDim.x);
            stamp(p, t, 5);
        }
        if (p.phase == 1) {
            // statistics of this GPU's rows -> the caller's collective; residuals survive the launch in global memory
            if (writer)
                for (int e = tid; e < NST; e += blockDim.x) p.stats_ext[e] = tot_p[e];
            for (int i = tid; i < nrows; i += blockDim.x) p.e_ext[(int64_t)tb * TILE + i] = ebuf[i];
            return;
        }
        if (p.phase == 2) {
            for (int e = tid; e < NST; e += blockDim.x) tot_p[e] = p.stats_ext[e];
            __syncthreads();
        }
        small_update<R, GJ_THREADS, GL, LL>(p, sh, tid, lane, warp, series, t, writer, blockDim.x, RHOV ? totv : nullptr);
        stamp(p, t, 6);
    }

    // apply the pending rank-1 update of the last step so that C in HBM is the filtered C_T
    for (int tile = tb + warp; tile < te; tile += NW) {
        const int rl = (tile - tb) * TILE + lane;
        T* gt = Cs + (int64_t)tile * (R * TILE);
        const double ep = ebuf[rl];
#pragma unroll
        for (int j = 0; j < R; ++j) gt[tile_pos(j, lane)] = (T)fma(ep, sh.g[j], (double)gt[tile_pos(j, lane)]);
        if (evalon) eval_cover(ev, eb, rl, sh.sc[7], sh.sc[1], sh.sc[2], robust, p.sig);   // the last step of the launch
    }
    if (evalon) {
        __syncthreads();
        eval_writeout<NW>(p, ev, red, series, part, tid);
    }
    if (writer) {
        for (int i = tid; i < R * R; i += blockDim.x) {
            stg[st_P(R) + i] = sh.P[i];
            stg[st_V(R) + i] = sh.V[i];
            stg[st_Q(R) + i] = sh.Q[i];
        }
        if (tid < R) {
            stg[st_x(R) + tid] = sh.x[tid];
            if (p.grad_out != nullptr && !glin_on<GL, LL>(p)) p.grad_out[(int64_t)series * R + tid] = sh.grad[tid];
        }
        if (tid == 0) {
            stg[st_rho(R)] = sh.rho;
            stg[st_lam(R)] = sh.lam;
        }
    }
    if constexpr (GL)
        if (writer && glin_on<GL, LL>(p) && p.grad_out != nullptr) lin_grad_writeout<R>(p.grad_out + (int64_t)series * (R * R + R), glin_acc(p), sh.grad, tid, blockDim.x);
}

}  // namespace psmf
