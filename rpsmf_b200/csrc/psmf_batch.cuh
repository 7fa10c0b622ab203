// Resident batch kernel (sm_100a): independent series, one CTA per series, C in shared memory for the whole launch.
//
// BASELINE.json configs[4] (4096 series of d = 512, r = 8, T = 5k split over the GPUs with no communication; the
// reference analogue is the 100-repeat loop of the imputation experiment, ExperimentImpute/rPSMF.py:194-232) and
// every single series whose dictionary fits one CTA's shared memory (the imputation datasets, d = 27 ... 505).
//
//   prologue   ONE bulk asynchronous copy (cp.async.bulk, SASS UBLKCP) brings the tiled C of the series (32 kB at
//              d = 512, r = 8, fp64) from HBM into shared memory, completing on an mbarrier; it stays there for all
//              n_steps filter steps and goes back with one bulk store at the end: C costs no HBM or L2 traffic per step.
//   step       pass over the resident tiles (one warp per 32-row tile, lane = row: pending rank-1 update, y_hat, e,
//              statistics; Gram by fp64 DMMA straight from the resident tile -- no staging copy) -> warp sums ->
//              __syncthreads -> CTA sum in fixed order -> r x r solve and update (small_update, shared with the other
//              kernels) -> next step.  No grid barrier, no global scratch, no atomics: series never talk to each other.
//              y_t / m_t of step t+1 are loaded into registers during step t (V3_PF tiles per warp), so the HBM
//              latency of the only per-step global reads is off the chain.
//   occupancy  NW = 4 warps and <= 102 registers at r <= 8: five series per SM share the fp64 pipe and hide each
//              other's latency chain (pass -> barrier -> Gauss-Jordan -> update); the grid is simply n_series CTAs.
//
// The statistics, the r x r algebra, the evaluation metrics and the masks are the same code as in psmf_filter.cuh, so
// a series filtered here is bit-identical to the same series filtered alone by the direct-load kernel with one CTA
// and the same number of warps... up to the warp count, which fixes the summation tree (NW is part of the result).
#pragma once
#include "psmf_stream.cuh"      // mbarrier / bulk-copy PTX wrappers

namespace psmf {

template <typename T>
struct YMreg {
    T y;
    unsigned char m;
};

template <int R, typename T, int NW, bool GL = false, bool LL = false>
__global__ void __launch_bounds__(NW * 32, batch_min_ctas(R, NW)) psmf_batch_kernel(const KParams p) {
    constexpr int NSP = nstat_pad(R), NST = nstat(R), NTHR = NW * 32;
    // elimination threads: all but one warp, which computes the inverse-free half of the r x r update meanwhile
    constexpr int NGJ = (NTHR - 32) < GJ_THREADS ? (NTHR - 32) : GJ_THREADS;
    extern __shared__ __align__(128) unsigned char dyn_smem_b[];
    __shared__ Smem<R> sh;
    __shared__ double red[NW * nstat_pad(R)];
    __shared__ __align__(8) uint64_t cbar;

    const int tid = threadIdx.x, lane = tid & 31, warp = uniform_warp_id();
    const int series = blockIdx.x;
    const int ntiles = (int)((p.d + TILE - 1) / TILE);
    const int nrows = ntiles * TILE;
    const size_t cbytes = (size_t)ntiles * R * TILE * sizeof(T);
    T* Ct = reinterpret_cast<T*>(dyn_smem_b);
    double* ebuf = reinterpret_cast<double*>(dyn_smem_b + batch_c_bytes(ntiles, R, sizeof(T)));
    const bool evalon = p.E != nullptr;
    EvalBuf eb;
    eb.yh = ebuf + nrows;
    eb.yo = eb.yh + nrows;
    eb.fl = reinterpret_cast<unsigned char*>(eb.yo + nrows);
    EvalAcc ev;
    const bool robust = (p.flags & F_ROBUST) != 0;

    T* Cs = reinterpret_cast<T*>(p.C) + (int64_t)series * p.c_series_stride;
    double* stg = p.state + (int64_t)series * st_size(R);

    // ---- prologue: C -> shared memory with one bulk copy; small state -> shared memory ----
    if (tid == 0) {
        mbar_init(&cbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(&cbar, (uint32_t)cbytes);
        bulk_load(Ct, Cs, (uint32_t)cbytes, &cbar);
    }
    for (int i = tid; i < R * R; i += NTHR) {
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
    for (int i = tid; i < nrows; i += NTHR) ebuf[i] = 0.0;
    if (evalon)
        for (int i = tid; i < nrows; i += NTHR) eb.fl[i] = 0;
    __syncthreads();
    predict_cta<R>(p, sh, tid, p.k0, series, NTHR);

    const T* __restrict__ Ys = reinterpret_cast<const T*>(p.Y) + (int64_t)series * p.ysst;
    const uint8_t* __restrict__ Ms = p.M ? p.M + (int64_t)series * p.msst : nullptr;
    const bool nanm = (p.flags & F_NAN_MASK) != 0;

    // y / m of this warp's first V3_PF tiles for step 0 (raw: converting at load time would stall on the load)
    YMreg<T> pf[V3_PF];
#pragma unroll
    for (int q = 0; q < V3_PF; ++q) {
        const int64_t row = (int64_t)(warp + q * NW) * TILE + lane;
        pf[q].y = (T)0; pf[q].m = 1;
        if (row < p.d) {
            pf[q].y = __ldg(Ys + row);
            if (Ms != nullptr) pf[q].m = __ldg(Ms + row);
        }
    }
    mbar_wait(p, &cbar, 0u, 0);                                                // C has landed

    for (int64_t t = 0; t < p.n_steps; ++t) {
        const T* __restrict__ Yt = Ys + t * p.ldy;
        const uint8_t* __restrict__ Mt = Ms ? Ms + t * p.ldm : nullptr;
        T* Yrec_t = p.Yrec ? reinterpret_cast<T*>(p.Yrec) + (int64_t)series * p.recsst + t * p.ldrec : nullptr;
        const T* __restrict__ Yo_t = evalon ? reinterpret_cast<const T*>(p.Yorig) + (int64_t)series * p.ysst + t * p.ldy : nullptr;
        const uint8_t* __restrict__ Et = evalon ? p.E + (int64_t)series * p.esst + t * p.lde : nullptr;
        const double w1 = sh.w1, w0 = sh.w0;
        stamp(p, t, 0);
        TileAcc<R> acc;
        acc.zero();
        // the current values leave the prefetch registers, the loads of step t+1 take their place
        YMreg<T> cur[V3_PF];
#pragma unroll
        for (int q = 0; q < V3_PF; ++q) cur[q] = pf[q];
        if (t + 1 < p.n_steps) {
#pragma unroll
            for (int q = 0; q < V3_PF; ++q) {
                const int64_t row = (int64_t)(warp + q * NW) * TILE + lane;
                if (row < p.d) {
                    pf[q].y = __ldg(Yt + p.ldy + row);
                    if (Mt != nullptr) pf[q].m = __ldg(Mt + p.ldm + row);
                }
            }
        }
        // ---- the pass: one warp per resident tile, lane = row.  r <= 8: TWO tiles per iteration, written load / compute /
        // store stage by stage so that the two independent instruction streams interleave (the tile is latency-bound: at
        // 14 warps per SM a single stream leaves the shared-memory and fp64 pipes two thirds idle); their Gram DMMAs go to
        // two accumulators.  Tiles of a warp: warp, warp + NW, ...
        auto load_tile = [&](int q, double (&c)[R], double& ep, double& yi, bool& mi, bool& inb, int& rl, int64_t& row) -> T* {
            const int tile = warp + q * NW;
            row = (int64_t)tile * TILE + lane;
            rl = tile * TILE + lane;
            inb = row < p.d;
            T* tl = Ct + (size_t)tile * (R * TILE);
#pragma unroll
            for (int j = 0; j < R; ++j) c[j] = (double)tl[tile_pos(j, lane)];
            ep = ebuf[rl];
            if (q < V3_PF) {
                // select the prefetched pair without dynamic register indexing
                T yr = cur[0].y;
                unsigned char mr = cur[0].m;
#pragma unroll
                for (int k = 1; k < V3_PF; ++k)
                    if (q == k) { yr = cur[k].y; mr = cur[k].m; }
                yi = inb ? (double)yr : 0.0;
                mi = inb;
                if (Mt != nullptr) mi = inb && mr != 0;
                else if (nanm) { mi = inb && !isnan(yi); yi = mi ? yi : 0.0; }
            } else {
                observe<T>(p, Yt, Mt, row, inb, yi, mi);
            }
            return tl;
        };
        auto store_tile = [&](T* tl, const double (&c)[R], double e, double yh, bool mi, bool inb, int rl, int64_t row) {
#pragma unroll
            for (int j = 0; j < R; ++j) tl[tile_pos(j, lane)] = (T)c[j];
            ebuf[rl] = e;
            if (Yrec_t != nullptr && inb) Yrec_t[row] = (T)yh;
            if (evalon) eval_row(ev, eb, rl, inb && Et[row] != 0, mi, yh, inb ? (double)Yo_t[row] : 0.0);
        };
        constexpr bool PAIR = R <= 8;
#pragma unroll 1
        for (int q = 0; warp + q * NW < ntiles; q += PAIR ? 2 : 1) {
            bool paired = false;
            if constexpr (PAIR) paired = warp + (q + 1) * NW < ntiles;
            if constexpr (PAIR) if (paired) {
                double cA[R], cB[R], epA, epB, yiA, yiB, eA, eB, yhA, yhB;
                bool miA, miB, inbA, inbB;
                int rlA, rlB;
                int64_t rowA, rowB;
                T* tlA = load_tile(q, cA, epA, yiA, miA, inbA, rlA, rowA);
                T* tlB = load_tile(q + 1, cB, epB, yiB, miB, inbB, rlB, rowB);
                if (evalon && t > 0) {
                    eval_cover(ev, eb, rlA, sh.sc[7], sh.sc[1], sh.sc[2], robust, p.sig);
                    eval_cover(ev, eb, rlB, sh.sc[7], sh.sc[1], sh.sc[2], robust, p.sig);
                }
                row_stats<R>(acc, sh, cA, epA, inbA, miA, yiA, w1, w0, eA, yhA);
                row_stats<R>(acc, sh, cB, epB, inbB, miB, yiB, w1, w0, eB, yhB);
                store_tile(tlA, cA, eA, yhA, miA, inbA, rlA, rowA);
                store_tile(tlB, cB, eB, yhB, miB, inbB, rlB, rowB);
                const unsigned mbA = __ballot_sync(FULL, miA), mbB = __ballot_sync(FULL, miB);
                __syncwarp();
                tile_gram2<R, T>(acc, tlA, mbA, tlB, mbB, lane);     // straight from the resident tiles
                __syncwarp();
            }
            if (!paired) {
                double c[R], ep, yi, e, yh;
                bool mi, inb;
                int rl;
                int64_t row;
                T* tl = load_tile(q, c, ep, yi, mi, inb, rl, row);
                if (evalon && t > 0) eval_cover(ev, eb, rl, sh.sc[7], sh.sc[1], sh.sc[2], robust, p.sig);
                row_stats<R>(acc, sh, c, ep, inb, mi, yi, w1, w0, e, yh);
                store_tile(tl, c, e, yh, mi, inb, rl, row);
                const unsigned mbits = __ballot_sync(FULL, mi);
                __syncwarp();
                tile_gram<R, T>(acc, tl, mbits, lane);               // straight from the resident tile
                __syncwarp();
            }
        }
        stamp(p, t, 1);
        acc_writeout<R>(acc, red + warp * NSP, w1, lane);
        __syncthreads();
        stamp(p, t, 2);
        if (tid < NST) {                                         // CTA total: fixed order over the warps
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < NW; ++w) s += red[w * NSP + tid];
            sh.tot[tid] = s;
        }
        if (NST > NTHR) {
            for (int e2 = NTHR + tid; e2 < NST; e2 += NTHR) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < NW; ++w) s += red[w * NSP + e2];
                sh.tot[e2] = s;
            }
        }
        __syncthreads();
        stamp(p, t, 5);
        small_update<R, NGJ, GL, LL>(p, sh, tid, lane, warp, series, t, true, NTHR);
        stamp(p, t, 6);
    }

    // pending rank-1 update of the last step, then C goes back to HBM with one bulk store
#pragma unroll 1
    for (int tile = warp; tile < ntiles; tile += NW) {
        const int rl = tile * TILE + lane;
        T* tl = Ct + (size_t)tile * (R * TILE);
        const double ep = ebuf[rl];
#pragma unroll
        for (int j = 0; j < R; ++j) tl[tile_pos(j, lane)] = (T)fma(ep, sh.g[j], (double)tl[tile_pos(j, lane)]);
        if (evalon) eval_cover(ev, eb, rl, sh.sc[7], sh.sc[1], sh.sc[2], robust, p.sig);
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
        bulk_store(Cs, Ct, (uint32_t)cbytes);
        bulk_commit();
    }
    if (evalon) eval_writeout<NW>(p, ev, red, series, 0, tid);
    for (int i = tid; i < R * R; i += NTHR) {
        stg[st_P(R) + i] = sh.P[i];
        stg[st_V(R) + i] = sh.V[i];
        stg[st_Q(R) + i] = sh.Q[i];
    }
    if (tid < R) {
        stg[st_x(R) + tid] = sh.x[tid];
        if (p.grad_out != nullptr && !glin_on<GL, LL>(p)) p.grad_out[(int64_t)series * R + tid] = sh.grad[tid];
    }
    if constexpr (GL)
        if (glin_on<GL, LL>(p) && p.grad_out != nullptr) lin_grad_writeout<R>(p.grad_out + (int64_t)series * (R * R + R), glin_acc(p), sh.grad, tid, NTHR);
    if (tid == 0) {
        stg[st_rho(R)] = sh.rho;
        stg[st_lam(R)] = sh.lam;
        bulk_wait<0>();                                          // the store has completed before the CTA retires
    }
}

}  // namespace psmf
