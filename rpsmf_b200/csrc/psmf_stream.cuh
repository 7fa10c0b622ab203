// TMA-staged, software-pipelined PSMF / rPSMF filter kernel (sm_100a): the large-d path.
//
// One cooperative launch of (data CTAs + 1 control CTA), one CTA per SM:
//
//   data CTA     producer warp (one thread): moves contiguous CHUNKS of the tiled C between HBM and a ring of
//                shared-memory slots with bulk asynchronous copies (cp.async.bulk, the 1-D TMA path: UBLKCP in
//                SASS) that complete on mbarriers, and bulk-stores updated chunks back.
//                   streaming (chunks of the CTA > slots): ring, every chunk loaded and stored once per step;
//                   resident  (chunks <= slots): C is loaded once and stays in shared memory for the launch.
//                14 pass warps (12 used when streaming): one warp per 32-row tile, all warps independent (lane =
//                row for the rank-1 update / y_hat / e, fp64 DMMA fragments for the Gram-type sums); at the end
//                of a pass a warp leaves its sums in shared memory, arrives on an mbarrier and moves on.
//                reduce warp: adds the per-warp sums in fixed order, writes the CTA partial to global memory
//                and bumps a global arrival counter; once all CTAs have arrived it sums ITS share of the
//                entries over all CTAs (fixed order: deterministic) and publishes the totals as tagged cells.
//                (One SM ingests only ~40 GB/s: a single CTA summing the ~200 kB of partials costs >= 5 us.)
//   control CTA  warps 8-15 poll the totals, exchange them with the other GPUs over NVLink and hand them to
//                warps 0-7, which run the r x r solve and publish {g_t, xbar_{t+1}} as tagged cells as soon as
//                x_t exists; the rest of the update follows off the critical path.  It is the only CTA that
//                holds V, P, Q, x, lambda.  A dedicated SM keeps the latency-bound solve away from the DMMA
//                traffic of the pass warps (measured: 3 us alone vs 8-23 us when it shared an SM with them)
//                and there is no grid barrier anywhere.
//
// Software pipeline.  The statistics of step t are sums over C_t = C_{t-1} + e_{t-1} g_{t-1}', and g_{t-1}
// only exists after the solve of step t-1.  Expanding the rank-1 term,
//
//     A_t  = sum m_t c c' = A0 + u g' + g u' + kappa g g'        A0 = sum m_t c c',  u = sum m_t e c
//     h_t  = sum m_t y_t c = h0 + psi g                          h0 = sum m_t y_t c, psi = sum m_t y_t e
//     bu_t = sum m_t e_t c = h_t - A_t xbar_t                     (e_t = y_t - m_t c.xbar_t)
//     q1_t = sum m_t e_t^2 = gamma - 2 xbar_t' h_t + xbar_t' A_t xbar_t,   gamma = sum m_t y_t^2
//
// with c = rows of C_{t-1}, e = e_{t-1}, g = g_{t-1}: every sum on the right is independent of the solve of
// step t-1.  So pass P_t (which turns C_{t-2} in HBM into C_{t-1}, computes e_{t-1} and the sums for step t)
// only needs the solve of step t-2 and runs CONCURRENTLY with the reduction / solve of step t-1; the solve of
// step t assembles A_t, bu_t, q1_t from the reduced sums in O(r^2) and proceeds as in psmf_filter.cuh.  The
// step time becomes max(pass, (pass + reduce + solve) / 2) instead of pass + reduce + solve (two steps in flight).  One extra
// read of y_t / m_t per step (+3 % HBM bytes) pays for it; C is still read and written once per step.
//
// Parameter sets: set s = {g_{s-1}, xbar_s} (set 0 = {0, xbar_0} from the state entering the launch); pass p
// needs set p-1, the flush pass n needs sets n-1 and n.  The control CTA publishes set t+1 after the solve
// of step t as tagged cells (tag t+2) at gparams[(t+1) & 1].
//
// Requirements checked by the host (else the direct-load kernel of psmf_filter.cuh is used): one series,
// d a multiple of 16, at least two SMs.
#pragma once
#include "psmf_filter.cuh"

namespace psmf {

constexpr int MAXSLOT = 64;
constexpr int V2_PASS_WARPS = V2_CWARPS;                           // 14 pass warps + reduce warp + producer warp per data CTA

__host__ __device__ constexpr int s_threads() { return (V2_CWARPS + 2) * 32; }

__host__ __device__ constexpr size_t round128(size_t x) { return (x + 127) / 128 * 128; }
template <int R, typename T>
struct SlotLayout {
    static constexpr int TS = v2_ts(R, (int)sizeof(T));
    static constexpr size_t TILE_BYTES = (size_t)R * TILE * sizeof(T);
    static constexpr size_t SLOT = round128(TS * TILE_BYTES);     // a slot holds one chunk of C, nothing else
};

// ---- mbarrier / bulk-copy PTX ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint64_t* bar, uint32_t n) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(n) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(const KParams& p, uint64_t* bar, uint32_t parity, long long step) {
    Spin sp;
    while (!mbar_try_wait(bar, parity)) {
        if (sp.expired(p, SPIN_MBAR, step)) break;
    }
}
// a wait that spans the whole launch (resident producer): no clock, it only gives up when the grid is aborting (the
// waits of the pass warps it depends on are the bounded ones), and it sleeps between attempts to stay off the pipes
__device__ __forceinline__ void mbar_wait_launch(const KParams& p, uint64_t* bar, uint32_t parity) {
    unsigned n = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++n & 15u) == 0u && *reinterpret_cast<volatile unsigned long long*>(p.bar + ABORT_WORD) != 0ULL) break;
        __nanosleep(500);
    }
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// shared state of a data CTA
template <int R>
struct DataSmem {
    static constexpr int NSP2 = nstat2_pad(R);
    double par[2][2 * R];          // par[s & 1] = parameter set s = {g_{s-1} (R), xbar_s (R)}
    double red[V2_PASS_WARPS * NSP2];   // per-warp partial sums of the current pass
    uint64_t full[MAXSLOT];        // slot loaded            (producer -> pass warps)
    uint64_t done[MAXSLOT];        // slot processed         (pass warps -> producer)
    uint64_t par_full[2];          // par[s & 1] copied from global memory   (pass warp 0 -> pass warps)
    volatile int gen[MAXSLOT];     // streaming: lap (load count) of the chunk the producer last requested for the slot
    uint64_t red_full;             // all pass warps have written red[]      (pass warps -> reduce warp)
    uint64_t red_free;             // red[] has been read                    (reduce warp -> pass warps)
};

// per-warp accumulators of one pipelined pass
struct PassAcc {
    double g00[2], g01[2], g11[2];   // fragments of A0 = sum m_t c c'
    double u0[2], u1[2];             // per-lane partial sums {u, h0} of column lane/4 (u0) and 8 + lane/4 (u1) over rows = lane%4 mod 4
    double v[5];                     // per-lane: kappa, psi, gamma, q0, n_obs
    __device__ __forceinline__ void zero() {
        g00[0] = g00[1] = g01[0] = g01[1] = g11[0] = g11[1] = u0[0] = u0[1] = u1[0] = u1[1] = 0.0;
#pragma unroll
        for (int i = 0; i < 5; ++i) v[i] = 0.0;
    }
};

// ---- pass warp: pass `pass` over the tiles tl = wp, wp + NPW, ... of the CTA ---------------------------
//   pass p in [0, n):  C_{p-2} -> C_{p-1} in the slot, e_{p-1} -> ebuf, Yrec_{p-1}, sums for step p
//   pass n (FLUSH):    C_{n-2} -> C_n (both pending rank-1 updates), Yrec_{n-1}
// y / m of steps p-1 and p are read with coalesced global loads, prefetched one tile ahead (the producer
// thread is latency-bound per bulk operation, so the slots carry C only).
template <typename T>
struct YM {              // RAW loaded values: converting at load time would stall on the load right away
    T yp, yc;            // y_{p-1}[row], y_p[row]
    unsigned char mp, mc;
};
template <typename T>
__device__ __forceinline__ YM<T> load_ym(const KParams& p, const T* __restrict__ Yb, const uint8_t* __restrict__ Mb, int64_t pass,
                                         int64_t row, bool has_prev, bool has_cur) {
    YM<T> r;
    r.yp = (T)0; r.yc = (T)0; r.mp = 1; r.mc = 1;
    if (row < p.d) {
        if (has_prev) {
            r.yp = __ldg(Yb + (pass - 1) * p.ldy + row);
            if (Mb != nullptr) r.mp = __ldg(Mb + (pass - 1) * p.ldm + row);
        }
        if (has_cur) {
            r.yc = __ldg(Yb + pass * p.ldy + row);
            if (Mb != nullptr) r.mc = __ldg(Mb + pass * p.ldm + row);
        }
    }
    return r;
}

template <int R, typename T, bool FLUSH>
__device__ __forceinline__ void s_warp_pass(const KParams& p, DataSmem<R>& ps, double* __restrict__ ebuf,
                                            unsigned char* __restrict__ slots, T* __restrict__ Yrec_prev,
                                            const T* __restrict__ Yb, const uint8_t* __restrict__ Mb, int tb, int nt, int nslot,
                                            int64_t pass, int wp, int lane, int NPW, YM<T>& nx) {
    using L = SlotLayout<R, T>;
    constexpr int TS = L::TS, NSP2 = nstat2_pad(R);
    const int nchunks = (nt + TS - 1) / TS;
    const bool streaming = nchunks > nslot;
    // parameter set pass-1 = {g_{pass-2}, xbar_{pass-1}}; the flush pass also needs g_{n-1} from set n
    const double* gp = ps.par[(pass - 1) & 1];
    const double* xbp = ps.par[(pass - 1) & 1] + R;
    const double* gl = ps.par[pass & 1];
    const bool has_prev = pass >= 1, has_cur = !FLUSH;
    const bool first_touch = pass == 0;      // FLUSH of an empty launch (n = 0) is pass 0 as well
    PassAcc acc;
    acc.zero();
    long long wait_full = 0;

    // nx = y / m of this warp's first tile, loaded before the wait for the parameter set
    for (int tl = wp; tl < nt; tl += NPW) {
        const YM<T> ym = nx;
        if (tl + NPW < nt)                                             // prefetch y / m of this warp's next tile
            nx = load_ym<T>(p, Yb, Mb, pass, (int64_t)(tb + tl + NPW) * TILE + lane, has_prev, has_cur);
        const int k = tl / TS, i = tl - k * TS;
        const int64_t kk = pass * nchunks + k;
        const int slot = streaming ? (int)(kk % nslot) : k;
        const uint32_t parity = (uint32_t)(streaming ? (kk / nslot) & 1 : 0);
        unsigned char* sb = slots + (size_t)slot * L::SLOT;
        const long long c0 = clock64();
        // mbarrier waits only know the parity of a phase.  Bulk loads complete out of order, so a warp that jumps
        // NPW / TS chunks ahead could reach a slot whose PREVIOUS load is still pending and would take that older
        // phase (same parity as two laps back) for its own.  The producer therefore publishes the lap it has
        // requested for the slot; once that is ours, the previous phase is complete and the parity is unambiguous.
        if (streaming) {
            const int lap = (int)(kk / nslot);
            Spin sp;
            while (ps.gen[slot] < lap) {
                if (sp.expired(p, SPIN_RING, pass)) break;
            }
        }
        // resident: tile tl belongs to this warp in every pass and nobody else touches it between the initial load and the
        // final store, so only the first pass waits for the load (phase 0 of full[k]) and only the flush pass releases it
        if (streaming || first_touch) mbar_wait(p, &ps.full[slot], parity, pass);
        wait_full += clock64() - c0;
        const int64_t row = (int64_t)(tb + tl) * TILE + lane;
        const int rl = tl * TILE + lane;
        const bool inb = row < p.d;
        T* tile = reinterpret_cast<T*>(sb) + (size_t)i * (R * TILE);

#ifdef PSMF_DEBUG
        if ((p.flags & F_DBG_NOCOMPUTE) != 0) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0 && (streaming || FLUSH)) {
                const int ntc = min(TS, nt - k * TS);
                mbar_arrive_n(&ps.done[slot], (i == ntc - 1) ? (uint32_t)(TS - ntc + 1) : 1u);
            }
            continue;
        }
#endif
        // ---- phase 1, lane = row ----
        // observation of steps p-1 and p: mask byte, or NaN-encoded missing entries (PSMF_NAN_MASK)
        double ypv = (double)ym.yp, ycv = (double)ym.yc;
        bool mpo = ym.mp != 0, mco = ym.mc != 0;
        if ((p.flags & F_NAN_MASK) != 0) {
            mpo = !isnan(ypv); mco = !isnan(ycv);
            ypv = mpo ? ypv : 0.0; ycv = mco ? ycv : 0.0;
        }
        double c[R];
#pragma unroll
        for (int j = 0; j < R; ++j) c[j] = (double)tile[tile_pos(j, lane)];
        double e = 0.0;
        if (pass >= 2) {                                           // C_{p-1} = C_{p-2} + e_{p-2} g_{p-2}'   (rPSMF.py:111)
            const double epp = ebuf[rl];
#pragma unroll
            for (int j = 0; j < R; ++j) c[j] = fma(epp, gp[j], c[j]);
        }
        if (pass >= 1) {                                           // e_{p-1} = y_{p-1} - m_{p-1} C_{p-1} xbar_{p-1}
            double yh4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int j = 0; j < R; ++j) yh4[j & 3] = fma(c[j], xbp[j], yh4[j & 3]);     // rPSMF.py:89
            const double yh = (yh4[0] + yh4[1]) + (yh4[2] + yh4[3]);
            e = ypv - ((inb && mpo) ? yh : 0.0);                   // rPSMF.py:101
            if (Yrec_prev != nullptr && inb) Yrec_prev[row] = (T)yh;
        }
        if constexpr (FLUSH) {                                     // C_n = C_{n-1} + e_{n-1} g_{n-1}'
#pragma unroll
            for (int j = 0; j < R; ++j) c[j] = fma(e, gl[j], c[j]);
#pragma unroll
            for (int j = 0; j < R; ++j) tile[tile_pos(j, lane)] = (T)c[j];
        } else {
#pragma unroll
            for (int j = 0; j < R; ++j) tile[tile_pos(j, lane)] = (T)c[j];
            ebuf[rl] = e;
            const bool mi = inb && mco;
            const double yi = ycv;
            acc.v[0] += mi ? e * e : 0.0;                          // kappa
            acc.v[1] += mi ? yi * e : 0.0;                         // psi
            acc.v[2] += mi ? yi * yi : 0.0;                        // gamma
            acc.v[3] += mi ? 0.0 : yi * yi;                        // q0 (rows missing at step p: e_p = y_p)
            acc.v[4] += mi ? 1.0 : 0.0;                            // n_obs
            const double me = mi ? e : 0.0, my = mi ? yi : 0.0;   // B columns 0 / 1 of the [u | h0] product
            __syncwarp();
            // ---- phase 2: A0 += sum m c c', [u | h0] += sum m c [e, y]  (fp64 DMMA, k = row) ----
            const unsigned mbits = __ballot_sync(FULL, mi);
            const int kq = lane & 3, mm = lane >> 2;
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                const int r4 = 4 * s + kq;
                const bool mrow = (mbits >> r4) & 1u;
                const int pos = r4 ^ (mm << 2);
                const double a0 = (mm < R) ? (double)tile[mm * 32 + pos] : 0.0;
                const double b0 = mrow ? a0 : 0.0;
                // [u | h0]: plain FMAs on the element this lane holds anyway (an 8x8x4 DMMA would waste 6 of its 8
                // columns: 16 fp64-pipe cycles against 2 per FMA)
                const double se = __shfl_sync(FULL, me, r4), sy = __shfl_sync(FULL, my, r4);
                dmma884(acc.g00, a0, b0);
                acc.u0[0] = fma(a0, se, acc.u0[0]);
                acc.u0[1] = fma(a0, sy, acc.u0[1]);
                if constexpr (R > 8) {
                    const double a1 = (8 + mm < R) ? (double)tile[(8 + mm) * 32 + pos] : 0.0;
                    const double b1 = mrow ? a1 : 0.0;
                    dmma884(acc.g01, a0, b1);
                    dmma884(acc.g11, a1, b1);
                    acc.u1[0] = fma(a1, se, acc.u1[0]);
                    acc.u1[1] = fma(a1, sy, acc.u1[1]);
                }
            }
        }
        // this warp is done with its tile: make the generic-proxy writes visible to the bulk store and
        // release the slot (the owner of the last tile of a partial chunk also signs for the missing tiles)
        if (streaming || FLUSH) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                const int ntc = min(TS, nt - k * TS);
                mbar_arrive_n(&ps.done[slot], (i == ntc - 1) ? (uint32_t)(TS - ntc + 1) : 1u);
            }
        }
    }
    if constexpr (!FLUSH) {
        if (wp == 0 && lane == 0) {
            stamp_pass(p, pass, 10, (unsigned long long)wait_full, false);
            stamp_pass(p, pass, 14, 0, true);
        }
        __syncwarp();
        // y / m of the first tile of the next pass: in flight while this pass is reduced and the next
        // parameter set is awaited
        if (pass + 1 <= p.n_steps)
            nx = load_ym<T>(p, Yb, Mb, pass + 1, (int64_t)(tb + wp) * TILE + lane, true, pass + 1 < p.n_steps);
        // per-warp sums -> ps.red; the reduce warp adds them and takes it from there, this warp moves on
        if (pass >= 1) mbar_wait(p, &ps.red_free, (uint32_t)((pass - 1) & 1), pass);
        double* r0 = ps.red + wp * NSP2;
        const int kq = lane & 3, mm = lane >> 2;
#pragma unroll
        for (int x = 0; x < 2; ++x) {
            const int n = 2 * kq + x;
            if (mm <= n && n < R) r0[gram_off(R, mm) + (n - mm)] = acc.g00[x];
            if constexpr (R > 8) {
                if (8 + n < R) r0[gram_off(R, mm) + (8 + n - mm)] = acc.g01[x];
                if (mm <= n && 8 + n < R) r0[gram_off(R, 8 + mm) + (n - mm)] = acc.g11[x];
            }
        }
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {                          // sum over the four row classes kq (fixed order)
            acc.u0[0] += __shfl_xor_sync(FULL, acc.u0[0], o);
            acc.u0[1] += __shfl_xor_sync(FULL, acc.u0[1], o);
            if constexpr (R > 8) {
                acc.u1[0] += __shfl_xor_sync(FULL, acc.u1[0], o);
                acc.u1[1] += __shfl_xor_sync(FULL, acc.u1[1], o);
            }
        }
        if (kq == 0) {                                             // u_mm, h0_mm
            if (mm < R) {
                r0[ngram(R) + mm] = acc.u0[0];
                r0[ngram(R) + R + mm] = acc.u0[1];
            }
            if constexpr (R > 8) {
                if (8 + mm < R) {
                    r0[ngram(R) + 8 + mm] = acc.u1[0];
                    r0[ngram(R) + R + 8 + mm] = acc.u1[1];
                }
            }
        }
        int base = 0, lim = 5;
        bfly<5, 16, 5>(acc.v, lane, base, lim);
        if (base < lim) r0[ngram(R) + 2 * R + base] = acc.v[0];
        __syncwarp();
        if (lane == 0) mbar_arrive(&ps.red_full);
        __syncwarp();
        if (wp == 0 && lane == 0) stamp_pass(p, pass, 15, 0, true);
        __syncwarp();
    }
}

// ---- producer: one thread drives all bulk copies of the CTA (C chunks only) ------------------------------
// The loop is latency-bound per iteration (~0.6 us measured, scratch/bulkbench.cu): one bulk store and one
// bulk load of a 16 KB chunk per iteration is what sustains the HBM rate, so nothing else goes through it.
template <int R, typename T>
__device__ void s_producer(const KParams& p, DataSmem<R>& ps, unsigned char* slots, T* Cs, int tb, int nt, int nslot) {
    using L = SlotLayout<R, T>;
    constexpr int TS = L::TS;
    const int nchunks = (nt + TS - 1) / TS;
    const bool streaming = nchunks > nslot;
    const int64_t npass = p.n_steps + 1;
    const uint32_t last_bytes = (uint32_t)((nt - (nchunks - 1) * TS) * L::TILE_BYTES);
    const uint32_t full_bytes = (uint32_t)(TS * L::TILE_BYTES);
    T* Cb = Cs + (size_t)tb * (R * TILE);
    constexpr size_t CHUNK_ELEMS = (size_t)TS * R * TILE;
    if (streaming) {
        // Ring of nslot slots over the chunk sequence (consumption order: pass-major).  Chunk j is stored as soon
        // as the pass warps release it and its slot is reloaded with chunk j + nslot right after the store has
        // left shared memory.
        const int64_t total = npass * nchunks;
        const int gap = nchunks - nslot;              // >= 1: store groups committed since the previous version of the chunk loaded next
        int lk = 0;                                   // chunk-in-pass index of the next load
        int64_t lc = 0;                               // global index of the next load
        for (; lc < total && lc < nslot; ++lc) {
            const uint32_t bytes = lk == nchunks - 1 ? last_bytes : full_bytes;
            mbar_arrive_expect_tx(&ps.full[lc], bytes);                 // ps.gen[lc] = 0 (lap 0) from the CTA prologue
            bulk_load(slots + (size_t)lc * L::SLOT, Cb + (size_t)lk * CHUNK_ELEMS, bytes, &ps.full[lc]);
            if (++lk == nchunks) lk = 0;
        }
        int sk = 0, slot = 0;                         // chunk-in-pass index / slot of the next store
        uint32_t par = 0;
        for (int64_t j = 0; j < total; ++j) {
            mbar_wait(p, &ps.done[slot], par, j);                                     // chunk j processed
            unsigned char* sb = slots + (size_t)slot * L::SLOT;
#ifdef PSMF_DEBUG
            if ((p.flags & F_DBG_NOSTORE) == 0)
#endif
                bulk_store(Cb + (size_t)sk * CHUNK_ELEMS, sb, sk == nchunks - 1 ? last_bytes : full_bytes);
            bulk_commit();
            if (lc < total) {
                bulk_wait_read<0>();                                               // the store has left shared memory
                // the previous version of the chunk loaded now (one pass ago) was stored `gap` groups ago: it has landed
                // once at most gap - 1 newer groups are pending
                if (gap > 8) bulk_wait<8>(); else if (gap > 4) bulk_wait<4>(); else if (gap > 2) bulk_wait<2>(); else if (gap > 1) bulk_wait<1>(); else bulk_wait<0>();
                const uint32_t bytes = lk == nchunks - 1 ? last_bytes : full_bytes;
                ps.gen[slot] = (int)(lc / nslot);                                   // lap of the chunk requested now
                __threadfence_block();
                mbar_arrive_expect_tx(&ps.full[slot], bytes);
                bulk_load(sb, Cb + (size_t)lk * CHUNK_ELEMS, bytes, &ps.full[slot]);
                if (++lk == nchunks) lk = 0;
                ++lc;
            }
            if (++sk == nchunks) sk = 0;
            if (++slot == nslot) { slot = 0; par ^= 1u; }
        }
    } else {
        for (int k = 0; k < nchunks; ++k) {
            const uint32_t bytes = k == nchunks - 1 ? last_bytes : full_bytes;
            mbar_arrive_expect_tx(&ps.full[k], bytes);
            bulk_load(slots + (size_t)k * L::SLOT, Cb + (size_t)k * CHUNK_ELEMS, bytes, &ps.full[k]);
        }
        // C stays resident: the pass warps only sign off after the flush pass (phase 0 of done[k])
        for (int k = 0; k < nchunks; ++k) {
            mbar_wait_launch(p, &ps.done[k], 0u);
            bulk_store(Cb + (size_t)k * CHUNK_ELEMS, slots + (size_t)k * L::SLOT, k == nchunks - 1 ? last_bytes : full_bytes);
            bulk_commit();
        }
    }
    bulk_wait<0>();
}

// ---- parameter sets {g_{s-1}, xbar_s}: control CTA -> data CTAs through global memory --------------------
// One 16-byte cell per double, {lo, tag, hi, tag} with tag = s + 1: every 8-byte half carries its own tag, so
// a reader that polls the cell needs no separate flag (one L2 round trip instead of two) and never sees a torn
// value.  p.gparams = [2 parities][2R] cells, zeroed by the host before every launch.
// named barriers of the control CTA
constexpr int CB_GJ = 1;           // elimination threads
constexpr int CB_S = 2;            // solver group
constexpr int CB_R = 3;            // reducer group
constexpr int CB_FULL = 4;         // +parity: reducers arrive, solvers wait     (statistics of a step are complete)
constexpr int CB_EMPTY = 6;        // +parity: solvers arrive, reducers wait     (statistics buffer may be overwritten)
constexpr int C_SOLVERS = 256;     // threads [0, 256): r x r update;  [256, blockDim): totals + NVLink exchange
constexpr int C_GJ = 192;          // elimination threads; the two remaining solver warps do the side computations

__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int R>
struct ControlSmem {
    Smem<R> sh;
    double tot2[2][nstat2_pad(R)];   // reduced (and exchanged) pipelined sums of step t in tot2[t & 1]
    double Mw[R][R + 1];             // copy of I + Pbar G for the one-warp solve of K b (the CTA-wide elimination overwrites aug)
    double a2[nstat2_pad(R)];        // A_t packed, h_t, gamma, q0, n_obs (solvers)
    double kb[R];                    // K b
};

// ---- K b on the critical path: Gauss-Jordan on [M | rhs] by ONE warp, entirely in registers ----------------------
// The data CTAs wait for x_t = x_bar + K b only; the full K (16 right-hand sides, for P_t) is needed a whole step
// later.  So one warp solves M z = Pbar b alone while the CTA-wide elimination produces K off the critical path: no
// shared-memory round trip and no barrier per pivot (shuffles only), ~110 cycles per pivot instead of ~280.
// Lane (row i = lane & 15, half h = lane >> 4) holds columns [h HC, (h+1) HC) of row i of M, half 0 also the rhs.
// Partial pivoting as in gauss_jordan_cta (integer max over the high words of |a_ik|, ties -> lowest row); rows are not
// swapped and pivot rows are not normalised: unknown k = rhs[p_k] / a[p_k][k] at the end.  All 32 lanes must call.
// Measured (scratch/solve_bench.cu, trace.py): 179 cycles per pivot alone on an SM, but ~2x that next to the CTA-wide
// elimination it was meant to overtake (shuffles share the MIO pipe with the elimination's shared-memory traffic) -- the
// data CTAs got x_t 0.5 us LATER than from the 192-thread elimination.  Kept for reference, off by default.
#ifndef PSMF_WARP_SOLVE
#define PSMF_WARP_SOLVE 0
#endif
constexpr bool WARP_SOLVE = PSMF_WARP_SOLVE != 0;

template <int R>
__device__ __forceinline__ void warp_solve(const double (*Mw)[R + 1], double rhs, double* __restrict__ z_out, int lane) {
    static_assert(R <= 16, "one warp holds at most 16 rows");
    constexpr int HC = (R + 1) / 2;
    const int i = lane & 15, h = lane >> 4;
    const bool rowok = i < R;
    double m[HC];
#pragma unroll
    for (int c = 0; c < HC; ++c) {
        const int gc = h * HC + c;
        m[c] = (rowok && gc < R) ? Mw[i][gc] : 0.0;
    }
    double r = (h == 0 && rowok) ? rhs : 0.0;
    int mycol = -1;                                    // the unknown this lane's row became the pivot row of
    double myinv = 0.0;
#pragma unroll
    for (int k = 0; k < R; ++k) {
        const int hk = k / HC, kl = k - hk * HC;                             // compile-time after unrolling
        const double colk = __shfl_sync(FULL, m[kl], i + 16 * hk);           // a_ik of this lane's row
        const int hi = __double2hiint(fabs(colk));
        const int key = (!rowok || mycol >= 0) ? -1 : ((hi & 0x7ffffff0) | (15 - i));
        const double cinv = fast_rcp(colk);
        const int pi = 15 - (__reduce_max_sync(FULL, key) & 15);
        const double inv = __shfl_sync(FULL, cinv, pi);
        const double f = (i == pi) ? 0.0 : colk * inv;                        // the pivot row itself stays
#pragma unroll
        for (int c = 0; c < HC; ++c) {
            if (HC + c > k) {                                                 // column still live in at least one half
                const double rp = __shfl_sync(FULL, m[c], pi + 16 * h);
                m[c] = fma(-f, rp, m[c]);
            }
        }
        const double rr = __shfl_sync(FULL, r, pi + 16 * h);
        r = fma(-f, rr, r);
        if (i == pi) {
            mycol = k;
            myinv = inv;
        }
    }
    if (h == 0 && rowok && mycol >= 0) z_out[mycol] = r * myinv;
}

// ---- reducer half of the control CTA -------------------------------------------------------------------
// One SM ingests only ~40 GB/s, so the ~200 kB of CTA partials of a step (147 CTAs x 173 doubles at r = 16) are
// not summed by the control CTA: the reduce warp of data CTA c sums entries c, c + ndata, .. over all CTAs
// (fixed order: deterministic) and publishes each total as a tagged cell; the control CTA polls the cells.
template <int R>
__device__ void reduce_warp(const KParams& p, DataSmem<R>& ps, int lane, int NPW) {
    constexpr int NSP2 = nstat2_pad(R), NST2 = nstat2(R);
    constexpr int NE = (NST2 + 31) / 32;
    const int ndata = p.cps, pstr = (ndata + 7) & ~7, cta = blockIdx.x;
    uint4* totals = reinterpret_cast<uint4*>(p.gparams) + 4 * MAXR;
    uint4* pcells = reinterpret_cast<uint4*>(p.partials);
    for (int64_t t = 0; t < p.n_steps; ++t) {
        const int b = (int)(t & 1);
        // the partial cells outlive the launch: their tags count the steps of the engine, not of the launch
        const uint32_t ptag = tag_of(p.step_base + (unsigned long long)t + 1ULL);
        uint4* base = pcells + (size_t)b * NSP2 * pstr;
        // (1) CTA partial of pass t: per-warp sums in fixed warp order -> tagged cells [parity][entry][cta]
        mbar_wait(p, &ps.red_full, (uint32_t)b, t);
        {
            double sum[NE];
#pragma unroll
            for (int i = 0; i < NE; ++i) sum[i] = 0.0;
            for (int w = 0; w < NPW; ++w) {
#pragma unroll
                for (int i = 0; i < NE; ++i) sum[i] += ps.red[w * NSP2 + min(lane + 32 * i, NSP2 - 1)];
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&ps.red_free);
#pragma unroll
            for (int i = 0; i < NE; ++i)
                if (lane + 32 * i < NST2) cell_store(base + (size_t)(lane + 32 * i) * pstr + cta, sum[i], ptag);
            if (lane == 0) stamp_pass(p, t, 9, 0, true);
            __syncwarp();
        }
        // (2) this CTA's share of the grid reduction: entries cta, cta + ndata, .. summed over all CTAs.  The warp polls
        // the cells of up to TWO entries together (lanes over the CTAs; all loads of both rows are in flight before any tag
        // is examined): one L2 round trip per attempt whether the CTA owns one entry or two.  Each total goes to the local
        // control CTA and -- row sharding -- straight into the mailbox of every peer GPU (lane = destination rank), so the
        // NVLink hop runs next to the local L2 hop instead of behind it.
        const unsigned long long gstep = p.step_base + (unsigned long long)t;
        const int mslot = (int)(gstep % MBOX_DEPTH);
        const uint32_t xtag = tag_of(gstep + 1ULL);
        const int nj = (ndata + 31) >> 5;                          // 32-cell groups per entry row (<= 8)
        for (int e = cta; e < NST2; e += 2 * ndata) {
            const int e2 = e + ndata;
            const bool has2 = e2 < NST2;
            const uint4* row = base + (size_t)e * pstr;
            const uint4* row2 = base + (size_t)(has2 ? e2 : e) * pstr;
            double v[8], w[8];
            bool ok;
            Spin sp;
            do {
                ok = true;
                uint32_t lo[8], hi[8], t0[8], t1[8], lo2[8], hi2[8], t02[8], t12[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    lo[j] = hi[j] = lo2[j] = hi2[j] = 0u;
                    t0[j] = t1[j] = t02[j] = t12[j] = ptag;
                    if (j < nj) {
                        const int c = min(lane + 32 * j, pstr - 1);
                        asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(lo[j]), "=r"(t0[j]), "=r"(hi[j]), "=r"(t1[j]) : "l"(row + c) : "memory");
                        if (has2)
                            asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                                         : "=r"(lo2[j]), "=r"(t02[j]), "=r"(hi2[j]), "=r"(t12[j]) : "l"(row2 + c) : "memory");
                    }
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = lane + 32 * j;
                    const bool in = c < ndata;
                    ok = ok && (!in || (t0[j] == ptag && t1[j] == ptag && t02[j] == ptag && t12[j] == ptag));
                    v[j] = in ? __hiloint2double((int)hi[j], (int)lo[j]) : 0.0;
                    w[j] = in ? __hiloint2double((int)hi2[j], (int)lo2[j]) : 0.0;
                }
                if (!ok) {
                    if (sp.expired(p, SPIN_PARTIALS, t)) ok = true;
                    else if (POLL_BACKOFF_NS > 0) __nanosleep(POLL_BACKOFF_NS);
                }
            } while (!__all_sync(FULL, ok));
            const double sum = warp_allsum(((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7])));
            const double sum2 = has2 ? warp_allsum(((w[0] + w[1]) + (w[2] + w[3])) + ((w[4] + w[5]) + (w[6] + w[7]))) : 0.0;
            if (lane < p.world) {
                if (lane == p.rank) {
                    cell_store(totals + (size_t)b * NSP2 + e, sum, tag_of((unsigned long long)t + 1ULL));
                    if (has2) cell_store(totals + (size_t)b * NSP2 + e2, sum2, tag_of((unsigned long long)t + 1ULL));
                } else {
                    uint4* dst = reinterpret_cast<uint4*>(p.mbox_peer[lane]) + ((size_t)mslot * MAX_PEERS + p.rank) * MBOX_SLOT;
                    cell_store_sys(dst + e, sum, xtag);
                    if (has2) cell_store_sys(dst + e2, sum2, xtag);
                }
            }
            __syncwarp();
        }
    }
}

// ---- reducer half of the control CTA: gather every entry over the local reduce warps and the peer GPUs ---------
// Thread e polls the local total of entry e and the world - 1 mailbox cells the peers' reduce warps stored, all at once
// (gather_ranks), and adds them in rank order: the same order on every GPU, so the replicated state stays bit-identical.
template <int R>
__device__ void control_reduce(const KParams& p, ControlSmem<R>& cs) {
    constexpr int NSP2 = nstat2_pad(R), NST2 = nstat2(R);
    const int tid = threadIdx.x - C_SOLVERS;
    const int NTHR = (int)blockDim.x - C_SOLVERS;
    const uint4* totals = reinterpret_cast<const uint4*>(p.gparams) + 4 * MAXR;
    for (int64_t t = 0; t < p.n_steps; ++t) {
        const int b = (int)(t & 1);
        double* tot2 = cs.tot2[b];
        if (t >= 2) named_bar_sync(CB_EMPTY + b, (int)blockDim.x);   // the solvers are done with the sums of step t-2
        stamp(p, t, 2, C_SOLVERS);
        const unsigned long long gstep = p.step_base + (unsigned long long)t;
        const uint4* slots = reinterpret_cast<const uint4*>(p.mbox_local) + (size_t)(gstep % MBOX_DEPTH) * MAX_PEERS * MBOX_SLOT;
        for (int e = tid; e < NST2; e += NTHR)
            tot2[e] = gather_ranks(p, slots, e, tag_of(gstep + 1ULL), totals + (size_t)b * NSP2 + e, tag_of((unsigned long long)t + 1ULL), 0.0, t);
        if (p.world > 1 && t == 0 && tid == NTHR - 1) mailbox_check_peers(p, 2, NST2, t);
        stamp(p, t, 4, C_SOLVERS);
        sync_n<CB_R>(NTHR);
        stamp(p, t, 13, C_SOLVERS);
        __threadfence_block();
        named_bar_arrive(CB_FULL + b, (int)blockDim.x);
    }
}

// ---- solver half of the control CTA --------------------------------------------------------------------
// Per step: assemble the statistics of step t from the pipelined sums (+ g_{t-1}, xbar_t), solve for K, update
// x and publish {g_t, xbar_{t+1}} as early as possible (that is all the data CTAs wait for); the rest of the
// r x r update (omega, phi, P, V, Q, rho, lambda, the next predict) follows off the critical path.
// rPSMF.py:102-115,133-135 with the statistics in the sufficient-statistic form of psmf_filter.cuh.
template <int R, bool GL, bool LL>
__device__ void control_solve(const KParams& p, ControlSmem<R>& cs) {
    constexpr int NGm = ngram(R);
    constexpr int NTHR = C_SOLVERS;
    constexpr int FIN = R & 1;
    Smem<R>& sh = cs.sh;
    double* a2 = cs.a2;
    const int tid = threadIdx.x, lane = tid & 31, warp = uniform_warp_id();
    const int64_t n = p.n_steps;
    const bool simp = (p.flags & F_SIMPLIFIED) != 0;
    const bool robust = (p.flags & F_ROBUST) != 0;
    const double dg = (double)p.d_global;
    double* stg = p.state;
    uint4* cells = reinterpret_cast<uint4*>(p.gparams);

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
    sync_n<CB_S>(NTHR);
    predict_cta<R, CB_S>(p, sh, tid, p.k0, 0, NTHR);               // xbar_0, Pbar_0, a_0, w1/w0
    if (tid < R) {                                                 // set 0 = {0, xbar_0}
        cell_store(cells + tid, 0.0, tag_of(1ULL));
        cell_store(cells + R + tid, sh.xb[tid], tag_of(1ULL));
    }

    for (int64_t t = 0; t < n; ++t) {
        const int b = (int)(t & 1);
        const double* t2 = cs.tot2[b];
        stamp(p, t, 0);
        named_bar_sync(CB_FULL + b, (int)blockDim.x);
        stamp(p, t, 1);
        // (A) A_t = A0 + u g' + g u' + kappa g g' (packed upper triangle), h_t = h0 + psi g, scalars
        {
            const double kappa = t2[NGm + 2 * R + 0], psi = t2[NGm + 2 * R + 1];
            for (int idx = tid; idx < R * R; idx += NTHR) {
                const int j = idx / R, k = idx % R;
                if (j <= k) {
                    const double gj = sh.g[j], gk = sh.g[k];
                    a2[gram_off(R, j) + (k - j)] = t2[gram_off(R, j) + (k - j)] + (t2[NGm + j] * gk + gj * t2[NGm + k]) + kappa * gj * gk;
                }
            }
            if (tid >= NTHR - R) {
                const int j = tid - (NTHR - R);
                a2[NGm + j] = fma(psi, sh.g[j], t2[NGm + R + j]);
            }
            if (tid < 3) a2[NGm + R + tid] = t2[NGm + 2 * R + 2 + tid];     // gamma, q0, n_obs
        }
        sync_n<CB_S>(NTHR);
        named_bar_arrive(CB_EMPTY + b, (int)blockDim.x);                        // cs.tot2[b] may be refilled (step t+2)
        // (B) augmented matrix [I + Pbar G | Pbar], G = w1 A_t
        if (!simp) {
            const double w1 = sh.w1;
            for (int idx = tid; idx < R * R; idx += NTHR) {
                const int i = idx / R, j = idx % R;
                double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
                for (int k = 0; k < R; k += 2) {
                    const int lo = k < j ? k : j, hi = k < j ? j : k;
                    acc0 = fma(sh.Pb[i * R + k], a2[gram_off(R, lo) + hi - lo], acc0);
                    if (k + 1 < R) {
                        const int lo1 = k + 1 < j ? k + 1 : j, hi1 = k + 1 < j ? j : k + 1;
                        acc1 = fma(sh.Pb[i * R + k + 1], a2[gram_off(R, lo1) + hi1 - lo1], acc1);
                    }
                }
                const double mij = fma(w1, acc0 + acc1, (i == j) ? 1.0 : 0.0);
                sh.aug[0][i][j] = mij;
                cs.Mw[i][j] = mij;
                sh.aug[0][i][R + j] = sh.Pb[i * R + j];
            }
            sync_n<CB_S>(NTHR);
        }
        // (C) elimination (C_GJ threads) next to the side computations (two warps)
        if (warp < C_GJ / 32) {
            // aug[FIN][perm[k]][R..2R) = K[k][:]   (measured: 128 and 192 threads tie at 2.3 us, 64: 5.8, 32: 9.1)
            if (!simp) gauss_jordan_cta<R, C_GJ, CB_GJ, 2 * R, LL>(sh, tid);
        } else if (warp == C_GJ / 32) {
            // b = w1 (h - A xbar), q1 = gamma - 2 xbar'h + xbar'A xbar, s = w1 q1 + w0 q0
            double ax = 0.0, hj = 0.0, xj = 0.0;
            if (lane < R) {
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int k = 0; k < R; k += 2) {
                    const int lo = k < lane ? k : lane, hi = k < lane ? lane : k;
                    s0 = fma(a2[gram_off(R, lo) + hi - lo], sh.xb[k], s0);
                    if (k + 1 < R) {
                        const int lo1 = k + 1 < lane ? k + 1 : lane, hi1 = k + 1 < lane ? lane : k + 1;
                        s1 = fma(a2[gram_off(R, lo1) + hi1 - lo1], sh.xb[k + 1], s1);
                    }
                }
                ax = s0 + s1;
                hj = a2[NGm + lane];
                xj = sh.xb[lane];
            }
            const double xh = warp_allsum(xj * hj);
            const double xax = warp_allsum(xj * ax);
            const double w1 = sh.w1, w0 = sh.w0;
            // q1 is rebuilt from raw second moments: when the residual is far below the signal the three terms cancel
            // and the rounding error (eps * gamma) can leave q1 slightly negative -> clamp
            const double q1 = fmax(a2[NGm + R + 0] - 2.0 * xh + xax, 0.0);
            const double q0 = a2[NGm + R + 1];
            if (lane < R) sh.tot[NGm + lane] = w1 * (hj - ax);                 // b = w1 sum m e c
            if (lane == 0) {
                sh.tot[NGm + R + 0] = w1 * q1 + (q0 != 0.0 ? w0 * q0 : 0.0);  // s = diff' Ri diff (a = 0: w0 = inf only matters with missing rows)
                sh.tot[NGm + R + 1] = q1;
                sh.tot[NGm + R + 2] = q0;
                sh.tot[NGm + R + 3] = a2[NGm + R + 2];
            }
            if (WARP_SOLVE && !simp) {
                // K b by this warp alone (warp_solve), then x_t and the publication of xbar_{t+1}: the data CTAs do not
                // wait for the CTA-wide elimination any more
                __syncwarp();
                double rhs = 0.0;
                if (lane < R) {
                    double s0 = 0.0, s1 = 0.0;
#pragma unroll
                    for (int k = 0; k < R; k += 2) {
                        s0 = fma(sh.Pb[lane * R + k], sh.tot[NGm + k], s0);
                        if (k + 1 < R) s1 = fma(sh.Pb[lane * R + k + 1], sh.tot[NGm + k + 1], s1);
                    }
                    rhs = s0 + s1;
                }
                warp_solve<R>(cs.Mw, rhs, cs.kb, lane);
                __syncwarp();
                const double xn = lane < R ? sh.xb[lane] + cs.kb[lane] : 0.0;  // rPSMF.py:104
                double xnext = xn;                                             // identity; external: set n is never used
                if (p.dynamics == DYN_LINEAR) {
                    // x_bar_{t+1} = A x_t + c in the operation order of linear_predict (predict_cta recomputes it from sh.x
                    // and must get the same bits: the data CTAs see this copy, the control CTA its own)
                    double acc = (lane < R && p.lin_c != nullptr) ? p.lin_c[lane] : 0.0;
#pragma unroll
                    for (int k = 0; k < R; ++k) {
                        const double xk = __shfl_sync(FULL, xn, k);
                        if (lane < R) acc = fma(p.lin_A[lane * R + k], xk, acc);
                    }
                    xnext = acc;
                } else if (p.dynamics == DYN_COS && lane < R) {
                    xnext = cos(__dadd_rn(__dmul_rn(__dmul_rn(6.283185307179586, sh.th[lane]), (double)(p.k0 + t + 1)), xn));
                }
                if (lane < R) cell_store(cells + (size_t)((t + 1) & 1) * 2 * R + R + lane, xnext, tag_of((unsigned long long)t + 2ULL));
                stamp(p, t, 6, C_GJ);
            }
        } else {
            // eta = (rho n_obs + (rho + a) tr(Pbar G)) / d, N = a + eta, g_t = V x_bar / N   (rPSMF.py:108-111)
            const double a = sh.a, rho = sh.rho;
            double eta;
            if (simp) {
                eta = rho;                                                     // synthetic_psmf.py:86-87
            } else {
                double tr = 0.0;
                if (lane < R) {
                    double s0 = 0.0, s1 = 0.0;
#pragma unroll
                    for (int i = 0; i < R; i += 2) {
                        const int lo = i < lane ? i : lane, hi = i < lane ? lane : i;
                        s0 = fma(sh.Pb[i * R + lane], a2[gram_off(R, lo) + hi - lo], s0);
                        if (i + 1 < R) {
                            const int lo1 = i + 1 < lane ? i + 1 : lane, hi1 = i + 1 < lane ? lane : i + 1;
                            s1 = fma(sh.Pb[(i + 1) * R + lane], a2[gram_off(R, lo1) + hi1 - lo1], s1);
                        }
                    }
                    tr = s0 + s1;
                }
                const double trpg = sh.w1 * warp_allsum(tr);
                eta = (rho * a2[NGm + R + 2] + (rho + a) * trpg) / dg;
            }
            const double N = a + eta;
            if (lane < R) {
                const double gl = (((p.flags & F_CUPDATE_VT) != 0) ? sh.vx[lane] : sh.vxt[lane]) / N;   // rPSMF.py:111 / PSMF.py:80
                sh.g[lane] = gl;
                if (WARP_SOLVE && !simp) cell_store(cells + (size_t)((t + 1) & 1) * 2 * R + lane, gl, tag_of((unsigned long long)t + 2ULL));
            }
            if (lane == 0) {
                sh.sc[1] = eta;
                sh.sc[2] = N;
            }
        }
        sync_n<CB_S>(NTHR);
        stamp(p, t, 7);
        // (D) x_t = xbar_t + K b, xbar_{t+1} = f(x_t); publish set t+1 = {g_t, xbar_{t+1}}   (warp 0)
        if (warp == 0) {
            const bool early = WARP_SOLVE && !simp;       // K b, x_t and the publication were done by the solver warp
            double kbj = 0.0;
            if (early) {
                kbj = lane < R ? cs.kb[lane] : 0.0;
            } else {
                const int j = lane & 15, half = lane >> 4;
                if (!simp && j < R) {
                    const double* Krow = &sh.aug[FIN][sh.perm[j]][R];
                    double s0 = 0.0, s1 = 0.0;
                    constexpr int H = (R + 1) / 2;
#pragma unroll
                    for (int k = 0; k < H; k += 2) {
                        const int k0 = half * H + k;
                        if (k0 < R) s0 = fma(Krow[k0], sh.tot[NGm + k0], s0);
                        if (k + 1 < H && k0 + 1 < R) s1 = fma(Krow[k0 + 1], sh.tot[NGm + k0 + 1], s1);
                    }
                    kbj = s0 + s1;
                }
                kbj += __shfl_xor_sync(FULL, kbj, 16);
            }
            double xn = 0.0, xnext = 0.0;
            if (lane < R) xn = sh.xb[lane] + kbj;                              // rPSMF.py:104 (simplified: x = x_bar)
            if (p.dynamics == DYN_LINEAR) {
                // x_bar_{t+1} = A x_t + c in the operation order of linear_predict (predict_cta recomputes it from sh.x
                // and must get the same bits: the data CTAs see this copy, the control CTA its own)
                double acc = (lane < R && p.lin_c != nullptr) ? p.lin_c[lane] : 0.0;
#pragma unroll
                for (int k = 0; k < R; ++k) {
                    const double xk = __shfl_sync(FULL, xn, k);
                    if (lane < R) acc = fma(p.lin_A[lane * R + k], xk, acc);
                }
                xnext = acc;
            }
            if (lane < R) {
                if (p.dynamics == DYN_COS) {
                    const double arg = __dadd_rn(__dmul_rn(__dmul_rn(6.283185307179586, sh.th[lane]), (double)(p.k0 + t + 1)), xn);
                    xnext = cos(arg);
                } else if (p.dynamics != DYN_LINEAR) {
                    xnext = xn;                        // external dynamics run one step per launch: set n is never used
                }
                if (!early) {
                    cell_store(cells + (size_t)((t + 1) & 1) * 2 * R + lane, sh.g[lane], tag_of((unsigned long long)t + 2ULL));
                    cell_store(cells + (size_t)((t + 1) & 1) * 2 * R + R + lane, xnext, tag_of((unsigned long long)t + 2ULL));
                }
            }
            if (!early) stamp(p, t, 6);
            // (E) off the critical path: omega, phi, gradient of the step log-likelihood (F_GRAD_LINEAR: with respect to
            // A and c, from the x_{t-1} still in sh.x), F_LOGLIK: its value and the one-step predictive log-density
            const double a = sh.a, rho = sh.rho, lam = sh.lam;
            const double s = sh.tot[NGm + R], q1 = sh.tot[NGm + R + 1], q0 = sh.tot[NGm + R + 2], nobs = sh.tot[NGm + R + 3];
            const double eta = sh.sc[1], N = sh.sc[2];
            const double bkb = warp_allsum((lane < R && !simp) ? sh.tot[NGm + lane] * kbj : 0.0);
            const double sSe = s - bkb;                                        // diff' CPinv diff (simplified: s)
            const double omega = robust ? (lam + sSe) / (lam + dg) : 1.0;      // rPSMF.py:105
            const double phi = robust ? (lam + q1 / N + (q0 != 0.0 ? q0 / eta : 0.0)) / (lam + dg) : 1.0;
            const bool lgrad = glin_on<GL, LL>(p) && p.grad_out != nullptr;
            double gfl = 0.0, xo = 0.0;
            if (lane < R) {
                xo = sh.x[lane];
                sh.x[lane] = xn;
                if (p.X_out != nullptr) p.X_out[t * R + lane] = xn;
                if (p.grad_out != nullptr && (p.dynamics == DYN_COS || lgrad)) {
                    // d ell_k / d theta = J_theta' d ell_k / d f; C'Me = b (rho + a)
                    const double cte = sh.tot[NGm + lane] * (rho + a);
                    const double gf = dll_df(p.flags, sh.vx[lane], sh.vxt[lane], cte, q1, nobs, lam, N);
                    if (lgrad) gfl = gf;
                    sh.grad[lane] += lgrad ? gf : gf * (6.283185307179586 * (double)(p.k0 + t) * sh.fd[lane]);
                }
            }
            if (lgrad) lin_grad_accum<R>(glin_acc(p), gfl, xo, lane);                // G_c += gf (above), G_A += gf x_{t-1}'
            if (lane == 0) {
                sh.sc[0] = omega; sh.sc[3] = phi; sh.sc[4] = sSe;
                sh.sc[5] = p.alpha * phi; sh.sc[6] = p.beta * omega;
                if (p.scal_out != nullptr) {
                    double* so = p.scal_out + t * (LL ? NSCAL_LL : NSCAL);
                    so[0] = a; so[1] = eta; so[2] = N; so[3] = omega; so[4] = phi; so[5] = sSe; so[6] = lam; so[7] = rho;
                }
                if (!(isfinite(N) && isfinite(omega) && isfinite(phi) && isfinite(xn)) || N == 0.0)
                    atomicCAS((unsigned long long*)p.status, ~0ULL, (unsigned long long)t);
            }
            if constexpr (LL) {
                if (p.scal_out != nullptr) {           // as in small_update (psmf_filter.cuh), uniform R
                    const double piv = (!simp && lane < R) ? sh.aug[0][lane][2 * R + 1] : 1.0;
                    double nll, lp;
                    step_loglik(p.flags, piv, nobs, N, q1, lam, nobs * log(rho + a), sh.w1 * q1 - bkb, lane, nll, lp);
                    if (lane == 0) {
                        p.scal_out[t * NSCAL_LL + 8] = nll;
                        p.scal_out[t * NSCAL_LL + 9] = lp;
                    }
                }
            }
            __syncwarp();
        }
        sync_n<CB_S>(NTHR);
        {
            const double omega = sh.sc[0], N = sh.sc[2], aphi = sh.sc[5], bom = sh.sc[6];
            for (int idx = tid; idx < R * R; idx += NTHR) {
                const int i = idx / R, j = idx % R;
                const double pn = simp ? sh.Pb[idx] : bom * sh.aug[FIN][sh.perm[i]][R + j];      // rPSMF.py:106
                const double vn = aphi * (sh.V[idx] - sh.vx[i] * sh.vxt[j] / N);                 // rPSMF.py:115
                sh.P[idx] = pn;
                sh.V[idx] = vn;
                if (!simp) sh.Q[idx] = omega * sh.Q[idx];                                        // rPSMF.py:133
            }
            if (tid == NTHR - 32) {
                const double lam = sh.lam;
                sh.rho = omega * sh.rho;                                                         // rPSMF.py:134
                sh.lam = (robust && (p.flags & F_FIXED_LAMBDA) == 0) ? lam + dg : lam;           // rPSMF.py:135
            }
        }
        sync_n<CB_S>(NTHR);
        if (t + 1 < n) predict_cta<R, CB_S>(p, sh, tid, p.k0 + t + 1, 0, NTHR);
        stamp(p, t, 12);
    }
    for (int i = tid; i < R * R; i += NTHR) {
        stg[st_P(R) + i] = sh.P[i];
        stg[st_V(R) + i] = sh.V[i];
        stg[st_Q(R) + i] = sh.Q[i];
    }
    if (tid < R) {
        stg[st_x(R) + tid] = sh.x[tid];
        if (p.grad_out != nullptr && !glin_on<GL, LL>(p)) p.grad_out[tid] = sh.grad[tid];
    }
    if (tid == 0) {
        stg[st_rho(R)] = sh.rho;
        stg[st_lam(R)] = sh.lam;
    }
    if (glin_on<GL, LL>(p) && p.grad_out != nullptr) {
        sync_n<CB_S>(NTHR);
        for (int i = tid; i < R * R + R; i += NTHR) p.grad_out[i] = i < R * R ? glin_acc(p)[i] : sh.grad[i - R * R];
    }
}

// pass warp 0 polls parameter set `set` in global memory into ps.par[set & 1] and releases the other warps
template <int R>
__device__ __forceinline__ void fetch_params(const KParams& p, DataSmem<R>& ps, int64_t set, int wp, int lane) {
    if (wp == 0) {
        const uint4* cells = reinterpret_cast<const uint4*>(p.gparams) + (size_t)(set & 1) * 2 * R;
        for (int i = lane; i < 2 * R; i += 32) ps.par[set & 1][i] = cell_poll<false>(p, cells + i, tag_of((unsigned long long)set + 1ULL), set);   // the whole CTA waits on this: no backoff
        __threadfence_block();
        __syncwarp();
        if (lane == 0) mbar_arrive(&ps.par_full[set & 1]);
    }
    mbar_wait(p, &ps.par_full[set & 1], (uint32_t)((set >> 1) & 1), set);
}

template <int R, typename T, bool GL = false, bool LL = false>
__global__ void __launch_bounds__(s_threads(), 1) psmf_stream_kernel(const KParams p) {
    if (p.trace != nullptr && threadIdx.x == 0 && (int)blockIdx.x < p.trace_steps) {   // debug: SM id of every CTA (row 159)
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        p.trace[(size_t)p.trace_steps * 16 + (size_t)159 * p.trace_steps + blockIdx.x] = smid;
    }
    // a CTA is either the control CTA or a data CTA: their static shared state shares one buffer
    constexpr size_t SBYTES = sizeof(ControlSmem<R>) > sizeof(DataSmem<R>) ? sizeof(ControlSmem<R>) : sizeof(DataSmem<R>);
    __shared__ __align__(16) unsigned char static_smem[SBYTES];
    extern __shared__ __align__(128) unsigned char dyn_smem_s[];
    if (blockIdx.x == gridDim.x - 1) {       // ---- control CTA ----
        ControlSmem<R>& cs = *reinterpret_cast<ControlSmem<R>*>(static_smem);
        // F_GRAD_LINEAR: the accumulator G_A is at the start of the control CTA's dynamic shared memory (p.glin_off = 0),
        // which it has no other use for
        if (uniform_warp_id() < C_SOLVERS / 32) control_solve<R, GL, LL>(p, cs);
        else control_reduce<R>(p, cs);
        return;
    }
    using L = SlotLayout<R, T>;
    const int NPW = p.npw;                                         // active pass warps (<= V2_PASS_WARPS)
    DataSmem<R>& ps = *reinterpret_cast<DataSmem<R>*>(static_smem);

    const int tid = threadIdx.x, lane = tid & 31, warp = uniform_warp_id();
    const int part = blockIdx.x;                                   // data CTA index, p.cps data CTAs
    const int ntiles = (int)((p.d + TILE - 1) / TILE);
    const int tb = (int)((int64_t)ntiles * part / p.cps);
    const int te = (int)((int64_t)ntiles * (part + 1) / p.cps);
    const int nt = te - tb;
    const int nslot = p.nslot;
    const int64_t n = p.n_steps;

    unsigned char* slots = dyn_smem_s;
    double* ebuf = reinterpret_cast<double*>(dyn_smem_s + (size_t)nslot * L::SLOT);
    T* Cs = reinterpret_cast<T*>(p.C);

    if (tid == 0) {
        for (int s = 0; s < nslot; ++s) {
            mbar_init(&ps.full[s], 1);
            mbar_init(&ps.done[s], L::TS);
        }
        mbar_init(&ps.par_full[0], 1);
        mbar_init(&ps.par_full[1], 1);
        for (int s2 = 0; s2 < MAXSLOT; ++s2) ps.gen[s2] = 0;
        mbar_init(&ps.red_full, (uint32_t)p.npw);
        mbar_init(&ps.red_free, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < nt * TILE; i += blockDim.x) ebuf[i] = 0.0;
    __syncthreads();

    if (warp == V2_PASS_WARPS) {             // ---- reduce warp ----
        reduce_warp<R>(p, ps, lane, p.npw);
        return;
    }
    if (warp == V2_PASS_WARPS + 1) {         // ---- producer warp ----
        if (lane == 0) s_producer<R, T>(p, ps, slots, Cs, tb, nt, nslot);
        return;
    }

    // ---- pass warps ----
    const int wp = warp;
    if (wp >= NPW) return;
    const T* Yb = reinterpret_cast<const T*>(p.Y);
    const uint8_t* Mb = p.M;
    YM<T> nx = load_ym<T>(p, Yb, Mb, 0, (int64_t)(tb + wp) * TILE + lane, false, true);
    for (int64_t pass = 0; pass < n; ++pass) {
        if (wp == 0 && lane == 0) stamp_pass(p, pass, 11, 0, true);
        if (pass >= 1) fetch_params<R>(p, ps, pass - 1, wp, lane);   // {g_{pass-2}, xbar_{pass-1}}
        if (wp == 0 && lane == 0) {
            stamp_pass(p, pass, 8, 0, true);
            if (p.trace != nullptr && pass < p.trace_steps) {      // per-CTA pass start times (second block)
                unsigned long long v;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
                p.trace[(size_t)p.trace_steps * (16 + 160) + (size_t)blockIdx.x * p.trace_steps + pass] = v;
            }
        }
        T* Yrec_prev = (p.Yrec && pass >= 1) ? reinterpret_cast<T*>(p.Yrec) + (pass - 1) * p.ldrec : nullptr;
        s_warp_pass<R, T, false>(p, ps, ebuf, slots, Yrec_prev, Yb, Mb, tb, nt, nslot, pass, wp, lane, NPW, nx);
        if (wp == 0 && lane == 0) {
            if (p.trace != nullptr && pass < p.trace_steps) {      // per-CTA pass end times behind the 16-entry rows
                unsigned long long v;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
                p.trace[(size_t)p.trace_steps * 16 + (size_t)blockIdx.x * p.trace_steps + pass] = v;
            }
        }
    }
    // flush: both pending rank-1 updates -> C_n; needs the parameter sets n-1 (fetched for pass n-1.. or now) and n
    fetch_params<R>(p, ps, n - 1, wp, lane);
    fetch_params<R>(p, ps, n, wp, lane);
    {
        T* Yrec_prev = p.Yrec ? reinterpret_cast<T*>(p.Yrec) + (n - 1) * p.ldrec : nullptr;
        s_warp_pass<R, T, true>(p, ps, ebuf, slots, Yrec_prev, Yb, Mb, tb, nt, nslot, n, wp, lane, NPW, nx);
    }
}

}  // namespace psmf
