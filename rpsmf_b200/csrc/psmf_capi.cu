// C ABI of the B200-native PSMF / rPSMF filter (include/psmf_b200.h).
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <cstdint>
#include <new>
#include <string>

#include "../../include/psmf_b200.h"
#include "psmf_common.cuh"
#include "psmf_tools.cuh"

PSMF_DECLARE_R(1) PSMF_DECLARE_R(2) PSMF_DECLARE_R(3) PSMF_DECLARE_R(4)
PSMF_DECLARE_R(5) PSMF_DECLARE_R(6) PSMF_DECLARE_R(7) PSMF_DECLARE_R(8)
PSMF_DECLARE_R(9) PSMF_DECLARE_R(10) PSMF_DECLARE_R(11) PSMF_DECLARE_R(12)
PSMF_DECLARE_R(13) PSMF_DECLARE_R(14) PSMF_DECLARE_R(15) PSMF_DECLARE_R(16)

namespace psmf {

static const launch_fn LAUNCH[MAXR + 1] = {
    nullptr,           launch_filter_r1,  launch_filter_r2,  launch_filter_r3,  launch_filter_r4,  launch_filter_r5,
    launch_filter_r6,  launch_filter_r7,  launch_filter_r8,  launch_filter_r9,  launch_filter_r10, launch_filter_r11,
    launch_filter_r12, launch_filter_r13, launch_filter_r14, launch_filter_r15, launch_filter_r16};
static const launch_fn LAUNCH_S[MAXR + 1] = {
    nullptr,           launch_stream_r1,  launch_stream_r2,  launch_stream_r3,  launch_stream_r4,  launch_stream_r5,
    launch_stream_r6,  launch_stream_r7,  launch_stream_r8,  launch_stream_r9,  launch_stream_r10, launch_stream_r11,
    launch_stream_r12, launch_stream_r13, launch_stream_r14, launch_stream_r15, launch_stream_r16};
static const shape_fn SHAPE_S[MAXR + 1] = {
    nullptr,          shape_stream_r1,  shape_stream_r2,  shape_stream_r3,  shape_stream_r4,  shape_stream_r5,
    shape_stream_r6,  shape_stream_r7,  shape_stream_r8,  shape_stream_r9,  shape_stream_r10, shape_stream_r11,
    shape_stream_r12, shape_stream_r13, shape_stream_r14, shape_stream_r15, shape_stream_r16};
static const launch_fn LAUNCH_V[MAXR + 1] = {
    nullptr,            launch_filterv_r1,  launch_filterv_r2,  launch_filterv_r3,  launch_filterv_r4,  launch_filterv_r5,
    launch_filterv_r6,  launch_filterv_r7,  launch_filterv_r8,  launch_filterv_r9,  launch_filterv_r10, launch_filterv_r11,
    launch_filterv_r12, launch_filterv_r13, launch_filterv_r14, launch_filterv_r15, launch_filterv_r16};
static const shape_fn SHAPE_V[MAXR + 1] = {
    nullptr,           shape_filterv_r1,  shape_filterv_r2,  shape_filterv_r3,  shape_filterv_r4,  shape_filterv_r5,
    shape_filterv_r6,  shape_filterv_r7,  shape_filterv_r8,  shape_filterv_r9,  shape_filterv_r10, shape_filterv_r11,
    shape_filterv_r12, shape_filterv_r13, shape_filterv_r14, shape_filterv_r15, shape_filterv_r16};
static const launch_fn LAUNCH_B[MAXR + 1] = {
    nullptr,          launch_batch_r1,  launch_batch_r2,  launch_batch_r3,  launch_batch_r4,  launch_batch_r5,
    launch_batch_r6,  launch_batch_r7,  launch_batch_r8,  launch_batch_r9,  launch_batch_r10, launch_batch_r11,
    launch_batch_r12, launch_batch_r13, launch_batch_r14, launch_batch_r15, launch_batch_r16};
static const shape_fn SHAPE_B4[MAXR + 1] = {
    nullptr,          shape_batch4_r1,  shape_batch4_r2,  shape_batch4_r3,  shape_batch4_r4,  shape_batch4_r5,
    shape_batch4_r6,  shape_batch4_r7,  shape_batch4_r8,  shape_batch4_r9,  shape_batch4_r10, shape_batch4_r11,
    shape_batch4_r12, shape_batch4_r13, shape_batch4_r14, shape_batch4_r15, shape_batch4_r16};
static const shape_fn SHAPE_B8[MAXR + 1] = {
    nullptr,          shape_batch8_r1,  shape_batch8_r2,  shape_batch8_r3,  shape_batch8_r4,  shape_batch8_r5,
    shape_batch8_r6,  shape_batch8_r7,  shape_batch8_r8,  shape_batch8_r9,  shape_batch8_r10, shape_batch8_r11,
    shape_batch8_r12, shape_batch8_r13, shape_batch8_r14, shape_batch8_r15, shape_batch8_r16};
static size_t batch_dyn(int64_t ntiles, int R, size_t esize, bool eval) { return batch_dyn_bytes(ntiles, R, esize, eval); }
static const shape_fn SHAPE[MAXR + 1] = {
    nullptr,          shape_filter_r1,  shape_filter_r2,  shape_filter_r3,  shape_filter_r4,  shape_filter_r5,
    shape_filter_r6,  shape_filter_r7,  shape_filter_r8,  shape_filter_r9,  shape_filter_r10, shape_filter_r11,
    shape_filter_r12, shape_filter_r13, shape_filter_r14, shape_filter_r15, shape_filter_r16};

// (n_series, d, R) row-major  <->  tiled [tile][R][32]
template <typename T>
__global__ void pack_C(const T* __restrict__ src, T* __restrict__ dst, int64_t d, int R, int64_t ntiles, int64_t total) {
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int l = (int)(idx % TILE);
        const int j = (int)((idx / TILE) % R);
        const int64_t tile = (idx / (TILE * (int64_t)R)) % ntiles;
        const int64_t s = idx / (TILE * (int64_t)R * ntiles);
        const int64_t row = tile * TILE + (l ^ ((j & 7) << 2));        // inverse of tile_pos (XOR swizzle)
        dst[idx] = row < d ? src[(s * d + row) * R + j] : (T)0;
    }
}
// F_RHO_VECTOR: caller's diag(R) (n_series, d) -> padded copy (whole tiles, 1.0 in the padding) + its mean per series;
// the state scalar rho becomes the scale (1.0)
__global__ void rho_pack(const double* __restrict__ src, double* __restrict__ dst, double* __restrict__ mean, double* __restrict__ state,
                         int64_t d, int64_t ld, int R) {
    __shared__ double red[256];
    const int s = blockIdx.x;
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < ld; i += blockDim.x) {
        const double v = i < d ? src[(int64_t)s * d + i] : 1.0;
        dst[(int64_t)s * ld + i] = v;
        acc += i < d ? v : 0.0;
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        mean[s] = red[0] / (double)d;
        state[(int64_t)s * st_size(R) + st_rho(R)] = 1.0;
    }
}
__global__ void rho_unpack(const double* __restrict__ src, const double* __restrict__ state, double* __restrict__ dst, int64_t d, int64_t ld, int R) {
    const int s = blockIdx.y;
    const double scale = state[(int64_t)s * st_size(R) + st_rho(R)];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < d; i += (int64_t)gridDim.x * blockDim.x)
        dst[(int64_t)s * d + i] = scale * src[(int64_t)s * ld + i];
}

template <typename T>
__global__ void unpack_C(const T* __restrict__ src, T* __restrict__ dst, int64_t d, int R, int64_t ntiles, int64_t total) {
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int l = (int)(idx % TILE);
        const int j = (int)((idx / TILE) % R);
        const int64_t tile = (idx / (TILE * (int64_t)R)) % ntiles;
        const int64_t s = idx / (TILE * (int64_t)R * ntiles);
        const int64_t row = tile * TILE + (l ^ ((j & 7) << 2));
        if (row < d) dst[(s * d + row) * R + j] = src[idx];
    }
}

}  // namespace psmf

using namespace psmf;

struct psmf_engine {
    psmf_config cfg;
    int R = 0;
    int S = 1;
    int64_t d = 0, ntiles = 0;
    size_t esize = 8;
    void* C = nullptr;
    double* state = nullptr;
    double* partials = nullptr;
    unsigned long long* bar = nullptr;
    double* gparams = nullptr;
    long long* status = nullptr;
    int cps = 1, threads = 0, launches_last = 0, num_sms = 0;
    size_t dyn_smem = 0;
    bool cooperative = false;
    // TMA-staged kernel configuration (cps2 == 0: not available for this shape)
    int cps2 = 0, threads2 = 0, nslot = 0;
    size_t dyn_smem2 = 0;
    bool resident2 = false;
    int last_kernel = 0;
    // resident batch kernel (one CTA per series, C in shared memory): available when the dictionary of a series fits
    bool batch_ok = false, batch_nw8 = false;
    int threads3 = 0;
    size_t dyn_smem3 = 0, last_dyn = 0;
    int maxsmem = 0;
    double* eval_part = nullptr;       // [S][cps][NEVAL] per-CTA evaluation sums of a launch
    double* stats_ext = nullptr;       // PSMF_XCHG_EXTERNAL: statistics of one step / residuals between the two launches
    double* e_ext = nullptr;
    double* rho_vec = nullptr;         // PSMF_RHO_VECTOR: caller's diag(R), (S, ntiles * 32) padded, and its mean per series
    double* rho_mean = nullptr;
    double* lin = nullptr;             // PSMF_DYN_LINEAR: A (R * R) then c (R)
    bool lin_set = false, lin_has_c = false;
    double* tool_buf = nullptr;        // scratch of psmf_eval_full / psmf_predict
    size_t tool_bytes = 0;
    unsigned long long* trace = nullptr;
    int trace_steps = 0;
    // NVLink mailbox (world_size > 1): [2 parities][MAX_PEERS][192] tagged 16-byte cells (psmf_filter.cuh gpu_exchange)
    void* mbox = nullptr;
    void* peer_mbox[PSMF_MAX_PEERS] = {nullptr};
    bool connected = false;
    int agreed_kernel = 0;             // world_size > 1: kernel all ranks agreed on in psmf_mailbox_connect (1 or 2)
    unsigned long long spin_ns = 10ULL * 1000000000ULL;   // bounded waits of the kernels (env PSMF_SPIN_TIMEOUT_MS)
    unsigned long long step_base = 0;
    cudaStream_t last_stream = nullptr;
    std::string err;
};

static std::string g_create_error;

static size_t mbox_bytes() { return (size_t)4 * PSMF_MAX_PEERS * MBOX_SLOT * 16; }   // [MBOX_DEPTH][peers] slots of MBOX_SLOT cells

static int fail(psmf_engine* h, int code, const std::string& msg) {
    if (h)
        h->err = msg;
    else
        g_create_error = msg;
    return code;
}
#define CK(h, call)                                                                                          \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess)                                                                              \
            return fail(h, PSMF_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));                \
    } while (0)

extern "C" int psmf_version(void) { return 200; }

extern "C" const char* psmf_last_error(psmf_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static void free_engine(psmf_engine* e) {
    if (!e) return;
    cudaFree(e->C);
    cudaFree(e->state);
    cudaFree(e->partials);
    cudaFree(e->bar);
    cudaFree(e->gparams);
    cudaFree(e->status);
    cudaFree(e->eval_part);
    cudaFree(e->stats_ext);
    cudaFree(e->e_ext);
    cudaFree(e->lin);
    cudaFree(e->rho_vec);
    cudaFree(e->rho_mean);
    cudaFree(e->tool_buf);
    for (int i = 0; i < PSMF_MAX_PEERS; ++i)
        if (e->peer_mbox[i] && i != e->cfg.rank) cudaIpcCloseMemHandle(e->peer_mbox[i]);
    cudaFree(e->mbox);
    delete e;
}

extern "C" int psmf_create(psmf_handle* out, const psmf_config* cfg) {
    if (!out || !cfg) return fail(nullptr, PSMF_E_INVALID, "null argument");
    *out = nullptr;
    if (cfg->r < 1 || cfg->r > PSMF_MAX_RANK) return fail(nullptr, PSMF_E_INVALID, "rank r must be in 1..16");
    if (cfg->d < 1) return fail(nullptr, PSMF_E_INVALID, "d must be >= 1");
    if (cfg->n_series < 1) return fail(nullptr, PSMF_E_INVALID, "n_series must be >= 1");
    if (cfg->dtype != PSMF_F64 && cfg->dtype != PSMF_F32) return fail(nullptr, PSMF_E_INVALID, "dtype must be PSMF_F64 or PSMF_F32");
    if (cfg->dynamics != PSMF_DYN_IDENTITY && cfg->dynamics != PSMF_DYN_COS && cfg->dynamics != PSMF_DYN_EXTERNAL &&
        cfg->dynamics != PSMF_DYN_LINEAR)
        return fail(nullptr, PSMF_E_INVALID, "unknown dynamics id");
    if (cfg->kernel < 0 || cfg->kernel > 3) return fail(nullptr, PSMF_E_INVALID, "kernel must be PSMF_KERNEL_AUTO / DIRECT / STREAM / BATCH");
    if (cfg->exchange != PSMF_XCHG_NVLINK && cfg->exchange != PSMF_XCHG_EXTERNAL)
        return fail(nullptr, PSMF_E_INVALID, "exchange must be PSMF_XCHG_NVLINK or PSMF_XCHG_EXTERNAL");
    if ((cfg->flags & PSMF_RHO_VECTOR) && (cfg->world_size > 1 || cfg->kernel == 2 || cfg->kernel == 3))
        return fail(nullptr, PSMF_E_INVALID, "PSMF_RHO_VECTOR (non-uniform diagonal R) runs on the direct-load kernel of one GPU: "
                                             "world_size 1, kernel AUTO or DIRECT");
    // the caller-driven exchange exists to shard one series by rows, which a non-uniform R does not support; its longer
    // statistics vector (nstat_v) would not fit the exchange buffer nor match the count psmf_stats_buffer reports
    if ((cfg->flags & PSMF_RHO_VECTOR) && cfg->exchange == PSMF_XCHG_EXTERNAL)
        return fail(nullptr, PSMF_E_INVALID, "PSMF_RHO_VECTOR (non-uniform diagonal R) runs on one GPU without row sharding: "
                                             "not with PSMF_XCHG_EXTERNAL");
    if ((cfg->flags & PSMF_GRAD_LINEAR) && cfg->dynamics != PSMF_DYN_LINEAR)
        return fail(nullptr, PSMF_E_INVALID, "PSMF_GRAD_LINEAR is the gradient with respect to A and c: it needs PSMF_DYN_LINEAR");
    if (cfg->exchange == PSMF_XCHG_EXTERNAL && cfg->n_series > 1)
        return fail(nullptr, PSMF_E_INVALID, "PSMF_XCHG_EXTERNAL shards ONE series by rows (n_series must be 1)");
    if (cfg->world_size < 1 || cfg->world_size > PSMF_MAX_PEERS || cfg->rank < 0 || cfg->rank >= cfg->world_size)
        return fail(nullptr, PSMF_E_INVALID, "bad world_size / rank");
    if (cfg->world_size > 1 && cfg->n_series > 1)
        return fail(nullptr, PSMF_E_INVALID, "row sharding (world_size > 1) and batching (n_series > 1) are exclusive");
    const int64_t dg = cfg->d_global > 0 ? cfg->d_global : cfg->d;
    if (dg < cfg->d) return fail(nullptr, PSMF_E_INVALID, "d_global < d");

    cudaError_t ce = cudaSetDevice(cfg->device);
    if (ce != cudaSuccess) return fail(nullptr, PSMF_E_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(ce));
    psmf_engine* e = new (std::nothrow) psmf_engine();
    if (!e) return fail(nullptr, PSMF_E_NOMEM, "host allocation failed");
    e->cfg = *cfg;
    e->cfg.d_global = dg;
    e->R = cfg->r;
    e->S = cfg->n_series;
    e->d = cfg->d;
    e->ntiles = (cfg->d + TILE - 1) / TILE;
    e->esize = cfg->dtype == PSMF_F64 ? 8 : 4;
    int sms = 0, maxsmem = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
    cudaDeviceGetAttribute(&maxsmem, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device);
    e->num_sms = sms;
    e->maxsmem = maxsmem;
    if (const char* ev = getenv("PSMF_SPIN_TIMEOUT_MS")) {              // how long a kernel waits for a silent peer GPU / CTA
        const long long ms = atoll(ev);
        if (ms >= 1) e->spin_ns = (unsigned long long)ms * 1000000ULL;
    }

    // ---- direct-load kernel: V1_WARPS warps per CTA, one staging tile per warp + the residual buffer ----
    int cps;
    if (e->S > 1) {
        cps = 1;
    } else if (cfg->ctas > 0) {
        cps = cfg->ctas;
    } else {
        int64_t want = e->ntiles / (2 * V1_WARPS);
        cps = (int)(want < 1 ? 1 : (want > sms ? sms : want));
    }
    if ((int64_t)cps > e->ntiles) cps = (int)e->ntiles;
    const size_t stage_bytes = (size_t)V1_WARPS * e->R * TILE * sizeof(double);
    LaunchShape shp;
    for (;;) {
        const int64_t tiles_per = (e->ntiles + cps - 1) / cps + 1;
        e->dyn_smem = stage_bytes + (size_t)tiles_per * TILE * sizeof(double);
        ce = ((cfg->flags & PSMF_RHO_VECTOR) ? SHAPE_V : SHAPE)[e->R](cfg->dtype, e->dyn_smem, &shp);
        if (ce == cudaSuccess && shp.max_ctas_per_sm >= 1) break;
        cudaGetLastError();
        // residual buffer does not fit: use more CTAs if allowed
        if (e->S == 1 && cfg->ctas <= 0 && cps < sms) {
            cps = cps * 2 > sms ? sms : cps * 2;
            continue;
        }
        free_engine(e);
        return fail(nullptr, PSMF_E_NOMEM, "d too large: per-CTA residual buffer exceeds shared memory");
    }
    // a forced grid larger than what fits on the device at once is cut to the co-resident count (cooperative launch);
    // fewer CTAs hold more tiles each, so the residual buffer is sized again for the grid that runs, until it is stable
    // (a larger buffer can lower the occupancy once more)
    while (e->S == 1 && cps > 1 && cps > sms * shp.max_ctas_per_sm) {
        cps = sms * shp.max_ctas_per_sm;
        const int64_t tiles_per = (e->ntiles + cps - 1) / cps + 1;
        e->dyn_smem = stage_bytes + (size_t)tiles_per * TILE * sizeof(double);
        ce = ((cfg->flags & PSMF_RHO_VECTOR) ? SHAPE_V : SHAPE)[e->R](cfg->dtype, e->dyn_smem, &shp);
        if (ce != cudaSuccess || shp.max_ctas_per_sm < 1) {
            cudaGetLastError();
            free_engine(e);
            return fail(nullptr, PSMF_E_NOMEM, "d too large: per-CTA residual buffer exceeds shared memory");
        }
    }
    e->cps = cps;
    e->threads = shp.threads;
    e->cooperative = cps > 1;

    // ---- TMA-staged kernel: slots of v2_ts(R, esize) tiles, residual buffer behind them ----
    if ((cfg->kernel == 0 || cfg->kernel == 2) && !(cfg->flags & PSMF_RHO_VECTOR) && cfg->exchange == PSMF_XCHG_NVLINK &&
        e->d % 16 == 0 && e->S == 1 && sms >= 2) {
        const int TS = v2_ts(e->R, (int)e->esize);
        auto r128 = [](size_t x) { return (x + 127) / 128 * 128; };
        const size_t slot = r128((size_t)TS * e->R * TILE * e->esize);     // psmf_stream.cuh SlotLayout: one chunk of C
        // data CTAs (one per SM) + one control CTA, all co-resident (cooperative launch)
        int cps2;
        if (cfg->ctas > 0) cps2 = cfg->ctas;
        else {
            int64_t want = e->ntiles / V2_CWARPS;                       // about one tile per pass warp and step
            cps2 = (int)(want < 1 ? 1 : want);
        }
        if ((int64_t)cps2 > e->ntiles) cps2 = (int)e->ntiles;
        if (cps2 > sms - 1) cps2 = sms - 1;
        if (cps2 > 256) cps2 = 256;                                    // control CTA sums <= 256 CTA partials per entry
        LaunchShape shp2;
        if (SHAPE_S[e->R](cfg->dtype, 0, &shp2) == cudaSuccess) {
            const int64_t tiles_max = (e->ntiles + cps2 - 1) / cps2;
            const int64_t nchunks_max = (tiles_max + TS - 1) / TS;
            const size_t ebuf = (size_t)tiles_max * TILE * sizeof(double);
            const int64_t avail = (int64_t)maxsmem - shp2.static_smem - (int64_t)ebuf - 256;
            int64_t nslot = avail > 0 ? avail / (int64_t)slot : 0;
            if (nslot > nchunks_max) nslot = nchunks_max;
            if (nslot > 64) nslot = 64;
#ifdef PSMF_DEBUG
            if (const char* ev = getenv("PSMF_NSLOT_MAX")) {            // debug knob (debug builds only)
                const int64_t cap = atoll(ev);
                if (cap >= 2 && nslot > cap) nslot = cap;
            }
#endif
            // a ring needs depth: with fewer than 5 slots the producer cannot keep loads, stores and the pass warps
            // apart (very large shards, where the residual buffer eats the shared memory) -> direct-load kernel
            const bool ring_ok = nchunks_max <= nslot || nslot >= 5;
            if (ring_ok && nslot >= (nchunks_max >= 2 ? 2 : 1)) {
                e->cps2 = cps2;
                e->nslot = (int)nslot;
                e->dyn_smem2 = (size_t)nslot * slot + ebuf;
                e->threads2 = shp2.threads;
                e->resident2 = nchunks_max <= nslot;
                if (SHAPE_S[e->R](cfg->dtype, e->dyn_smem2, &shp2) != cudaSuccess || shp2.max_ctas_per_sm < 1) e->cps2 = 0;
            }
        }
        cudaGetLastError();
    }
    if (cfg->kernel == 2 && e->cps2 == 0) {
        free_engine(e);
        return fail(nullptr, PSMF_E_INVALID, "TMA-staged kernel not available for this shape (needs d % 16 == 0, one series, and room for a ring of 5 chunk slots)");
    }
    // ---- resident batch kernel: one CTA per series, the whole dictionary of a series in shared memory ----
    if ((cfg->kernel == 0 || cfg->kernel == 3) && cfg->world_size == 1 && !(cfg->flags & PSMF_RHO_VECTOR)) {
        e->batch_nw8 = e->ntiles >= 8 && e->S <= 2 * sms;       // few series: more warps per series; many: more series per SM
        e->dyn_smem3 = batch_dyn(e->ntiles, e->R, e->esize, false);
        LaunchShape sb;
        if (e->dyn_smem3 <= (size_t)maxsmem &&
            (e->batch_nw8 ? SHAPE_B8 : SHAPE_B4)[e->R](cfg->dtype, e->dyn_smem3, &sb) == cudaSuccess && sb.max_ctas_per_sm >= 1) {
            e->batch_ok = true;
            e->threads3 = sb.threads;
        }
        cudaGetLastError();
    }
    if (cfg->kernel == 3 && !e->batch_ok) {
        free_engine(e);
        return fail(nullptr, PSMF_E_INVALID, "batch kernel not available: the dictionary of a series (d x r) must fit the shared memory of one CTA, world_size 1");
    }

    const size_t cbytes = (size_t)e->S * e->ntiles * TILE * e->R * e->esize;
    // >= nstat_pad(R): pipelined statistics (nstat2_pad), or the longer vector of a non-uniform diagonal R
    const int nsp = (cfg->flags & PSMF_RHO_VECTOR) ? nstat_v_pad(e->R) : (ngram(e->R) + 2 * e->R + 5 + 7) / 8 * 8;
#define CKC(call)                                                                                            \
    do {                                                                                                     \
        cudaError_t e__ = (call);                                                                            \
        if (e__ != cudaSuccess) {                                                                            \
            free_engine(e);                                                                                  \
            return fail(nullptr, e__ == cudaErrorMemoryAllocation ? PSMF_E_NOMEM : PSMF_E_CUDA,              \
                        std::string(#call) + ": " + cudaGetErrorString(e__));                                \
        }                                                                                                    \
    } while (0)
    CKC(cudaMalloc(&e->C, cbytes));
    CKC(cudaMemset(e->C, 0, cbytes));
    CKC(cudaMalloc(&e->state, (size_t)e->S * st_size(e->R) * sizeof(double)));
    CKC(cudaMemset(e->state, 0, (size_t)e->S * st_size(e->R) * sizeof(double)));
    {
        const int cmax = e->cps > e->cps2 ? e->cps : e->cps2;
        const size_t pstr = (size_t)((cmax + 7) & ~7) + 1;            // transposed partials + totals (grid_reduce)
        // direct kernel: doubles; pipelined kernel: [2][nstat2_pad][pstr] tagged 16-byte cells
        const size_t pbytes = (size_t)2 * nsp * (pstr > 17 ? pstr : 17) * 16;
        CKC(cudaMalloc(&e->partials, pbytes));
        CKC(cudaMemset(e->partials, 0, pbytes));
    }
    CKC(cudaMalloc(&e->bar, 8 * sizeof(unsigned long long)));
    CKC(cudaMalloc(&e->gparams, GPARAMS_BYTES));                        // 16-byte cells (psmf_stream.cuh): parameter sets [2][2R], totals [2][nstat2_pad]
    CKC(cudaMalloc(&e->status, sizeof(long long)));
    CKC(cudaMemset(e->status, 0xFF, sizeof(long long)));
    if (cfg->world_size > 1 && cfg->exchange == PSMF_XCHG_NVLINK) {
        CKC(cudaMalloc(&e->mbox, mbox_bytes()));
        CKC(cudaMemset(e->mbox, 0, mbox_bytes()));
    }
    if (cfg->exchange == PSMF_XCHG_EXTERNAL) {
        CKC(cudaMalloc(&e->stats_ext, (size_t)nstat_pad(MAXR) * sizeof(double)));
        CKC(cudaMemset(e->stats_ext, 0, (size_t)nstat_pad(MAXR) * sizeof(double)));
        CKC(cudaMalloc(&e->e_ext, (size_t)(e->ntiles + 1) * TILE * sizeof(double)));
        CKC(cudaMemset(e->e_ext, 0, (size_t)(e->ntiles + 1) * TILE * sizeof(double)));
    }
    CKC(cudaMalloc(&e->eval_part, (size_t)e->S * (e->cps > 1 ? e->cps : 1) * NEVAL * sizeof(double)));
    if (cfg->flags & PSMF_RHO_VECTOR) {
        CKC(cudaMalloc(&e->rho_vec, (size_t)e->S * e->ntiles * TILE * sizeof(double)));
        CKC(cudaMalloc(&e->rho_mean, (size_t)e->S * sizeof(double)));
    }
    CKC(cudaMalloc(&e->lin, (size_t)(e->R * e->R + e->R) * sizeof(double)));
    CKC(cudaMemset(e->lin, 0, (size_t)(e->R * e->R + e->R) * sizeof(double)));
#undef CKC
    *out = e;
    return PSMF_OK;
}

extern "C" int psmf_destroy(psmf_handle h) {
    if (!h) return PSMF_E_INVALID;
    cudaSetDevice(h->cfg.device);
    free_engine(h);
    return PSMF_OK;
}

static int copy_small(psmf_engine* h, bool set, double* user, int off, int n, cudaStream_t st) {
    if (!user) return PSMF_OK;
    const size_t pitch = (size_t)st_size(h->R) * sizeof(double);
    double* eng = h->state + off;
    if (set)
        CK(h, cudaMemcpy2DAsync(eng, pitch, user, n * sizeof(double), n * sizeof(double), h->S, cudaMemcpyDeviceToDevice, st));
    else
        CK(h, cudaMemcpy2DAsync(user, n * sizeof(double), eng, pitch, n * sizeof(double), h->S, cudaMemcpyDeviceToDevice, st));
    return PSMF_OK;
}

static int state_io(psmf_engine* h, bool set, void* C, double* V, double* P, double* x, double* Q, double* rho,
                    double* lambda, double* theta, cudaStream_t st) {
    if (!h) return PSMF_E_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    const int R = h->R;
    if (C) {
        const int64_t total = (int64_t)h->S * h->ntiles * TILE * R;
        const int blocks = (int)((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256);
        if (h->cfg.dtype == PSMF_F64) {
            if (set) pack_C<double><<<blocks, 256, 0, st>>>((const double*)C, (double*)h->C, h->d, R, h->ntiles, total);
            else unpack_C<double><<<blocks, 256, 0, st>>>((const double*)h->C, (double*)C, h->d, R, h->ntiles, total);
        } else {
            if (set) pack_C<float><<<blocks, 256, 0, st>>>((const float*)C, (float*)h->C, h->d, R, h->ntiles, total);
            else unpack_C<float><<<blocks, 256, 0, st>>>((const float*)h->C, (float*)C, h->d, R, h->ntiles, total);
        }
        CK(h, cudaGetLastError());
    }
    int rc;
    if ((rc = copy_small(h, set, x, st_x(R), R, st))) return rc;
    if ((rc = copy_small(h, set, P, st_P(R), R * R, st))) return rc;
    if ((rc = copy_small(h, set, V, st_V(R), R * R, st))) return rc;
    if ((rc = copy_small(h, set, Q, st_Q(R), R * R, st))) return rc;
    if ((rc = copy_small(h, set, theta, st_theta(R), R, st))) return rc;
    if (rho && (h->cfg.flags & PSMF_RHO_VECTOR)) {
        // diag(R) as a vector per series: the engine keeps the caller's vector and a scalar scale (R <- omega R, rPSMF.py:134)
        const int64_t ld = h->ntiles * TILE;
        if (set) {
            rho_pack<<<h->S, 256, 0, st>>>(rho, h->rho_vec, h->rho_mean, h->state, h->d, ld, R);
        } else {
            dim3 grid((unsigned)((h->d + 255) / 256 > 1024 ? 1024 : (h->d + 255) / 256), (unsigned)h->S);
            rho_unpack<<<grid, 256, 0, st>>>(h->rho_vec, h->state, rho, h->d, ld, R);
        }
        CK(h, cudaGetLastError());
    } else if ((rc = copy_small(h, set, rho, st_rho(R), 1, st))) return rc;
    if ((rc = copy_small(h, set, lambda, st_lam(R), 1, st))) return rc;
    return PSMF_OK;
}

extern "C" int psmf_set_state(psmf_handle h, const void* C, const double* V, const double* P, const double* x,
                              const double* Q, const double* rho, const double* lambda, const double* theta, void* stream) {
    return state_io(h, true, const_cast<void*>(C), const_cast<double*>(V), const_cast<double*>(P), const_cast<double*>(x),
                    const_cast<double*>(Q), const_cast<double*>(rho), const_cast<double*>(lambda),
                    const_cast<double*>(theta), (cudaStream_t)stream);
}

extern "C" int psmf_get_state(psmf_handle h, void* C, double* V, double* P, double* x, double* Q, double* rho,
                              double* lambda, double* theta, void* stream) {
    return state_io(h, false, C, V, P, x, Q, rho, lambda, theta, (cudaStream_t)stream);
}

static int run_impl(psmf_handle h, const psmf_io* io, int64_t n_steps, int64_t k0, void* stream, int phase) {
    if (!h || !io) return PSMF_E_INVALID;
    if (n_steps < 1) return fail(h, PSMF_E_INVALID, "n_steps must be >= 1");
    if (!io->Y) return fail(h, PSMF_E_INVALID, "Y is NULL");
    if (io->ldy < h->d) return fail(h, PSMF_E_INVALID, "ldy < d");
    if (io->M && io->ldm < h->d) return fail(h, PSMF_E_INVALID, "ldm < d");
    if (io->M && (h->cfg.flags & PSMF_NAN_MASK)) return fail(h, PSMF_E_INVALID, "PSMF_NAN_MASK: the mask is encoded in Y, M must be NULL");
    if (io->Yrec_out && io->ldrec < h->d) return fail(h, PSMF_E_INVALID, "ldrec < d");
    const bool eval = io->E != nullptr;
    if (eval && (!io->Yorig || !io->eval_out || io->lde < h->d))
        return fail(h, PSMF_E_INVALID, "fused evaluation needs E (lde >= d), Yorig and eval_out together");
    if (h->cfg.dynamics == PSMF_DYN_EXTERNAL) {
        if (n_steps != 1) return fail(h, PSMF_E_INVALID, "PSMF_DYN_EXTERNAL runs one step per call");
        if (!io->xbar_ext || (!io->F_ext && !(h->cfg.flags & PSMF_SIMPLIFIED)))
            return fail(h, PSMF_E_INVALID, "PSMF_DYN_EXTERNAL needs xbar_ext and F_ext");
    }
    if (h->cfg.dynamics == PSMF_DYN_LINEAR && !h->lin_set)
        return fail(h, PSMF_E_STATE, "PSMF_DYN_LINEAR: call psmf_set_linear_dynamics first");
    const bool external = h->cfg.exchange == PSMF_XCHG_EXTERNAL;
    if (external) {
        if (n_steps != 1) return fail(h, PSMF_E_INVALID, "PSMF_XCHG_EXTERNAL runs one step per psmf_run / psmf_run_finish pair");
        if (eval) return fail(h, PSMF_E_INVALID, "fused evaluation is not available with PSMF_XCHG_EXTERNAL");
    } else if (phase != 0) {
        return fail(h, PSMF_E_STATE, "psmf_run_finish needs an engine created with PSMF_XCHG_EXTERNAL");
    }
    cudaStream_t st = (cudaStream_t)stream;
    CK(h, cudaSetDevice(h->cfg.device));
    KParams p;
    memset(&p, 0, sizeof(p));
    p.C = h->C;
    p.c_series_stride = h->ntiles * TILE * h->R;
    p.state = h->state;
    p.Y = io->Y; p.ldy = io->ldy; p.ysst = io->y_series_stride;
    p.M = io->M; p.ldm = io->ldm; p.msst = io->m_series_stride;
    p.X_out = io->X_out;
    p.Yrec = io->Yrec_out; p.ldrec = io->ldrec; p.recsst = io->rec_series_stride;
    p.scal_out = io->scal_out;
    p.xbar_ext = io->xbar_ext; p.F_ext = io->F_ext;
    p.grad_out = io->grad_out;
    p.partials = h->partials;
    p.bar = h->bar;
    p.status = h->status;
    p.d = h->d; p.d_global = h->cfg.d_global;
    p.n_steps = n_steps; p.k0 = k0;
    p.n_series = h->S; p.cps = h->cps;
    p.flags = h->cfg.flags; p.dynamics = h->cfg.dynamics;
#ifdef PSMF_DEBUG
    if (const char* ev = getenv("PSMF_DEBUG_FLAGS")) p.flags |= (int)strtol(ev, nullptr, 0) & (7 << 20);
#endif
    p.spin_ns = h->spin_ns;
    p.alpha = h->cfg.alpha; p.beta = h->cfg.beta;
    p.world = external ? 1 : h->cfg.world_size; p.rank = h->cfg.rank;
    p.phase = phase;
    p.stats_ext = h->stats_ext; p.e_ext = h->e_ext;
    p.lin_A = h->lin; p.lin_c = h->lin_has_c ? h->lin + h->R * h->R : nullptr;
    p.rho_vec = h->rho_vec; p.rho_sst = h->ntiles * TILE; p.rho_mean = h->rho_mean;
    if (eval) {
        p.Yorig = io->Yorig; p.E = io->E; p.lde = io->lde; p.esst = io->e_series_stride; p.sig = io->sig;
        p.eval_part = h->eval_part;
    }
    if (p.world > 1) {
        if (!h->connected) return fail(h, PSMF_E_STATE, "world_size > 1: call psmf_mailbox_connect before psmf_run");
        p.mbox_local = (double*)h->mbox;
        for (int i = 0; i < p.world; ++i) {
            p.mbox_peer[i] = (double*)h->peer_mbox[i];
        }
    }
    p.step_base = h->step_base;       // steps filtered by this engine so far: tags of the mailbox / partial cells
    p.trace = h->trace; p.trace_steps = h->trace_steps;
    CK(h, cudaMemsetAsync(h->bar, 0, 8 * sizeof(unsigned long long), st));
    CK(h, cudaMemsetAsync(h->gparams, 0, GPARAMS_BYTES, st));
    if (phase != 2) CK(h, cudaMemsetAsync(h->status, 0xFF, sizeof(long long), st));
    // ---- which kernel ----
    // the resident batch kernel: independent series / one small series, C in shared memory for the whole launch
    bool use3 = h->batch_ok && !external &&
                (h->cfg.kernel == 3 || (h->cfg.kernel == 0 && h->cfg.ctas <= 0 && (h->S > 1 || h->ntiles <= 32)));
    size_t dyn3 = h->dyn_smem3;
    // PSMF_GRAD_LINEAR: the accumulator G_A (R * R doubles) goes behind the other dynamic shared memory of the direct-load and
    // batch kernels; the TMA-staged control CTA keeps it in its own dynamic shared memory, which is at least one chunk slot
    // (>= 512 R bytes > 8 R^2)
    const size_t glin = (h->cfg.flags & PSMF_GRAD_LINEAR) ? (size_t)h->R * h->R * sizeof(double) : 0;
    if (use3 && (eval || glin)) {
        dyn3 = batch_dyn(h->ntiles, h->R, h->esize, eval);
        p.glin_off = (int64_t)dyn3;
        dyn3 += glin;
        LaunchShape sb;
        if (dyn3 > (size_t)h->maxsmem ||
            (h->batch_nw8 ? SHAPE_B8 : SHAPE_B4)[h->R](h->cfg.dtype, dyn3, &sb) != cudaSuccess || sb.max_ctas_per_sm < 1) {
            cudaGetLastError();
            if (h->cfg.kernel == 3)
                return fail(h, PSMF_E_NOMEM, "batch kernel: no shared memory left for the evaluation buffers / the gradient accumulator");
            use3 = false;
        }
    }
    // the TMA-staged kernel needs 16-byte aligned rows of Y / M (bulk copies)
    const size_t es = h->esize;
    bool aligned = h->cps2 > 0 && ((uintptr_t)io->Y % 16 == 0) && ((size_t)io->ldy * es % 16 == 0) &&
                   ((size_t)io->y_series_stride * es % 16 == 0);
    if (io->M) aligned = aligned && ((uintptr_t)io->M % 16 == 0) && (io->ldm % 16 == 0) && (io->m_series_stride % 16 == 0);
    bool use2 = !use3 && aligned && !eval && !external && h->cfg.dynamics != PSMF_DYN_EXTERNAL &&
                (h->cfg.kernel == 2 || (h->cfg.kernel == 0 && h->ntiles >= 2 * (V2_CWARPS + 1)));
    if (h->cfg.kernel == 2 && !use2)
        return fail(h, PSMF_E_INVALID, "kernel=2 requested but Y/M are not 16-byte aligned, dynamics is external, or fused "
                                       "evaluation was requested (direct-load / batch kernels only)");
    if (p.world > 1) {
        // row sharding: the kernel is a collective decision (psmf_mailbox_connect) -- the two kernels exchange
        // different statistics vectors, so a rank must never pick one from local facts alone
        if (eval) return fail(h, PSMF_E_INVALID, "fused evaluation is per GPU: not available with row sharding");
        if (h->agreed_kernel == 2 && !aligned)
            return fail(h, PSMF_E_INVALID, "the ranks agreed on the TMA-staged kernel but this rank's Y/M are not 16-byte aligned "
                                           "(pad ldy/ldm to a multiple of 16 bytes, or create every engine with kernel=1)");
        use2 = h->agreed_kernel == 2;
    }
    if (use3) {
        p.cps = 1;
        CK(h, LAUNCH_B[h->R](p, h->cfg.dtype, h->S, dyn3, st, h->batch_nw8));
        h->last_kernel = 3;
        h->last_dyn = dyn3;
    } else if (use2) {
        p.cps = h->cps2;
        p.nslot = h->nslot;
        p.glin_off = 0;                   // G_A at the start of the control CTA's dynamic shared memory
        p.trace_cta = h->cps2;
        // streaming from HBM: 12 of the 14 pass warps (3 per scheduler; a multiple of the 4 tiles of a chunk) keep up
        // with the ring and leave issue slots to the producer -- measured optimum at r = 16 under the power cap;
        // resident in shared memory: every warp helps
        // fp32 storage halves the bytes per tile: the pass is bound by the fp64 pipe, not by the ring -> all 14 warps
        p.npw = (h->resident2 || h->cfg.dtype == PSMF_F32) ? V2_CWARPS : 12;
#ifdef PSMF_DEBUG
        if (const char* ev = getenv("PSMF_NPW")) { const int v = atoi(ev); if (v >= 1 && v <= V2_CWARPS) p.npw = v; }
#endif
        p.gparams = h->gparams;
        CK(h, LAUNCH_S[h->R](p, h->cfg.dtype, h->cps2 + 1, h->dyn_smem2, st, true));
        h->last_kernel = 2;
        h->last_dyn = h->dyn_smem2;
    } else {
        size_t dyn1 = h->dyn_smem;
        if (eval || glin) {
            const int64_t tiles_per = (h->ntiles + h->cps - 1) / h->cps + 1;
            if (eval) dyn1 += (size_t)tiles_per * TILE * 17 + 16;
            p.glin_off = (int64_t)dyn1;
            dyn1 += glin;
            LaunchShape sh1;
            if (((h->cfg.flags & PSMF_RHO_VECTOR) ? SHAPE_V : SHAPE)[h->R](h->cfg.dtype, dyn1, &sh1) != cudaSuccess || sh1.max_ctas_per_sm < 1 ||
                (h->cooperative && h->cps > h->num_sms * sh1.max_ctas_per_sm)) {
                cudaGetLastError();
                return fail(h, PSMF_E_NOMEM, "no shared memory left for the evaluation buffers / the gradient accumulator at this d / grid");
            }
        }
        CK(h, ((h->cfg.flags & PSMF_RHO_VECTOR) ? LAUNCH_V : LAUNCH)[h->R](p, h->cfg.dtype, h->S * h->cps, dyn1, st, h->cooperative));
        h->last_kernel = 1;
        h->last_dyn = dyn1;
    }
    if (eval) {
        eval_part_finish<<<h->S, 32, 0, st>>>(h->eval_part, p.cps, io->eval_out);
        CK(h, cudaGetLastError());
    }
    h->launches_last = eval ? 2 : 1;
    h->last_stream = st;
    if (phase != 1) h->step_base += (unsigned long long)n_steps;
    return PSMF_OK;
}

extern "C" int psmf_run(psmf_handle h, const psmf_io* io, int64_t n_steps, int64_t k0, void* stream) {
    if (!h) return PSMF_E_INVALID;
    return run_impl(h, io, n_steps, k0, stream, h->cfg.exchange == PSMF_XCHG_EXTERNAL ? 1 : 0);
}

extern "C" int psmf_run_finish(psmf_handle h, const psmf_io* io, int64_t k0, void* stream) {
    if (!h) return PSMF_E_INVALID;
    return run_impl(h, io, 1, k0, stream, 2);
}

extern "C" int psmf_stats_buffer(psmf_handle h, double** dev_ptr, int32_t* count) {
    if (!h || !dev_ptr || !count) return PSMF_E_INVALID;
    if (!h->stats_ext) return fail(h, PSMF_E_STATE, "engine was not created with PSMF_XCHG_EXTERNAL");
    *dev_ptr = h->stats_ext;
    *count = nstat(h->R);
    return PSMF_OK;
}

extern "C" int psmf_set_linear_dynamics(psmf_handle h, const double* A, const double* c, void* stream) {
    if (!h || !A) return PSMF_E_INVALID;
    if (h->cfg.dynamics != PSMF_DYN_LINEAR) return fail(h, PSMF_E_STATE, "engine was not created with PSMF_DYN_LINEAR");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    CK(h, cudaMemcpyAsync(h->lin, A, (size_t)h->R * h->R * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (c) CK(h, cudaMemcpyAsync(h->lin + h->R * h->R, c, (size_t)h->R * sizeof(double), cudaMemcpyDeviceToDevice, st));
    h->lin_set = true;
    h->lin_has_c = c != nullptr;
    return PSMF_OK;
}

static int tool_scratch(psmf_engine* h, size_t bytes) {
    if (h->tool_bytes >= bytes) return PSMF_OK;
    cudaFree(h->tool_buf);
    h->tool_buf = nullptr;
    h->tool_bytes = 0;
    CK(h, cudaMalloc(&h->tool_buf, bytes));
    h->tool_bytes = bytes;
    return PSMF_OK;
}

extern "C" int psmf_predict(psmf_handle h, int64_t n_pred, int64_t k0, const double* Xpred_in, double* Xpred_out, void* Ypred_out,
                            int64_t ldp, int64_t pred_series_stride, void* stream) {
    if (!h) return PSMF_E_INVALID;
    if (n_pred < 1) return fail(h, PSMF_E_INVALID, "n_pred must be >= 1");
    if (Ypred_out && ldp < h->d) return fail(h, PSMF_E_INVALID, "ldp < d");
    if (h->cfg.dynamics == PSMF_DYN_EXTERNAL && !Xpred_in)
        return fail(h, PSMF_E_INVALID, "PSMF_DYN_EXTERNAL: the caller owns f, pass the rolled-out states in Xpred_in");
    if (h->cfg.dynamics == PSMF_DYN_LINEAR && !h->lin_set && !Xpred_in)
        return fail(h, PSMF_E_STATE, "PSMF_DYN_LINEAR: call psmf_set_linear_dynamics first");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const double* Xp = Xpred_in;
    if (!Xp) {
        double* dst = Xpred_out;
        if (!dst) {
            int rc = tool_scratch(h, (size_t)h->S * n_pred * h->R * sizeof(double));
            if (rc) return rc;
            dst = h->tool_buf;
        }
        rollout_kernel<<<h->S, 32, 0, st>>>(h->state, h->R, h->cfg.dynamics, h->lin, h->lin_has_c ? h->lin + h->R * h->R : nullptr, k0,
                                           n_pred, dst);
        CK(h, cudaGetLastError());
        Xp = dst;
    } else if (Xpred_out && Xpred_out != Xpred_in) {
        CK(h, cudaMemcpyAsync(Xpred_out, Xpred_in, (size_t)h->S * n_pred * h->R * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    if (Ypred_out) {
        const int64_t groups = (h->ntiles + TOOL_WARPS - 1) / TOOL_WARPS;
        dim3 grid((unsigned)(groups > 1024 ? 1024 : groups), (unsigned)h->S);
        if (h->cfg.dtype == PSMF_F64)
            project_kernel<double><<<grid, TOOL_WARPS * 32, 0, st>>>((const double*)h->C, h->ntiles * TILE * h->R, h->d, h->R, Xp, n_pred,
                                                                    (double*)Ypred_out, ldp, pred_series_stride);
        else
            project_kernel<float><<<grid, TOOL_WARPS * 32, 0, st>>>((const float*)h->C, h->ntiles * TILE * h->R, h->d, h->R, Xp, n_pred,
                                                                   (float*)Ypred_out, ldp, pred_series_stride);
        CK(h, cudaGetLastError());
    }
    h->last_stream = st;
    return PSMF_OK;
}

extern "C" int psmf_eval_full(psmf_handle h, const double* X, int64_t n_steps, const void* Yorig, int64_t ldy, int64_t y_series_stride,
                              const uint8_t* E, int64_t lde, int64_t e_series_stride, double* out, void* stream) {
    if (!h || !X || !Yorig || !E || !out) return PSMF_E_INVALID;
    if (n_steps < 1 || ldy < h->d || lde < h->d) return fail(h, PSMF_E_INVALID, "bad n_steps / ldy / lde");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t groups = (h->ntiles + TOOL_WARPS - 1) / TOOL_WARPS;
    const int nparts = (int)(groups > 256 ? 256 : groups);
    int rc = tool_scratch(h, (size_t)h->S * nparts * 2 * sizeof(double));
    if (rc) return rc;
    dim3 grid((unsigned)nparts, (unsigned)h->S);
    if (h->cfg.dtype == PSMF_F64)
        eval_full_kernel<double><<<grid, TOOL_WARPS * 32, 0, st>>>((const double*)h->C, h->ntiles * TILE * h->R, h->d, h->R, X, n_steps,
                                                                  (const double*)Yorig, ldy, y_series_stride, E, lde, e_series_stride, h->tool_buf);
    else
        eval_full_kernel<float><<<grid, TOOL_WARPS * 32, 0, st>>>((const float*)h->C, h->ntiles * TILE * h->R, h->d, h->R, X, n_steps,
                                                                 (const float*)Yorig, ldy, y_series_stride, E, lde, e_series_stride, h->tool_buf);
    CK(h, cudaGetLastError());
    eval_full_finish<<<h->S, 32, 0, st>>>(h->tool_buf, nparts, out);
    CK(h, cudaGetLastError());
    h->last_stream = st;
    return PSMF_OK;
}

// ---- handle-free tools: ingest and the missing-segment generator ------------------------------------------------
static int tool_fail(cudaError_t e, const char* what) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(e);
    return PSMF_E_CUDA;
}
#define TCK(call)                                                     \
    do {                                                              \
        cudaError_t e__ = (call);                                     \
        if (e__ != cudaSuccess) return tool_fail(e__, #call);         \
    } while (0)

extern "C" int psmf_ingest(int32_t device, const double* src, int64_t d, int64_t n, int32_t dtype, int32_t keep_nan, void* Y_out,
                           int64_t ldy, uint8_t* M_out, int64_t ldm, void* stream) {
    if (!src || d < 1 || n < 1 || (!Y_out && !M_out) || (Y_out && ldy < d) || (M_out && ldm < d) ||
        (dtype != PSMF_F64 && dtype != PSMF_F32))
        return fail(nullptr, PSMF_E_INVALID, "psmf_ingest: bad arguments");
    TCK(cudaSetDevice(device));
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((d + 31) / 32)), block(32, 8);
    if (grid.y > 65535) return fail(nullptr, PSMF_E_INVALID, "psmf_ingest: d too large for one call (split the rows)");
    const int mode = keep_nan ? INGEST_KEEP_NAN : 0;
    if (dtype == PSMF_F64)
        ingest_kernel<double><<<grid, block, 0, (cudaStream_t)stream>>>(src, d, n, mode, (double*)Y_out, ldy, M_out, ldm);
    else
        ingest_kernel<float><<<grid, block, 0, (cudaStream_t)stream>>>(src, d, n, mode, (float*)Y_out, ldy, M_out, ldm);
    TCK(cudaGetLastError());
    return PSMF_OK;
}

extern "C" int psmf_transpose_mask(int32_t device, const uint8_t* src, int64_t d, int64_t n, uint8_t* dst, int64_t ld, void* stream) {
    if (!src || !dst || d < 1 || n < 1 || ld < d) return fail(nullptr, PSMF_E_INVALID, "psmf_transpose_mask: bad arguments");
    TCK(cudaSetDevice(device));
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((d + 31) / 32)), block(32, 8);
    if (grid.y > 65535) return fail(nullptr, PSMF_E_INVALID, "psmf_transpose_mask: d too large for one call (split the rows)");
    transpose_mask_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(src, d, n, dst, ld);
    TCK(cudaGetLastError());
    return PSMF_OK;
}

extern "C" int psmf_missing_segments(int32_t device, int32_t dtype, void* Y, int64_t ldy, uint8_t* E, int64_t lde, int64_t d, int64_t n,
                                     const int64_t* starts, int32_t seg, uint64_t* count_dev, void* stream) {
    if (!Y || !E || !starts || !count_dev || d < 1 || n < 1 || ldy < d || lde < d || seg < 1 || (dtype != PSMF_F64 && dtype != PSMF_F32))
        return fail(nullptr, PSMF_E_INVALID, "psmf_missing_segments: bad arguments");
    TCK(cudaSetDevice(device));
    const unsigned blocks = (unsigned)((d + 255) / 256);
    if (dtype == PSMF_F64)
        missing_segments_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((double*)Y, ldy, E, lde, d, n, starts, seg,
                                                                                 (unsigned long long*)count_dev);
    else
        missing_segments_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((float*)Y, ldy, E, lde, d, n, starts, seg,
                                                                                (unsigned long long*)count_dev);
    TCK(cudaGetLastError());
    return PSMF_OK;
}

extern "C" int psmf_count_nan(int32_t device, int32_t dtype, const void* Y, int64_t ldy, int64_t d, int64_t n, uint64_t* count_dev,
                              void* stream) {
    if (!Y || !count_dev || d < 1 || n < 1 || ldy < d || (dtype != PSMF_F64 && dtype != PSMF_F32))
        return fail(nullptr, PSMF_E_INVALID, "psmf_count_nan: bad arguments");
    TCK(cudaSetDevice(device));
    const int64_t total = d * n;
    const unsigned blocks = (unsigned)((total + 255) / 256 > 2048 ? 2048 : (total + 255) / 256);
    if (dtype == PSMF_F64)
        count_nan_kernel<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double*)Y, ldy, d, n, (unsigned long long*)count_dev);
    else
        count_nan_kernel<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)Y, ldy, d, n, (unsigned long long*)count_dev);
    TCK(cudaGetLastError());
    return PSMF_OK;
}

extern "C" int psmf_status(psmf_handle h, int64_t* first_bad_step) {
    if (!h) return PSMF_E_INVALID;
    CK(h, cudaSetDevice(h->cfg.device));
    CK(h, cudaStreamSynchronize(h->last_stream));
    long long v = -1;
    CK(h, cudaMemcpy(&v, h->status, sizeof(v), cudaMemcpyDeviceToHost));
    if (v >= 0 && (v & (STATUS_TIMEOUT | STATUS_MISMATCH)) != 0) {
        const long long step = v & 0xFFFFFFFFFFFFLL;
        if (first_bad_step) *first_bad_step = (int64_t)step;
        if (v & STATUS_TIMEOUT) {
            static const char* const SITE[] = {"?", "tagged cell", "NVLink mailbox (peer GPU)", "mbarrier", "grid barrier",
                                               "chunk ring", "CTA partials"};
            const int where = (int)((v >> 48) & 0xFF);
            char buf[256];
            snprintf(buf, sizeof(buf), "a kernel wait made no progress for %.1f s at step %lld (%s): a peer GPU or CTA is gone; "
                     "the results of this launch are invalid", (double)h->spin_ns * 1e-9, step, SITE[where < 7 ? where : 0]);
            return fail(h, PSMF_E_STATE, buf);
        }
        return fail(h, PSMF_E_STATE, "a peer GPU runs a different kernel / statistics layout (mailbox header mismatch at step " +
                                         std::to_string(step) + ")");
    }
    if (first_bad_step) *first_bad_step = (int64_t)v;
    return PSMF_OK;
}

extern "C" int psmf_launch_info(psmf_handle h, int32_t* ctas, int32_t* threads, int32_t* smem_bytes, int32_t* launches) {
    if (!h) return PSMF_E_INVALID;
    const int k = h->last_kernel;
    if (ctas) *ctas = k == 2 ? h->cps2 + 1 : (k == 3 ? 1 : h->cps);
    if (threads) *threads = k == 2 ? h->threads2 : (k == 3 ? h->threads3 : h->threads);
    if (smem_bytes) *smem_bytes = (int32_t)h->last_dyn;
    if (launches) *launches = h->launches_last;
    return PSMF_OK;
}

extern "C" int psmf_launch_info2(psmf_handle h, int32_t* kernel, int32_t* nslot, int32_t* resident) {
    if (!h) return PSMF_E_INVALID;
    if (kernel) *kernel = h->last_kernel;
    if (nslot) *nslot = h->last_kernel == 2 ? h->nslot : 0;
    if (resident) *resident = h->last_kernel == 2 && h->resident2 ? 1 : 0;
    return PSMF_OK;
}

extern "C" int psmf_set_trace(psmf_handle h, uint64_t* dev_buf, int32_t steps) {
    if (!h) return PSMF_E_INVALID;
    h->trace = (unsigned long long*)dev_buf;
    h->trace_steps = dev_buf ? steps : 0;
    return PSMF_OK;
}

// Plan record that travels with the IPC handle (bytes 64..127 of the blob): every rank sees every record and
// derives the same decision from them, so the ranks can never run different kernels against each other.
struct plan_record {
    int32_t version, r, dtype, flags, dynamics, world, kernel_pref, eligible2, auto2, rank;
    int64_t d_global;
    int32_t pad[4];
};
static_assert(sizeof(plan_record) <= 64, "plan record must fit the second half of the blob");

static plan_record make_plan(const psmf_engine* h) {
    plan_record r;
    memset(&r, 0, sizeof(r));
    r.version = psmf_version();
    r.r = h->R; r.dtype = h->cfg.dtype; r.flags = h->cfg.flags; r.dynamics = h->cfg.dynamics; r.world = h->cfg.world_size;
    r.kernel_pref = h->cfg.kernel; r.rank = h->cfg.rank; r.d_global = h->cfg.d_global;
    r.eligible2 = (h->cps2 > 0 && h->cfg.dynamics != PSMF_DYN_EXTERNAL) ? 1 : 0;
    r.auto2 = (r.eligible2 && h->ntiles >= 2 * (V2_CWARPS + 1)) ? 1 : 0;
    return r;
}

extern "C" int psmf_mailbox_export(psmf_handle h, void* blob_128B) {
    if (!h || !blob_128B) return PSMF_E_INVALID;
    if (h->cfg.world_size < 2 || !h->mbox) return fail(h, PSMF_E_STATE, "engine was created with world_size == 1");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(h, cudaSetDevice(h->cfg.device));
    cudaIpcMemHandle_t hd;
    CK(h, cudaIpcGetMemHandle(&hd, h->mbox));
    memset(blob_128B, 0, PSMF_MAILBOX_BLOB_BYTES);
    memcpy(blob_128B, &hd, sizeof(hd));
    const plan_record pr = make_plan(h);
    memcpy((char*)blob_128B + 64, &pr, sizeof(pr));
    return PSMF_OK;
}

extern "C" int psmf_mailbox_connect(psmf_handle h, const void* all_blobs, int32_t n) {
    if (!h || !all_blobs) return PSMF_E_INVALID;
    if (n != h->cfg.world_size || n < 2) return fail(h, PSMF_E_INVALID, "need one blob per rank");
    CK(h, cudaSetDevice(h->cfg.device));
    const char* blobs = (const char*)all_blobs;
    // ---- collective plan: same inputs on every rank -> same decision on every rank ----
    const plan_record mine = make_plan(h);
    bool any_forced1 = false, any_forced2 = false, all_eligible2 = true, all_auto2 = true;
    for (int i = 0; i < n; ++i) {
        plan_record pr;
        memcpy(&pr, blobs + (size_t)i * PSMF_MAILBOX_BLOB_BYTES + 64, sizeof(pr));
        if (pr.version != mine.version || pr.r != mine.r || pr.dtype != mine.dtype || pr.flags != mine.flags ||
            pr.dynamics != mine.dynamics || pr.world != mine.world || pr.d_global != mine.d_global || pr.rank != i)
            return fail(h, PSMF_E_INVALID, "rank " + std::to_string(i) + " was created with a different configuration "
                                           "(version / r / dtype / flags / dynamics / world_size / d_global / rank order)");
        any_forced1 = any_forced1 || pr.kernel_pref == 1;
        any_forced2 = any_forced2 || pr.kernel_pref == 2;
        all_eligible2 = all_eligible2 && pr.eligible2 != 0;
        all_auto2 = all_auto2 && (pr.auto2 != 0 || (pr.kernel_pref == 2 && pr.eligible2 != 0));
    }
    if (any_forced1 && any_forced2) return fail(h, PSMF_E_INVALID, "ranks disagree: kernel=1 and kernel=2 were both forced");
    if (any_forced2 && !all_eligible2)
        return fail(h, PSMF_E_INVALID, "kernel=2 was forced but not every rank's shard is eligible for the TMA-staged kernel");
    h->agreed_kernel = any_forced2 ? 2 : (any_forced1 ? 1 : (all_auto2 ? 2 : 1));
    for (int i = 0; i < n; ++i) {
        if (i == h->cfg.rank) {
            h->peer_mbox[i] = h->mbox;
            continue;
        }
        cudaIpcMemHandle_t hd;
        memcpy(&hd, blobs + (size_t)i * PSMF_MAILBOX_BLOB_BYTES, sizeof(hd));
        void* ptr = nullptr;
        CK(h, cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
        h->peer_mbox[i] = ptr;
    }
    h->connected = true;
    return PSMF_OK;
}
