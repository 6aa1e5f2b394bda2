// music_b200.cu - C-ABI shim (include/music_b200.h) over the sm_100a MUSIC DOA kernels.
//
// Host-side responsibilities only: argument checks (the reference's constructor asserts,
// /root/reference/lib/baz_music_doa.cc:45-50, made real), device buffers, the steering-table
// double buffer (set_array_response semantics, :60-70), chunking and host<->device staging.
// No CPU compute path exists here: without an sm_100 device create() fails.
#include "../../include/music_b200.h"

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "music_kernels.cuh"
#include "music_fused.cuh"
#include "music_covn.cuh"
#include "music_fused8.cuh"
#include "music_steer.cuh"
#include "music_planar.cuh"
#include "music_reduce.cuh"

using namespace music;

namespace {

std::mutex g_err_mutex;
std::string g_create_error;

struct DeviceTable {
    float *c64 = nullptr;   // [K][M] (re, im)
    double *soa = nullptr;  // [ntiles][2M+1][TILE]
    unsigned char *fz = nullptr;  // fused kernel's tensor-core screen layout (music_fused.cuh, M = 4 only)
    float *na_max = nullptr;      // max ||a||^2 over the table rows (screen threshold)
};

struct Workspace {
    double *R = nullptr, *ev = nullptr, *Vt = nullptr, *P64 = nullptr;
    uint32_t cap = 0, p64_cap = 0;
    cudaEvent_t scan_done = nullptr;
    bool used = false;
};

constexpr int NSLOT = 2;  // workspace slots: one per host staging stream (process_device on a caller stream shares slot 0)

}  // namespace

struct music_b200 {
    uint32_t m = 0, n = 0, nsamples = 0, K = 0, N = 0;
    int device = 0;
    int sm_count = 0;
    std::mutex mutex;        // serialises process_*() and set_table(), like d_mutex (:67, :101)
    std::mutex err_mutex;    // guards `error` alone: fail() may run before `mutex` is taken (argument checks)
    std::string error;
    std::atomic<uint64_t> launches{0};

    DeviceTable table[2];
    int cur_table = 0;
    double *steer_pos = nullptr;   // device copy of the element positions (set_geometry)
    unsigned *steer_count = nullptr;
    int *steer_list = nullptr;
    float *steer_vals = nullptr;
    int peak_mode = MUSIC_B200_PEAKS_TOP_BINS;  // set_peak_mode()
    uint32_t peak_excl = 0;
    unsigned steer_guarded = 0;    // entries of the last built table re-evaluated with the host libm

    // fp64 workspace slots (R, eigenvalues, sorted eigenvectors, optional strengths) of the three-kernel path
    Workspace ws[NSLOT];
    unsigned *work_ctr = nullptr;      // persistent kernels: ring of self-resetting (window tickets, finished CTAs) pairs, CTR_RING per slot
    unsigned ctr_seq[2] = {0, 0};      // next ring entry per slot
    bool fused_spec = true;            // the spectrum port on the fused M = 4 kernel (MUSIC_B200_FUSED_SPEC=0: three-kernel path)
    bool pdl = true;                   // fused M = 4 kernel: programmatic dependent launch (MUSIC_B200_PDL=0 turns it off)
    cudaEvent_t fused_done = nullptr;  // orders persistent launches that share a ticket counter but not a stream
    bool fused_used[2] = {false, false};
    bool eig_mode = false;            // fused kernels: false principal eigenvector by squaring (default), true Jacobi for every window (MUSIC_B200_EIG=jacobi)
    unsigned *f8_stats = nullptr;     // fused M = 8 kernel: windows solved by squaring / by the Jacobi fallback
    int mma_fin_max = 3;              // fused kernel: no tensor-core pass starts once the tickets have run out and this many covariance warps are done (MUSIC_B200_MMA_FIN; 0: at ticket exhaustion, -1: fp64 drain only)
    long long *fused_trace = nullptr;  // MUSIC_B200_TRACE=1: per-CTA clock64 trace of the fused kernel (tools/fused_trace.py)
    bool fused = true;       // MUSIC_B200_FUSED=0 forces the three-kernel path
    // optional per-stage timing (bench.py's roofline leg): events around K1/K2/K3/top-n per chunk
    bool timing = false;
    std::vector<cudaEvent_t> tev;   // 5 events per timed chunk
    size_t tev_used = 0;    // done[0] marks the end of the last process_device() on its stream

    // host path staging
    cudaStream_t streams[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr};
    float *d_in[2] = {nullptr, nullptr};
    float *d_ang[2] = {nullptr, nullptr}, *d_lvl[2] = {nullptr, nullptr}, *d_spec[2] = {nullptr, nullptr};
    int32_t *d_bins[2] = {nullptr, nullptr};
    // pinned host mirrors of d_ang/d_lvl/d_bins: device->host copies into caller memory would be synchronous when that
    // memory is pageable (numpy arrays, GNU Radio buffers) and stall the enqueue of the next chunk's upload
    float *p_ang[2] = {nullptr, nullptr}, *p_lvl[2] = {nullptr, nullptr};
    int32_t *p_bins[2] = {nullptr, nullptr};
    uint32_t slot_w0[2] = {0, 0}, slot_W[2] = {0, 0};
    uint32_t host_chunk = 0;
    bool host_spec_alloc = false;
    cudaStream_t last_fused_stream[2] = {nullptr, nullptr};  // per ticket counter: launches on one stream need no event

    // caller memory registered for DMA (cudaHostRegister), newest last: GNU Radio hands work() the same pageable
    // circular buffers over and over, so a range is pinned once and found again on every later call
    struct HostReg { uintptr_t base; size_t len; };
    std::vector<HostReg> hostregs;
    bool hostreg = true;   // MUSIC_B200_HOSTREG=0: never register (pageable copies go through the driver's staging)

    // multi-device handle (music_b200_create_multi): one child per device, windows dealt w -> child w mod G
    std::vector<music_b200 *> kids;

    // fused all-gather of the peak bins (music_b200_gather_*): peer-mapped buffers, epoch flags
    int32_t *gather_buf = nullptr;
    unsigned *gather_flags = nullptr;
    size_t gather_cap = 0;
    int32_t *peer_bins[MAX_PEERS] = {};
    unsigned *peer_flags[MAX_PEERS] = {};
    bool peer_ipc[MAX_PEERS] = {};
    int gather_G = 0, gather_rank = 0;
    unsigned gather_epoch = 0;
};

namespace {

int fail(music_b200 *h, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) {
        std::lock_guard<std::mutex> g(h->err_mutex);
        h->error = buf;
    } else {
        std::lock_guard<std::mutex> g(g_err_mutex);
        g_create_error = buf;
    }
    return code;
}

#define CU(h, expr)                                                                             \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return fail((h), e_ == cudaErrorMemoryAllocation ? MUSIC_B200_ENOMEM : MUSIC_B200_ECUDA, \
                        "%s failed: %s", #expr, cudaGetErrorString(e_));                        \
    } while (0)

// Table rows are padded (||a||^2 = +inf) to whole TILE-row tiles.
uint32_t table_tiles(uint32_t K) { return (uint32_t)((K + TILE - 1) / TILE); }
size_t soa_doubles(uint32_t K, uint32_t M) { return (size_t)table_tiles(K) * (2 * M + 1) * TILE; }

// derived layouts (fp64 SoA tiles, TF32 hi/lo MMA fragments) of the c64 table already in t.c64
int finish_table(music_b200 *h, int slot, cudaStream_t st)
{
    DeviceTable &t = h->table[slot];
    const int ntiles = (int)table_tiles(h->K);
    prep_table_kernel<<<ntiles, TILE, 0, st>>>(reinterpret_cast<const float2 *>(t.c64), t.soa, (int)h->K, (int)h->m);
    h->launches++;
    if (t.fz) {
        const int threads = (FZ_NDEC + fused_tiles((int)h->K)) * (FZ_BINS / 16) * 32;
        CU(h, cudaMemsetAsync(t.na_max, 0, sizeof(float), st));
        prep_table_tc_kernel<<<(threads + 255) / 256, 256, 0, st>>>(t.c64, t.fz, t.na_max, (int)h->K);
        h->launches++;
    }
    CU(h, cudaGetLastError());
    CU(h, cudaStreamSynchronize(st));
    return MUSIC_B200_OK;
}

int upload_table(music_b200 *h, int slot, const float *table_c64, cudaStream_t st)
{
    CU(h, cudaMemcpyAsync(h->table[slot].c64, table_c64, (size_t)h->K * h->m * 2 * sizeof(float), cudaMemcpyHostToDevice, st));
    return finish_table(h, slot, st);
}

// Steering table built on the device from the element positions (music_steer.cuh), then patched at the
// few entries whose float32 rounding could depend on the libm in use.
int build_table(music_b200 *h, int slot, const double *pos_xy, double lambda, cudaStream_t st)
{
    DeviceTable &t = h->table[slot];
    const int K = (int)h->K, M = (int)h->m;
    if (!h->steer_pos) {
        CU(h, cudaMalloc(&h->steer_pos, sizeof(double) * 2 * MUSIC_B200_MAX_M));
        CU(h, cudaMalloc(&h->steer_count, sizeof(unsigned)));
        CU(h, cudaMalloc(&h->steer_list, sizeof(int) * STEER_GUARD_CAP));
        CU(h, cudaMalloc(&h->steer_vals, sizeof(float) * 2 * STEER_GUARD_CAP));
    }
    CU(h, cudaMemcpyAsync(h->steer_pos, pos_xy, sizeof(double) * 2 * M, cudaMemcpyHostToDevice, st));
    CU(h, cudaMemsetAsync(h->steer_count, 0, sizeof(unsigned), st));
    steer_table_kernel<<<(K * M + 255) / 256, 256, 0, st>>>(h->steer_pos, lambda, K, M, reinterpret_cast<float2 *>(t.c64),
                                                           h->steer_count, h->steer_list);
    h->launches++;
    CU(h, cudaGetLastError());
    unsigned cnt = 0;
    CU(h, cudaMemcpyAsync(&cnt, h->steer_count, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    h->steer_guarded = cnt;
    if (cnt > (unsigned)STEER_GUARD_CAP) {
        // more boundary cases than the list holds (a degenerate geometry, e.g. all elements at the origin, makes
        // every entry exactly (1, 0)): evaluate every entry the literal way
        std::vector<float> full((size_t)K * M * 2);
        for (int k = 0; k < K; ++k)
            for (int a = 0; a < M; ++a) steer_entry_host(pos_xy, lambda, K, k, a, &full[2 * ((size_t)k * M + a)], &full[2 * ((size_t)k * M + a) + 1]);
        CU(h, cudaMemcpyAsync(t.c64, full.data(), full.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        CU(h, cudaStreamSynchronize(st));
    } else if (cnt) {
        std::vector<int> list(cnt);
        CU(h, cudaMemcpyAsync(list.data(), h->steer_list, sizeof(int) * cnt, cudaMemcpyDeviceToHost, st));
        CU(h, cudaStreamSynchronize(st));
        std::vector<float> vals(2 * (size_t)cnt);
        for (unsigned i = 0; i < cnt; ++i) steer_entry_host(pos_xy, lambda, K, list[i] / M, list[i] % M, &vals[2 * i], &vals[2 * i + 1]);
        CU(h, cudaMemcpyAsync(h->steer_vals, vals.data(), vals.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        steer_patch_kernel<<<(cnt + 255) / 256, 256, 0, st>>>(reinterpret_cast<float2 *>(t.c64), h->steer_list,
                                                            reinterpret_cast<const float2 *>(h->steer_vals), (int)cnt);
        h->launches++;
        CU(h, cudaGetLastError());
        CU(h, cudaStreamSynchronize(st));  // vals is a local
    }
    return finish_table(h, slot, st);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// 3-D tensor map over the M-antenna input d_in viewed as rows of 128 bytes (16 / M snapshots each; with SWIZZLE_128B a
// narrower inner box would be padded to the 128-byte span): {32 floats, N * M / 16 rows, W windows}, box {32, box_rows, 1}.
// False when the driver cannot encode it.
bool encode_row_map(CUtensorMap *tm, const float *d_in, int M, int N, uint32_t W, int box_rows)
{
    const EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t gdim[3] = {32u, (cuuint64_t)(N / (16 / M)), (cuuint64_t)W};
    const cuuint64_t gstr[2] = {128u, (cuuint64_t)(8 * M) * (cuuint64_t)N};
    const cuuint32_t box[3] = {32u, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(d_in), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Inside the chunk loops of the host entry points an error must not skip the common tail (stream syncs, slot
// reset): record it in rc and leave the loop instead of returning.
#define CU_BREAK(h, rc, expr)                                                                    \
    {                                                                                            \
        cudaError_t e_ = (expr);                                                                 \
        if (e_ != cudaSuccess) {                                                                 \
            rc = fail((h), e_ == cudaErrorMemoryAllocation ? MUSIC_B200_ENOMEM : MUSIC_B200_ECUDA, \
                      "%s failed: %s", #expr, cudaGetErrorString(e_));                           \
            break;                                                                               \
        }                                                                                        \
    }

constexpr unsigned CTR_RING = 256;  // ticket-counter pairs per slot (see ticket_counter)

// Windows per sub-batch bounding one workspace slot to ~384 MiB.
uint32_t max_sub_windows(const music_b200 *h, bool need_p64)
{
    const size_t per_win = (size_t)h->m * h->m * 2 * 8 * 2 + h->m * 8 + (need_p64 ? (size_t)h->K * 8 : 0);
    size_t c = ((size_t)384 << 20) / per_win;
    c = std::max<size_t>(SCAN_B, std::min<size_t>(c, 1u << 20));
    return (uint32_t)(c / SCAN_B * SCAN_B);
}

int ensure_slot(music_b200 *h, Workspace &ws, uint32_t windows, bool need_p64)
{
    if (windows > ws.cap) {
        // the slot may still be in use by an earlier call on another stream
        if (ws.used) CU(h, cudaEventSynchronize(ws.scan_done));
        cudaFree(ws.R); cudaFree(ws.ev); cudaFree(ws.Vt);
        ws.R = ws.ev = ws.Vt = nullptr; ws.cap = 0;
        const size_t mm = (size_t)h->m * h->m * 2;
        CU(h, cudaMalloc(&ws.R, windows * mm * sizeof(double)));
        CU(h, cudaMalloc(&ws.Vt, windows * mm * sizeof(double)));
        CU(h, cudaMalloc(&ws.ev, (size_t)windows * h->m * sizeof(double)));
        ws.cap = windows;
    }
    if (need_p64 && windows > ws.p64_cap) {
        if (ws.used) CU(h, cudaEventSynchronize(ws.scan_done));
        cudaFree(ws.P64); ws.P64 = nullptr; ws.p64_cap = 0;
        CU(h, cudaMalloc(&ws.P64, (size_t)windows * h->K * sizeof(double)));
        ws.p64_cap = windows;
    }
    return MUSIC_B200_OK;
}

template <int MT>
void launch_scan(music_b200 *h, const Workspace &ws, const double *soa, uint32_t W, bool argmax, bool p64, bool spec,
                 PeakOut po, float *d_spec, double *d_p64, cudaStream_t st)
{
    const int grid = (W + SCAN_B - 1) / SCAN_B;
    const size_t smem = (size_t)SCAN_B * h->m * h->m * 2 * sizeof(double);
#define SCAN_CASE(A, P, S)                                                                              \
    if (argmax == A && p64 == P && spec == S)                                                           \
        scan_kernel<MT, A, P, S><<<grid, TILE, smem, st>>>(soa, ws.Vt, (int)h->m, (int)h->n, (int)h->K,  \
                                                           (int)W, po, d_spec, d_p64);
    if constexpr (MT == 0) {  // (M = 4, 8, 16 take scan_peak1_kernel for this case)
        SCAN_CASE(true, false, false)
    }
    SCAN_CASE(true, false, true)
    SCAN_CASE(true, true, false)
    SCAN_CASE(true, true, true)
    SCAN_CASE(false, true, false)
    SCAN_CASE(false, true, true)
#undef SCAN_CASE
    h->launches++;
}

cudaEvent_t *timing_events(music_b200 *h)
{
    if (!h->timing) return nullptr;
    if (h->tev_used + 5 > h->tev.size()) {
        for (int i = 0; i < 5; ++i) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
            h->tev.push_back(e);
        }
    }
    cudaEvent_t *p = h->tev.data() + h->tev_used;
    h->tev_used += 5;
    return p;
}

// Ticket counter pair `slot` (0 / 1) for a persistent kernel about to be launched on `st`.  The counters re-arm
// themselves at the end of a launch, so launches that share a pair must not overlap: on one stream that is stream
// order; when the stream changes, the new stream first waits for everything enqueued on the previous one.
unsigned *ticket_counter(music_b200 *h, int slot, cudaStream_t st)
{
    slot &= 1;
    if (h->fused_used[slot] && h->last_fused_stream[slot] != st) {
        if (cudaEventRecord(h->fused_done, h->last_fused_stream[slot]) != cudaSuccess ||
            cudaStreamWaitEvent(st, h->fused_done, 0) != cudaSuccess) {
            cudaGetLastError();        // e.g. the previous stream no longer exists
            cudaDeviceSynchronize();
        }
    }
    h->fused_used[slot] = true;
    h->last_fused_stream[slot] = st;
    // Every launch draws its own pair from the slot's ring: with programmatic dependent launch the CTAs of launch k + 1
    // start on the SMs launch k has left while k's last CTAs are still running, so the two must not share tickets.  A
    // pair is reused CTR_RING launches later; launches on one stream overlap only with their neighbours, and each
    // persistent CTA owns a whole SM, so fewer than CTR_RING launches are ever resident together.
    const unsigned e = h->ctr_seq[slot]++ % CTR_RING;
    return h->work_ctr + 2 * ((size_t)slot * CTR_RING + e);
}

// K1: covariance of W windows into ws.R, on `st`.
void launch_cov(music_b200 *h, const Workspace &ws, const float *d_in, uint32_t W, cudaStream_t st, int ctr_slot)
{
    const int M = (int)h->m, N = (int)h->N;
    CUtensorMap tm;
    if (M == 4) {
        // persistent, one CTA per SM, per-warp TMA ring (see cov4_tma_kernel)
        const int grid = std::min<int>(h->sm_count, (int)((W + COV_WARPS - 1) / COV_WARPS));
        cov4_tma_kernel<<<grid, COV_WARPS * 32, COV_SMEM, st>>>(d_in, ws.R, (int)W, N);
        h->launches++;
    } else if ((M == 8 || M == 16) && N >= 128 && N % (16 / M) == 0 &&
               encode_row_map(&tm, d_in, M, N, W, M == 8 ? 32 * CovNJobs<8>::STEPS * 8 * 8 / 128 : 32 * CovNJobs<16>::STEPS * 8 * 16 / 128)) {
        // TMA-tiled, window staged once per group of warps (music_covn.cuh); the box is one stage
        constexpr int groups8 = CN_WARPS / CovNJobs<8>::J, groups16 = CN_WARPS / CovNJobs<16>::J;
        const int groups = M == 8 ? groups8 : groups16;
        const int grid = std::min<int>(h->sm_count, (int)((W + groups - 1) / groups));
        unsigned *ctr = ticket_counter(h, ctr_slot, st);
        if (M == 8) covN_tma_kernel<8><<<grid, CN_WARPS * 32, CN_SMEM, st>>>(tm, ws.R, (int)W, N, ctr);
        else covN_tma_kernel<16><<<grid, CN_WARPS * 32, CN_SMEM, st>>>(tm, ws.R, (int)W, N, ctr);
        h->launches++;
    } else if (M % 4 == 0) {
        const int T = M / 4;
        const int wpb = 8;
        {
            const long long items = (long long)W * T;
            cov_tile_kernel<false><<<(unsigned)((items + wpb - 1) / wpb), wpb * 32, 0, st>>>(d_in, ws.R, (int)W, N, M);
            h->launches++;
        }
        if (T > 1) {
            const long long items = (long long)W * (T * (T - 1) / 2);
            cov_tile_kernel<true><<<(unsigned)((items + wpb - 1) / wpb), wpb * 32, 0, st>>>(d_in, ws.R, (int)W, N, M);
            h->launches++;
        }
    } else {
        const int E = M * (M + 1) / 2;
        const int S = 256 / E;
        cov_generic_kernel<<<W, 256, (size_t)S * E * 2 * sizeof(double), st>>>(d_in, ws.R, (int)W, N, M);
        h->launches++;
    }
}

// Output descriptor of a batch whose first window is local window w0 of the call: local pointers as given, plus the
// peers' gather buffers (music_b200_gather_attach / process_device_sharded) advanced to the same stream position.
PeakOut make_peak_out(const music_b200 *h, float *d_ang, float *d_lvl, int32_t *d_bins, size_t w0)
{
    PeakOut po;
    po.angles = d_ang; po.levels = d_lvl; po.bins = d_bins;
    po.npeer = h->gather_G; po.rank = h->gather_rank; po.n = (int)h->n;
    for (int p = 0; p < MAX_PEERS; ++p)
        po.peer[p] = (p < h->gather_G && h->peer_bins[p]) ? h->peer_bins[p] + w0 * (size_t)h->gather_G * h->n : nullptr;
    return po;
}

GatherFlags make_gather_flags(const music_b200 *h, bool signal)
{
    GatherFlags gf;
    for (int p = 0; p < MAX_PEERS; ++p) gf.peer[p] = p < h->gather_G ? h->peer_flags[p] : nullptr;
    gf.epoch = (signal && h->gather_G > 0 && h->peer_flags[0]) ? h->gather_epoch : 0u;
    return gf;
}

// raises this GPU's epoch flag at every peer once everything before it on the stream is done (unfused paths; the
// fused kernel signals from its last CTA)
__global__ void gather_signal_kernel(const GatherFlags gf, int npeer, int rank)
{
    if ((int)threadIdx.x < npeer) {
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(gf.peer[threadIdx.x] + rank), "r"(gf.epoch) : "memory");
    }
}

// consumer side: returns when every peer's flag in THIS GPU's array has reached `epoch`
__global__ void gather_wait_kernel(const unsigned *flags, int npeer, unsigned epoch)
{
    if ((int)threadIdx.x < npeer) {
        unsigned v;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + threadIdx.x) : "memory");
            if ((int)(v - epoch) >= 0) break;
            __nanosleep(200);
        } while (true);
    }
}

// K2 + K3 (+ top-n) of W windows from ws.R, on `st`.  tev (optional) = timing events [1..4].
int launch_eig_scan(music_b200 *h, const Workspace &ws, uint32_t W, const PeakOut &po, float *d_spec,
                    double *d_P64_out, double *d_R_out, double *d_ev_out, cudaStream_t st, cudaEvent_t *tev)
{
    const int M = (int)h->m;
    const double *soa = h->table[h->cur_table].soa;
    {
        const int grid = (W + 127) / 128;
        switch (M) {
        case 4: eig_kernel<4, true><<<grid, 128, 0, st>>>(ws.R, ws.ev, ws.Vt, M, (int)W); break;
        case 8: eig_coop_kernel<8><<<(W + EIGC_WARPS - 1) / EIGC_WARPS, EIGC_WARPS * 32, 0, st>>>(ws.R, ws.ev, ws.Vt, (int)W); break;
        case 12: eig_coop_kernel<12><<<(W + EIGC_WARPS - 1) / EIGC_WARPS, EIGC_WARPS * 32, 0, st>>>(ws.R, ws.ev, ws.Vt, (int)W); break;
        case 16: eig_coop_kernel<16><<<(W + EIGC_WARPS - 1) / EIGC_WARPS, EIGC_WARPS * 32, 0, st>>>(ws.R, ws.ev, ws.Vt, (int)W); break;
        default:
            if (M <= 8) eig_kernel<8, false><<<grid, 128, 0, st>>>(ws.R, ws.ev, ws.Vt, M, (int)W);
            else eig_kernel<MAXM, false><<<grid, 128, 0, st>>>(ws.R, ws.ev, ws.Vt, M, (int)W);
            break;
        }
        h->launches++;
    }
    if (tev) cudaEventRecord(tev[2], st);
    const bool local = h->peak_mode == MUSIC_B200_PEAKS_LOCAL_MAXIMA;
    const bool argmax = (h->n == 1) && !local;
    const bool need_p64 = !argmax || d_P64_out != nullptr;
    double *p64 = d_P64_out ? d_P64_out : ws.P64;
    const bool fast = argmax && !need_p64 && !d_spec && (M == 4 || M == 8 || M == 16);
    if (fast) {
        const int grid = (W + SCAN_B - 1) / SCAN_B;
        if (M == 4) scan_peak1_kernel<4><<<grid, TILE, 0, st>>>(soa, ws.Vt, (int)h->K, (int)W, po);
        else if (M == 8) scan_peak1_kernel<8><<<grid, TILE, 0, st>>>(soa, ws.Vt, (int)h->K, (int)W, po);
        else scan_peak1_kernel<16><<<grid, TILE, 0, st>>>(soa, ws.Vt, (int)h->K, (int)W, po);
        h->launches++;
    } else {
        switch (M) {
        case 4: launch_scan<4>(h, ws, soa, W, argmax, need_p64, d_spec != nullptr, po, d_spec, p64, st); break;
        case 8: launch_scan<8>(h, ws, soa, W, argmax, need_p64, d_spec != nullptr, po, d_spec, p64, st); break;
        case 16: launch_scan<16>(h, ws, soa, W, argmax, need_p64, d_spec != nullptr, po, d_spec, p64, st); break;
        default: launch_scan<0>(h, ws, soa, W, argmax, need_p64, d_spec != nullptr, po, d_spec, p64, st); break;
        }
    }
    if (tev) cudaEventRecord(tev[3], st);
    if (!argmax) {
        if (local) topn_local_kernel<<<(W + 7) / 8, 256, 0, st>>>(p64, (int)h->n, (int)h->K, (int)W, (int)h->peak_excl, po);
        else topn_kernel<<<(W + 7) / 8, 256, 0, st>>>(p64, (int)h->n, (int)h->K, (int)W, po);
        h->launches++;
    }
    if (tev) cudaEventRecord(tev[4], st);
    if (d_R_out)
        CU(h, cudaMemcpyAsync(d_R_out, ws.R, (size_t)W * M * M * 2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (d_ev_out)
        CU(h, cudaMemcpyAsync(d_ev_out, ws.ev, (size_t)W * M * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CU(h, cudaGetLastError());
    return MUSIC_B200_OK;
}

// K1 on planar streams (music_planar.cuh): windows first .. first + W - 1 of the call
void launch_cov_planar(music_b200 *h, const Workspace &ws, const PlanarStreams &S, unsigned long long first_snapshot,
                       unsigned hop, uint32_t W, cudaStream_t st)
{
    const int M = (int)h->m, N = (int)h->N, T = (M + 3) / 4, wpb = 8;
    cov_planar_kernel<false><<<(unsigned)(((long long)W * T + wpb - 1) / wpb), wpb * 32, 0, st>>>(S, first_snapshot, hop, ws.R, (int)W, N, M);
    h->launches++;
    if (T > 1) {
        const long long items = (long long)W * (T * (T - 1) / 2);
        cov_planar_kernel<true><<<(unsigned)((items + wpb - 1) / wpb), wpb * 32, 0, st>>>(S, first_snapshot, hop, ws.R, (int)W, N, M);
        h->launches++;
    }
}

// Enqueue `nwindows` windows on `st`: one persistent launch where a fused kernel covers the call, otherwise the three-kernel
// path in sub-batches of at most max_sub_windows() windows through workspace slot `slot`.  `slot` (0 / 1) also picks the
// ticket-counter ring of the persistent kernels.
int enqueue_device(music_b200 *h, const float *d_in, uint32_t nwindows, float *d_ang, float *d_lvl, float *d_spec,
                   int32_t *d_bins, double *d_P64, double *d_R, double *d_ev, cudaStream_t st, int slot,
                   const PlanarStreams *planar = nullptr, unsigned hop = 0)
{
    if (nwindows == 0) return MUSIC_B200_OK;
    if ((!planar && !d_in) || !d_ang) return fail(h, MUSIC_B200_EINVAL, "d_in_c64 and d_angles must not be NULL");
    if (!planar && (reinterpret_cast<uintptr_t>(d_in) & 15u) != 0) return fail(h, MUSIC_B200_EINVAL, "d_in_c64 must be 16-byte aligned");
    // planar streams can take the fused path when the 16-byte granularity of bulk copies allows it
    bool planar_fusable = false;
    if (planar) {
        planar_fusable = (hop % 2 == 0) && (h->N % 2 == 0);
        for (uint32_t r = 0; r < h->m; ++r) planar_fusable = planar_fusable && (reinterpret_cast<uintptr_t>(planar->p[r]) & 15u) == 0;
    }
    const bool local_peaks = h->peak_mode == MUSIC_B200_PEAKS_LOCAL_MAXIMA;
    if ((!planar || planar_fusable) && h->fused && !local_peaks && h->m == 4 && h->n == 1 && (!d_spec || h->fused_spec) && !d_P64 && !d_R && !d_ev) {
        // whole call in one persistent launch (music_fused.cuh); no workspace involved
        cudaEvent_t *tev = timing_events(h);
        if (tev) cudaEventRecord(tev[0], st);
        const int grid = std::min<int>(h->sm_count, (int)((nwindows + FZ_COV_WARPS - 1) / FZ_COV_WARPS));
        unsigned *ctr = ticket_counter(h, slot, st);
        const DeviceTable &tb = h->table[h->cur_table];
        const PeakOut po = make_peak_out(h, d_ang, d_lvl, d_bins, 0);
        const GatherFlags gf = make_gather_flags(h, true);
        // Programmatic dependent launch: when the previous operation on `st` is another launch of this kernel, the new
        // CTAs are placed as soon as the old ones leave their SMs (every CTA signals launch_dependents at its start) instead
        // of after the whole grid has drained; the kernel orders its own output writes behind the previous grid with
        // griddepcontrol.wait.  After any other kind of operation the launch is an ordinary stream-ordered one.
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(FZ_THREADS); lc.dynamicSmemBytes = FZ_SMEM; lc.stream = st;
        cudaLaunchAttribute la[1];
        la[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        la[0].val.programmaticStreamSerializationAllowed = 1;
        lc.attrs = la; lc.numAttrs = h->pdl ? 1 : 0;
        const int W_i = (int)nwindows, N_i = (int)h->N, K_i = (int)h->K;
        const bool tr = h->fused_trace != nullptr;  // MUSIC_B200_TRACE=1: the instantiation with the clock64 trace
        // drain workers: 100 ns idle sleep, 16 chunks per group, no early drain (DESIGN.md section 5)
        const unsigned char *fz = tb.fz;
        const float *c64 = tb.c64, *na_max = tb.na_max;
        cudaError_t le;
        if (planar) {
            auto kern = tr ? music4_fused_kernel<true, true> : music4_fused_kernel<true, false>;
            le = cudaLaunchKernelEx(&lc, kern, (const float *)nullptr, *planar, 0ull, (unsigned)hop, fz, c64, na_max, W_i, N_i, K_i, po, ctr,
                                    h->fused_trace, (int)h->eig_mode, gf, h->mma_fin_max, 100u, 16, 0, d_spec);
        } else {
            auto kern = tr ? music4_fused_kernel<false, true> : music4_fused_kernel<false, false>;
            le = cudaLaunchKernelEx(&lc, kern, d_in, PlanarStreams{}, 0ull, 0u, fz, c64, na_max, W_i, N_i, K_i, po, ctr, h->fused_trace,
                                    (int)h->eig_mode, gf, h->mma_fin_max, 100u, 16, 0, d_spec);
        }
        CU(h, le);
        h->launches++;
        if (tev) for (int i = 1; i < 5; ++i) cudaEventRecord(tev[i], st);
        CU(h, cudaGetLastError());
        return MUSIC_B200_OK;
    }
    CUtensorMap tm;
    if (!planar && h->fused && !local_peaks && h->m == 8 && h->n == 1 && !d_spec && !d_P64 && !d_R && !d_ev && h->N >= 128 &&
        h->N % 2 == 0 && encode_row_map(&tm, d_in, 8, (int)h->N, nwindows, F8_STAGE / 128)) {
        // M = 8: whole call in one persistent launch (music_fused8.cuh); R and the eigenvectors stay in shared memory
        cudaEvent_t *tev = timing_events(h);
        if (tev) cudaEventRecord(tev[0], st);
        const int grid = std::min<int>(h->sm_count, (int)((nwindows + F8_WARPS - 1) / F8_WARPS));
        unsigned *ctr = ticket_counter(h, slot, st);
        music8_fused_kernel<<<grid, F8_WARPS * 32, F8_SMEM, st>>>(tm, h->table[h->cur_table].soa, (int)nwindows, (int)h->N, (int)h->K,
                                                                 make_peak_out(h, d_ang, d_lvl, d_bins, 0), ctr, make_gather_flags(h, true),
                                                                 h->eig_mode, h->f8_stats);
        h->launches++;
        if (tev) for (int i = 1; i < 5; ++i) cudaEventRecord(tev[i], st);
        CU(h, cudaGetLastError());
        return MUSIC_B200_OK;
    }
    const bool internal_p64 = (h->n != 1 || local_peaks) && !d_P64;
    const uint32_t sub = std::min((nwindows + SCAN_B - 1) / SCAN_B * SCAN_B, max_sub_windows(h, internal_p64));
    Workspace &ws = h->ws[slot];
    int rc = ensure_slot(h, ws, sub, internal_p64);
    if (rc) return rc;
    if (ws.used) CU(h, cudaStreamWaitEvent(st, ws.scan_done, 0));  // the slot's last user may be another stream
    for (uint32_t w0 = 0; w0 < nwindows; w0 += sub) {
        const uint32_t W = std::min(sub, nwindows - w0);
        cudaEvent_t *tev = timing_events(h);
        if (tev) cudaEventRecord(tev[0], st);
        if (planar) launch_cov_planar(h, ws, *planar, (unsigned long long)w0 * hop, hop, W, st);
        else launch_cov(h, ws, d_in + (size_t)w0 * h->nsamples * 2, W, st, slot);
        if (tev) cudaEventRecord(tev[1], st);
        rc = launch_eig_scan(h, ws, W,
                             make_peak_out(h, d_ang + (size_t)w0 * h->n, d_lvl ? d_lvl + (size_t)w0 * h->n : nullptr,
                                           d_bins ? d_bins + (size_t)w0 * h->n : nullptr, w0),
                             d_spec ? d_spec + (size_t)w0 * h->K : nullptr,
                             d_P64 ? d_P64 + (size_t)w0 * h->K : nullptr, d_R ? d_R + (size_t)w0 * h->m * h->m * 2 : nullptr,
                             d_ev ? d_ev + (size_t)w0 * h->m : nullptr, st, tev);
        if (rc) return rc;
        CU(h, cudaEventRecord(ws.scan_done, st));
        ws.used = true;
    }
    if (h->gather_G > 0) {
        const GatherFlags gf = make_gather_flags(h, true);
        if (gf.epoch) {
            gather_signal_kernel<<<1, 32, 0, st>>>(gf, h->gather_G, h->gather_rank);
            h->launches++;
        }
    }
    return MUSIC_B200_OK;
}

struct NvtxRange {  // SURVEY.md section 5 tracing hook: ranges show up in nsys / ncu timelines, free when no tool is attached
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// Makes [ptr, ptr + bytes) DMA-able if it is ordinary pageable memory: page-aligned cudaHostRegister, remembered in
// the handle (at most 16 ranges, oldest evicted).  Memory that is already pinned (cudaHostAlloc, registered by the
// caller) or that cannot be registered is left alone - the copies then take the driver's staged path.
void host_register(music_b200 *h, const void *ptr, size_t bytes, bool read_only)
{
    if (!h->hostreg || !ptr || bytes < ((size_t)1 << 20)) return;
    const uintptr_t a = reinterpret_cast<uintptr_t>(ptr), page = 4096;
    const uintptr_t lo = a & ~(page - 1), hi = (a + bytes + page - 1) & ~(page - 1);
    for (size_t i = 0; i < h->hostregs.size(); ++i)
        if (h->hostregs[i].base <= lo && hi <= h->hostregs[i].base + h->hostregs[i].len) return;  // already ours
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) == cudaSuccess) {
        if (at.type != cudaMemoryTypeUnregistered) return;  // pinned by the caller (or not host memory at all)
    } else {
        cudaGetLastError();
    }
    NvtxRange r("music_b200: cudaHostRegister");
    // ranges of ours that overlap the new one (a circular buffer seen at a shifted offset): drop them first
    for (size_t i = 0; i < h->hostregs.size();) {
        const music_b200::HostReg &g = h->hostregs[i];
        if (g.base < hi && lo < g.base + g.len) {
            cudaHostUnregister(reinterpret_cast<void *>(g.base));
            h->hostregs.erase(h->hostregs.begin() + i);
        } else {
            ++i;
        }
    }
    cudaError_t e = cudaHostRegister(reinterpret_cast<void *>(lo), hi - lo, cudaHostRegisterPortable | (read_only ? cudaHostRegisterReadOnly : 0));
    if (e != cudaSuccess && read_only) {
        cudaGetLastError();
        e = cudaHostRegister(reinterpret_cast<void *>(lo), hi - lo, cudaHostRegisterPortable);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();  // not registrable (e.g. a read-only mapping): pageable copies still work
        return;
    }
    if (h->hostregs.size() >= 16) {
        cudaHostUnregister(reinterpret_cast<void *>(h->hostregs.front().base));
        h->hostregs.erase(h->hostregs.begin());
    }
    h->hostregs.push_back(music_b200::HostReg{lo, (size_t)(hi - lo)});
}

void free_host_staging(music_b200 *h)
{
    for (int i = 0; i < 2; ++i) {
        cudaFree(h->d_in[i]); cudaFree(h->d_ang[i]); cudaFree(h->d_lvl[i]); cudaFree(h->d_spec[i]); cudaFree(h->d_bins[i]);
        cudaFreeHost(h->p_ang[i]); cudaFreeHost(h->p_lvl[i]); cudaFreeHost(h->p_bins[i]);
        h->d_in[i] = h->d_ang[i] = h->d_lvl[i] = h->d_spec[i] = nullptr;
        h->d_bins[i] = nullptr;
        h->p_ang[i] = h->p_lvl[i] = nullptr;
        h->p_bins[i] = nullptr;
        h->slot_W[i] = 0;
    }
    h->host_chunk = 0;
    h->host_spec_alloc = false;
}

int ensure_host_staging(music_b200 *h, uint32_t chunk, bool spec)
{
    if (chunk <= h->host_chunk && (!spec || h->host_spec_alloc)) return MUSIC_B200_OK;
    const uint32_t cap = std::max(chunk, h->host_chunk);
    free_host_staging(h);
    for (int i = 0; i < 2; ++i) {
        CU(h, cudaMalloc(&h->d_in[i], (size_t)cap * h->nsamples * 2 * sizeof(float)));
        CU(h, cudaMalloc(&h->d_ang[i], (size_t)cap * h->n * sizeof(float)));
        CU(h, cudaMalloc(&h->d_lvl[i], (size_t)cap * h->n * sizeof(float)));
        CU(h, cudaMalloc(&h->d_bins[i], (size_t)cap * h->n * sizeof(int32_t)));
        CU(h, cudaHostAlloc(&h->p_ang[i], (size_t)cap * h->n * sizeof(float), cudaHostAllocDefault));
        CU(h, cudaHostAlloc(&h->p_lvl[i], (size_t)cap * h->n * sizeof(float), cudaHostAllocDefault));
        CU(h, cudaHostAlloc(&h->p_bins[i], (size_t)cap * h->n * sizeof(int32_t), cudaHostAllocDefault));
        if (spec) CU(h, cudaMalloc(&h->d_spec[i], (size_t)cap * h->K * sizeof(float)));
    }
    h->host_chunk = cap;
    h->host_spec_alloc = spec;
    return MUSIC_B200_OK;
}

// results of the chunk last computed in staging slot s: pinned mirror -> caller memory (the slot's stream is idle).
// The chunk holds the windows w = (slot_w0 + i) * G + g of the call (G = 1, g = 0 on a single-device handle).
void flush_host_slot(music_b200 *h, int s, float *angles, float *levels, int32_t *bins, uint32_t G = 1, uint32_t g = 0)
{
    const uint32_t W = h->slot_W[s];
    if (!W) return;
    const size_t n = h->n;
    if (G == 1) {
        const size_t off = (size_t)h->slot_w0[s] * n, cnt = (size_t)W * n;
        memcpy(angles + off, h->p_ang[s], cnt * sizeof(float));
        if (levels) memcpy(levels + off, h->p_lvl[s], cnt * sizeof(float));
        if (bins) memcpy(bins + off, h->p_bins[s], cnt * sizeof(int32_t));
    } else {
        for (uint32_t i = 0; i < W; ++i) {
            const size_t off = ((size_t)(h->slot_w0[s] + i) * G + g) * n;
            for (size_t r = 0; r < n; ++r) {
                angles[off + r] = h->p_ang[s][i * n + r];
                if (levels) levels[off + r] = h->p_lvl[s][i * n + r];
                if (bins) bins[off + r] = h->p_bins[s][i * n + r];
            }
        }
    }
    h->slot_W[s] = 0;
}

// device -> pinned mirrors of slot s (asynchronous on st whatever memory the caller's outputs live in)
int download_host_slot(music_b200 *h, int s, uint32_t w0, uint32_t W, bool levels, bool bins, cudaStream_t st)
{
    CU(h, cudaMemcpyAsync(h->p_ang[s], h->d_ang[s], (size_t)W * h->n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (levels) CU(h, cudaMemcpyAsync(h->p_lvl[s], h->d_lvl[s], (size_t)W * h->n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (bins) CU(h, cudaMemcpyAsync(h->p_bins[s], h->d_bins[s], (size_t)W * h->n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    h->slot_w0[s] = w0;
    h->slot_W[s] = W;
    return MUSIC_B200_OK;
}


}  // namespace

extern "C" {

int music_b200_version(void) { return 2; }

const char *music_b200_last_error(const music_b200 *h)
{
    static thread_local std::string copy;  // the returned text stays valid until this thread's next call
    if (h) {
        music_b200 *hm = const_cast<music_b200 *>(h);
        std::lock_guard<std::mutex> g(hm->err_mutex);
        copy = hm->error;
        return copy.c_str();
    }
    std::lock_guard<std::mutex> g(g_err_mutex);
    copy = g_create_error;
    return copy.c_str();
}

uint64_t music_b200_launch_count(const music_b200 *h)
{
    if (!h) return 0;
    uint64_t n = h->launches.load();
    for (const music_b200 *c : h->kids) n += c->launches.load();
    return n;
}

int music_b200_debug_fused_trace(music_b200 *h, long long *host_out, int max_ctas)
{
    if (h && !h->kids.empty()) return music_b200_debug_fused_trace(h->kids[0], host_out, max_ctas);  // multi-device handle: device 0 serves this entry
    if (!h || !host_out || !h->fused_trace) return MUSIC_B200_EINVAL;
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaDeviceSynchronize());
    CU(h, cudaMemcpy(host_out, h->fused_trace, (size_t)std::min(max_ctas, 1024) * FZ_TRACE * sizeof(long long), cudaMemcpyDeviceToHost));
    return MUSIC_B200_OK;
}

int music_b200_debug_fused8_stats(music_b200 *h, uint64_t *out2)
{
    if (h && !h->kids.empty()) return music_b200_debug_fused8_stats(h->kids[0], out2);
    if (!h || !out2 || !h->f8_stats) return MUSIC_B200_EINVAL;
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    unsigned v[2];
    CU(h, cudaMemcpy(v, h->f8_stats, sizeof v, cudaMemcpyDeviceToHost));
    out2[0] = v[0];
    out2[1] = v[1];
    return MUSIC_B200_OK;
}

int music_b200_set_stage_timing(music_b200 *h, int enable)
{
    if (h && !h->kids.empty()) return music_b200_set_stage_timing(h->kids[0], enable);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    std::lock_guard<std::mutex> g(h->mutex);
    h->timing = enable != 0;
    h->tev_used = 0;
    return MUSIC_B200_OK;
}

int music_b200_get_stage_times(music_b200 *h, double *ms4, uint64_t *chunks)
{
    if (h && !h->kids.empty()) return music_b200_get_stage_times(h->kids[0], ms4, chunks);  // multi-device handle: device 0 serves this entry
    if (!h || !ms4) return MUSIC_B200_EINVAL;
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    for (int i = 0; i < 4; ++i) ms4[i] = 0.0;
    const size_t nch = h->tev_used / 5;
    for (size_t c = 0; c < nch; ++c) {
        cudaEvent_t *e = h->tev.data() + 5 * c;
        CU(h, cudaEventSynchronize(e[4]));
        for (int i = 0; i < 4; ++i) {
            float ms = 0.f;
            CU(h, cudaEventElapsedTime(&ms, e[i], e[i + 1]));
            ms4[i] += ms;
        }
    }
    if (chunks) *chunks = nch;
    h->tev_used = 0;
    return MUSIC_B200_OK;
}

int music_b200_create(music_b200 **out, uint32_t m, uint32_t n, uint32_t nsamples, uint32_t resolution,
                      const float *table_c64, int device)
{
    if (!out) return fail(nullptr, MUSIC_B200_EINVAL, "out must not be NULL");
    *out = nullptr;
    // reference asserts, lib/baz_music_doa.cc:45-50 (+ n >= 1, n < m, see header)
    if (m == 0 || m > MUSIC_B200_MAX_M) return fail(nullptr, MUSIC_B200_EINVAL, "m must be in 1..%d (got %u)", MUSIC_B200_MAX_M, m);
    if (n == 0 || n >= m) return fail(nullptr, MUSIC_B200_EINVAL, "need 1 <= n < m (got n=%u, m=%u)", n, m);
    if (nsamples == 0 || nsamples % m != 0) return fail(nullptr, MUSIC_B200_EINVAL, "nsamples must be a positive multiple of m (got %u)", nsamples);
    if (resolution == 0) return fail(nullptr, MUSIC_B200_EINVAL, "resolution must be > 0");
    if (!table_c64) return fail(nullptr, MUSIC_B200_EINVAL, "array response table must not be NULL");

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, MUSIC_B200_ENODEVICE, "no CUDA device (%s); this library has no CPU path", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, MUSIC_B200_ENODEVICE, "device %d out of range (0..%d)", device, ndev - 1);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
        return fail(nullptr, MUSIC_B200_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, MUSIC_B200_ENODEVICE, "device %d is sm_%d%d; this build targets sm_100a only", device, prop.major, prop.minor);

    music_b200 *h = new (std::nothrow) music_b200();
    if (!h) return fail(nullptr, MUSIC_B200_ENOMEM, "out of host memory");
    h->m = m; h->n = n; h->nsamples = nsamples; h->K = resolution; h->N = nsamples / m;
    h->device = device; h->sm_count = prop.multiProcessorCount;

    int rc = MUSIC_B200_OK;
    auto init = [&]() -> int {
        CU(h, cudaSetDevice(device));
        for (int i = 0; i < 2; ++i) {
            CU(h, cudaStreamCreateWithFlags(&h->streams[i], cudaStreamNonBlocking));
            CU(h, cudaEventCreateWithFlags(&h->done[i], cudaEventDisableTiming));
            CU(h, cudaMalloc(&h->table[i].c64, (size_t)resolution * m * 2 * sizeof(float)));
            CU(h, cudaMalloc(&h->table[i].soa, soa_doubles(resolution, m) * sizeof(double)));
            if (m == 4) {
                CU(h, cudaMalloc(&h->table[i].fz, fused_table_bytes((int)resolution)));
                CU(h, cudaMalloc(&h->table[i].na_max, sizeof(float)));
            }
        }
        for (int i = 0; i < NSLOT; ++i) CU(h, cudaEventCreateWithFlags(&h->ws[i].scan_done, cudaEventDisableTiming));
        // scan kernels with M = 16 need 32 KiB dynamic smem (< 48 KiB default), nothing to opt in.
        if (const char *e = getenv("MUSIC_B200_FUSED")) h->fused = atoi(e) != 0;
        if (const char *e = getenv("MUSIC_B200_EIG")) h->eig_mode = !strcmp(e, "jacobi");
        if (const char *e = getenv("MUSIC_B200_PDL")) h->pdl = atoi(e) != 0;
        if (const char *e = getenv("MUSIC_B200_FUSED_SPEC")) h->fused_spec = atoi(e) != 0;
        if (const char *e = getenv("MUSIC_B200_MMA_FIN")) h->mma_fin_max = std::max(-1, std::min(8, atoi(e)));
        CU(h, cudaFuncSetAttribute(covN_tma_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CN_SMEM));
        CU(h, cudaFuncSetAttribute(covN_tma_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CN_SMEM));
        CU(h, cudaFuncSetAttribute(music8_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F8_SMEM));
        CU(h, cudaMalloc(&h->f8_stats, 2 * sizeof(unsigned)));
        CU(h, cudaMemset(h->f8_stats, 0, 2 * sizeof(unsigned)));
        CU(h, cudaEventCreateWithFlags(&h->fused_done, cudaEventDisableTiming));
        CU(h, cudaMalloc(&h->work_ctr, 2 * CTR_RING * 2 * sizeof(unsigned)));  // self-resetting (tickets, finished CTAs) pairs
        CU(h, cudaMemset(h->work_ctr, 0, 2 * CTR_RING * 2 * sizeof(unsigned)));
        if (const char *e = getenv("MUSIC_B200_HOSTREG")) h->hostreg = atoi(e) != 0;
        if (getenv("MUSIC_B200_TRACE")) {
            CU(h, cudaMalloc(&h->fused_trace, FZ_TRACE * sizeof(long long) * 1024));
            CU(h, cudaMemset(h->fused_trace, 0, FZ_TRACE * sizeof(long long) * 1024));
        }
        CU(h, cudaFuncSetAttribute(music4_fused_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FZ_SMEM));
        CU(h, cudaFuncSetAttribute(music4_fused_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FZ_SMEM));
        CU(h, cudaFuncSetAttribute(music4_fused_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FZ_SMEM));
        CU(h, cudaFuncSetAttribute(music4_fused_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FZ_SMEM));
        CU(h, cudaFuncSetAttribute(cov4_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)COV_SMEM));
        return upload_table(h, 0, table_c64, h->streams[0]);
    };
    rc = init();
    if (rc != MUSIC_B200_OK) {
        fail(nullptr, rc, "%s", std::string(h->error).c_str());
        music_b200_destroy(h);
        return rc;
    }
    h->cur_table = 0;
    *out = h;
    return MUSIC_B200_OK;
}

int music_b200_set_table(music_b200 *h, const float *table_c64)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (!table_c64) return fail(h, MUSIC_B200_EINVAL, "array response table must not be NULL");
    std::lock_guard<std::mutex> g(h->mutex);
    if (!h->kids.empty()) {  // multi-device handle: every device holds a full copy of the table (SURVEY.md section 8e)
        for (music_b200 *c : h->kids) {
            const int rc = music_b200_set_table(c, table_c64);
            if (rc) return fail(h, rc, "%s", music_b200_last_error(c));
        }
        return MUSIC_B200_OK;
    }
    CU(h, cudaSetDevice(h->device));
    // Work enqueued by earlier process_device() calls may still be reading the current slot on
    // a caller stream; fill the other slot and flip.  (The slot being overwritten was retired
    // two set_table() calls ago; synchronise the device once to be safe - retunes are rare.)
    CU(h, cudaDeviceSynchronize());
    const int slot = h->cur_table ^ 1;
    int rc = upload_table(h, slot, table_c64, h->streams[0]);
    if (rc) return rc;
    h->cur_table = slot;
    return MUSIC_B200_OK;
}

int music_b200_process_planar_device(music_b200 *h, const float *const *d_streams, uint32_t hop, uint32_t nwindows,
                                     float *d_angles, float *d_levels, float *d_spectrum, int32_t *d_bins, void *stream)
{
    if (h && !h->kids.empty()) return music_b200_process_planar_device(h->kids[0], d_streams, hop, nwindows, d_angles, d_levels, d_spectrum, d_bins, stream);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    if (nwindows == 0) return MUSIC_B200_OK;
    if (!d_streams) return fail(h, MUSIC_B200_EINVAL, "d_streams must not be NULL");
    if (hop == 0) return fail(h, MUSIC_B200_EINVAL, "hop must be >= 1 snapshot");
    PlanarStreams S;
    for (uint32_t r = 0; r < MAXM; ++r) S.p[r] = nullptr;
    for (uint32_t r = 0; r < h->m; ++r) {
        if (!d_streams[r] || (reinterpret_cast<uintptr_t>(d_streams[r]) & 7u) != 0)
            return fail(h, MUSIC_B200_EINVAL, "antenna stream %u must be a non-NULL, 8-byte aligned device pointer", r);
        S.p[r] = reinterpret_cast<const float2 *>(d_streams[r]);
    }
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    return enqueue_device(h, nullptr, nwindows, d_angles, d_levels, d_spectrum, d_bins, nullptr, nullptr, nullptr,
                          static_cast<cudaStream_t>(stream), 0, &S, hop);
}

int music_b200_process_planar_host(music_b200 *h, const float *const *streams, uint32_t hop, uint32_t nwindows,
                                   float *angles, float *levels, float *spectrum, int32_t *bins)
{
    if (h && !h->kids.empty()) return music_b200_process_planar_host(h->kids[0], streams, hop, nwindows, angles, levels, spectrum, bins);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    if (nwindows == 0) return MUSIC_B200_OK;
    if (!streams || !angles) return fail(h, MUSIC_B200_EINVAL, "streams and angles must not be NULL");
    if (hop == 0) return fail(h, MUSIC_B200_EINVAL, "hop must be >= 1 snapshot");
    for (uint32_t r = 0; r < h->m; ++r)
        if (!streams[r]) return fail(h, MUSIC_B200_EINVAL, "antenna stream %u must not be NULL", r);
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    // staging holds cap * m * N samples; a chunk of C windows needs m * ((C - 1) * hop + N) of them, laid out planar
    const size_t N = h->N;
    size_t cap = std::max<size_t>(SCAN_B, ((size_t)32 << 20) / std::max((size_t)h->nsamples * 8, spectrum ? (size_t)h->K * sizeof(float) : (size_t)0));
    cap = std::max<size_t>(cap, ((size_t)hop + N - 1) / N + 1);  // at least one window when hop > N
    h->slot_W[0] = h->slot_W[1] = 0;  // nothing pending from an earlier (possibly failed) call
    int rc = ensure_host_staging(h, (uint32_t)cap, spectrum != nullptr);
    if (rc) return rc;
    cap = h->host_chunk;
    uint32_t chunk = (uint32_t)std::min<size_t>(cap, 1 + (cap * N - N) / hop);
    chunk = std::min(chunk, (nwindows + 1) / 2 > SCAN_B ? (nwindows + 1) / 2 : nwindows);
    chunk = std::max<uint32_t>(1, chunk);
    int it = 0;
    rc = MUSIC_B200_OK;
    for (uint32_t w0 = 0; w0 < nwindows && rc == MUSIC_B200_OK; w0 += chunk, ++it) {
        const int s = it & 1;
        const uint32_t W = std::min(chunk, nwindows - w0);
        cudaStream_t st = h->streams[s];
        if (it >= 2) {
            CU_BREAK(h, rc, cudaStreamSynchronize(st));
            flush_host_slot(h, s, angles, levels, bins);
        }
        const size_t seg = (size_t)(W - 1) * hop + N;  // snapshots of each stream this chunk touches
        PlanarStreams S;
        for (uint32_t r = 0; r < MAXM; ++r) S.p[r] = nullptr;
        for (uint32_t r = 0; r < h->m && rc == MUSIC_B200_OK; ++r) {
            float *dst = h->d_in[s] + (size_t)r * seg * 2;
            CU_BREAK(h, rc, cudaMemcpyAsync(dst, streams[r] + ((size_t)w0 * hop) * 2, seg * 2 * sizeof(float), cudaMemcpyHostToDevice, st));
            S.p[r] = reinterpret_cast<const float2 *>(dst);
        }
        if (rc) break;
        rc = enqueue_device(h, nullptr, W, h->d_ang[s], h->d_lvl[s], spectrum ? h->d_spec[s] : nullptr, h->d_bins[s],
                            nullptr, nullptr, nullptr, st, s, &S, hop);
        if (rc) break;
        rc = download_host_slot(h, s, w0, W, levels != nullptr, bins != nullptr, st);
        if (rc) break;
        if (spectrum) CU_BREAK(h, rc, cudaMemcpyAsync(spectrum + (size_t)w0 * h->K, h->d_spec[s], (size_t)W * h->K * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    cudaError_t e0 = cudaStreamSynchronize(h->streams[0]);
    cudaError_t e1 = cudaStreamSynchronize(h->streams[1]);
    if (rc || e0 != cudaSuccess || e1 != cudaSuccess) h->slot_W[0] = h->slot_W[1] = 0;  // nothing valid to hand out
    if (rc) return rc;
    if (e0 != cudaSuccess || e1 != cudaSuccess)
        return fail(h, MUSIC_B200_ECUDA, "stream sync failed: %s", cudaGetErrorString(e0 != cudaSuccess ? e0 : e1));
    flush_host_slot(h, 0, angles, levels, bins);
    flush_host_slot(h, 1, angles, levels, bins);
    return MUSIC_B200_OK;
}

int music_b200_reduce_angles_device(music_b200 *h, const float *d_angles, const float *d_levels, uint32_t nwindows, int weighted,
                                    float *d_mean_deg, float *d_resultant, float *d_weight_sum, void *stream)
{
    if (h && !h->kids.empty()) return music_b200_reduce_angles_device(h->kids[0], d_angles, d_levels, nwindows, weighted, d_mean_deg, d_resultant, d_weight_sum, stream);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    if (!d_angles || !d_mean_deg) return fail(h, MUSIC_B200_EINVAL, "d_angles and d_mean_deg must not be NULL");
    if (weighted && !d_levels) return fail(h, MUSIC_B200_EINVAL, "level weighting needs d_levels");
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    reduce_angles_kernel<<<h->n, REDUCE_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(d_angles, d_levels, (int)nwindows, (int)h->n,
                                                                                      weighted ? 1 : 0, d_mean_deg, d_resultant, d_weight_sum);
    h->launches++;
    CU(h, cudaGetLastError());
    return MUSIC_B200_OK;
}

int music_b200_reduce_spectrum_device(music_b200 *h, const float *d_spectrum, uint32_t nwindows, float *d_mean, void *stream)
{
    if (h && !h->kids.empty()) return music_b200_reduce_spectrum_device(h->kids[0], d_spectrum, nwindows, d_mean, stream);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    if (!d_spectrum || !d_mean) return fail(h, MUSIC_B200_EINVAL, "d_spectrum and d_mean must not be NULL");
    if (nwindows == 0) return fail(h, MUSIC_B200_EINVAL, "nwindows must be >= 1");
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    reduce_spectrum_kernel<<<(h->K + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_spectrum, (int)nwindows, (int)h->K, d_mean);
    h->launches++;
    CU(h, cudaGetLastError());
    return MUSIC_B200_OK;
}

// host-buffer conveniences: upload, reduce, download (GUI-rate calls; not a throughput path)
int music_b200_reduce_angles_host(music_b200 *h, const float *angles, const float *levels, uint32_t nwindows, int weighted,
                                  float *mean_deg, float *resultant, float *weight_sum)
{
    if (h && !h->kids.empty()) return music_b200_reduce_angles_host(h->kids[0], angles, levels, nwindows, weighted, mean_deg, resultant, weight_sum);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    if (!angles || !mean_deg) return fail(h, MUSIC_B200_EINVAL, "angles and mean_deg must not be NULL");
    if (weighted && !levels) return fail(h, MUSIC_B200_EINVAL, "level weighting needs levels");
    float *d_a = nullptr, *d_l = nullptr, *d_o = nullptr;
    const size_t nb = (size_t)nwindows * h->n * sizeof(float);
    int rc = MUSIC_B200_OK;
    {
        std::lock_guard<std::mutex> g(h->mutex);
        CU(h, cudaSetDevice(h->device));
        if (cudaMalloc(&d_a, std::max<size_t>(nb, 4)) != cudaSuccess || cudaMalloc(&d_o, 3 * h->n * sizeof(float)) != cudaSuccess ||
            (levels && cudaMalloc(&d_l, std::max<size_t>(nb, 4)) != cudaSuccess)) {
            cudaFree(d_a); cudaFree(d_o); cudaFree(d_l);
            return fail(h, MUSIC_B200_ENOMEM, "cudaMalloc failed for the reducer buffers");
        }
        cudaMemcpy(d_a, angles, nb, cudaMemcpyHostToDevice);
        if (levels) cudaMemcpy(d_l, levels, nb, cudaMemcpyHostToDevice);
    }
    rc = music_b200_reduce_angles_device(h, d_a, d_l, nwindows, weighted, d_o, d_o + h->n, d_o + 2 * h->n, nullptr);
    if (rc == MUSIC_B200_OK) {
        std::vector<float> out(3 * h->n);
        const cudaError_t e = cudaMemcpy(out.data(), d_o, out.size() * sizeof(float), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(h, MUSIC_B200_ECUDA, "reducer failed: %s", cudaGetErrorString(e));
        else {
            for (uint32_t i = 0; i < h->n; ++i) {
                mean_deg[i] = out[i];
                if (resultant) resultant[i] = out[h->n + i];
                if (weight_sum) weight_sum[i] = out[2 * h->n + i];
            }
        }
    }
    cudaFree(d_a); cudaFree(d_o); cudaFree(d_l);
    return rc;
}

int music_b200_reduce_spectrum_host(music_b200 *h, const float *spectrum, uint32_t nwindows, float *mean)
{
    if (h && !h->kids.empty()) return music_b200_reduce_spectrum_host(h->kids[0], spectrum, nwindows, mean);  // multi-device handle: device 0 serves this entry
    if (!h) return MUSIC_B200_EINVAL;
    if (!spectrum || !mean) return fail(h, MUSIC_B200_EINVAL, "spectrum and mean must not be NULL");
    if (nwindows == 0) return fail(h, MUSIC_B200_EINVAL, "nwindows must be >= 1");
    float *d_s = nullptr, *d_m = nullptr;
    const size_t nb = (size_t)nwindows * h->K * sizeof(float);
    {
        std::lock_guard<std::mutex> g(h->mutex);
        CU(h, cudaSetDevice(h->device));
        if (cudaMalloc(&d_s, nb) != cudaSuccess || cudaMalloc(&d_m, h->K * sizeof(float)) != cudaSuccess) {
            cudaFree(d_s); cudaFree(d_m);
            return fail(h, MUSIC_B200_ENOMEM, "cudaMalloc failed for the reducer buffers");
        }
        cudaMemcpy(d_s, spectrum, nb, cudaMemcpyHostToDevice);
    }
    int rc = music_b200_reduce_spectrum_device(h, d_s, nwindows, d_m, nullptr);
    if (rc == MUSIC_B200_OK) {
        const cudaError_t e = cudaMemcpy(mean, d_m, h->K * sizeof(float), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(h, MUSIC_B200_ECUDA, "reducer failed: %s", cudaGetErrorString(e));
    }
    cudaFree(d_s); cudaFree(d_m);
    return rc;
}

int music_b200_set_peak_mode(music_b200 *h, int mode, uint32_t exclusion_bins)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (mode != MUSIC_B200_PEAKS_TOP_BINS && mode != MUSIC_B200_PEAKS_LOCAL_MAXIMA) return fail(h, MUSIC_B200_EINVAL, "unknown peak mode %d", mode);
    if (exclusion_bins >= h->K) return fail(h, MUSIC_B200_EINVAL, "exclusion_bins must be < resolution");
    std::lock_guard<std::mutex> g(h->mutex);
    for (music_b200 *c : h->kids) {
        const int rc = music_b200_set_peak_mode(c, mode, exclusion_bins);
        if (rc) return fail(h, rc, "%s", music_b200_last_error(c));
    }
    h->peak_mode = mode;
    h->peak_excl = exclusion_bins;
    return MUSIC_B200_OK;
}

int music_b200_set_geometry(music_b200 *h, const double *positions_xy, double wavelength, uint32_t *guarded)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (!positions_xy) return fail(h, MUSIC_B200_EINVAL, "element positions must not be NULL");
    if (!(wavelength > 0.0) || !std::isfinite(wavelength)) return fail(h, MUSIC_B200_EINVAL, "wavelength must be positive and finite");
    for (uint32_t i = 0; i < 2 * h->m; ++i)
        if (!std::isfinite(positions_xy[i])) return fail(h, MUSIC_B200_EINVAL, "element positions must be finite");
    std::lock_guard<std::mutex> g(h->mutex);
    if (!h->kids.empty()) {
        for (music_b200 *c : h->kids) {
            const int rc = music_b200_set_geometry(c, positions_xy, wavelength, guarded);
            if (rc) return fail(h, rc, "%s", music_b200_last_error(c));
        }
        return MUSIC_B200_OK;
    }
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaDeviceSynchronize());  // as in set_table(): the slot being rebuilt must be idle
    const int slot = h->cur_table ^ 1;
    int rc = build_table(h, slot, positions_xy, wavelength, h->streams[0]);
    if (rc) return rc;
    h->cur_table = slot;
    if (guarded) *guarded = h->steer_guarded;
    return MUSIC_B200_OK;
}

void music_b200_steer_entry_host(const double *positions_xy, double wavelength, uint32_t resolution, uint32_t step,
                                 uint32_t antenna, float *re_im)
{
    steer_entry_host(positions_xy, wavelength, (int)resolution, (int)step, (int)antenna, &re_im[0], &re_im[1]);
}

int music_b200_get_table(music_b200 *h, float *table_c64)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (!table_c64) return fail(h, MUSIC_B200_EINVAL, "output table must not be NULL");
    if (!h->kids.empty()) return music_b200_get_table(h->kids[0], table_c64);
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaMemcpy(table_c64, h->table[h->cur_table].c64, (size_t)h->K * h->m * 2 * sizeof(float), cudaMemcpyDeviceToHost));
    return MUSIC_B200_OK;
}

int music_b200_process_device_ex(music_b200 *h, const float *d_in_c64, uint32_t nwindows, float *d_angles,
                                 float *d_levels, float *d_spectrum, int32_t *d_bins, double *d_P64, double *d_R,
                                 double *d_eigvals, void *stream)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (!h->kids.empty()) {
        // multi-device handle: the call goes to the child on whose device the input lives
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, d_in_c64) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            return fail(h, MUSIC_B200_EINVAL, "d_in_c64 is not a device pointer");
        }
        for (music_b200 *c : h->kids)
            if (c->device == at.device) {
                const int rc = music_b200_process_device_ex(c, d_in_c64, nwindows, d_angles, d_levels, d_spectrum, d_bins, d_P64, d_R, d_eigvals, stream);
                if (rc) fail(h, rc, "%s", music_b200_last_error(c));
                return rc;
            }
        return fail(h, MUSIC_B200_EINVAL, "d_in_c64 lives on device %d, which this handle does not own", at.device);
    }
    std::lock_guard<std::mutex> g(h->mutex);
    NvtxRange range("music_b200_process_device");
    CU(h, cudaSetDevice(h->device));
    if (h->gather_G > 0) {
        if ((size_t)nwindows * h->gather_G * h->n > h->gather_cap) return fail(h, MUSIC_B200_EINVAL, "gather buffer holds %zu entries, the call needs %zu", h->gather_cap, (size_t)nwindows * h->gather_G * h->n);
        ++h->gather_epoch;
    }
    return enqueue_device(h, d_in_c64, nwindows, d_angles, d_levels, d_spectrum, d_bins, d_P64, d_R, d_eigvals,
                          static_cast<cudaStream_t>(stream), 0);
}

int music_b200_process_device(music_b200 *h, const float *d_in_c64, uint32_t nwindows, float *d_angles,
                              float *d_levels, float *d_spectrum, int32_t *d_bins, void *stream)
{
    return music_b200_process_device_ex(h, d_in_c64, nwindows, d_angles, d_levels, d_spectrum, d_bins, nullptr, nullptr,
                                        nullptr, stream);
}

int music_b200_process_host(music_b200 *h, const float *in_c64, uint32_t nwindows, float *angles, float *levels,
                            float *spectrum, int32_t *bins)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (nwindows == 0) return MUSIC_B200_OK;
    if (!in_c64 || !angles) return fail(h, MUSIC_B200_EINVAL, "in_c64 and angles must not be NULL");
    std::lock_guard<std::mutex> g(h->mutex);
    NvtxRange range("music_b200_process_host");
    // lanes: the handle itself, or the per-device children of a multi-device handle; lane g takes the windows
    // w = i * G + g (round-robin at window granularity, SURVEY.md section 8e) - every lane feeds its own PCIe link
    music_b200 *self[1] = {h};
    music_b200 *const *lanes = h->kids.empty() ? self : h->kids.data();
    const uint32_t G = h->kids.empty() ? 1u : (uint32_t)h->kids.size();
    const size_t win_bytes = (size_t)h->nsamples * 2 * sizeof(float);
    // chunk: ~32 MiB of input per copy, so that H2D of chunk i+1 overlaps compute of chunk i (with the spectrum port
    // connected a window also returns K floats: bound the chunk by the larger of the two)
    const size_t per_win = std::max(win_bytes, spectrum ? (size_t)h->K * sizeof(float) : (size_t)0);
    const uint32_t per_lane = (nwindows + G - 1) / G;
    uint32_t chunk = (uint32_t)std::max<size_t>(SCAN_B, ((size_t)32 << 20) / per_win);
    chunk = std::min(chunk, (per_lane + 1) / 2 > SCAN_B ? (per_lane + 1) / 2 : per_lane);
    chunk = std::max<uint32_t>(1, chunk);
    // pageable caller memory (GNU Radio's circular buffers, numpy arrays) is pinned once and found again on later calls
    CU(h, cudaSetDevice(lanes[0]->device));
    host_register(h, in_c64, (size_t)nwindows * win_bytes, true);
    if (spectrum) host_register(h, spectrum, (size_t)nwindows * h->K * sizeof(float), false);
    int rc = MUSIC_B200_OK;
    for (uint32_t l = 0; l < G && rc == MUSIC_B200_OK; ++l) {
        music_b200 *c = lanes[l];
        if (cudaSetDevice(c->device) != cudaSuccess) { rc = fail(h, MUSIC_B200_ECUDA, "cudaSetDevice(%d) failed", c->device); break; }
        c->slot_W[0] = c->slot_W[1] = 0;  // nothing pending from an earlier (possibly failed) call
        rc = ensure_host_staging(c, chunk, spectrum != nullptr);
        if (rc && c != h) fail(h, rc, "%s", std::string(c->error).c_str());
    }
    // Each of a lane's two copy streams computes in its own workspace slot and with its own ticket counter, so H2D,
    // kernels and D2H of consecutive chunks overlap freely (the path is PCIe-bound by ~100x).
    for (uint32_t it = 0; rc == MUSIC_B200_OK && (uint64_t)it * chunk < per_lane; ++it) {
        const int s = (int)(it & 1);
        for (uint32_t l = 0; l < G && rc == MUSIC_B200_OK; ++l) {
            music_b200 *c = lanes[l];
            const uint32_t Wl = l < nwindows ? (nwindows - l + G - 1) / G : 0;  // windows of this lane
            const uint32_t i0 = it * chunk;
            if (i0 >= Wl) continue;
            const uint32_t W = std::min(chunk, Wl - i0);
            cudaStream_t st = c->streams[s];
            CU_BREAK(h, rc, cudaSetDevice(c->device));
            if (it >= 2) {
                CU_BREAK(h, rc, cudaStreamSynchronize(st));  // slot buffers free again (its D2H finished)
                flush_host_slot(c, s, angles, levels, bins, G, l);
            }
            const float *src = in_c64 + ((size_t)i0 * G + l) * h->nsamples * 2;
            {
                NvtxRange r("music_b200: H2D");
                if (G == 1) { CU_BREAK(h, rc, cudaMemcpyAsync(c->d_in[s], src, (size_t)W * win_bytes, cudaMemcpyHostToDevice, st)); }
                else { CU_BREAK(h, rc, cudaMemcpy2DAsync(c->d_in[s], win_bytes, src, (size_t)G * win_bytes, win_bytes, W, cudaMemcpyHostToDevice, st)); }
            }
            {
                NvtxRange r("music_b200: kernels");
                rc = enqueue_device(c, c->d_in[s], W, c->d_ang[s], c->d_lvl[s], spectrum ? c->d_spec[s] : nullptr, c->d_bins[s],
                                    nullptr, nullptr, nullptr, st, s);
                if (rc && c != h) fail(h, rc, "%s", std::string(c->error).c_str());
                if (rc) break;
            }
            NvtxRange r("music_b200: D2H");
            rc = download_host_slot(c, s, i0, W, levels != nullptr, bins != nullptr, st);
            if (rc && c != h) fail(h, rc, "%s", std::string(c->error).c_str());
            if (rc) break;
            if (spectrum) {
                float *dst = spectrum + ((size_t)i0 * G + l) * h->K;
                const size_t row = (size_t)h->K * sizeof(float);
                if (G == 1) { CU_BREAK(h, rc, cudaMemcpyAsync(dst, c->d_spec[s], (size_t)W * row, cudaMemcpyDeviceToHost, st)); }
                else { CU_BREAK(h, rc, cudaMemcpy2DAsync(dst, (size_t)G * row, c->d_spec[s], row, row, W, cudaMemcpyDeviceToHost, st)); }
            }
        }
    }
    // common tail, also after an error: every stream idle, nothing left pending in the slots
    cudaError_t e_sync = cudaSuccess;
    for (uint32_t l = 0; l < G; ++l) {
        music_b200 *c = lanes[l];
        cudaSetDevice(c->device);
        for (int s = 0; s < 2; ++s) {
            const cudaError_t e = cudaStreamSynchronize(c->streams[s]);
            if (e != cudaSuccess && e_sync == cudaSuccess) e_sync = e;
        }
    }
    if (rc == MUSIC_B200_OK && e_sync != cudaSuccess) rc = fail(h, MUSIC_B200_ECUDA, "stream sync failed: %s", cudaGetErrorString(e_sync));
    for (uint32_t l = 0; l < G; ++l) {
        music_b200 *c = lanes[l];
        if (rc == MUSIC_B200_OK) {
            flush_host_slot(c, 0, angles, levels, bins, G, l);
            flush_host_slot(c, 1, angles, levels, bins, G, l);
        } else {
            c->slot_W[0] = c->slot_W[1] = 0;  // nothing valid to hand out
        }
    }
    return rc;
}

int music_b200_create_multi(music_b200 **out, uint32_t m, uint32_t n, uint32_t nsamples, uint32_t resolution,
                            const float *table_c64, const int *devices, int ndev)
{
    if (!out) return fail(nullptr, MUSIC_B200_EINVAL, "out must not be NULL");
    *out = nullptr;
    if (!devices || ndev < 1 || ndev > MAX_PEERS) return fail(nullptr, MUSIC_B200_EINVAL, "need 1..%d devices (got %d)", MAX_PEERS, ndev);
    for (int i = 0; i < ndev; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return fail(nullptr, MUSIC_B200_EINVAL, "device %d listed twice", devices[i]);
    music_b200 *h = new (std::nothrow) music_b200();
    if (!h) return fail(nullptr, MUSIC_B200_ENOMEM, "out of host memory");
    h->m = m; h->n = n; h->nsamples = nsamples; h->K = resolution; h->N = m ? nsamples / m : 0;
    h->device = devices[0];
    if (const char *e = getenv("MUSIC_B200_HOSTREG")) h->hostreg = atoi(e) != 0;
    for (int i = 0; i < ndev; ++i) {
        music_b200 *c = nullptr;
        const int rc = music_b200_create(&c, m, n, nsamples, resolution, table_c64, devices[i]);  // (sets the create error text)
        if (rc != MUSIC_B200_OK) {
            music_b200_destroy(h);
            return rc;
        }
        h->kids.push_back(c);
    }
    // peer access between every pair (the sharded device entry stores peak bins straight into the peers' buffers)
    for (int i = 0; i < ndev; ++i) {
        cudaSetDevice(devices[i]);
        for (int j = 0; j < ndev; ++j) {
            if (i == j) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) == cudaSuccess && can) {
                const cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
                if (e != cudaSuccess) cudaGetLastError();  // already enabled is fine
            }
        }
    }
    *out = h;
    return MUSIC_B200_OK;
}

int music_b200_device_count(const music_b200 *h) { return h ? (h->kids.empty() ? 1 : (int)h->kids.size()) : 0; }

/* ---- fused all-gather of the peak bins across processes (one GPU per process) ---- */
int music_b200_gather_create(music_b200 *h, uint32_t total_windows, unsigned char *ipc_handles /* [2][64] */)
{
    if (!h || !ipc_handles) return MUSIC_B200_EINVAL;
    if (!h->kids.empty()) return fail(h, MUSIC_B200_EINVAL, "gather_create applies to single-device handles (a multi-device handle gathers in process_device_sharded)");
    std::lock_guard<std::mutex> g(h->mutex);
    CU(h, cudaSetDevice(h->device));
    if (h->gather_buf) return fail(h, MUSIC_B200_EINVAL, "gather buffer already created");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    const size_t elems = (size_t)total_windows * h->n;
    CU(h, cudaMalloc(&h->gather_buf, std::max<size_t>(elems, 1) * sizeof(int32_t)));
    CU(h, cudaMalloc(&h->gather_flags, MAX_PEERS * sizeof(unsigned)));
    CU(h, cudaMemset(h->gather_buf, 0xff, std::max<size_t>(elems, 1) * sizeof(int32_t)));
    CU(h, cudaMemset(h->gather_flags, 0, MAX_PEERS * sizeof(unsigned)));
    h->gather_cap = elems;
    cudaIpcMemHandle_t hb, hf;
    CU(h, cudaIpcGetMemHandle(&hb, h->gather_buf));
    CU(h, cudaIpcGetMemHandle(&hf, h->gather_flags));
    memcpy(ipc_handles, &hb, 64);
    memcpy(ipc_handles + 64, &hf, 64);
    return MUSIC_B200_OK;
}

int music_b200_gather_attach(music_b200 *h, int nranks, int rank, const unsigned char *all_handles /* [nranks][2][64] */)
{
    if (!h || !all_handles) return MUSIC_B200_EINVAL;
    if (nranks < 1 || nranks > MAX_PEERS || rank < 0 || rank >= nranks) return fail(h, MUSIC_B200_EINVAL, "need 1 <= nranks <= %d and 0 <= rank < nranks", MAX_PEERS);
    std::lock_guard<std::mutex> g(h->mutex);
    if (!h->gather_buf) return fail(h, MUSIC_B200_EINVAL, "call gather_create first");
    CU(h, cudaSetDevice(h->device));
    for (int p = 0; p < nranks; ++p) {
        if (p == rank) {
            h->peer_bins[p] = h->gather_buf;
            h->peer_flags[p] = h->gather_flags;
            continue;
        }
        cudaIpcMemHandle_t hb, hf;
        memcpy(&hb, all_handles + (size_t)p * 128, 64);
        memcpy(&hf, all_handles + (size_t)p * 128 + 64, 64);
        void *pb = nullptr, *pf = nullptr;
        CU(h, cudaIpcOpenMemHandle(&pb, hb, cudaIpcMemLazyEnablePeerAccess));
        CU(h, cudaIpcOpenMemHandle(&pf, hf, cudaIpcMemLazyEnablePeerAccess));
        h->peer_bins[p] = static_cast<int32_t *>(pb);
        h->peer_flags[p] = static_cast<unsigned *>(pf);
        h->peer_ipc[p] = true;
    }
    h->gather_G = nranks;
    h->gather_rank = rank;
    h->gather_epoch = 0;
    return MUSIC_B200_OK;
}

int music_b200_gather_wait(music_b200 *h, void *stream)
{
    if (!h) return MUSIC_B200_EINVAL;
    std::lock_guard<std::mutex> g(h->mutex);
    if (h->gather_G <= 0 || !h->gather_flags) return fail(h, MUSIC_B200_EINVAL, "no gather attached");
    CU(h, cudaSetDevice(h->device));
    gather_wait_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(h->gather_flags, h->gather_G, h->gather_epoch);
    h->launches++;
    CU(h, cudaGetLastError());
    return MUSIC_B200_OK;
}

const int32_t *music_b200_gather_buffer(const music_b200 *h) { return h ? h->gather_buf : nullptr; }

int music_b200_gather_read(music_b200 *h, int32_t *host_out, uint32_t count)
{
    if (!h || !host_out) return MUSIC_B200_EINVAL;
    std::lock_guard<std::mutex> g(h->mutex);
    if (!h->gather_buf || count > h->gather_cap) return fail(h, MUSIC_B200_EINVAL, "gather buffer holds %zu entries", h->gather_cap);
    CU(h, cudaSetDevice(h->device));
    CU(h, cudaMemcpy(host_out, h->gather_buf, (size_t)count * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return MUSIC_B200_OK;
}

/* ---- one call, G devices, inputs resident: shard g holds the windows w = i * G + g ---- */
int music_b200_process_device_sharded(music_b200 *h, const float *const *d_in_c64, uint32_t nwindows_total, float *const *d_angles,
                                      float *const *d_levels, int32_t *const *d_bins_all, void *const *streams)
{
    if (!h) return MUSIC_B200_EINVAL;
    if (h->kids.empty()) return fail(h, MUSIC_B200_EINVAL, "process_device_sharded needs a handle from music_b200_create_multi");
    if (!d_in_c64 || !d_angles) return fail(h, MUSIC_B200_EINVAL, "d_in_c64 and d_angles must not be NULL");
    std::lock_guard<std::mutex> g(h->mutex);
    NvtxRange range("music_b200_process_device_sharded");
    const int G = (int)h->kids.size();
    int rc = MUSIC_B200_OK;
    for (int l = 0; l < G && rc == MUSIC_B200_OK; ++l) {
        music_b200 *c = h->kids[l];
        const uint32_t Wl = (uint32_t)l < nwindows_total ? (nwindows_total - l + G - 1) / G : 0;
        if (!Wl) continue;
        CU_BREAK(h, rc, cudaSetDevice(c->device));
        // the scan epilogue of shard l stores its peak bins at stream position w = i * G + l of EVERY device's array
        c->gather_G = d_bins_all ? G : 0;
        c->gather_rank = l;
        for (int p = 0; p < G; ++p) { c->peer_bins[p] = d_bins_all ? d_bins_all[p] : nullptr; c->peer_flags[p] = nullptr; }
        rc = enqueue_device(c, d_in_c64[l], Wl, d_angles[l], d_levels ? d_levels[l] : nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                            streams ? static_cast<cudaStream_t>(streams[l]) : nullptr, 0);
        c->gather_G = 0;
        if (rc) fail(h, rc, "%s", std::string(c->error).c_str());
    }
    return rc;
}

void music_b200_destroy(music_b200 *h)
{
    if (!h) return;
    for (music_b200 *c : h->kids) music_b200_destroy(c);
    h->kids.clear();
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (const music_b200::HostReg &r : h->hostregs) cudaHostUnregister(reinterpret_cast<void *>(r.base));
    h->hostregs.clear();
    for (int p = 0; p < MAX_PEERS; ++p)
        if (h->peer_ipc[p]) { cudaIpcCloseMemHandle(h->peer_bins[p]); cudaIpcCloseMemHandle(h->peer_flags[p]); }
    cudaFree(h->gather_buf);
    cudaFree(h->gather_flags);
    cudaGetLastError();
    free_host_staging(h);
    for (int i = 0; i < NSLOT; ++i) {
        Workspace &ws = h->ws[i];
        cudaFree(ws.R); cudaFree(ws.ev); cudaFree(ws.Vt); cudaFree(ws.P64);
        if (ws.scan_done) cudaEventDestroy(ws.scan_done);
    }
    cudaFree(h->fused_trace);
    cudaFree(h->f8_stats);
    cudaFree(h->work_ctr);
    cudaFree(h->steer_pos); cudaFree(h->steer_count); cudaFree(h->steer_list); cudaFree(h->steer_vals);
    if (h->fused_done) cudaEventDestroy(h->fused_done);
    for (int i = 0; i < 2; ++i) {
        cudaFree(h->table[i].c64); cudaFree(h->table[i].soa); cudaFree(h->table[i].fz); cudaFree(h->table[i].na_max);
        if (h->streams[i]) cudaStreamDestroy(h->streams[i]);
        if (h->done[i]) cudaEventDestroy(h->done[i]);
    }
    for (cudaEvent_t e : h->tev) cudaEventDestroy(e);
    delete h;
}

}  // extern "C"
