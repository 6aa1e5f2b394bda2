// music_kernels.cuh - sm_100a kernels for the MUSIC DOA hot path (v1: three-stage pipeline).
//
// Stage map (reference = /root/reference/lib/baz_music_doa.cc):
//   K1 cov_tile_kernel / cov_generic_kernel  <- :74-85  widen c64->f64, R = x x^H / N
//   K2 eig_kernel                            <- :88-93  Hermitian eig, ascending, noise/signal split
//   K3 scan_kernel (+ topn_kernel)           <- :103-155 pseudospectrum, top-n, float casts
//   prep_table_kernel                        <- :110-112 (table widening, hoisted out of the loop)
//
// All arithmetic is fp64 (fp32 inputs are widened exactly; fp32 x fp32 products are exact in
// fp64), because P(theta) = 1/||G^H a||^2 is ill-conditioned at the peak (DESIGN.md).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace music {

constexpr int MAXM = 16;
constexpr int TILE = 256;        // angles per steering-table tile == scan CTA size
constexpr int SCAN_B = 8;        // windows per scan CTA
constexpr double COMPLEMENT_GUARD = 0.0078125;  // 2^-7: below this fraction of ||a||^2 use the direct form

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float4 ldg_stream(const float4 *p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

// ------------------------------------------------------------------------------------------
// K1: covariance, one warp per (window, 4x4 antenna tile).  Lanes stride over snapshots with
// 128-bit coalesced loads (a snapshot's 4-antenna group is one 32-byte sector), accumulate the
// tile in fp64 registers, then a warp-shuffle reduction.  R is written as full M x M complex
// (row-major, interleaved re/im), lower triangle by conjugate symmetry.
//   DIAG tile (I == I): Hermitian half only - 4 real diagonals + 6 complex = 16 accumulators,
//                        32 DFMA per snapshot (2*M^2 for M = 4).
//   OFF  tile (I <  J): full 4x4 complex block = 32 accumulators, 64 DFMA per snapshot.
// ------------------------------------------------------------------------------------------
template <bool OFF>
__global__ void __launch_bounds__(256) cov_tile_kernel(const float *__restrict__ in, double *__restrict__ R,
                                                       int W, int N, int M)
{
    const int T = M >> 2;                                   // tiles per dimension
    const int tiles = OFF ? (T * (T - 1)) / 2 : T;          // tiles of this kind per window
    const long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (item >= (long long)W * tiles) return;
    const int w = (int)(item / tiles);
    int t = (int)(item % tiles);
    int I, J;
    if (OFF) {  // enumerate I < J
        I = 0;
        while (t >= T - 1 - I) { t -= T - 1 - I; ++I; }
        J = I + 1 + t;
    } else {
        I = J = t;
    }
    const float4 *base = reinterpret_cast<const float4 *>(in) + (size_t)w * N * (M >> 1);
    const int rowq = M >> 1;  // float4 per snapshot

    double acc[OFF ? 32 : 16];
#pragma unroll
    for (int i = 0; i < (OFF ? 32 : 16); ++i) acc[i] = 0.0;

    constexpr int U = 4;  // snapshots in flight per lane
    for (int c0 = lane; c0 < N; c0 += 32 * U) {
        float4 xa[U][2], xb[U][2];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + 32 * u;
            if (c < N) {
                const float4 *p = base + (size_t)c * rowq;
                xa[u][0] = ldg_stream(p + 2 * I);
                xa[u][1] = ldg_stream(p + 2 * I + 1);
                if (OFF) {
                    xb[u][0] = ldg_stream(p + 2 * J);
                    xb[u][1] = ldg_stream(p + 2 * J + 1);
                }
            } else {
                xa[u][0] = xa[u][1] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (OFF) xb[u][0] = xb[u][1] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            double ar[4], ai[4];
            ar[0] = xa[u][0].x; ai[0] = xa[u][0].y; ar[1] = xa[u][0].z; ai[1] = xa[u][0].w;
            ar[2] = xa[u][1].x; ai[2] = xa[u][1].y; ar[3] = xa[u][1].z; ai[3] = xa[u][1].w;
            if (OFF) {
                double br[4], bi[4];
                br[0] = xb[u][0].x; bi[0] = xb[u][0].y; br[1] = xb[u][0].z; bi[1] = xb[u][0].w;
                br[2] = xb[u][1].x; bi[2] = xb[u][1].y; br[3] = xb[u][1].z; bi[3] = xb[u][1].w;
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {  // x_i * conj(y_j)
                        acc[2 * (i * 4 + j)] = fma(ar[i], br[j], fma(ai[i], bi[j], acc[2 * (i * 4 + j)]));
                        acc[2 * (i * 4 + j) + 1] = fma(ai[i], br[j], fma(-ar[i], bi[j], acc[2 * (i * 4 + j) + 1]));
                    }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i] = fma(ar[i], ar[i], fma(ai[i], ai[i], acc[i]));
                int e = 4;
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = i + 1; j < 4; ++j) {
                        acc[e] = fma(ar[i], ar[j], fma(ai[i], ai[j], acc[e]));
                        acc[e + 1] = fma(ai[i], ar[j], fma(-ar[i], ai[j], acc[e + 1]));
                        e += 2;
                    }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < (OFF ? 32 : 16); ++i) acc[i] = warp_sum(acc[i]);

    if (lane == 0) {
        const double dn = (double)N;
        double *Rw = R + (size_t)w * M * M * 2;
        if (OFF) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const double re = acc[2 * (i * 4 + j)] / dn, im = acc[2 * (i * 4 + j) + 1] / dn;
                    const int r = 4 * I + i, c = 4 * J + j;
                    Rw[2 * (r * M + c)] = re;  Rw[2 * (r * M + c) + 1] = im;
                    Rw[2 * (c * M + r)] = re;  Rw[2 * (c * M + r) + 1] = -im;
                }
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = 4 * I + i;
                Rw[2 * (r * M + r)] = acc[i] / dn;
                Rw[2 * (r * M + r) + 1] = 0.0;
            }
            int e = 4;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = i + 1; j < 4; ++j) {
                    const double re = acc[e] / dn, im = acc[e + 1] / dn;
                    const int r = 4 * I + i, c = 4 * I + j;
                    Rw[2 * (r * M + c)] = re;  Rw[2 * (r * M + c) + 1] = im;
                    Rw[2 * (c * M + r)] = re;  Rw[2 * (c * M + r) + 1] = -im;
                    e += 2;
                }
        }
    }
}

// ------------------------------------------------------------------------------------------
// K1 (M = 4, the headline shape): TMA-staged covariance.  Persistent CTAs (one per SM), one warp
// per window, and a private ring of COV_STAGES x COV_CHUNK bytes per warp filled by 1-D bulk
// async copies (cp.async.bulk, SASS UBLKCP) that complete on mbarriers.  The producer is lane 0
// of the same warp, so "slot free" is just program order (__syncwarp) and only "slot full"
// needs a barrier.  The ring runs across window boundaries, i.e. the next window's first
// chunks are already in flight during the warp-shuffle reduction of the current one.
// Per snapshot and lane: 2 LDS.128, 8 F2F (exact widening), 32 DFMA into 16 accumulators
// (Hermitian half of x x^H).  Bytes in flight per SM = 8 warps x (STAGES-1) x 4 KiB.
// ------------------------------------------------------------------------------------------
constexpr int COV_CHUNK = 4096;  // bytes per stage = 128 snapshots of 4 antennas
constexpr int COV_WARPS = 8;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// L2 eviction policies.  The input stream is read exactly once (1.3 GB per launch through a 126 MB L2): marking it
// evict_first keeps it from pushing out the steering tables, which every SM re-reads but some only at the end of a launch
// (the fp64 table of the drain workers came back from DRAM at ~3 k cycles per row without this).
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ double ldg_f64_hint(const double *p, uint64_t policy)
{
    double v;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(policy));
    return v;
}
__device__ __forceinline__ float4 ldg_f32x4_hint(const float4 *p, uint64_t policy)
{
    float4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(policy));
    return v;
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ void cov4_accumulate(double (&acc)[16], const float4 a, const float4 b)
{
    const double r0 = a.x, i0 = a.y, r1 = a.z, i1 = a.w, r2 = b.x, i2 = b.y, r3 = b.z, i3 = b.w;
    acc[0] = fma(r0, r0, fma(i0, i0, acc[0]));
    acc[1] = fma(r1, r1, fma(i1, i1, acc[1]));
    acc[2] = fma(r2, r2, fma(i2, i2, acc[2]));
    acc[3] = fma(r3, r3, fma(i3, i3, acc[3]));
    // R_ij += x_i conj(x_j), i < j
    acc[4] = fma(r0, r1, fma(i0, i1, acc[4]));    acc[5] = fma(i0, r1, fma(-r0, i1, acc[5]));    // 01
    acc[6] = fma(r0, r2, fma(i0, i2, acc[6]));    acc[7] = fma(i0, r2, fma(-r0, i2, acc[7]));    // 02
    acc[8] = fma(r0, r3, fma(i0, i3, acc[8]));    acc[9] = fma(i0, r3, fma(-r0, i3, acc[9]));    // 03
    acc[10] = fma(r1, r2, fma(i1, i2, acc[10]));  acc[11] = fma(i1, r2, fma(-r1, i2, acc[11]));  // 12
    acc[12] = fma(r1, r3, fma(i1, i3, acc[12]));  acc[13] = fma(i1, r3, fma(-r1, i3, acc[13]));  // 13
    acc[14] = fma(r2, r3, fma(i2, i3, acc[14]));  acc[15] = fma(i2, r3, fma(-r2, i3, acc[15]));  // 23
}

template <int STAGES>
__global__ void __launch_bounds__(COV_WARPS * 32, 1) cov4_tma_kernel(const float *__restrict__ in, double *__restrict__ R,
                                                                     int W, int N)
{
    extern __shared__ __align__(128) unsigned char cov_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(cov_smem) + warp * STAGES;  // first 1 KiB: barriers
    unsigned char *ring = cov_smem + 1024 + (size_t)warp * STAGES * COV_CHUNK;
    const uint32_t bar0 = smem_u32(bars), ring0 = smem_u32(ring);

    const int gw = blockIdx.x * COV_WARPS + warp, total_warps = gridDim.x * COV_WARPS;
    const size_t win_bytes = (size_t)N * 32;
    const int cpw = (int)((win_bytes + COV_CHUNK - 1) / COV_CHUNK);  // chunks per window
    const int nwin = gw < W ? (W - gw + total_warps - 1) / total_warps : 0;
    const long long total = (long long)nwin * cpw;
    const unsigned char *src0 = reinterpret_cast<const unsigned char *>(in);

    if (lane == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();

    const uint64_t pol_stream = l2_policy_evict_first();
    auto issue = [&](long long c) {  // lane 0 only
        const int j = (int)(c / cpw), q = (int)(c % cpw);
        const size_t off = (size_t)q * COV_CHUNK;
        const uint32_t bytes = (uint32_t)min((size_t)COV_CHUNK, win_bytes - off);
        const int slot = (int)(c % STAGES);
        const unsigned char *src = src0 + ((size_t)gw + (size_t)j * total_warps) * win_bytes + off;
        mbar_expect_tx(bar0 + 8 * slot, bytes);
        bulk_g2s_hint(ring0 + slot * COV_CHUNK, src, bytes, bar0 + 8 * slot, pol_stream);
    };
    if (lane == 0)
        for (long long c = 0; c < total && c < STAGES; ++c) issue(c);

    double acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.0;

    int q = 0, j = 0, slot = 0;
    uint32_t parity = 0;
    for (long long c = 0; c < total; ++c) {
        while (!mbar_try_wait(bar0 + 8 * slot, parity)) {}
        const size_t off = (size_t)q * COV_CHUNK;
        const int nsnap = (int)(min((size_t)COV_CHUNK, win_bytes - off) >> 5);
        const float4 *buf = reinterpret_cast<const float4 *>(ring + (size_t)slot * COV_CHUNK);
        if (nsnap == COV_CHUNK / 32) {
            float4 xa[4], xb[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                xa[u] = buf[2 * (lane + 32 * u)];
                xb[u] = buf[2 * (lane + 32 * u) + 1];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) cov4_accumulate(acc, xa[u], xb[u]);
        } else {
            for (int s = lane; s < nsnap; s += 32) cov4_accumulate(acc, buf[2 * s], buf[2 * s + 1]);
        }
        __syncwarp();  // every lane is done reading the slot -> it may be refilled
        if (lane == 0 && c + STAGES < total) issue(c + STAGES);
        if (++slot == STAGES) { slot = 0; parity ^= 1; }
        if (++q == cpw) {
            q = 0;
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = warp_sum(acc[i]);
            if (lane == 0) {
                const double dn = (double)N;
                double *Rw = R + ((size_t)gw + (size_t)j * total_warps) * 32;
                Rw[0] = acc[0] / dn;   Rw[1] = 0.0;   // (0,0)
                Rw[10] = acc[1] / dn;  Rw[11] = 0.0;  // (1,1)
                Rw[20] = acc[2] / dn;  Rw[21] = 0.0;  // (2,2)
                Rw[30] = acc[3] / dn;  Rw[31] = 0.0;  // (3,3)
                int e = 4;
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = a + 1; b < 4; ++b) {
                        const double re = acc[e] / dn, im = acc[e + 1] / dn;
                        Rw[2 * (a * 4 + b)] = re;  Rw[2 * (a * 4 + b) + 1] = im;
                        Rw[2 * (b * 4 + a)] = re;  Rw[2 * (b * 4 + a) + 1] = -im;
                        e += 2;
                    }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = 0.0;
            ++j;
        }
    }
}

// Generic-M covariance (any 2 <= M <= MAXM, used when M % 4 != 0): one CTA per window, thread
// (entry e, slice s) accumulates R_ij over snapshots c = s, s+S, ...; slices summed in smem.
__global__ void __launch_bounds__(256) cov_generic_kernel(const float *__restrict__ in, double *__restrict__ R,
                                                          int W, int N, int M)
{
    extern __shared__ double sm[];  // [S][E][2]
    const int w = blockIdx.x;
    const int E = M * (M + 1) / 2;
    const int S = blockDim.x / E;
    const int e = threadIdx.x % E, s = threadIdx.x / E;
    int i = 0, rem = e;
    while (rem >= M - i) { rem -= M - i; ++i; }
    const int j = i + rem;
    const float2 *x = reinterpret_cast<const float2 *>(in) + (size_t)w * N * M;
    double re = 0.0, im = 0.0;
    if (s < S) {
        for (int c = s; c < N; c += S) {
            const float2 a = x[(size_t)c * M + i], b = x[(size_t)c * M + j];
            const double ar = a.x, ai = a.y, br = b.x, bi = b.y;
            re = fma(ar, br, fma(ai, bi, re));
            im = fma(ai, br, fma(-ar, bi, im));
        }
        sm[2 * (s * E + e)] = re;
        sm[2 * (s * E + e) + 1] = im;
    }
    __syncthreads();
    if (threadIdx.x < E) {
        re = 0.0; im = 0.0;
        for (int q = 0; q < S; ++q) { re += sm[2 * (q * E + e)]; im += sm[2 * (q * E + e) + 1]; }
        re /= (double)N; im /= (double)N;
        double *Rw = R + (size_t)w * M * M * 2;
        if (i == j) im = 0.0;
        Rw[2 * (i * M + j)] = re;  Rw[2 * (i * M + j) + 1] = im;
        Rw[2 * (j * M + i)] = re;  Rw[2 * (j * M + i) + 1] = -im;
    }
}

// ------------------------------------------------------------------------------------------
// K2: Hermitian eigendecomposition, cyclic two-sided complex Jacobi, one thread per window
// (SIMT over windows).  MT > 0: compile-time M (register arrays); MT == 0: runtime M <= MAXM.
// Output Vt[w][j][i] = component i of eigenvector j, eigenvalues ascending (stable on ties),
// so vectors 0..M-n-1 span the noise subspace G (:93) and M-n..M-1 the signal subspace.
// ------------------------------------------------------------------------------------------
template <int MA>
__device__ __forceinline__ void jacobi_rotate(double (&Ar)[MA][MA], double (&Ai)[MA][MA], double (&Vr)[MA][MA],
                                              double (&Vi)[MA][MA], const int p, const int q, const int M)
{
    const double gr = Ar[p][q], gi = Ai[p][q];
    const double g = sqrt(gr * gr + gi * gi);
    if (g == 0.0) return;
    const double app = Ar[p][p], aqq = Ar[q][q];
    const double er = gr / g, ei = gi / g;
    const double theta = (aqq - app) / (2.0 * g);
    double t = 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
    if (theta < 0.0) t = -t;
    const double c = 1.0 / sqrt(t * t + 1.0);
    const double s = t * c;
    const double swr = s * er, swi = s * ei;  // s * e,  e = a_pq / |a_pq|
#pragma unroll
    for (int k = 0; k < MA; ++k) {
        if (k >= M) break;
        if (k == p || k == q) continue;
        const double kpr = Ar[k][p], kpi = Ai[k][p], kqr = Ar[k][q], kqi = Ai[k][q];
        const double npr = c * kpr - (swr * kqr + swi * kqi);  // a_kp' = c a_kp - conj(s e) a_kq
        const double npi = c * kpi - (swr * kqi - swi * kqr);
        const double nqr = c * kqr + (swr * kpr - swi * kpi);  // a_kq' = (s e) a_kp + c a_kq
        const double nqi = c * kqi + (swr * kpi + swi * kpr);
        Ar[k][p] = npr; Ai[k][p] = npi; Ar[k][q] = nqr; Ai[k][q] = nqi;
        Ar[p][k] = npr; Ai[p][k] = -npi; Ar[q][k] = nqr; Ai[q][k] = -nqi;
    }
    Ar[p][p] = app - t * g; Ai[p][p] = 0.0;
    Ar[q][q] = aqq + t * g; Ai[q][q] = 0.0;
    Ar[p][q] = 0.0; Ai[p][q] = 0.0; Ar[q][p] = 0.0; Ai[q][p] = 0.0;
#pragma unroll
    for (int k = 0; k < MA; ++k) {
        if (k >= M) break;
        const double kpr = Vr[k][p], kpi = Vi[k][p], kqr = Vr[k][q], kqi = Vi[k][q];
        Vr[k][p] = c * kpr - (swr * kqr + swi * kqi);
        Vi[k][p] = c * kpi - (swr * kqi - swi * kqr);
        Vr[k][q] = c * kqr + (swr * kpr - swi * kpi);
        Vi[k][q] = c * kqi + (swr * kpi + swi * kpr);
    }
}

// Strict total order used for the ascending sort: by value, NaN last, ties by column index
// (stable).  A total order makes the ranks a permutation even for NaN eigenvalues, so every
// output slot is written.
__device__ __forceinline__ bool eig_before(double wl, int l, double wj, int j)
{
    const bool nl = wl != wl, nj = wj != wj;
    if (nl || nj) return (!nl && nj) || (nl && nj && l < j);
    return (wl < wj) || (wl == wj && l < j);
}

// Branch-free variant for the fully unrolled M = 4 solver: no early-out, reciprocal square roots
// instead of sqrt + divide (3 rsqrt + 1 reciprocal per rotation), so that the two disjoint
// rotations of a parallel-ordering step are one basic block and their dependent chains
// interleave.  The eigensolver is latency-bound (one lane per window), and in the fused kernel
// its latency is the pipeline's tail.
// The rotation arithmetic of the M = 4 solvers, written with explicit rounding intrinsics so that the one-lane solver
// (herm_eig_body<4, true>) and the four-lanes-per-window solver of the fused kernel (herm_eig4_coop) round identically
// whatever the compiler would contract: their eigenvectors are bit-identical (tests compare the two paths exactly).
__device__ __forceinline__ void jrot_params(const double gr, const double gi, const double app, const double aqq, double &c,
                                            double &swr, double &swi, double &t, double &g)
{
    const double gg = fma(gr, gr, __dmul_rn(gi, gi));
    const bool nz = gg > 0.0;                                  // false for 0 and NaN (NaN then propagates via g)
    const double rg = nz ? rsqrt(gg) : 0.0;                    // 1 / |a_pq|
    g = (gg != gg) ? gg : __dmul_rn(gg, rg);                   // |a_pq| (NaN stays NaN)
    const double er = __dmul_rn(gr, rg), ei = __dmul_rn(gi, rg);
    double theta = __dmul_rn(__dmul_rn(0.5, __dsub_rn(aqq, app)), rg);
    theta = fmin(fmax(theta, -1e150), 1e150);                  // keeps theta^2 finite; |t| ~ 1/(2|theta|) ~ 0 there
    const double q1 = fma(theta, theta, 1.0);
    const double sq = __dmul_rn(q1, rsqrt(q1));                // sqrt(theta^2 + 1)
    t = __ddiv_rn(1.0, __dadd_rn(fabs(theta), sq));
    t = nz ? copysign(t, theta) : 0.0;
    c = rsqrt(fma(t, t, 1.0));
    const double sn = __dmul_rn(t, c);
    swr = __dmul_rn(sn, er);                                   // s * e,  e = a_pq / |a_pq|
    swi = __dmul_rn(sn, ei);
}

// (kp, kq) -> (c kp - conj(sw) kq, c kq + sw kp)
__device__ __forceinline__ void jrot_mix(const double c, const double swr, const double swi, const double kpr, const double kpi,
                                         const double kqr, const double kqi, double &npr, double &npi, double &nqr, double &nqi)
{
    npr = fma(c, kpr, -fma(swr, kqr, __dmul_rn(swi, kqi)));
    npi = fma(c, kpi, -fma(swr, kqi, __dmul_rn(-swi, kqr)));
    nqr = fma(c, kqr, fma(swr, kpr, __dmul_rn(-swi, kpi)));
    nqi = fma(c, kqi, fma(swr, kpi, __dmul_rn(swi, kpr)));
}

// one half of jrot_mix with the same roundings: isq ? (c own + sw mate) : (c own - conj(sw) mate)
__device__ __forceinline__ void jrot_mix_half(const double c, const double swr, const double swi, const bool isq, const double ownr,
                                              const double owni, const double mr, const double mi, double &re, double &im)
{
    const double se = isq ? -swi : swi;
    const double inr = fma(swr, mr, __dmul_rn(se, mi));
    const double ini = fma(swr, mi, __dmul_rn(-se, mr));
    re = fma(c, ownr, isq ? inr : -inr);
    im = fma(c, owni, isq ? ini : -ini);
}

// eigenvector component times the phase that makes component 0 real
__device__ __forceinline__ void eig_out4(const double vr, const double vi, const double pr, const double pi, double &re, double &im)
{
    re = fma(vr, pr, -__dmul_rn(vi, pi));
    im = fma(vr, pi, __dmul_rn(vi, pr));
}

template <int MA>
__device__ __forceinline__ void jacobi_rotate_bf(double (&Ar)[MA][MA], double (&Ai)[MA][MA], double (&Vr)[MA][MA],
                                                 double (&Vi)[MA][MA], const int p, const int q)
{
    const double app = Ar[p][p], aqq = Ar[q][q];
    double c, swr, swi, t, g;
    jrot_params(Ar[p][q], Ai[p][q], app, aqq, c, swr, swi, t, g);
#pragma unroll
    for (int k = 0; k < MA; ++k) {
        if (k == p || k == q) continue;
        double npr, npi, nqr, nqi;
        jrot_mix(c, swr, swi, Ar[k][p], Ai[k][p], Ar[k][q], Ai[k][q], npr, npi, nqr, nqi);
        Ar[k][p] = npr; Ai[k][p] = npi; Ar[k][q] = nqr; Ai[k][q] = nqi;
        Ar[p][k] = npr; Ai[p][k] = -npi; Ar[q][k] = nqr; Ai[q][k] = -nqi;
    }
    Ar[p][p] = fma(-t, g, app); Ai[p][p] = 0.0;
    Ar[q][q] = fma(t, g, aqq);  Ai[q][q] = 0.0;
    Ar[p][q] = 0.0; Ai[p][q] = 0.0; Ar[q][p] = 0.0; Ai[q][p] = 0.0;
#pragma unroll
    for (int k = 0; k < MA; ++k) {
        double npr, npi, nqr, nqi;
        jrot_mix(c, swr, swi, Vr[k][p], Vi[k][p], Vr[k][q], Vi[k][q], npr, npi, nqr, nqi);
        Vr[k][p] = npr; Vi[k][p] = npi; Vr[k][q] = nqr; Vi[k][q] = nqi;
    }
}

// Unit phasor p = conj(v0)/|v0| that makes component 0 of an eigenvector real and >= 0 (any
// phase is a valid eigenvector; MUSIC only uses |e^H a| and the projector).  The scan kernels
// rely on Im(v0) == 0 to drop two multiply-adds per bin.
__device__ __forceinline__ void eig_phase(double v0r, double v0i, double &pr, double &pi)
{
    const double mag = sqrt(v0r * v0r + v0i * v0i);
    if (mag > 0.0) { pr = v0r / mag; pi = -v0i / mag; }
    else { pr = 1.0; pi = 0.0; }  // v0 == 0 (or NaN): leave the vector as it is
}

// MA = array extent; STATIC: M == MA at compile time, everything unrolled into registers
// (M = 4); otherwise runtime M <= MA with the matrices in local memory.
// Rw: M x M complex (row-major, interleaved) in global or shared memory; ew (may be null): M
// ascending eigenvalues; vw: Vt[j][i], eigenvector j contiguous.
// A covariance with an Inf entry (an Inf input sample) has ||R||_F^2 = Inf, and off <= c * fro holds for off = fro = Inf:
// without this check the Jacobi loops stop at once and hand out the identity's columns as eigenvectors, i.e. a finite
// spectrum and a peak.  The reference's eig_sym gets no decomposition there and work() inserts no peak; the solvers
// therefore return NaN eigenvalues and eigenvectors for any R whose ||R||_F^2 is not finite, as they already did for NaN.
constexpr double DBL_MAX_FRO = 1.7976931348623157e308;

template <int MA, bool STATIC>
__device__ __forceinline__ void herm_eig_body(const double *Rw, double *ew, double *vw, const int M)
{
    double Ar[MA][MA], Ai[MA][MA], Vr[MA][MA], Vi[MA][MA];
    if (STATIC) {
#pragma unroll
        for (int i = 0; i < MA; ++i)
#pragma unroll
            for (int j = 0; j < MA; ++j) {
                Ar[i][j] = Rw[2 * (i * MA + j)];
                Ai[i][j] = Rw[2 * (i * MA + j) + 1];
                Vr[i][j] = (i == j) ? 1.0 : 0.0;
                Vi[i][j] = 0.0;
            }
    } else {
        for (int i = 0; i < M; ++i)
            for (int j = 0; j < M; ++j) {
                Ar[i][j] = Rw[2 * (i * M + j)];
                Ai[i][j] = Rw[2 * (i * M + j) + 1];
                Vr[i][j] = (i == j) ? 1.0 : 0.0;
                Vi[i][j] = 0.0;
            }
    }
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, fro = 0.0;
        if (STATIC) {
#pragma unroll
            for (int i = 0; i < MA; ++i)
#pragma unroll
                for (int j = 0; j < MA; ++j) {
                    const double e2 = Ar[i][j] * Ar[i][j] + Ai[i][j] * Ai[i][j];
                    fro += e2;
                    if (i != j) off += e2;
                }
        } else {
            for (int i = 0; i < M; ++i)
                for (int j = 0; j < M; ++j) {
                    const double e2 = Ar[i][j] * Ar[i][j] + Ai[i][j] * Ai[i][j];
                    fro += e2;
                    if (i != j) off += e2;
                }
        }
        if (!(fro <= DBL_MAX_FRO)) {  // Inf / NaN in R: no eigenvectors (see DBL_MAX_FRO)
            if (STATIC) {
#pragma unroll
                for (int i = 0; i < MA; ++i)
#pragma unroll
                    for (int j = 0; j < MA; ++j) Ar[i][j] = Ai[i][j] = Vr[i][j] = Vi[i][j] = CUDART_NAN;
            } else {
                for (int i = 0; i < M; ++i)
                    for (int j = 0; j < M; ++j) Ar[i][j] = Ai[i][j] = Vr[i][j] = Vi[i][j] = CUDART_NAN;
            }
            break;
        }
        if (off <= (M > 4 ? 1e-29 : 1e-32) * fro || off == 0.0) break;  // see eig_coop_kernel for the M > 4 threshold
        if (STATIC && MA == 4) {
            // parallel (round-robin) ordering: the two rotations of a step touch disjoint rows/columns
            jacobi_rotate_bf<MA>(Ar, Ai, Vr, Vi, 0, 1); jacobi_rotate_bf<MA>(Ar, Ai, Vr, Vi, 2, 3);
            jacobi_rotate_bf<MA>(Ar, Ai, Vr, Vi, 0, 2); jacobi_rotate_bf<MA>(Ar, Ai, Vr, Vi, 1, 3);
            jacobi_rotate_bf<MA>(Ar, Ai, Vr, Vi, 0, 3); jacobi_rotate_bf<MA>(Ar, Ai, Vr, Vi, 1, 2);
        } else if (STATIC) {
#pragma unroll
            for (int p = 0; p < MA - 1; ++p)
#pragma unroll
                for (int q = p + 1; q < MA; ++q) jacobi_rotate<MA>(Ar, Ai, Vr, Vi, p, q, MA);
        } else {
#pragma unroll 1
            for (int p = 0; p < M - 1; ++p)
#pragma unroll 1
                for (int q = p + 1; q < M; ++q) jacobi_rotate<MA>(Ar, Ai, Vr, Vi, p, q, M);
        }
    }
    // ascending, stable: destination slot of column j = #{l : w_l < w_j} + #{l < j : w_l == w_j}
    if (STATIC) {
#pragma unroll
        for (int j = 0; j < MA; ++j) {
            int rank = 0;
#pragma unroll
            for (int l = 0; l < MA; ++l) rank += eig_before(Ar[l][l], l, Ar[j][j], j);
            if (ew) ew[rank] = Ar[j][j];
            double pr, pi;
            eig_phase(Vr[0][j], Vi[0][j], pr, pi);
#pragma unroll
            for (int i = 0; i < MA; ++i) {
                double re, im;
                eig_out4(Vr[i][j], Vi[i][j], pr, pi, re, im);
                vw[2 * (rank * MA + i)] = re;
                vw[2 * (rank * MA + i) + 1] = (i == 0) ? 0.0 : im;
            }
        }
    } else {
        for (int j = 0; j < M; ++j) {
            int rank = 0;
            for (int l = 0; l < M; ++l) rank += eig_before(Ar[l][l], l, Ar[j][j], j);
            if (ew) ew[rank] = Ar[j][j];
            double pr, pi;
            eig_phase(Vr[0][j], Vi[0][j], pr, pi);
            for (int i = 0; i < M; ++i) {
                vw[2 * (rank * M + i)] = Vr[i][j] * pr - Vi[i][j] * pi;
                vw[2 * (rank * M + i) + 1] = (i == 0) ? 0.0 : Vr[i][j] * pi + Vi[i][j] * pr;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// M = 4 eigensolver with FOUR LANES PER WINDOW (the fused kernel's eigensolver warp: 8 windows per round).
// The one-lane solver is a single dependent chain (~34 k cycles per round whatever the contention), and that latency
// is the tail of the fused kernel; here lane j of a group holds column j of A and of V in XOR-relative slots - slot t
// is row j ^ t - so that for the parallel-ordering step with pairs {j, j ^ X} every register index is a compile-time
// constant: own 2x2 block = slots {0, X}, the two rows of the other pair = slots {O, O ^ X}, and row k of the mate's
// column sits in the mate's slot t ^ X.  Both lanes of a pair compute the pair's rotation from identical inputs.
// Bit-identical to two sequential jacobi_rotate_bf calls per step (first the pair containing index 0), which
// tools/emulate_eig4_coop.py checks on the CPU and tests/test_gpu_parity.py (fused == unfused) on the GPU:
//   phase 1  lanes of the second pair apply the first rotation to their column (a local 2-row mix)
//   phase 2  exchange the two off-block rows with the mate
//   phase 3  column mix with the own pair's rotation; own 2x2 block := diag(app - t g, aqq + t g)
//   phase 4  lanes of the first pair apply the second rotation to their column
//   V        whole columns mix with the mate's column
// `live` freezes a window whose sweep test has passed while other windows of the warp go on.
// ------------------------------------------------------------------------------------------
template <int X>
__device__ __forceinline__ void eig4_coop_step(double (&ar)[4], double (&ai)[4], double (&vr)[4], double (&vi)[4], const int j,
                                               const bool live)
{
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int O = (X == 1) ? 2 : 1, O2 = O ^ X, HB = (X == 1) ? 1 : 2;
    const bool isq = (j & HB) != 0;           // the larger index of my pair
    const bool first = (j == 0) || (j == X);  // my pair is the one the sequential order rotates first
    const double dm = __shfl_xor_sync(FULL, ar[0], X);  // the mate's diagonal element
    const double app = isq ? dm : ar[0], aqq = isq ? ar[0] : dm;
    double c, swr, swi, t, g;
    jrot_params(ar[X], isq ? ai[X] : -ai[X], app, aqq, c, swr, swi, t, g);  // lane p holds conj(a_pq)
    const double c2 = __shfl_xor_sync(FULL, c, O), swr2 = __shfl_xor_sync(FULL, swr, O), swi2 = __shfl_xor_sync(FULL, swi, O);
    const bool o_is_p = ((j ^ O) & HB) == 0;  // which of my two off-block rows is the smaller index of the other pair
    auto other_pair = [&](const bool doit) {
        const double pr = o_is_p ? ar[O] : ar[O2], pi = o_is_p ? ai[O] : ai[O2];
        const double qr = o_is_p ? ar[O2] : ar[O], qi = o_is_p ? ai[O2] : ai[O];
        double npr, npi, nqr, nqi;
        jrot_mix(c2, swr2, swi2, pr, -pi, qr, -qi, npr, npi, nqr, nqi);  // my column holds the conjugates of rows p, q
        if (doit) {
            ar[O] = o_is_p ? npr : nqr;   ai[O] = o_is_p ? -npi : -nqi;
            ar[O2] = o_is_p ? nqr : npr;  ai[O2] = o_is_p ? -nqi : -npi;
        }
    };
    other_pair(live && !first);
    {
        const double mOr = __shfl_xor_sync(FULL, ar[O2], X), mOi = __shfl_xor_sync(FULL, ai[O2], X);   // mate's entry of my row (slot O)
        const double mO2r = __shfl_xor_sync(FULL, ar[O], X), mO2i = __shfl_xor_sync(FULL, ai[O], X);   // ... of my row (slot O2)
        double r0, i0, r1, i1;
        jrot_mix_half(c, swr, swi, isq, ar[O], ai[O], mOr, mOi, r0, i0);
        jrot_mix_half(c, swr, swi, isq, ar[O2], ai[O2], mO2r, mO2i, r1, i1);
        if (live) {
            ar[O] = r0; ai[O] = i0; ar[O2] = r1; ai[O2] = i1;
            ar[0] = isq ? fma(t, g, aqq) : fma(-t, g, app);
            ai[0] = 0.0; ar[X] = 0.0; ai[X] = 0.0;
        }
    }
    other_pair(live && first);
    double nr[4], ni[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const double mr = __shfl_xor_sync(FULL, vr[s ^ X], X), mi = __shfl_xor_sync(FULL, vi[s ^ X], X);
        jrot_mix_half(c, swr, swi, isq, vr[s], vi[s], mr, mi, nr[s], ni[s]);
    }
    if (live) {
#pragma unroll
        for (int s = 0; s < 4; ++s) { vr[s] = nr[s]; vi[s] = ni[s]; }
    }
}

// All 32 lanes must call this together; lane group g = lane >> 2 works on one window (active = group has one),
// j = lane & 3.  Rw: 4 x 4 complex, row-major interleaved (shared memory); vw: Vt[rank][i] like herm_eig_body.
__device__ __forceinline__ void herm_eig4_coop(const double *Rw, double *vw, const bool active, const int j)
{
    constexpr unsigned FULL = 0xffffffffu;
    double ar[4], ai[4], vr[4], vi[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const int row = j ^ s;
        ar[s] = active ? Rw[2 * (row * 4 + j)] : 0.0;
        ai[s] = active ? Rw[2 * (row * 4 + j) + 1] : 0.0;
        vr[s] = (s == 0) ? 1.0 : 0.0;
        vi[s] = 0.0;
    }
    bool live = active;
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0;
#pragma unroll
        for (int s = 1; s < 4; ++s) off += ar[s] * ar[s] + ai[s] * ai[s];
        double fro = off + (ar[0] * ar[0] + ai[0] * ai[0]);
        off += __shfl_xor_sync(FULL, off, 1);
        fro += __shfl_xor_sync(FULL, fro, 1);
        off += __shfl_xor_sync(FULL, off, 2);
        fro += __shfl_xor_sync(FULL, fro, 2);
        if (live && !(fro <= DBL_MAX_FRO)) {  // Inf / NaN in R, as in herm_eig_body
#pragma unroll
            for (int s = 0; s < 4; ++s) ar[s] = ai[s] = vr[s] = vi[s] = CUDART_NAN;
            live = false;
        }
        if (off <= 1e-32 * fro || off == 0.0) live = false;  // same test as herm_eig_body (NaN never passes)
        if (!__any_sync(FULL, live)) break;
        eig4_coop_step<1>(ar, ai, vr, vi, j, live);
        eig4_coop_step<2>(ar, ai, vr, vi, j, live);
        eig4_coop_step<3>(ar, ai, vr, vi, j, live);
    }
    // ascending, stable ranks from the four diagonals; phase from component 0 = slot j
    const double wj = ar[0];
    int rank = 0;
#pragma unroll
    for (int s = 1; s < 4; ++s) {
        const double wl = __shfl_xor_sync(FULL, wj, s);
        rank += eig_before(wl, j ^ s, wj, j);
    }
    const double v0r = j == 0 ? vr[0] : j == 1 ? vr[1] : j == 2 ? vr[2] : vr[3];
    const double v0i = j == 0 ? vi[0] : j == 1 ? vi[1] : j == 2 ? vi[2] : vi[3];
    double pr, pi;
    eig_phase(v0r, v0i, pr, pi);
    if (active) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int i = j ^ s;
            double re, im;
            eig_out4(vr[s], vi[s], pr, pi, re, im);
            vw[2 * (rank * 4 + i)] = re;
            vw[2 * (rank * 4 + i) + 1] = (i == 0) ? 0.0 : im;
        }
    }
}

template <int MA, bool STATIC>
__global__ void __launch_bounds__(128) eig_kernel(const double *__restrict__ R, double *__restrict__ evals,
                                                  double *__restrict__ Vt, int Mrt, int W)
{
    const int M = STATIC ? MA : Mrt;
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    herm_eig_body<MA, STATIC>(R + (size_t)w * M * M * 2, evals + (size_t)w * M, Vt + (size_t)w * M * M * 2, M);
}

// ------------------------------------------------------------------------------------------
// K2 for M = 8..16 (even M): warp-cooperative Jacobi with the matrices in shared memory, one warp
// per window.  The thread-per-window solver keeps A and V (2 x M x M complex) in local memory
// for M > 4 and is bound by that traffic (M = 16: ~0.5 M cycles per window per SM); here a sweep is
// M-1 parallel steps of M/2 disjoint rotations (round-robin ordering): lanes 0..M/2-1 compute the
// rotations, then all 32 lanes apply them to the columns of A and V and to the rows of A.
// Output layout and conventions are those of herm_eig_body (ascending, stable, real v[0]).
// ------------------------------------------------------------------------------------------
constexpr int EIGC_WARPS = 4;

// One warp, one window: A (M x M complex, row-major, shared memory) holds R on entry and the rotated matrix (its diagonal =
// the eigenvalues) on exit, V (M x M scratch) the eigenvectors as columns; rot / pair: M/2 entries of warp-private scratch.
// P = row pitch of A and V in complex entries.  P = M + 1 with the column phase running row-fastest over the lanes makes a
// quarter warp (8 lanes, one 128-bit wavefront) touch 8 different rows of ONE column: chunk (k P + p) mod 8 = (k + p) mod 8,
// all distinct - no bank conflicts; with P = M and pair-fastest lanes the 8 columns of one row collide pairwise
// (c and c + 8 share banks): 56.6 M conflicts per 4096 windows at M = 16 (profiles/r02_ncu_config5_kernels.txt).
template <int M, int P = M>
__device__ __forceinline__ void eig_coop_warp(double2 *A, double2 *V, double (*rot)[4], int (*pair)[2], const int lane)
{
    static_assert(M % 2 == 0 && M <= MAXM, "even M only");
    constexpr int H = M / 2;
    for (int i = lane; i < M * M; i += 32) V[(i / M) * P + i % M] = make_double2((i / M == i % M) ? 1.0 : 0.0, 0.0);
    __syncwarp();
    double prev_off = 1e300;
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, fro = 0.0;
        for (int i = lane; i < M * M; i += 32) {
            const double2 a = A[(i / M) * P + i % M];
            const double e2 = a.x * a.x + a.y * a.y;
            fro += e2;
            if (i / M != i % M) off += e2;
        }
        off = warp_sum(off);
        fro = warp_sum(fro);
        // rounding keeps the off-diagonal energy of an M x M iterate near 2 M eps^2 ||A||_F^2 (4e-31 at M = 16), so
        // the M = 4 threshold (1e-32) is unreachable here: stop at 1e-29, or when a sweep no longer helps
        if (!(fro <= DBL_MAX_FRO)) {  // Inf / NaN in R, as in herm_eig_body (fro is the same in every lane)
            for (int i = lane; i < M * M; i += 32) { A[(i / M) * P + i % M] = make_double2(CUDART_NAN, CUDART_NAN); V[(i / M) * P + i % M] = make_double2(CUDART_NAN, CUDART_NAN); }
            __syncwarp();
            break;
        }
        if (off <= 1e-29 * fro || off == 0.0 || (sweep > 2 && off <= 1e-24 * fro && off >= 0.25 * prev_off)) break;
        prev_off = off;
        for (int step = 0; step < M - 1; ++step) {
            if (lane < H) {  // rotation of pair `lane` (circle method: index M-1 stays, the others rotate)
                int p, q;
                if (lane == 0) { p = M - 1; q = step; }
                else { p = (step + lane) % (M - 1); q = (step - lane + (M - 1)) % (M - 1); }
                if (p > q) { const int t = p; p = q; q = t; }
                const double2 g2 = A[p * P + q];
                const double app = A[p * P + p].x, aqq = A[q * P + q].x;
                const double gg = fma(g2.x, g2.x, g2.y * g2.y);
                const bool nz = gg > 0.0;
                const double rg = nz ? rsqrt(gg) : 0.0;
                double theta = 0.5 * (aqq - app) * rg;
                theta = fmin(fmax(theta, -1e150), 1e150);
                const double q1 = fma(theta, theta, 1.0);
                const double sq = q1 * rsqrt(q1);
                double t = 1.0 / (fabs(theta) + sq);
                t = nz ? copysign(t, theta) : 0.0;
                if (gg != gg) t = gg;  // NaN input stays NaN
                const double c = rsqrt(fma(t, t, 1.0));
                const double sn = t * c;
                rot[lane][0] = c;
                rot[lane][1] = sn * g2.x * rg;
                rot[lane][2] = sn * g2.y * rg;
                pair[lane][0] = p;
                pair[lane][1] = q;
            }
            __syncwarp();
            // columns: B[k][p] = c A[k][p] - conj(sw) A[k][q],  B[k][q] = sw A[k][p] + c A[k][q]   (A and V)
            for (int it = lane; it < M * H; it += 32) {
                const int k = (P == M) ? it / H : it % M, i = (P == M) ? it % H : it / M;
                const int p = pair[i][0], q = pair[i][1];
                const double c = rot[i][0], swr = rot[i][1], swi = rot[i][2];
                {
                    const double2 ap = A[k * P + p], aq = A[k * P + q];
                    A[k * P + p] = make_double2(c * ap.x - (swr * aq.x + swi * aq.y), c * ap.y - (swr * aq.y - swi * aq.x));
                    A[k * P + q] = make_double2(c * aq.x + (swr * ap.x - swi * ap.y), c * aq.y + (swr * ap.y + swi * ap.x));
                }
                {
                    const double2 vp = V[k * P + p], vq = V[k * P + q];
                    V[k * P + p] = make_double2(c * vp.x - (swr * vq.x + swi * vq.y), c * vp.y - (swr * vq.y - swi * vq.x));
                    V[k * P + q] = make_double2(c * vq.x + (swr * vp.x - swi * vp.y), c * vq.y + (swr * vp.y + swi * vp.x));
                }
            }
            __syncwarp();
            // rows: A'[p][k] = c B[p][k] - sw B[q][k],  A'[q][k] = conj(sw) B[p][k] + c B[q][k]
            // (k fastest across lanes: a row is contiguous, so the accesses are bank-conflict free)
            for (int it = lane; it < M * H; it += 32) {
                const int i = it / M, k = it % M;
                const int p = pair[i][0], q = pair[i][1];
                const double c = rot[i][0], swr = rot[i][1], swi = rot[i][2];
                const double2 bp = A[p * P + k], bq = A[q * P + k];
                A[p * P + k] = make_double2(c * bp.x - (swr * bq.x - swi * bq.y), c * bp.y - (swr * bq.y + swi * bq.x));
                A[q * P + k] = make_double2(c * bq.x + (swr * bp.x + swi * bp.y), c * bq.y + (swr * bp.y - swi * bp.x));
            }
            __syncwarp();
            if (lane < H) {  // exact zeros / real diagonal where the rotation says so
                const int p = pair[lane][0], q = pair[lane][1];
                A[p * P + q] = make_double2(0.0, 0.0);
                A[q * P + p] = make_double2(0.0, 0.0);
                A[p * P + p].y = 0.0;
                A[q * P + q].y = 0.0;
            }
            __syncwarp();
        }
    }
}

// ascending, stable ranks; eigenvector j -> vw[rank(j)][.] (component i), phase fixed so that component 0 is real;
// ew (may be null): the eigenvalues in the same order
template <int M, int P = M>
__device__ __forceinline__ void eig_coop_store(const double2 *A, const double2 *V, double *ew, double2 *vw, const int lane)
{
    for (int it = lane; it < M * M; it += 32) {
        const int j = it / M, i = it % M;  // column j, component i
        const double wj = A[j * P + j].x;
        int rank = 0;
        for (int l = 0; l < M; ++l) rank += eig_before(A[l * P + l].x, l, wj, j);
        double pr, pi;
        eig_phase(V[0 * P + j].x, V[0 * P + j].y, pr, pi);
        const double2 v = V[i * P + j];
        vw[rank * M + i] = make_double2(v.x * pr - v.y * pi, i == 0 ? 0.0 : v.x * pi + v.y * pr);
        if (i == 0 && ew) ew[rank] = wj;
    }
}

template <int M>
__global__ void __launch_bounds__(EIGC_WARPS * 32) eig_coop_kernel(const double *__restrict__ R, double *__restrict__ evals,
                                                                   double *__restrict__ Vt, int W)
{
    constexpr int H = M / 2;
    constexpr int P = (M == 16) ? M + 1 : M;  // padded pitch where a row spans more than the 32 banks (see eig_coop_warp)
    __shared__ double2 sA[EIGC_WARPS][M * P];
    __shared__ double2 sV[EIGC_WARPS][M * P];
    __shared__ double sRot[EIGC_WARPS][H][4];  // c, Re(s w), Im(s w), unused
    __shared__ int sPair[EIGC_WARPS][H][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = blockIdx.x * EIGC_WARPS + warp;
    if (w >= W) return;
    double2 *A = sA[warp], *V = sV[warp];
    const double2 *Rw = reinterpret_cast<const double2 *>(R) + (size_t)w * M * M;
    for (int i = lane; i < M * M; i += 32) A[(i / M) * P + i % M] = Rw[i];
    eig_coop_warp<M, P>(A, V, sRot[warp], sPair[warp], lane);
    eig_coop_store<M, P>(A, V, evals + (size_t)w * M, reinterpret_cast<double2 *>(Vt) + (size_t)w * M * M, lane);
}

// ------------------------------------------------------------------------------------------
// Steering table preparation (once per set_table): c64 [K][M] -> fp64 SoA tiles
//   soa[tile][comp][TILE],  comp = 2i (Re a_i), 2i+1 (Im a_i), 2M (||a||^2); zero padded.
// Hoists the per-step c64 -> c128 widening of the reference (:110-112) out of the hot loop.
// ------------------------------------------------------------------------------------------
__global__ void prep_table_kernel(const float2 *__restrict__ tab, double *__restrict__ soa, int K, int M)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int tile = k / TILE, j = k % TILE;
    double *base = soa + (size_t)tile * (2 * M + 1) * TILE + j;
    double na = 0.0;
    for (int i = 0; i < M; ++i) {
        double re = 0.0, im = 0.0;
        if (k < K) { const float2 a = tab[(size_t)k * M + i]; re = a.x; im = a.y; }
        base[(size_t)(2 * i) * TILE] = re;
        base[(size_t)(2 * i + 1) * TILE] = im;
        na = fma(re, re, fma(im, im, na));
    }
    base[(size_t)(2 * M) * TILE] = (k < K) ? na : __longlong_as_double(0x7ff0000000000000LL);  // padding never wins
}

// ------------------------------------------------------------------------------------------
// K3: pseudospectrum scan.  One CTA per batch of SCAN_B windows; thread <-> angle bin within a
// 256-bin table tile (its 2M+1 doubles live in registers), inner loop over the batch's windows
// with the eigenvectors broadcast from shared memory.  Every bin is computed by the same
// instruction sequence, so bit-equal table rows give bit-equal strengths (mirror ties).
//
//   d_k = ||G^H a_k||^2 is evaluated through the signal-subspace complement
//         d = ||a||^2 - sum_s |e_s^H a|^2         (n < M-n: fewer flops)
//   and recomputed in the direct noise-subspace form wherever d < 2^-7 ||a||^2 (near the
//   peaks), so cancellation never costs more than ~2 digits.  P = 1.0 / d.
//
//   ARGMAX: n == 1 fused peak pick, ordered (P desc, bin asc), P > 0 strictly, NaN never.
// ------------------------------------------------------------------------------------------
constexpr int MAX_PEERS = 8;  // GPUs of one NVSwitch domain
struct PeakOut {
    float *angles;   // [W][n]
    float *levels;   // [W][n] or null
    int32_t *bins;   // [W][n] or null
    // Fused all-gather of the peak bins (SURVEY.md section 8e): with npeer = G > 0 this GPU holds the windows
    // w = i * G + rank of a round-robin sharded stream (i = local window index) and every kernel that writes a
    // peak bin also stores it at stream position w of EVERY peer's gather buffer (peer-mapped device memory, NVLink
    // stores straight from the scan epilogue; peer[rank] is this GPU's own buffer) - no collective kernel runs.
    int32_t *peer[MAX_PEERS];
    int npeer, rank, n;
};

struct GatherFlags {
    unsigned *peer[MAX_PEERS];  // peer[p][r] = last epoch in which GPU r finished writing its bins into GPU p's buffer
    unsigned epoch;             // 0: no signalling
};

// peak bin of local output slot o (= local window * n + r)
__device__ __forceinline__ void peak_store_bin(const PeakOut &out, const size_t o, const int kk)
{
    if (out.bins) out.bins[o] = kk;
    if (out.npeer > 0) {
        const size_t w = o / (size_t)out.n, r = o - w * (size_t)out.n;
        const size_t go = (w * (size_t)out.npeer + (size_t)out.rank) * (size_t)out.n + r;
        for (int p = 0; p < out.npeer; ++p) out.peer[p][go] = kk;
    }
}

__device__ __forceinline__ bool peak_better(double Pa, int ka, double Pb, int kb)
{
    return (Pa > Pb) || (Pa == Pb && ka >= 0 && (kb < 0 || ka < kb));
}

template <int MT>
__device__ __forceinline__ double strength_denominator(const double *ar, const double *ai, double na,
                                                       const double *sv, int M, int n, bool use_sig)
{
    double d;
    if (use_sig) {
        double acc = 0.0;
        for (int s = M - n; s < M; ++s) {
            double cr = 0.0, ci = 0.0;
#pragma unroll
            for (int i = 0; i < (MT ? MT : MAXM); ++i) {
                if (!MT && i >= M) break;
                const double2 e = *reinterpret_cast<const double2 *>(sv + 2 * (s * M + i));
                cr = fma(e.x, ar[i], fma(e.y, ai[i], cr));
                ci = fma(e.x, ai[i], fma(-e.y, ar[i], ci));
            }
            acc = fma(cr, cr, fma(ci, ci, acc));
        }
        d = na - acc;
        if (!(d < COMPLEMENT_GUARD * na)) return d;  // NaN falls through to the direct form (stays NaN)
    }
    double acc = 0.0;
    for (int s = 0; s < M - n; ++s) {
        double cr = 0.0, ci = 0.0;
#pragma unroll
        for (int i = 0; i < (MT ? MT : MAXM); ++i) {
            if (!MT && i >= M) break;
            const double2 e = *reinterpret_cast<const double2 *>(sv + 2 * (s * M + i));
            cr = fma(e.x, ar[i], fma(e.y, ai[i], cr));
            ci = fma(e.x, ai[i], fma(-e.y, ar[i], ci));
        }
        acc = fma(cr, cr, fma(ci, ci, acc));
    }
    d = acc;
    return d;
}

template <int MT, bool ARGMAX, bool WRITE_P64, bool WRITE_SPEC>
__global__ void __launch_bounds__(TILE) scan_kernel(const double *__restrict__ soa, const double *__restrict__ Vt,
                                                    int Mrt, int n, int K, int W, PeakOut out,
                                                    float *__restrict__ spectrum, double *__restrict__ P64)
{
    constexpr int MA = MT ? MT : MAXM;
    const int M = MT ? MT : Mrt;
    extern __shared__ __align__(16) double smem[];
    double *sV = smem;  // [SCAN_B][M*M*2]
    const int w0 = blockIdx.x * SCAN_B;
    const int nb = min(SCAN_B, W - w0);
    const int vsz = M * M * 2;
    for (int i = threadIdx.x; i < nb * vsz; i += blockDim.x) sV[i] = Vt[(size_t)w0 * vsz + i];
    __syncthreads();

    const bool use_sig = (n < M - n);
    // Peak-only path (no spectrum output): keep the running minimum of d = ||G^H a||^2 instead of
    // the maximum of P = 1/d, so the IEEE division leaves the inner loop.  The update rule is
    // exactly "P_new > P_best" (the reference's strict '>' on strengths, :132): a candidate that
    // is smaller by more than 2^-50 relative has a strictly larger reciprocal; inside that sliver
    // the two reciprocals are compared.  d is never negative (direct form is a sum of squares,
    // complement form is only kept above 2^-7 ||a||^2), NaN fails `d < best`.
    constexpr bool FAST = ARGMAX && !WRITE_P64 && !WRITE_SPEC;
    double best[SCAN_B];  // FAST: min d; otherwise: max P
    int bestk[SCAN_B];
#pragma unroll
    for (int b = 0; b < SCAN_B; ++b) { best[b] = FAST ? __longlong_as_double(0x7ff0000000000000LL) : 0.0; bestk[b] = -1; }

    const int ntiles = (K + TILE - 1) / TILE;
    for (int tile = 0; tile < ntiles; ++tile) {
        const int k = tile * TILE + threadIdx.x;
        const double *tb = soa + (size_t)tile * (2 * M + 1) * TILE + threadIdx.x;
        double ar[MA], ai[MA];
#pragma unroll
        for (int i = 0; i < MA; ++i) {
            if (!MT && i >= M) break;
            ar[i] = tb[(size_t)(2 * i) * TILE];
            ai[i] = tb[(size_t)(2 * i + 1) * TILE];
        }
        const double na = tb[(size_t)(2 * M) * TILE];
        if (k < K) {
#pragma unroll
            for (int b = 0; b < SCAN_B; ++b) {
                if (b < nb) {
                    const double d = strength_denominator<MT>(ar, ai, na, sV + b * vsz, M, n, use_sig);
                    if (FAST) {
                        if (d < best[b]) {
                            if (d < best[b] * 0.99999999999999911182 /* 1 - 2^-50 */ || 1.0 / d > 1.0 / best[b]) {
                                best[b] = d;
                                bestk[b] = k;
                            }
                        }
                    } else {
                        const double P = 1.0 / d;
                        if (WRITE_SPEC) spectrum[(size_t)(w0 + b) * K + k] = (float)P;
                        if (WRITE_P64) P64[(size_t)(w0 + b) * K + k] = P;
                        if (ARGMAX) {
                            if (P > best[b]) { best[b] = P; bestk[b] = k; }  // k ascending per thread: strict > keeps the lower bin
                        }
                    }
                }
            }
        }
    }
    if (ARGMAX) {
        __shared__ double rP[SCAN_B][TILE / 32];
        __shared__ int rk[SCAN_B][TILE / 32];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
        for (int b = 0; b < SCAN_B; ++b) {
            int kk = bestk[b];
            double P = FAST ? (kk >= 0 ? 1.0 / best[b] : 0.0) : best[b];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double Po = __shfl_xor_sync(0xffffffffu, P, o);
                const int ko = __shfl_xor_sync(0xffffffffu, kk, o);
                if (peak_better(Po, ko, P, kk)) { P = Po; kk = ko; }
            }
            if (lane == 0) { rP[b][wid] = P; rk[b][wid] = kk; }
        }
        __syncthreads();
        if (threadIdx.x < nb) {
            const int b = threadIdx.x;
            double P = rP[b][0];
            int kk = rk[b][0];
            for (int q = 1; q < TILE / 32; ++q)
                if (peak_better(rP[b][q], rk[b][q], P, kk)) { P = rP[b][q]; kk = rk[b][q]; }
            const size_t o = (size_t)(w0 + b);  // n == 1
            if (kk >= 0) {
                out.angles[o] = (float)((double)kk * 360.0 / (double)K);  // :134, :153
                if (out.levels) out.levels[o] = (float)P;                 // :154
            } else {
                out.angles[o] = 0.f;                                      // (0,0) initial pair, :95
                if (out.levels) out.levels[o] = 0.f;
            }
            peak_store_bin(out, o, kk);
        }
    }
}

// ------------------------------------------------------------------------------------------
// K3 fast path: peak-only scan for n == 1 < M-1 (no spectrum output), branch-free hot loop.
//   per (bin, window): 4*M DFMA for c = e^H a, 2 DFMA for d = ||a||^2 - |c|^2, and an integer
//   compare of the fp64 bit patterns (positive doubles order like their bits) on the ALU pipe,
//   so the FP64 pipe - the bottleneck - only sees the 4M+2 DFMAs.
//   Rare events are hoisted out of the unrolled window loop:
//     * complement guard (d < 2^-7 ||a||^2): one branch per tile, direct noise-subspace form;
//     * candidates within 8 ulps of the running minimum: exact comparison of the reciprocals
//       (keeps the rule identical to the reference's strict '>' on P = 1/d, :132).
//   Table rows beyond K are padded with ||a||^2 = +inf (d = +inf never wins), windows beyond W
//   in the last batch recompute the last valid window (results discarded).
// ------------------------------------------------------------------------------------------
// Shared-memory load the compiler may not hoist: the eigenvectors are loop invariant across
// table tiles, and hoisting 8 windows x M complex into registers spills everything.
__device__ __forceinline__ double2 lds_f64x2(uint32_t addr)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}

template <int M>
__device__ __forceinline__ double direct_denominator(const double *ar, const double *ai, uint32_t sv)
{
    double acc = 0.0;
#pragma unroll 1
    for (int s = 0; s < M - 1; ++s) {
        double cr = 0.0, ci = 0.0;
#pragma unroll
        for (int i = 0; i < M; ++i) {
            const double2 e = lds_f64x2(sv + 16 * (s * M + i));
            cr = fma(e.x, ar[i], fma(e.y, ai[i], cr));
            ci = fma(e.x, ai[i], fma(-e.y, ar[i], ci));
        }
        acc = fma(cr, cr, fma(ci, ci, acc));
    }
    return acc;
}

// Thread mapping: 256 threads = SCAN_G window groups x SCAN_BINS bins; a thread owns one bin of
// the current 128-bin half tile and SCAN_WPT windows (state in registers), so that 3-4 CTAs fit
// per SM and every SMSP has >= 6 warps of independent DFMA chains to hide the FP64 latency.
constexpr int SCAN_WPT = 4;                   // windows per thread
constexpr int SCAN_G = SCAN_B / SCAN_WPT;     // window groups per CTA
constexpr int SCAN_BINS = TILE / SCAN_G;      // bins per CTA iteration

template <int M>
__device__ __forceinline__ double complement_denominator(const double *ar, const double *ai, double na, uint32_t e)
{
    // component 0 of every eigenvector is real (eig_kernel fixes the phase): 2 DMUL, not 4 DFMA
    const double2 e0 = lds_f64x2(e);
    double cr = e0.x * ar[0], ci = e0.x * ai[0];
#pragma unroll
    for (int i = 1; i < M; ++i) {
        const double2 ev = lds_f64x2(e + 16 * i);
        cr = fma(ev.x, ar[i], fma(ev.y, ai[i], cr));
        ci = fma(ev.x, ai[i], fma(-ev.y, ar[i], ci));
    }
    return fma(-cr, cr, fma(-ci, ci, na));
}

// Running peak state of WPT windows held by one thread.
template <int WPT>
struct PeakState {
    double bestd[WPT];   // running minimum of d = ||G^H a||^2
    unsigned hbm1[WPT];  // high word of bestd, minus one (saturating at 0): screening threshold
    int bestk[WPT];
    __device__ __forceinline__ void reset()
    {
#pragma unroll
        for (int b = 0; b < WPT; ++b) { bestd[b] = __longlong_as_double(0x7ff0000000000000LL); hbm1[b] = 0x7fefffffu; bestk[b] = -1; }
    }
};

// One steering-table row (bin k) against WPT windows.  ev[b]: shared address of window b's sorted
// eigenvector block (Vt layout).  The loops run antenna-outer / window-inner so that the 2*WPT
// dot-product chains are independent and interleave in issue order (the DFMA pipe has a long
// dependent-issue latency; two windows at a time leave it half idle).
//   hot path : complement form d = ||a||^2 - |e_s^H a|^2, 2 DMUL + 4(M-1)+2 DFMA per window, then a
//              screen on the high 32 bits of d on the ALU pipe:
//                hd <= hi(guard)               -> maybe inside the cancellation guard (or negative): cold
//                hd <  hi(best) - 1 (unsigned) -> below the running minimum by >= 2^-20 relative: accept
//                hd in {hi(best)-1, hi(best)}  -> ambiguous (includes exact ties): cold
//              NaNs and negative-signed values are large as unsigned and are never accepted.
//   cold path: exact evaluation (direct noise-subspace form inside the guard) and the reference's
//              rule "replace iff 1/d > 1/best" (strict '>' on the strengths, :132).
template <int M, int WPT>
__device__ __forceinline__ void scan_bin(const double (&ar)[M], const double (&ai)[M], const double na, const int k,
                                         const uint32_t (&ev)[WPT], PeakState<WPT> &ps)
{
    constexpr int sig = 16 * (M - 1) * M;  // byte offset of the signal vector (largest eigenvalue)
    double cr[WPT], ci[WPT];
#pragma unroll
    for (int b = 0; b < WPT; ++b) {
        double e0x;
        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(e0x) : "r"(ev[b] + sig));
        cr[b] = e0x * ar[0];
        ci[b] = e0x * ai[0];
    }
#pragma unroll
    for (int i = 1; i < M; ++i) {
#pragma unroll
        for (int b = 0; b < WPT; ++b) {
            // same association as complement_denominator (the cold path): fma(e.x, a, fma(e.y, a', c)), so that a bin
            // evaluated hot in one thread and cold in another rounds identically (exact mirror ties stay exact)
            const double2 e = lds_f64x2(ev[b] + sig + 16 * i);
            cr[b] = fma(e.y, ai[i], cr[b]);
            ci[b] = fma(-e.y, ar[i], ci[b]);
            cr[b] = fma(e.x, ar[i], cr[b]);
            ci[b] = fma(e.x, ai[i], ci[b]);
        }
    }
    const double gna = COMPLEMENT_GUARD * na;
    const int hg = __double2hiint(gna);
    unsigned cold = 0;
#pragma unroll
    for (int b = 0; b < WPT; ++b) {
        const double d = fma(-cr[b], cr[b], fma(-ci[b], ci[b], na));
        const int hds = __double2hiint(d);
        const unsigned hd = (unsigned)hds;
        const bool guard = hds <= hg;
        if ((hd - ps.hbm1[b]) <= 1u || guard) cold |= 1u << b;
        if (hd < ps.hbm1[b] && !guard) { ps.bestd[b] = d; ps.bestk[b] = k; ps.hbm1[b] = max(hd, 1u) - 1u; }
    }
    if (cold) {
#pragma unroll
        for (int b = 0; b < WPT; ++b) {
            if (cold & (1u << b)) {
                double d = complement_denominator<M>(ar, ai, na, ev[b] + sig);
                if (d < gna) d = direct_denominator<M>(ar, ai, ev[b]);
                if (d < ps.bestd[b]) {
                    if (d < ps.bestd[b] * 0.99999999999999911182 /* 1 - 2^-50 */ || 1.0 / d > 1.0 / ps.bestd[b]) {
                        ps.bestd[b] = d;
                        ps.bestk[b] = k;
                        ps.hbm1[b] = max((unsigned)__double2hiint(d), 1u) - 1u;
                    }
                }
            }
        }
    }
}

template <int M>
__global__ void __launch_bounds__(TILE, 3) scan_peak1_kernel(const double *__restrict__ soa, const double *__restrict__ Vt,
                                                             int K, int W, PeakOut out)
{
    constexpr int vsz = M * M * 2;
    __shared__ __align__(16) double sV[SCAN_B * vsz];
    const int w0 = blockIdx.x * SCAN_B;
    const int nb = min(SCAN_B, W - w0);
    for (int i = threadIdx.x; i < SCAN_B * vsz; i += blockDim.x) {
        const int b = min(i / vsz, nb - 1);
        sV[i] = Vt[(size_t)(w0 + b) * vsz + (i % vsz)];
    }
    __syncthreads();

    const int g = threadIdx.x / SCAN_BINS, t = threadIdx.x % SCAN_BINS;
    uint32_t ev[SCAN_WPT];
#pragma unroll
    for (int b = 0; b < SCAN_WPT; ++b) ev[b] = smem_u32(sV) + 8 * ((g * SCAN_WPT + b) * vsz);
    PeakState<SCAN_WPT> ps;
    ps.reset();

    const int niter = (K + SCAN_BINS - 1) / SCAN_BINS;
    for (int it = 0; it < niter; ++it) {
        const int k = it * SCAN_BINS + t;  // table is padded to a multiple of TILE with ||a||^2 = +inf
        const double *tb = soa + (size_t)(k / TILE) * (2 * M + 1) * TILE + (k % TILE);
        double ar[M], ai[M];
#pragma unroll
        for (int i = 0; i < M; ++i) {
            ar[i] = tb[(size_t)(2 * i) * TILE];
            ai[i] = tb[(size_t)(2 * i + 1) * TILE];
        }
        const double na = tb[(size_t)(2 * M) * TILE];
        scan_bin<M, SCAN_WPT>(ar, ai, na, k, ev, ps);
    }
    // per-window merge over the SCAN_BINS threads of the group, order (P desc, bin asc)
    constexpr int WPG = SCAN_BINS / 32;  // warps per group
    __shared__ double rP[SCAN_B][WPG];
    __shared__ int rk[SCAN_B][WPG];
    const int lane = threadIdx.x & 31, wig = (threadIdx.x >> 5) % WPG;
#pragma unroll
    for (int b = 0; b < SCAN_WPT; ++b) {
        int kk = ps.bestk[b];
        double P = kk >= 0 ? 1.0 / ps.bestd[b] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double Po = __shfl_xor_sync(0xffffffffu, P, o);
            const int ko = __shfl_xor_sync(0xffffffffu, kk, o);
            if (peak_better(Po, ko, P, kk)) { P = Po; kk = ko; }
        }
        if (lane == 0) { rP[g * SCAN_WPT + b][wig] = P; rk[g * SCAN_WPT + b][wig] = kk; }
    }
    __syncthreads();
    if (threadIdx.x < nb) {
        const int b = threadIdx.x;
        double P = rP[b][0];
        int kk = rk[b][0];
        for (int q = 1; q < WPG; ++q)
            if (peak_better(rP[b][q], rk[b][q], P, kk)) { P = rP[b][q]; kk = rk[b][q]; }
        const size_t o = (size_t)(w0 + b);
        if (kk >= 0) {
            out.angles[o] = (float)((double)kk * 360.0 / (double)K);  // :134, :153
            if (out.levels) out.levels[o] = (float)P;                 // :154
        } else {
            out.angles[o] = 0.f;                                      // (0,0) initial pair, :95
            if (out.levels) out.levels[o] = 0.f;
        }
        peak_store_bin(out, o, kk);
    }
}

// Top-n for n >= 2 from the fp64 strengths: one warp per window, n rounds of a warp arg-max in
// the reference's total order (P desc, bin asc; P > 0 strictly; NaN never) - equivalent to the
// insertion loop at :129-141.
__global__ void __launch_bounds__(256) topn_kernel(const double *__restrict__ P64, int n, int K, int W, PeakOut out)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= W) return;
    const double *P = P64 + (size_t)w * K;
    double prevP = 0.0;
    int prevk = -1;
    bool first = true;
    for (int r = 0; r < n; ++r) {
        double bP = 0.0;
        int bk = -1;
        if (first || prevk >= 0) {
            for (int k = lane; k < K; k += 32) {
                const double p = P[k];
                const bool after = first || (p < prevP) || (p == prevP && k > prevk);
                if (after && p > 0.0 && p > bP) { bP = p; bk = k; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double Po = __shfl_xor_sync(0xffffffffu, bP, o);
                const int ko = __shfl_xor_sync(0xffffffffu, bk, o);
                if (peak_better(Po, ko, bP, bk)) { bP = Po; bk = ko; }
            }
        }
        if (lane == 0) {
            const size_t o = (size_t)w * n + r;
            if (bk >= 0) {
                out.angles[o] = (float)((double)bk * 360.0 / (double)K);
                if (out.levels) out.levels[o] = (float)bP;
            } else {
                out.angles[o] = 0.f;
                if (out.levels) out.levels[o] = 0.f;
            }
            peak_store_bin(out, o, bk);
        }
        first = false;
        prevP = bP;
        prevk = bk;
    }
}

// Opt-in peak rule (not in the reference; SURVEY.md section 8(f) rank 3, oracle/music_oracle.py::pick_local_maxima):
// the n largest circular local maxima of P, at least `excl` + 1 bins apart.  One warp per window; pass r finds the
// best remaining candidate (P[k] > 0, P[k] > P[k-1], P[k] >= P[k+1], farther than excl bins from every peak taken
// so far; ties -> lowest k).
__global__ void __launch_bounds__(256) topn_local_kernel(const double *__restrict__ P64, int n, int K, int W, int excl, PeakOut out)
{
    __shared__ int taken_all[8][MAXM];  // per warp: bins of the picks made so far
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= W) return;
    volatile int *taken = taken_all[threadIdx.x >> 5];
    const double *P = P64 + (size_t)w * K;
    bool dry = false;
    for (int r = 0; r < n; ++r) {
        double bP = 0.0;
        int bk = -1;
        if (!dry) {
            for (int k = lane; k < K; k += 32) {
                const double p = P[k];
                if (!(p > 0.0) || !(p > bP)) continue;  // also skips NaN; an equal p at a higher k never wins
                const double pl = P[k == 0 ? K - 1 : k - 1], pr = P[k == K - 1 ? 0 : k + 1];
                if (!(p > pl) || !(p >= pr)) continue;
                bool ok = true;
                for (int q = 0; q < r; ++q) {
                    const int t = taken[q];
                    int d = k > t ? k - t : t - k;
                    d = min(d, K - d);
                    ok = ok && d > excl;
                }
                if (ok) { bP = p; bk = k; }
            }
        }
        __syncwarp();  // lanes leave the k loop after different trip counts
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double Po = __shfl_xor_sync(0xffffffffu, bP, o);
            const int ko = __shfl_xor_sync(0xffffffffu, bk, o);
            if (peak_better(Po, ko, bP, bk)) { bP = Po; bk = ko; }
        }
        if (bk < 0) dry = true;
        if (lane == 0) {
            if (r < MAXM) taken[r] = bk;
            const size_t o = (size_t)w * n + r;
            if (bk >= 0) {
                out.angles[o] = (float)((double)bk * 360.0 / (double)K);
                if (out.levels) out.levels[o] = (float)bP;
            } else {
                out.angles[o] = 0.f;
                if (out.levels) out.levels[o] = 0.f;
            }
            peak_store_bin(out, o, bk);
        }
        __syncwarp();
    }
}

}  // namespace music
