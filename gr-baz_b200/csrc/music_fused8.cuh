// music_fused8.cuh - FUSED persistent kernel for M = 8 antennas, n = 1 source, peak outputs only (BASELINE configs[2], [3]):
// covariance + eigenvectors + pseudospectrum scan + peak pick in ONE launch; R and the eigenvectors never leave shared
// memory (the three-kernel path writes R, eigenvalues and eigenvectors to an fp64 HBM workspace and runs its FP64-only
// eigensolver and scan AFTER the HBM-bound covariance instead of under it).
//
// Unlike the M = 4 kernel (music_fused.cuh: warp-specialised, queues between the stages) every warp here owns its windows
// from the first byte to the peak bin - at M = 8 one warp's 64 fp64 accumulators per lane already fill the register file
// (8 warps x 250 registers), there is no room for dedicated eigensolver / scan warps, and none is needed:
//   1. covariance   exactly covN_tma_kernel<8> (music_covn.cuh): the window streams through a per-warp ring of 6 KiB stages
//                   filled by cp.async.bulk.tensor (UTMALDG, 128-byte swizzle), lane <-> snapshot, 128 DFMA per 16 F2F,
//                   transposing butterfly -> R (8 x 8 complex) in the warp's shared memory;
//   2. eigenvectors principal eigenvector by repeated squaring + two power steps + residual certificate + Householder basis
//                   of the complement - music_eig4p.cuh's algorithm with the whole warp on one 8 x 8 matrix (lane = row r,
//                   two columns); ~5 % of the covariance's DFMA count.  Windows without a dominant eigenvalue (noise only,
//                   NaN, all zero) run the warp-cooperative Jacobi solver of the unfused path (eig_coop_warp);
//   3. scan         after every 4th window (and at the end) the warp scans its 4 pending windows in fp64 with the unfused
//                   kernel's hot loop (scan_bin<8, 4>: lane <-> bin, 4 windows per table row so the 136-byte fp64 row from
//                   L2 is amortised), merges over the lanes and writes the peaks.
// While one warp is in phases 2-3 (about a fifth of its time) the other seven keep the HBM stream going; the stages' rings
// refill during the scan.  FP64 work per window: covariance 128 x N, scan 34 x K, eigenvectors ~2 % - the kernel needs
// ~85 % of the FP64 pipe at the HBM roof, so it runs just below the covariance-only kernel's speed.
// Bit-exactness: the scan is the unfused kernel's arithmetic; the eigenvectors differ from Jacobi's by ~1e-15, P by ~1e-12.
//
// Reference lines covered: /root/reference/lib/baz_music_doa.cc:74-155 (everything work() does per window except the
// optional spectrum port), M = 8, n = 1.
#pragma once
#include "music_covn.cuh"
#include "music_eig4p.cuh"

namespace music {

constexpr int F8_WARPS = 8;
constexpr int F8_STEPS = 3;                       // 32-snapshot steps per stage
constexpr int F8_ROWS = 32 * F8_STEPS;            // snapshots per stage
constexpr int F8_STAGE = F8_ROWS * 64;            // bytes per stage (6 KiB)
constexpr int F8_SG = 3;                          // stages per warp
constexpr int F8_RING = F8_WARPS * F8_SG * F8_STAGE;   // 144 KiB
constexpr int F8_BATCH = 4;                       // windows per scan (= scan_bin's windows per thread)
// per-warp scratch after the ring and the barriers: R (also the squaring scratch) | V scratch | eigenvectors of the batch |
// Jacobi rotation scratch
constexpr int F8_W_R = 0, F8_W_V = 1024, F8_W_VT = 2048, F8_W_ROT = 2048 + F8_BATCH * 1024, F8_W_PAIR = F8_W_ROT + 128;
constexpr int F8_WARP_BYTES = F8_W_PAIR + 64;     // 6336
constexpr size_t F8_OFF_BARS = F8_RING;           // uint64 full[24], empty[24]
constexpr size_t F8_OFF_WRING = F8_OFF_BARS + 2 * F8_WARPS * F8_SG * 8;  // int wring[8][8]
constexpr size_t F8_OFF_WARP = (F8_OFF_WRING + F8_WARPS * 8 * 4 + 127) / 128 * 128;
constexpr size_t F8_SMEM = F8_OFF_WARP + (size_t)F8_WARPS * F8_WARP_BYTES + 1024;  // + realignment slack
static_assert(F8_STAGE % 1024 == 0 && F8_SMEM <= 227 * 1024, "fused M = 8 kernel shared memory");

// Principal eigenvector + complement basis of the 8 x 8 Hermitian matrix in S (row-major, shared memory; destroyed).
// Lane owns the entries (r, c0), (r, c0 + 1) with r = lane >> 2, c0 = 2 (lane & 3).  Vt (64 complex) receives
// Vt[rank][i] like eig_coop_store: ranks 0..6 = complement basis, rank 7 = principal eigenvector.  On failure (returns
// false, warp-uniform) S holds the power-of-two scaled input again, ready for the Jacobi solver.
__device__ __forceinline__ bool eig8_principal_warp(double2 *S, double2 *Vt, const int lane)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int r = lane >> 2, c0 = 2 * (lane & 3);
    const bool diag_owner = c0 == (r & ~1);  // this lane holds (r, r): its entry number r & 1
    auto row_sum = [&](double v) {           // over the 4 lanes of a row
        v += __shfl_xor_sync(FULL, v, 1);
        v += __shfl_xor_sync(FULL, v, 2);
        return v;
    };
    auto col_sum = [&](double v) {           // over the 8 rows (lanes of equal lane & 3)
        v += __shfl_xor_sync(FULL, v, 4);
        v += __shfl_xor_sync(FULL, v, 8);
        v += __shfl_xor_sync(FULL, v, 16);
        return v;
    };
    double2 a0[2] = {S[r * 8 + c0], S[r * 8 + c0 + 1]}, a[2];
    bool okc;
    const double sc0 = eigp_pow2_scale(warp_sum(diag_owner ? ((r & 1) ? a0[1].x : a0[0].x) : 0.0), okc);
#pragma unroll
    for (int i = 0; i < 2; ++i) { a0[i].x *= sc0; a0[i].y *= sc0; a[i] = a0[i]; }
    int st = okc ? 0 : 3;  // 0 squaring, 1 rank-one test passed (one more squaring), 2 converged, 3 failed
    __syncwarp();
    for (int it = 0; it < EIGP_MAXSQ && st < 2; ++it) {
        S[r * 8 + c0] = a[0];
        S[r * 8 + c0 + 1] = a[1];
        __syncwarp();
        double2 n0 = make_double2(0.0, 0.0), n1 = make_double2(0.0, 0.0);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const double2 x = S[r * 8 + k], b0 = S[k * 8 + c0], b1 = S[k * 8 + c0 + 1];
            n0.x = fma(x.x, b0.x, n0.x); n0.x = fma(-x.y, b0.y, n0.x);
            n0.y = fma(x.x, b0.y, n0.y); n0.y = fma(x.y, b0.x, n0.y);
            n1.x = fma(x.x, b1.x, n1.x); n1.x = fma(-x.y, b1.y, n1.x);
            n1.y = fma(x.x, b1.y, n1.y); n1.y = fma(x.y, b1.x, n1.y);
        }
        __syncwarp();
        if (diag_owner) { if (r & 1) n1.y = 0.0; else n0.y = 0.0; }
        const double t = warp_sum(diag_owner ? ((r & 1) ? n1.x : n0.x) : 0.0);
        const double f = warp_sum(fma(n0.x, n0.x, fma(n0.y, n0.y, fma(n1.x, n1.x, n1.y * n1.y))));
        bool oks;
        const double sc = eigp_pow2_scale(t, oks);
        const bool pass = f >= 0.999999999 * (t * t);
        a[0] = make_double2(n0.x * sc, n0.y * sc);
        a[1] = make_double2(n1.x * sc, n1.y * sc);
        st = !oks ? 3 : (st == 1 ? 2 : (pass ? 1 : 0));
    }
    bool ok = st == 2;
    // the column with the largest diagonal (ties: lowest index) is mu e conj(e_j*): conj of row j*
    S[r * 8 + c0] = a[0];
    S[r * 8 + c0 + 1] = a[1];
    __syncwarp();
    int js = 0;
    double dm = S[0].x;
#pragma unroll
    for (int k = 1; k < 8; ++k) {
        const double d = S[k * 9].x;
        if (d > dm) { dm = d; js = k; }
    }
    double ur[8], ui[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const double2 b = S[js * 8 + c];
        ur[c] = b.x; ui[c] = -b.y;
    }
    __syncwarp();
    // two power steps with the original (scaled) matrix, then one more product for the certificate
    const bool hi0 = (lane & 3) >= 2, odd0 = (lane & 1) != 0;  // c0 = 4 hi0 + 2 odd0
    for (int step = 0; step < 3; ++step) {
        // u at my two columns (static register indices via selects)
        const double x0r = hi0 ? (odd0 ? ur[6] : ur[4]) : (odd0 ? ur[2] : ur[0]), x0i = hi0 ? (odd0 ? ui[6] : ui[4]) : (odd0 ? ui[2] : ui[0]);
        const double x1r = hi0 ? (odd0 ? ur[7] : ur[5]) : (odd0 ? ur[3] : ur[1]), x1i = hi0 ? (odd0 ? ui[7] : ui[5]) : (odd0 ? ui[3] : ui[1]);
        double wr = fma(a0[0].x, x0r, -(a0[0].y * x0i)), wi = fma(a0[0].x, x0i, a0[0].y * x0r);
        wr = fma(a0[1].x, x1r, wr); wr = fma(-a0[1].y, x1i, wr);
        wi = fma(a0[1].x, x1i, wi); wi = fma(a0[1].y, x1r, wi);
        wr = row_sum(wr);
        wi = row_sum(wi);  // w_r, identical in the 4 lanes of row r
        // u_r (static selects again)
        const int rr = r;
        const double urr = rr == 0 ? ur[0] : rr == 1 ? ur[1] : rr == 2 ? ur[2] : rr == 3 ? ur[3] : rr == 4 ? ur[4] : rr == 5 ? ur[5] : rr == 6 ? ur[6] : ur[7];
        const double uir = rr == 0 ? ui[0] : rr == 1 ? ui[1] : rr == 2 ? ui[2] : rr == 3 ? ui[3] : rr == 4 ? ui[4] : rr == 5 ? ui[5] : rr == 6 ? ui[6] : ui[7];
        if (step == 2) {
            const double lam = col_sum(fma(urr, wr, uir * wi));
            const double qr = fma(-lam, urr, wr), qi = fma(-lam, uir, wi);
            const double res2 = col_sum(fma(qr, qr, qi * qi));
            ok = ok && (res2 <= 1e-24 * (lam * lam)) && lam > 0.0;
            break;
        }
        const double inv = 1.0 / sqrt(col_sum(fma(wr, wr, wi * wi)));
        if ((lane & 3) == 0) S[r] = make_double2(wr * inv, wi * inv);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 8; ++c) { ur[c] = S[c].x; ui[c] = S[c].y; }
        __syncwarp();
    }
    if (!ok) {  // hand the (scaled) input back to the caller for the Jacobi solver
        S[r * 8 + c0] = a0[0];
        S[r * 8 + c0 + 1] = a0[1];
        __syncwarp();
        return false;
    }
    double pr, pi;
    eig_phase(ur[0], ui[0], pr, pi);
    double er[8], ei[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) eig_out4(ur[c], ui[c], pr, pi, er[c], ei[c]);
    ei[0] = 0.0;
    const double h = 1.0 / (1.0 + er[0]);
    // my two entries of Vt: rank = r (7: the eigenvector, rho < 7: g_q with q = rho + 1), components i = c0, c0 + 1
    const int q = r + 1;
    const double eqr = q == 1 ? er[1] : q == 2 ? er[2] : q == 3 ? er[3] : q == 4 ? er[4] : q == 5 ? er[5] : q == 6 ? er[6] : er[7];
    const double eqi = q == 1 ? ei[1] : q == 2 ? ei[2] : q == 3 ? ei[3] : q == 4 ? ei[4] : q == 5 ? ei[5] : q == 6 ? ei[6] : ei[7];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int i = c0 + s;
        const double eir = s == 0 ? (hi0 ? (odd0 ? er[6] : er[4]) : (odd0 ? er[2] : er[0])) : (hi0 ? (odd0 ? er[7] : er[5]) : (odd0 ? er[3] : er[1]));
        const double eii = s == 0 ? (hi0 ? (odd0 ? ei[6] : ei[4]) : (odd0 ? ei[2] : ei[0])) : (hi0 ? (odd0 ? ei[7] : ei[5]) : (odd0 ? ei[3] : ei[1]));
        double2 out;
        if (r == 7) {
            out = make_double2(eir, eii);
        } else if (i == 0) {
            out = make_double2(-eqr, eqi);  // -conj(e_q)
        } else {
            const double pr2 = fma(eir, eqr, eii * eqi), pi2 = fma(eii, eqr, -(eir * eqi));  // e_i conj(e_q)
            out = make_double2(fma(-pr2, h, i == q ? 1.0 : 0.0), -(pi2 * h));
        }
        Vt[r * 8 + i] = out;
    }
    __syncwarp();
    return true;
}

__global__ void __launch_bounds__(F8_WARPS * 32, 1)
music8_fused_kernel(const __grid_constant__ CUtensorMap tm, const double *__restrict__ soa, int W, int N, int K, const PeakOut out,
                    unsigned *__restrict__ work_ctr, const GatherFlags gather_flags, const bool eig_mode /* false: squaring; true: Jacobi */,
                    unsigned *__restrict__ stats /* optional [2]: windows solved by squaring / by Jacobi */)
{
    const unsigned long long tm_addr = reinterpret_cast<unsigned long long>(&tm);
    constexpr int M = 8;
    extern __shared__ __align__(1024) unsigned char f8_smem_raw[];
    unsigned char *smem = f8_smem_raw + ((1024u - (smem_u32(f8_smem_raw) & 1023u)) & 1023u);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + F8_OFF_BARS);
    volatile int *wring = reinterpret_cast<volatile int *>(smem + F8_OFF_WRING) + warp * 8;
    unsigned char *ring = smem + (size_t)warp * F8_SG * F8_STAGE;
    unsigned char *wsm = smem + F8_OFF_WARP + (size_t)warp * F8_WARP_BYTES;
    double2 *Rw = reinterpret_cast<double2 *>(wsm + F8_W_R), *Vs = reinterpret_cast<double2 *>(wsm + F8_W_V);
    double2 *Vb = reinterpret_cast<double2 *>(wsm + F8_W_VT);
    double(*rot)[4] = reinterpret_cast<double(*)[4]>(wsm + F8_W_ROT);
    int(*pair)[2] = reinterpret_cast<int(*)[2]>(wsm + F8_W_PAIR);
    const uint32_t full0 = smem_u32(bars + warp * F8_SG), ring0 = smem_u32(ring);
    if (lane == 0) {
        for (int s = 0; s < F8_SG; ++s) mbar_init(full0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();

    const int cpw = (N + F8_ROWS - 1) / F8_ROWS;  // chunks per window (the last one is zero-filled beyond N)
    // producer state (lane 0): next chunk to request = chunk iq of window iw
    int iq = 0, iw = -1, wr = 0;
    unsigned issued = 0;
    auto claim = [&]() {
        const unsigned tkt = atomicAdd(&work_ctr[0], 1u);
        iw = tkt < (unsigned)W ? (int)tkt : -1;
        wring[wr & 7] = iw;
        ++wr;
    };
    const uint64_t pol_stream = l2_policy_evict_first();
    auto issue = [&]() {  // the slot is free: the only consumer is this warp, in program order
        const int slot = (int)(issued % F8_SG);
        mbar_expect_tx(full0 + 8 * slot, F8_STAGE);
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;"
                     ::"r"(ring0 + slot * F8_STAGE), "l"(tm_addr), "r"(0), "r"(iq * (F8_STAGE / 128)), "r"(iw), "r"(full0 + 8 * slot), "l"(pol_stream)
                     : "memory");  // evict_first: the stream is read once and must not push the steering table out of L2
        ++issued;
        if (++iq == cpw) { iq = 0; claim(); }
    };
    if (lane == 0) {
        claim();
        for (int s = 0; s < F8_SG && iw >= 0; ++s) issue();
    }
    __syncwarp();

    const int Kpad = (K + TILE - 1) / TILE * TILE;
    int nb = 0;          // windows waiting in the batch
    int wid[F8_BATCH];   // their window numbers
#pragma unroll
    for (int b = 0; b < F8_BATCH; ++b) wid[b] = 0;
    unsigned n_sq = 0, n_jac = 0;

    auto scan_batch = [&]() {
        uint32_t ev[F8_BATCH];
#pragma unroll
        for (int b = 0; b < F8_BATCH; ++b) ev[b] = smem_u32(Vb + 64 * min(b, nb - 1));
        PeakState<F8_BATCH> ps;
        ps.reset();
        for (int k = lane; k < Kpad; k += 32) {
            const double *tb = soa + (size_t)(k / TILE) * (2 * M + 1) * TILE + (k % TILE);
            double ar[M], ai[M];
#pragma unroll
            for (int i = 0; i < M; ++i) {
                ar[i] = __ldg(tb + (size_t)(2 * i) * TILE);
                ai[i] = __ldg(tb + (size_t)(2 * i + 1) * TILE);
            }
            const double na = __ldg(tb + (size_t)(2 * M) * TILE);
            scan_bin<M, F8_BATCH>(ar, ai, na, k, ev, ps);
        }
#pragma unroll
        for (int b = 0; b < F8_BATCH; ++b) {
            int kk = ps.bestk[b];
            double P = kk >= 0 ? 1.0 / ps.bestd[b] : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double Po = __shfl_xor_sync(0xffffffffu, P, o);
                const int ko = __shfl_xor_sync(0xffffffffu, kk, o);
                if (peak_better(Po, ko, P, kk)) { P = Po; kk = ko; }
            }
            if (lane == b && b < nb) {
                const size_t o = (size_t)wid[b];
                if (kk >= 0) {
                    out.angles[o] = (float)((double)kk * 360.0 / (double)K);  // reference :134, :153
                    if (out.levels) out.levels[o] = (float)P;                 // reference :154
                } else {
                    out.angles[o] = 0.f;                                      // (0,0) initial pair, reference :95
                    if (out.levels) out.levels[o] = 0.f;
                }
                peak_store_bin(out, o, kk);
            }
        }
        __syncwarp();
        nb = 0;
    };

    unsigned consumed = 0;
    for (int rd = 0;; ++rd) {
        const int wcur = wring[rd & 7];
        if (wcur < 0) break;
        double acc[64];  // (not live across the eigenvector / scan phases below)
#pragma unroll
        for (int i = 0; i < 64; ++i) acc[i] = 0.0;
        for (int q = 0; q < cpw; ++q, ++consumed) {
            const int slot = (int)(consumed % F8_SG);
            while (!mbar_try_wait(full0 + 8 * slot, (consumed / F8_SG) & 1)) {}
            const unsigned char *stage = ring + (size_t)slot * F8_STAGE;
#pragma unroll
            for (int rr = 0; rr < F8_STEPS; ++rr) {
                const int r = lane + 32 * rr;
                const CovnQuad a = covn_quad<M>(stage, r, 0), b = covn_quad<M>(stage, r, 1);
                covn_acc_off(acc, a, b);
                covn_acc_diag(acc + 32, a);
                covn_acc_diag(acc + 48, b);
            }
            __syncwarp();  // every lane is done reading the slot -> it may be refilled
            if (lane == 0 && iw >= 0) issue();
        }
        __syncwarp();  // lane 0's ring writes (claims during this window) become visible to the next read
        // transposing butterfly (music_covn.cuh): lane l ends up owning entries 2l and 2l + 1
#pragma unroll
        for (int o = 16, n = 32; o >= 1; o >>= 1, n >>= 1) {
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < n; ++i) {
                const double send = upper ? acc[i] : acc[i + n];
                const double keep = upper ? acc[i + n] : acc[i];
                acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
        }
        {
            const double dn = (double)N;
            const double v0 = acc[0] / dn, v1 = acc[1] / dn;
            if (lane < 16) {  // complex entry (i, j) of the off-diagonal block (0, 1)
                const int r = lane >> 2, c = 4 + (lane & 3);
                Rw[r * M + c] = make_double2(v0, v1);
                Rw[c * M + r] = make_double2(v0, -v1);
            } else {  // diagonal half of block I: lanes 0-1 of the octet hold the 4 real diagonals, lanes 2-7 the 6 pairs
                const int I = lane < 24 ? 0 : 1, e = lane & 7;
                if (e < 2) {
                    const int r = 4 * I + 2 * e;
                    Rw[r * M + r] = make_double2(v0, 0.0);
                    Rw[(r + 1) * M + r + 1] = make_double2(v1, 0.0);
                } else {
                    const int p = e - 2;  // (0,1) (0,2) (0,3) (1,2) (1,3) (2,3)
                    const int i = p < 3 ? 0 : (p < 5 ? 1 : 2), j = p < 3 ? p + 1 : (p < 5 ? p - 1 : 3);
                    const int r = 4 * I + i, c = 4 * I + j;
                    Rw[r * M + c] = make_double2(v0, v1);
                    Rw[c * M + r] = make_double2(v0, -v1);
                }
            }
        }
        __syncwarp();
        // eigenvectors of this window -> batch slot nb
        double2 *Vt = Vb + 64 * nb;
        bool solved = false;
        if (!eig_mode) solved = eig8_principal_warp(Rw, Vt, lane);
        if (solved) {
            ++n_sq;
        } else {
            eig_coop_warp<M>(Rw, Vs, rot, pair, lane);
            eig_coop_store<M>(Rw, Vs, nullptr, Vt, lane);
            __syncwarp();
            ++n_jac;
        }
#pragma unroll
        for (int b = 0; b < F8_BATCH; ++b)
            if (b == nb) wid[b] = wcur;
        if (++nb == F8_BATCH) scan_batch();
    }
    if (nb > 0) scan_batch();
    if (stats && lane == 0) {
        if (n_sq) atomicAdd(&stats[0], n_sq);
        if (n_jac) atomicAdd(&stats[1], n_jac);
    }
    // the last CTA to finish re-arms the ticket counter (launches that share it are ordered by the host) and, when the
    // peak bins went to peer GPUs, raises this GPU's epoch flag at every peer
    __syncthreads();
    if (threadIdx.x == 0) {
        if (out.npeer > 0) __threadfence_system(); else __threadfence();
        if (atomicAdd(&work_ctr[1], 1u) == gridDim.x - 1) {
            work_ctr[0] = 0;
            work_ctr[1] = 0;
            __threadfence();
            if (out.npeer > 0 && gather_flags.epoch) {
                __threadfence_system();
                for (int p = 0; p < out.npeer; ++p)
                    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(gather_flags.peer[p] + out.rank), "r"(gather_flags.epoch) : "memory");
            }
        }
    }
}

}  // namespace music
