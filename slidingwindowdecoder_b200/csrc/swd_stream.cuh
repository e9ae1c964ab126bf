// swd_stream.cuh — full-window min-sum BP for graphs whose messages do not fit one SM's shared memory
// (8 * nnz > ~220 KB: e.g. the un-windowed [[144,12,12]] DEM, 936 x 8784 with 30672 edges, IBM.ipynb:122-123).
//
// Same arithmetic as pre_bp_kernel (bp_guessing_decoder.pyx:48-139 / osd_window.pyx:381-485), different mapping:
// one THREAD per shot, a warp = 32 consecutive shots, and the messages live in HBM in a shot-interleaved layout
//     msg[p * G + g]        p = CSR position of the edge, g = the thread's index in the tile of G shots
// so that every message access of a warp is one fully coalesced 256-byte line and the graph indices are
// warp-uniform (broadcast loads through L1): no bank conflicts, no barriers, no divergence except shots that have
// already converged (their lanes stop issuing loads and stores).  Per iteration and shot the kernel moves exactly the
// algorithmic bytes of SURVEY 8(d): read E + write E in the check pass, read E + write E in the variable pass
// (E * 32 bytes) plus 8 n bytes of posterior history - HBM is the roof that binds here.
// The parity of the hard decisions is kept as bit words in shared memory ([word][thread]), the syndrome as bit words in HBM.
#pragma once
#include "swd_device.cuh"

struct StreamWs {
    double *msg;        // [nnz][G]
    double *hs;         // [4][n][G]   posterior ring (slot = iteration & 3)
    u32 *decw;          // [ceil(n/32)][G] hard decisions, bit v & 31 of word v >> 5
    u32 *syndw;         // [ceil(m/32)][G] syndrome bit words
    int *itdone;        // [G] iterations executed
    u8 *conv;           // [G]
    long long G;        // shots per tile = threads of the launch
    const double *llrT; // [n][G] per-shot priors of the tile, transposed like hs (per-shot calls only)
};

// Memory-level parallelism is what this kernel lives on.  Both passes read the messages in a sequence that is known in
// advance (check pass: CSR positions 0, 1, 2, ...; variable pass: cpos[0], cpos[1], ...), so every thread keeps SWD_SK
// asynchronous 8-byte copies (cp.async, LDGSTS) in flight into its own ring of shared-memory slots, SWD_SK edges ahead of
// the one it is working on: a warp has 16 coalesced 256-byte lines outstanding all the time instead of one batch per
// variable node (ncu: first version 7 % of the HBM roof, register-batched loads 27 %).  A thread only ever reads the slots
// it filled itself, so there is no barrier and no mbarrier - cp.async.wait_group orders each copy before its use.
#ifndef SWD_SK
#define SWD_SK 16          /* 32 measured 7 % slower: the ring is not what limits the lines in flight */
#endif
#ifndef SWD_STREAM_MINB
#define SWD_STREAM_MINB 2
#endif
__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// SHOT = true: priors from sw.llrT (the tile's rows of g.llr_shot, transposed by llr_transpose_kernel): one coalesced line
// per warp, as the messages, where a row-major read would cost one sector per lane.
template <int DM, bool SHOT = false>
__global__ void __launch_bounds__(256, SWD_STREAM_MINB)
pre_bp_stream_kernel(GraphDev g, const u8 *__restrict__ synd, long long B, long long tile_base, int max_iter, double alpha,
                     StreamWs sw, int full_hist, u64 *stats) {
    constexpr int K = SWD_SK;
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = blockDim.x, tid = threadIdx.x;
    const int m = g.m, n = g.n, nnz = g.nnz, MW = (m + 31) >> 5;
    double *ring = (double *)smem + tid;       // [K][T] doubles: slot s of this thread = ring[s * T]
    u32 *s_par = (u32 *)(smem + (size_t)8 * K * T);    // [MW][T] parity of H * e per check, bit words
    const long long gid = (long long)blockIdx.x * T + tid;
    const long long shot = tile_base + gid;
    const long long G = sw.G;
    const bool live = shot < B;
    double *msg = sw.msg + gid;
    u32 *g_synd = sw.syndw + gid;              // [MW][G] syndrome bit words (HBM / L2: one coalesced word per 32 rows)
    // ---- syndrome bytes -> bit words
    for (int w = 0; w < MW; w++) {
        u32 word = 0;
        if (live) {
            const int r1 = min(32, m - 32 * w);
            for (int b = 0; b < r1; b++) word |= (u32)(synd[shot * m + 32 * w + b] & 1u) << b;
        }
        g_synd[(size_t)w * G] = word;
    }
    bool done = !live;
    int iters = 0, conv = 0;
    u64 edge_passes = 0;
    for (int it = 0; it < max_iter; it++) {
        if (__all_sync(FULLMASK, done)) break;
        if (done) continue;
        // ---- check pass: min1 / min2 / argmin / parity (pyx:62-96); iteration 1 reads the priors (pyx:55-60)
        if (it > 0) {
#pragma unroll
            for (int i = 0; i < K; i++) { if (i < nnz) cp_async8(ring + i * T, msg + (size_t)i * G); cp_async_commit(); }
        }
        u32 sword = 0;
        for (int r = 0; r < m; r++) {
            const int p0 = __ldg(g.rp + r), p1 = __ldg(g.rp + r + 1);
            double m1 = SWD_BIG, m2 = SWD_BIG; int arg = -1;
            if ((r & 31) == 0) sword = g_synd[(size_t)(r >> 5) * G];
            u32 par = (sword >> (r & 31)) & 1u;
            u64 neg = 0;
#pragma unroll 4
            for (int p = p0; p < p1; p++) {
                double b;
                if (it == 0) b = SHOT ? sw.llrT[(size_t)__ldg(g.rc + p) * G + gid] : __ldg(g.llr + __ldg(g.rc + p));
                else {
                    cp_async_wait<K - 1>();
                    b = ring[(p & (K - 1)) * T];
                    if (p + K < nnz) cp_async8(ring + (p & (K - 1)) * T, msg + (size_t)(p + K) * G);
                    cp_async_commit();
                }
                double a = fabs(b);
                a = (a > SWD_CLIP) ? SWD_CLIP : a;
                const bool lt = a < m1;
                const double hi = lt ? m1 : a;
                m2 = (hi < m2) ? hi : m2;
                m1 = lt ? a : m1;
                arg = lt ? p : arg;
                const u32 ng = (u32)(b <= 0.0);
                par ^= ng;
                if (p - p0 < 64) neg |= (u64)ng << (p - p0);
            }
            const double q1 = m1 * alpha, q2 = m2 * alpha;
#pragma unroll 4
            for (int p = p0; p < p1; p++) {
                u32 ng;
                if (p - p0 < 64) ng = (u32)((neg >> (p - p0)) & 1ull);
                else ng = (u32)(((it == 0) ? (SHOT ? sw.llrT[(size_t)__ldg(g.rc + p) * G + gid] : __ldg(g.llr + __ldg(g.rc + p)))
                                           : msg[(size_t)p * G]) <= 0.0);   // rows longer than 64: re-read (not yet overwritten)
                msg[(size_t)p * G] = flip_sign((p == arg) ? q2 : q1, par ^ ng);
            }
        }
        cp_async_wait<0>();
        // ---- variable pass: ordered prefix / suffix sums (pyx:98-127), hard decisions, parity of H * e
        for (int w = 0; w < MW; w++) s_par[w * T + tid] = 0;
        const bool keep = full_hist || (it >= max_iter - 4);
        double *hs = sw.hs + ((size_t)(it & 3) * n) * G + gid;
        u32 decw = 0;
#pragma unroll
        for (int i = 0; i < K; i++) { if (i < nnz) cp_async8(ring + i * T, msg + (size_t)__ldg(g.cpos + i) * G); cp_async_commit(); }
        for (int v = 0; v < n; v++) {
            const int e0 = __ldg(g.cp + v), d = __ldg(g.cp + v + 1) - e0;
            double cc[DM], pre[DM]; int pp[DM];
            double t = SHOT ? sw.llrT[(size_t)v * G + gid] : __ldg(g.llr + v);
#pragma unroll
            for (int k = 0; k < DM; k++) {
                if (k < d) {
                    const int e = e0 + k;
                    pp[k] = __ldg(g.cpos + e);
                    cp_async_wait<K - 1>();
                    cc[k] = ring[(e & (K - 1)) * T];
                    if (e + K < nnz) cp_async8(ring + (e & (K - 1)) * T, msg + (size_t)__ldg(g.cpos + e + K) * G);
                    cp_async_commit();
                    pre[k] = t; t += cc[k];
                }
            }
            const u32 hard = (u32)(t <= 0.0);
            decw |= hard << (v & 31);
            if ((v & 31) == 31 || v == n - 1) { sw.decw[(size_t)(v >> 5) * G + gid] = decw; decw = 0; }
            if (hard) {
#pragma unroll 1
                for (int k = 0; k < d; k++) { const int r = __ldg(g.cr + e0 + k); s_par[(r >> 5) * T + tid] ^= 1u << (r & 31); }
            }
            double s = 0.0;
#pragma unroll
            for (int k = DM - 1; k >= 0; k--) if (k < d) { msg[(size_t)pp[k] * G] = pre[k] + s; s += cc[k]; }
            if (keep) hs[(size_t)v * G] = t;
        }
        cp_async_wait<0>();
        iters = it + 1;
        edge_passes++;
        u32 mism = 0;
        for (int w = 0; w < MW; w++) mism |= s_par[w * T + tid] ^ g_synd[(size_t)w * G];
        if (!mism) { conv = 1; done = true; }
    }
    if (live) { sw.itdone[gid] = iters; sw.conv[gid] = (u8)conv; }
    // work counter: edge-iterations (warp-reduced)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) edge_passes += __shfl_xor_sync(FULLMASK, edge_passes, o);
    if ((tid & 31) == 0 && edge_passes) atomicAdd(&stats[0], edge_passes * (u64)g.nnz);
}

// One warp per shot of the tile: unpacks the hard decisions to bytes, appends non-converged shots to the work list with
// their posterior-history sums (the sort keys), writes the osd_window outputs (history, iteration count).
__global__ void pre_bp_stream_finish_kernel(GraphDev g, long long B, long long tile_base, StreamWs sw, u8 *__restrict__ dec_out,
                                            u8 *__restrict__ conv_out, Workspace ws, int *iter_out, double *lpr_out) {
    const int lane = threadIdx.x & 31;
    const long long wglobal = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int n = g.n;
    const long long G = sw.G;
    for (long long gi = wglobal; gi < G && tile_base + gi < B; gi += nwarps) {
        const long long shot = tile_base + gi;
        const int it = sw.itdone[gi], conv = sw.conv[gi];
        int slot = -1;
        if (!conv) {
            if (lane == 0) { slot = atomicAdd(&ws.counters[0], 1); ws.gdg_list[slot] = (int)shot; }
            slot = __shfl_sync(FULLMASK, slot, 0);
        }
        if (lane == 0) { conv_out[shot] = (u8)conv; if (iter_out) iter_out[shot] = it; }
        for (int v = lane; v < n; v += 32) {
            dec_out[shot * n + v] = (u8)((sw.decw[(size_t)(v >> 5) * G + gi] >> (v & 31)) & 1u);
            if (!conv || lpr_out) {
                double h4[4];
#pragma unroll
                for (int s = 0; s < 4; s++) h4[s] = (s < it) ? sw.hs[((size_t)s * n + v) * G + gi] : 0.0;     // fresh ring: unwritten slots are 0
                if (!conv) {
                    ws.sum[(size_t)slot * n + v] = ((h4[0] + h4[1]) + h4[2]) + h4[3];
                    if (ws.hist) {
#pragma unroll
                        for (int s = 0; s < 4; s++) ws.hist[((size_t)slot * n + v) * 4 + s] = h4[s];
                    }
                }
                if (lpr_out) {
#pragma unroll
                    for (int s = 0; s < 4; s++) lpr_out[((size_t)shot * n + v) * 4 + s] = h4[s];
                }
            }
        }
    }
}

// Per-shot priors of one tile, [nb][n] row-major (rows tile_base.. of g.llr_shot) -> llrT [n][G]: 32 x 32 blocks through
// shared memory, coalesced on both sides.  Rows past the batch are left unwritten (their lanes never read them).
__global__ void __launch_bounds__(256)
llr_transpose_kernel(const double *__restrict__ llr_shot, long long B, long long tile_base, int n, long long G, double *__restrict__ llrT) {
    __shared__ double t[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 8 rows of 32
    const long long s0 = tile_base + (long long)blockIdx.y * 32;     // first shot of the block
    const int v0 = blockIdx.x * 32;
    for (int i = ty; i < 32; i += 8) {
        const long long shot = s0 + i; const int v = v0 + tx;
        if (shot < B && v < n) t[i][tx] = llr_shot[(size_t)shot * n + v];
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int v = v0 + i; const long long shot = s0 + tx;
        if (shot < B && v < n) llrT[(size_t)v * G + (shot - tile_base)] = t[tx][i];
    }
}
