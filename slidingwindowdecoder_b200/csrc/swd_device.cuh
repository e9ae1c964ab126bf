// swd_device.cuh — device-side building blocks of the B200 window decoder.
//
// Semantics follow the reference's BPGD class (src/include/bpgd.cpp) but none of its
// structure: the Tanner graph is flat CSR/CSC, a branch path is executed by one CTA,
// messages live in ONE shared-memory array that alternately holds bit-to-check and
// check-to-bit values, decided variables are marked by a NaN in their message slots,
// and the posterior history ring lives in registers of the thread that owns the VN.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

typedef uint16_t u16;
typedef uint8_t  u8;
typedef int8_t   i8;
typedef uint32_t u32;
typedef unsigned long long u64;

#define SWD_BIG     1e308       /* empty-min sentinel, bpgd.cpp:106 */
#define SWD_CLIP    50.0        /* bpgd.cpp:120-121 */
#define SWD_MAX_PM  10000.0     /* bpgd.cpp:11 */
#define FULLMASK    0xffffffffu
#define SWD_CPT     4           /* checks owned per thread in path kernels: m <= SWD_CPT * blockDim */
#ifndef SWD_DIET
#define SWD_DIET    1           /* 1: cvn, the reset snapshot and the tree backup stay in HBM (L2), not in shared memory */
#endif

// ----------------------------------------------------------------------------------------------
// layouts (byte offsets), computed once on the host
// ----------------------------------------------------------------------------------------------
struct SubLayout {              // per-slot "sub-graph blob": shortened graph + reset snapshot
    int nn, m, es_max;          // es_max: edge capacity of THIS layout (shared-memory tiers differ)
    int lcap;                   // max row length of the window graph
    int off_prior;              // double[nn]
    int off_col;                // u16[nn]     original column of sub-VN j (sorted order)
    int off_voff;               // u16[nn+1]
    int off_coff;               // u16[m+1]    first message slot of the check with rank q (rows padded to odd length)
    int off_crank;              // u16[m]      rank q of check r (checks ranked by row length, descending)
    int off_synd;               // u8[m]
    int off_vnmask;             // i8[nn]      state after reset (bpgd.cpp:199-239)
    int off_cnmask;             // i8[m]
    int off_cndeg;              // u8[m]
    int off_vperm;              // u16[nn]     VN ownership order (sorted by degree: uniform work per warp)
    int off_cperm;              // u16[m]      check ownership order (sorted by row length)
    int fixed_bytes;            // multiple of 16: header + all of the above
    int off_vrow, off_vpos, off_cvn;   // u16[es_max] each, 16-byte aligned; vpos / cvn use jagged-diagonal slots
    int blob_bytes;             // multiple of 16
};
struct BlobHeader { int es; int status; int bad_rows; int shot; };   // 16 bytes at offset 0

struct PathSmem {               // dynamic shared memory of path_kernel, offsets after the blob image
    int off_msg;                // double[es_max]
    int off_vnmask, off_error, off_dec;       // i8[nn]
    int off_cnmask;             // i8[m]
    int off_cndeg, off_flip;    // u8[m]
    int off_upar;               // u32[m]
    int off_bvn, off_bcn, off_bdeg;           // backup snapshot (tree paths)
    int off_red;                // reduction scratch: 64 doubles + 64 ints
    int off_misc;               // ints: broadcast slots
    int off_bar;                // mbarrier (8 bytes)
    int total;
};

struct GraphDev {               // static window graph (device pointers)
    int m, n, nnz;
    const int *rp;              // [m+1]  CSR row pointer
    const u16 *rc;              // [nnz]  CSR column index
    const int *cp;              // [n+1]  CSC column pointer
    const u16 *cr;              // [nnz]  CSC row index (ascending)
    const u16 *cpos;            // [nnz]  CSC entry -> CSR position
    const u16 *vord;            // [n]    columns in descending degree order (ownership order of the pre-BP kernel)
    const double *llr;          // [n]
    const u32 *vrec;            // [n]    per ownership slot: first CSC entry | degree << 16   (pre-BP kernel)
    const double *llr_s;        // [n]    llr in ownership-slot order
    // first check pass of the full-window min-sum BP for an all-zero syndrome: in iteration 1 every bit-to-check message
    // is its column's prior (pyx:55-60), so the check-to-bit magnitudes do not depend on the shot and a syndrome bit
    // only flips the sign of its row.  nullptr: not available (product-sum, osd-only graphs).
    const double *c2b1;         // [nphys]  physical slot order of the pre-BP kernel (pads: 0)
    const u16 *rowof;           // [nphys]  physical slot -> row (pads: 0)
    // Physical message layout of the pre-BP kernel (swd_api.cu: pre_layout).  The graph is the same for every shot, so the
    // slot of every edge is chosen once on the host such that BOTH passes are (nearly) bank-conflict free: rows start on
    // distinct 8-byte banks within every 16 consecutive rows (check pass: thread r reads prow[r] + k), and the order of the
    // slots inside a row - free, ties between equal magnitudes give q1 = q2 - is picked so that the 16 edges a half-warp of
    // the variable pass touches in step k fall on 16 distinct banks.
    int nphys;                  // message slots incl. the few pad slots between rows
    const u32 *prow;            // [m]    first physical slot | row length << 16
    const u16 *cpj;             // [nnz]  jagged-diagonal map: cpj[jb[k] + sl] = physical slot of the k-th edge of the column at
                                //        ownership slot sl (sl < number of columns of degree > k): lane-contiguous 16-bit loads
    int jb[17];
    // per-shot priors of the current chunk: row b = channel LLRs of chunk shot b (row-major [B][n], column order of the graph).
    // nullptr: every shot uses `llr`.  Set per launch by the *_llr entry points; read by the SHOT instantiations only.
    const double *llr_shot;
};

struct GdgDev {                 // parameters of the decimation tree
    int num_iter, max_step, T, S, tree_step, side_step, low_error, n_tree, n_side, n_rec;
    double factor;
    int rec_stride;             // bytes per result record
    int side_stride;            // bytes per side snapshot
    int kind;                   // SWD_KIND_*
    int multi_thread;
    int post_max_iter;
    // shared-prefix tree: the first shared_T decimation steps are identical for all branch paths with the same
    // prefix of favour/flip decisions, so they are computed once per prefix ("nodes") instead of once per path
    int shared_T, n_nodes, node_stride;
    int bak_stride;             // bytes per tree-path backup (vn_mask, cn_mask, cn_deg)
    int count_work;             // 1 while profiling is enabled (swd_set_profiling): the min-sum calls count their work
    int node_off_err, node_off_cn, node_off_deg, node_off_flip, node_off_msg, node_off_hist;
};

struct Workspace {              // per-batch device buffers
    int *counters;              // [0] gdg_count, [1..] tickets
    int *gdg_list;              // [cap] shot id per slot
    double *sum;                // [cap][n]      posterior-history sums (sort keys)
    double *hist;               // [cap][n][4]   pre-BP history (osd_window only) or NULL
    u8 *blob;                   // [cap][blob_bytes]
    u8 *rec;                    // [cap][n_rec][rec_stride]
    u8 *side;                   // [cap][n_side][side_stride]
    u8 *node;                   // [cap][n_nodes][node_stride] shared-prefix snapshots (masks, messages, history)
    u64 *stats;                 // device counters: [0] pre edge-iters [1] path edge-iters [2] paths [3] bp calls [4] osd shots
                                // [5] gdg shots [6] vn iters [7] cn iters [8] check-pass slots scanned [9] osd columns scanned [10] osd pivots
    // work lists of the branch-path launches: list `l` holds counters[SWD_WL_CNT + l] packed items at wl + l * wl_stride.
    // A launch only draws tickets for work that exists (a node that died or converged lists no children), and the item
    // itself carries what the set-up needs first (slot, branch path, message-slot count), so the shot's graph can be
    // requested from HBM right after the item is read.
    u64 *wl;
    long long wl_stride;
    u8 *bak;                    // [cap][n_tree][bak_stride] tree paths' backup state (bpgd.cpp:476-484), SWD_DIET only
};
#define SWD_WL_CNT   32          /* counters[32 ..]: list lengths */
#define SWD_WL_MAX   20
// item: bits 0..27 slot, 28..43 message slots (es), 44 bad_rows, 48..63 branch path
__device__ __forceinline__ u64 wl_pack(int slot, int es, int bad, int path) {
    return (u64)(u32)slot | ((u64)(u32)es << 28) | ((u64)(bad ? 1u : 0u) << 44) | ((u64)(u32)path << 48);
}
__device__ __forceinline__ void wl_push(const Workspace &ws, int list, u64 item) {
    const int pos = atomicAdd(&ws.counters[SWD_WL_CNT + list], 1);
    ws.wl[(size_t)list * ws.wl_stride + pos] = item;
}
// list ids (tier t = 0 typical shots / 1 oversized shortened graphs): node level l: 2 l + t; with T = shared_T:
// main path 2 T + t, other paths from depth T: 2 T + 2 + t, side branches 2 T + 4 + t.  Kinds without the shared-prefix
// tree use list t for their first (phase 0) launch.

// ----------------------------------------------------------------------------------------------
// small helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u64 *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 phase) {
    u32 ok = 0;
    while (!ok) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
    }
}
// L2 prefetch of a global range (16-byte aligned, size % 16 == 0): warms the cache for a TMA load issued later
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, u32 bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// TMA 1-D bulk copy global -> shared (SASS: UBLKCP); dst/src 16-byte aligned, bytes % 16 == 0
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, u32 bytes, u64 *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Shared-memory array bases are kept as opaque 32-bit shared-window addresses: the empty asm stops the compiler from
// re-deriving them from kernel parameters at every access (LDC + IADD3 + the S2R-based window base, ~40 % of the
// instructions of the min-sum loop before), so one register per hot array holds the base and accesses are LDS/STS [R+..].
__device__ __forceinline__ u32 pin_u32(u32 x) { asm volatile("" : "+r"(x)); return x; }
template <typename T>
__device__ __forceinline__ T *pinned_smem(const void *p) { return (T *)__cvta_shared_to_generic((size_t)pin_u32(smem_u32(p))); }

__device__ __forceinline__ double dnan() { return __longlong_as_double(0x7ff8000000000000LL); }

// lexicographic (value, index) minimum across the CTA. Result broadcast to all threads.
// red_d[>=32], red_i[>=32] shared scratch.  Contains __syncthreads().
__device__ __forceinline__ void block_argmin(double &v, int &idx, double *red_d, int *red_i) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(FULLMASK, v, o);
        int oi = __shfl_xor_sync(FULLMASK, idx, o);
        if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
    __syncthreads();                    // scratch may still be read from a previous call
    if (lane == 0) { red_d[wid] = v; red_i[wid] = idx; }
    __syncthreads();
    double bv = red_d[0]; int bi = red_i[0];
#pragma unroll 1
    for (int w = 1; w < nw; w++) {
        double ov = red_d[w]; int oi = red_i[w];
        if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    v = bv; idx = bi;
}

// exclusive scan over a[0..L] in shared memory (L+1 entries; a[L] should be 0 on entry and
// receives the total).  wt: >= 33 u32 of shared scratch.  Contains __syncthreads().
__device__ __forceinline__ void block_excl_scan(u32 *a, int L1, u32 *wt) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = (T + 31) >> 5;
    const int per = (L1 + T - 1) / T;
    int s = tid * per, e = s + per; if (e > L1) e = L1; if (s > L1) s = L1;
    u32 sum = 0;
    for (int i = s; i < e; i++) sum += a[i];
    u32 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { u32 t = __shfl_up_sync(FULLMASK, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) wt[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        u32 v = lane < nw ? wt[lane] : 0, iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { u32 t = __shfl_up_sync(FULLMASK, iv, o); if (lane >= o) iv += t; }
        wt[lane] = iv - v;
    }
    __syncthreads();
    u32 base = wt[wid] + incl - sum;
    for (int i = s; i < e; i++) { u32 t = a[i]; a[i] = base; base += t; }
    __syncthreads();
}

// stable ascending argsort of (key, idx) pairs held in shared memory (bitonic network on NP2
// elements; ties broken by idx, which makes it equal to std::stable_sort with operator<,
// bpgd.cpp:384-389).  Contains __syncthreads().
__device__ __forceinline__ void block_bitonic_sort(double *key, u16 *idx, int NP2) {
    const int T = blockDim.x, tid = threadIdx.x;
    for (int k = 2; k <= NP2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (NP2 >> 1); t += T) {
                int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                int hi = lo | j;
                bool asc = ((lo & k) == 0);
                double a = key[lo], b = key[hi];
                u16 ia = idx[lo], ib = idx[hi];
                bool gt = (b < a) || (!(a < b) && ib < ia);      // (a,ia) > (b,ib)
                if (gt == asc) { key[lo] = b; key[hi] = a; idx[lo] = ib; idx[hi] = ia; }
            }
            __syncthreads();
        }
    }
}

// The same argsort with E = NP2 / blockDim.x elements per thread held in registers (element i = tid * E + e): strides
// below E are compare-exchanges between registers, strides below 32 E are warp shuffles, and only the strides that cross
// warps go through shared memory (conflict-free transposed image, two barriers each): 6 block-wide exchange stages
// instead of 66 barrier-separated passes for NP2 = 2048.  (key, idx) is a strict total order on the real entries, so any
// correct network returns the order of std::stable_sort.  Loads the keys itself: src[0..n) (global), padded with
// (+inf, 0xffff); leaves the sorted idx[] (and key[]) in shared memory in natural order.  Contains __syncthreads().
__device__ __forceinline__ bool pair_less(double a, u32 ia, double b, u32 ib) { return (a < b) || (!(b < a) && ia < ib); }

template <int E>
__device__ __forceinline__ void block_bitonic_sort_regs(double *key, u16 *idx, int NP2, const double *__restrict__ src, int n) {
    const int T = blockDim.x, tid = threadIdx.x;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    double k_[E]; u32 i_[E];
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int i = tid * E + e;
        k_[e] = (i < n) ? src[i] : inf;
        i_[e] = (i < n) ? (u32)i : 0xffffu;
    }
    // runs up to length E: registers only
#pragma unroll
    for (int k = 2; k <= E; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int e = 0; e < E; e++) {
                if ((e & j) == 0) {
                    const bool asc = (((tid * E + e) & k) == 0);
                    const bool gt = pair_less(k_[e | j], i_[e | j], k_[e], i_[e]);
                    if (gt == asc) { const double tk = k_[e]; k_[e] = k_[e | j]; k_[e | j] = tk; const u32 ti = i_[e]; i_[e] = i_[e | j]; i_[e | j] = ti; }
                }
            }
        }
    }
    for (int k = 2 * E; k <= NP2; k <<= 1) {
        const bool asc = (((tid * E) & k) == 0);
        for (int j = k >> 1; j >= E; j >>= 1) {
            const int dj = j / E;                                  // distance in threads
            const bool keep_min = (((tid & dj) == 0) == asc);
            if (dj < 32) {
#pragma unroll
                for (int e = 0; e < E; e++) {
                    const double pk = __shfl_xor_sync(FULLMASK, k_[e], dj);
                    const u32 pi = __shfl_xor_sync(FULLMASK, i_[e], dj);
                    const bool pl = pair_less(pk, pi, k_[e], i_[e]);
                    const bool sl = pair_less(k_[e], i_[e], pk, pi);
                    if (keep_min ? pl : sl) { k_[e] = pk; i_[e] = pi; }
                }
            } else {
#pragma unroll
                for (int e = 0; e < E; e++) { key[e * T + tid] = k_[e]; idx[e * T + tid] = (u16)i_[e]; }
                __syncthreads();
                const int pt = tid ^ dj;
#pragma unroll
                for (int e = 0; e < E; e++) {
                    const double pk = key[e * T + pt];
                    const u32 pi = idx[e * T + pt];
                    const bool pl = pair_less(pk, pi, k_[e], i_[e]);
                    const bool sl = pair_less(k_[e], i_[e], pk, pi);
                    if (keep_min ? pl : sl) { k_[e] = pk; i_[e] = pi; }
                }
                __syncthreads();
            }
        }
#pragma unroll
        for (int j = E >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int e = 0; e < E; e++) {
                if ((e & j) == 0) {
                    const bool gt = pair_less(k_[e | j], i_[e | j], k_[e], i_[e]);
                    if (gt == asc) { const double tk = k_[e]; k_[e] = k_[e | j]; k_[e | j] = tk; const u32 ti = i_[e]; i_[e] = i_[e | j]; i_[e | j] = ti; }
                }
            }
        }
    }
#pragma unroll
    for (int e = 0; e < E; e++) { key[tid * E + e] = k_[e]; idx[tid * E + e] = (u16)i_[e]; }
    __syncthreads();
}

// The GDG kinds keep only the nn columns with the smallest keys (BPGD::reset copies the first new_n sorted columns,
// bpgd.cpp:199-209; the dropped ones are zeroed whatever their order), so a full argsort of n keys is not needed:
// radix-select the nn-th smallest on the order-preserving integer image of the keys (11 + 11 leading bits, two shared-
// memory histograms), compact the candidates (everything up to and including the boundary bucket, so ties stay
// together) and sort those CAP << n pairs.  idx[0..nn) then equals the first nn entries of the full stable argsort.
// Returns false (nothing written that matters) when the boundary bucket is too crowded - the caller sorts everything.
// E * blockDim.x >= n; key needs >= 2049 u32 and >= CAP u64; misc[4..7] and wt (>= 33 u32) are scratch.
__device__ __forceinline__ u64 ordered_key(double x) {
    if (x == 0.0) x = 0.0;                                          // -0.0 and +0.0 compare equal
    const u64 b = (u64)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

template <int E>
__device__ __forceinline__ bool block_select_sort(double *key, u16 *idx, u32 *wt, int *misc, const double *__restrict__ src,
                                                  int n, int nn, int CAP) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    u32 *hist = (u32 *)key; u64 *ckey = (u64 *)key;
    u64 k_[E];
#pragma unroll
    for (int e = 0; e < E; e++) { const int i = tid * E + e; k_[e] = (i < n) ? ordered_key(src[i]) : ~0ull; }
    for (int b = tid; b <= 2048; b += T) hist[b] = 0;
    __syncthreads();
#pragma unroll
    for (int e = 0; e < E; e++) if (tid * E + e < n) atomicAdd(&hist[(u32)(k_[e] >> 53)], 1u);
    __syncthreads();
    block_excl_scan(hist, 2049, wt);
    for (int b = tid; b < 2048; b += T) if ((int)hist[b] < nn && (int)hist[b + 1] >= nn) { misc[4] = b; misc[5] = (int)hist[b]; misc[6] = (int)hist[b + 1]; }
    __syncthreads();
    const u32 b1 = (u32)misc[4]; const int below = misc[5]; int upto = misc[6];
    u64 thr = b1; int sh = 53;
    if (upto > CAP) {                                                // refine inside the boundary bucket
        __syncthreads();
        for (int b = tid; b <= 2048; b += T) hist[b] = 0;
        __syncthreads();
#pragma unroll
        for (int e = 0; e < E; e++) if (tid * E + e < n && (u32)(k_[e] >> 53) == b1) atomicAdd(&hist[(u32)(k_[e] >> 42) & 0x7ffu], 1u);
        __syncthreads();
        block_excl_scan(hist, 2049, wt);
        const int need = nn - below;
        for (int b = tid; b < 2048; b += T) if ((int)hist[b] < need && (int)hist[b + 1] >= need) { misc[4] = b; misc[6] = below + (int)hist[b + 1]; }
        __syncthreads();
        thr = ((u64)b1 << 11) | (u32)misc[4]; sh = 42; upto = misc[6];
        if (upto > CAP) return false;
    }
    __syncthreads();
    if (tid == 0) misc[7] = 0;
    for (int p = upto + tid; p < CAP; p += T) { ckey[p] = ~0ull; idx[p] = (u16)0xffff; }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int i = tid * E + e;
        const bool cand = (i < n) && ((k_[e] >> sh) <= thr);
        const u32 bal = __ballot_sync(FULLMASK, cand);
        int base = 0;
        if (lane == 0 && bal) base = atomicAdd(&misc[7], __popc(bal));
        base = __shfl_sync(FULLMASK, base, 0);
        if (cand) { const int pos = base + __popc(bal & ((1u << lane) - 1)); ckey[pos] = k_[e]; idx[pos] = (u16)i; }
    }
    __syncthreads();
    for (int k = 2; k <= CAP; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (CAP >> 1); t += T) {
                const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;
                const bool asc = ((lo & k) == 0);
                const u64 a = ckey[lo], b = ckey[hi];
                const u16 ia = idx[lo], ib = idx[hi];
                const bool gt = (b < a) || (b == a && ib < ia);
                if (gt == asc) { ckey[lo] = b; ckey[hi] = a; idx[lo] = ib; idx[hi] = ia; }
            }
            __syncthreads();
        }
    }
    return true;
}

// The same selection for any n (keys re-read from global memory at every level instead of held in registers) and without a
// fall-back: the radix descent continues over all 64 key bits (11 bits per level, 9 at the last), and if the boundary
// bucket is still too crowded then all its keys are EQUAL - the stable order takes those with the smallest indices, which
// an index-ordered block scan ranks.  Always leaves idx[0..nn) = the first nn entries of the full stable argsort.
// key needs >= max(2049 u32, CAP u64); idx >= CAP u16; misc[4..7], wt scratch.
__device__ __forceinline__ void block_select_sort_big(double *key, u16 *idx, u32 *wt, int *misc, const double *__restrict__ src,
                                                      int n, int nn, int CAP) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    u32 *hist = (u32 *)key; u64 *ckey = (u64 *)key;
    u64 prefix = 0;            // bits above `sh + bits` of the boundary key
    int below = 0, upto = 0, sh = 53, bits = 11;
    bool equal_tail = false;   // boundary bucket = keys exactly equal to `prefix` (all 64 bits fixed)
    for (int level = 0;; level++) {
        const u32 mask = (1u << bits) - 1u;
        __syncthreads();
        for (int b = tid; b <= 2048; b += T) hist[b] = 0;
        __syncthreads();
        for (int i = tid; i < n; i += T) {
            const u64 k = ordered_key(src[i]);
            if (level == 0 || (k >> (sh + bits)) == prefix) atomicAdd(&hist[(u32)(k >> sh) & mask], 1u);
        }
        __syncthreads();
        block_excl_scan(hist, 2049, wt);
        const int need = nn - below;
        for (int b = tid; b < 2048; b += T) if ((int)hist[b] < need && (int)hist[b + 1] >= need) { misc[4] = b; misc[5] = (int)hist[b]; misc[6] = (int)hist[b + 1]; }
        __syncthreads();
        const u32 bsel = (u32)misc[4];
        upto = below + misc[6]; below += misc[5];
        prefix = (prefix << bits) | bsel;
        if (upto <= CAP) break;
        if (sh == 0) { equal_tail = true; break; }
        if (sh >= 11) { sh -= 11; bits = 11; } else { bits = sh; sh = 0; }       // 53, 42, 31, 20, 9, then the last 9 bits
    }
    // prefix = the boundary key's bits from `sh` up; candidates: (k >> sh) < prefix, plus the boundary bucket itself
    // (all of it, or - equal keys - its nn - below smallest indices)
    __syncthreads();
    const int take = nn - below;       // entries wanted from the boundary bucket (equal_tail only)
    int rank_eq = 0;
    if (equal_tail) {
        u32 *cnt = hist;               // [T + 1] <= 2049: the histogram is dead
        const int per = (n + T - 1) / T;
        int c = 0;
        for (int e = 0; e < per; e++) { const int i = tid * per + e; if (i < n && ordered_key(src[i]) == prefix) c++; }
        cnt[tid] = (u32)c;
        if (tid == 0) cnt[T] = 0;
        __syncthreads();
        block_excl_scan(cnt, T + 1, wt);
        rank_eq = (int)cnt[tid];
        upto = below + take;
        __syncthreads();
    }
    if (tid == 0) misc[7] = 0;
    for (int p = upto + tid; p < CAP; p += T) { ckey[p] = ~0ull; idx[p] = (u16)0xffff; }
    __syncthreads();
    if (!equal_tail) {
        for (int base = 0; base < n; base += T) {
            const int i = base + tid;
            u64 k = 0; bool cand = false;
            if (i < n) { k = ordered_key(src[i]); cand = (k >> sh) <= prefix; }
            const u32 bal = __ballot_sync(FULLMASK, cand);
            int pb = 0;
            if (lane == 0 && bal) pb = atomicAdd(&misc[7], __popc(bal));
            pb = __shfl_sync(FULLMASK, pb, 0);
            if (cand) { const int pos = pb + __popc(bal & ((1u << lane) - 1)); ckey[pos] = k; idx[pos] = (u16)i; }
        }
    } else {
        const int per = (n + T - 1) / T;
        for (int e = 0; e < per; e++) {
            const int i = tid * per + e;
            if (i >= n) break;
            const u64 k = ordered_key(src[i]);
            bool cand = k < prefix;
            if (k == prefix) { cand = rank_eq < take; rank_eq++; }
            if (cand) { const int pos = atomicAdd(&misc[7], 1); ckey[pos] = k; idx[pos] = (u16)i; }
        }
    }
    __syncthreads();
    for (int k = 2; k <= CAP; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (CAP >> 1); t += T) {
                const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;
                const bool asc = ((lo & k) == 0);
                const u64 a = ckey[lo], b = ckey[hi];
                const u16 ia = idx[lo], ib = idx[hi];
                const bool gt = (b < a) || (b == a && ib < ia);
                if (gt == asc) { ckey[lo] = b; ckey[hi] = a; idx[lo] = ib; idx[hi] = ia; }
            }
            __syncthreads();
        }
    }
}

// ----------------------------------------------------------------------------------------------
// branch-path context (all pointers into shared memory)
// ----------------------------------------------------------------------------------------------
// Message slots: checks are ranked by row length (descending, rank q) and stored row after row in
// rank order, every row padded to an ODD number of slots (the pad is a permanently dead NaN slot).
// A warp that owns consecutive ranks runs loops of equal length L, and its 64-bit accesses
// base + lane*L + k are bank-conflict free because L is odd.
struct Ctx {
    int m, nn, es;
    int bad_rows;
    double factor;
    int low_error;
    int A, A_sum, C, D;                 // bpgd.hpp:15 thresholds (ints)
    double *msg;
    const double *prior;
    const u16 *voff, *vrow, *vpos, *cvn, *coff, *crank;
    const u16 *vperm, *cperm;
    const u8 *synd;
    i8 *vn_mask, *error, *cn_mask, *dec;
    u8 *cn_deg, *flip;
    u32 *upar;
    double *red_d; int *red_i; int *misc;
    int count_work;                     // accumulate the per-call work counters (edge / VN / CN / slot iterations)
    int zslot;                          // index (relative to msg) of a shared-memory double that always holds +0.0
};

// ownership: slot (tid, i) -> sorted index; odd rounds run backwards so that every warp gets a mix of
// heavy and light nodes (nodes are sorted by degree)
__device__ __forceinline__ int own_slot(int i, int tid, int T) { return (i & 1) ? i * T + (T - 1 - tid) : i * T + tid; }

// BPGD::vn_set_value (bpgd.cpp:51-80) executed by ONE warp; lane k handles the k-th check of vn.
template <bool HASMSG>
__device__ __forceinline__ int set_warp(Ctx &c, int vn, int val, int lane) {
    int cur = c.vn_mask[vn];
    if (cur >= 0) return (cur == val) ? 0 : -1;
    __syncwarp();
    if (lane == 0) { c.vn_mask[vn] = (i8)val; c.error[vn] = (i8)val; }
    const int e0 = c.voff[vn], d = c.voff[vn + 1] - e0;
    int fail = 0;
    if (lane < d) {
        const int r = c.vrow[e0 + lane];
        if (HASMSG) c.msg[c.vpos[e0 + lane]] = dnan();
        int cm = c.cn_mask[r], dg = c.cn_deg[r];
        if (cm < 0 || dg == 0) fail = 1;
        else {
            dg -= 1;
            if (val) cm ^= 1;
            c.cn_deg[r] = (u8)dg;
            if (dg == 0) { if (cm != 0) fail = 1; else cm = -1; }
            c.cn_mask[r] = (i8)cm;
        }
    }
    fail = __any_sync(FULLMASK, fail);
    __syncwarp();
    return fail ? -1 : 0;
}

// BPGD::peel (bpgd.cpp:13-49) executed by ONE warp in exactly the reference's sweep order:
// ballots find the next degree<=1 active check at or after the sweep position.
template <bool HASMSG>
__device__ __forceinline__ int peel_warp(Ctx &c, int lane) {
    for (;;) {
        bool clean = true;
        int cn = 0;
        while (cn < c.m) {
            int r = cn + lane;
            bool cand = false;
            if (r < c.m) cand = (c.cn_mask[r] >= 0) && (c.cn_deg[r] < 2);
            u32 b = __ballot_sync(FULLMASK, cand);
            if (!b) { cn += 32; continue; }
            r = cn + __ffs(b) - 1;
            if (c.cn_deg[r] == 0) {                 // bpgd.cpp:22-26
                if (!HASMSG) {
                    // reset-time peel (many emptied checks): retire every degree-0 candidate of this ballot window that comes
                    // before its first degree-1 candidate at once - they only get their mask cleared, in any order
                    const bool z = cand && (c.cn_deg[cn + lane] == 0);
                    const u32 zb = __ballot_sync(FULLMASK, z), ob = b & ~zb;
                    const u32 upto = ob ? ((1u << (__ffs(ob) - 1)) - 1u) : 0xffffffffu;
                    __syncwarp();
                    if (z && ((1u << lane) & upto)) c.cn_mask[cn + lane] = -1;
                    __syncwarp();
                    cn = ob ? cn + __ffs(ob) - 1 : cn + 32;
                    continue;
                }
                __syncwarp();
                if (lane == 0) c.cn_mask[r] = -1;
                __syncwarp();
                cn = r + 1; continue;
            }
            clean = false;
            const int q = c.crank[r], p0 = c.coff[q], len = c.coff[q + 1] - p0;
            int vn = -1;
            for (int kb = 0; kb < len && vn < 0; kb += 32) {
                int k = kb + lane, j = -1;
                bool und = false;
                if (k < len) { j = c.cvn[p0 + k]; und = (j != 0xffff) && (c.vn_mask[j] < 0); }
                u32 ub = __ballot_sync(FULLMASK, und);
                if (ub) vn = __shfl_sync(FULLMASK, j, __ffs(ub) - 1);
            }
            if (vn < 0) return -1;
            const int val = c.cn_mask[r];
            if (set_warp<HASMSG>(c, vn, val, lane) < 0) return -1;
            cn = r + 1;
        }
        if (clean) return 0;
    }
}

// BPGD::get_pm (bpgd.cpp:250-256): ordered fp64 sum over j ascending; every lane of the calling
// warp computes the same value.
__device__ __forceinline__ double pm_warp(const Ctx &c, int lane) {
    double pm = 0.0;
#pragma unroll 1
    for (int base = 0; base < c.nn; base += 32) {
        int j = base + lane;
        u32 b = __ballot_sync(FULLMASK, j < c.nn && c.error[j] != 0);
        while (b) { int k = __ffs(b) - 1; pm += c.prior[base + k]; b &= b - 1; }
    }
    return pm;
}

// BPGD::init (bpgd.cpp:82-95) + NaN marking of decided VNs.  Whole CTA; caller syncs.
template <int VPT>
__device__ __forceinline__ void init_msgs(Ctx &c) {
    const int T = blockDim.x, tid = threadIdx.x;
#pragma unroll 1
    for (int i = 0; i < VPT; i++) {
        const int sl = own_slot(i, tid, T);
        if (sl < c.nn) {
            const int j = c.vperm[sl];
            const int e0 = c.voff[j], e1 = c.voff[j + 1];
            const double v = (c.vn_mask[j] < 0) ? c.prior[j] : dnan();
#pragma unroll 1
            for (int e = e0; e < e1; e++) c.msg[c.vpos[e]] = v;
        }
    }
#pragma unroll 1
    for (int i = 0; i < SWD_CPT; i++) {
        const int q = own_slot(i, tid, T);
        if (q < c.m) { const int p1 = c.coff[q + 1]; if (p1 > c.coff[q] && c.cvn[p1 - 1] == 0xffff) c.msg[p1 - 1] = dnan(); }
    }
}

// sign-flip of a double by xor on the sign bit (mag * -f == -(mag * f) exactly in IEEE arithmetic)
__device__ __forceinline__ double flip_sign(double x, u32 flip) {
    return __hiloint2double(__double2hiint(x) ^ (int)(flip << 31), __double2loint(x));
}

// one message slot of the first check-update loop: running (min1, min2, argmin), sign and dead masks.
// Dead slots (decided VN, pad) hold a quiet NaN: every ordered compare is false for them, so they are neither clipped nor
// do they enter min1 / min2.  The masks are shifted in most-significant-first (one funnel shift each): after S slots,
// slot k sits at bit S - 1 - k.  neg: the sign bit (an exact +0.0, which also counts as "<= 0", bpgd.cpp:124, is caught by
// the caller: it makes min1 zero).  dead: exponent field all ones <=> (|hi| + 0x00100000) carries into bit 31.
#ifndef SWD_LATE_CLIP
#define SWD_LATE_CLIP 1
#endif
// CLIPPED = false: the +-50 clip of bpgd.cpp:119-121 is left to the caller - clipping is monotone, so the two smallest clipped
// magnitudes are the clipped two smallest magnitudes (check_update applies it to min1 / min2 once per row).
template <bool CLIPPED = true>
__device__ __forceinline__ void check_slot(const double b, const int k, double &m1, double &m2, int &arg, u32 &neg, u32 &dead) {
    const u32 hi = (u32)__double2hiint(b);
    const u32 ahi = hi & 0x7fffffffu;
    double a = __hiloint2double((int)ahi, __double2loint(b));
    if (CLIPPED) a = (a > SWD_CLIP) ? SWD_CLIP : a;              // bpgd.cpp:119-121
    const bool lt = a < m1;
    const double h = lt ? m1 : a;                                // max(m1, a); NaN stays NaN
    m2 = (h < m2) ? h : m2;
    m1 = lt ? a : m1;
    arg = lt ? k : arg;
    neg = __funnelshift_l(hi, neg, 1);
    dead = __funnelshift_l(ahi + 0x00100000u, dead, 1);
}

// rare: a message of the row is an exact zero - rebuild the sign mask with the reference's "<= 0" test
__device__ __noinline__ u32 check_neg_mask_exact(const double *row, int len) {
    u32 neg = 0;
#pragma unroll 1
    for (int k = 0; k < len; k++) neg = (neg << 1) | (u32)(row[k] <= 0.0);       // false for NaN
    return neg;
}

// rows longer than 32 slots (heavy checks of non-BB codes): out of line, so that the hot loop stays small
__device__ __noinline__ void check_update_long(double *row, int len, int cm, double fpos, double fneg) {
    double m1 = SWD_BIG, m2 = SWD_BIG; int arg = -1, par = cm;
#pragma unroll 1
    for (int k = 0; k < len; k++) {
        const double b = row[k];
        if (b != b) continue;
        double a = fabs(b); a = (a > SWD_CLIP) ? SWD_CLIP : a;
        if (a < m1) { m2 = m1; m1 = a; arg = k; } else if (a < m2) m2 = a;
        par ^= (b <= 0.0);
    }
#pragma unroll 1
    for (int k = 0; k < len; k++) {
        const double b = row[k];
        if (b != b) continue;
        const double mag = (k == arg) ? m2 : m1;
        row[k] = mag * ((par ^ (int)(b <= 0.0)) ? fneg : fpos);
    }
}

// one check update in min1/min2/argmin/parity form (== bpgd.cpp:103-148) on message slots p0 .. p0+len.
// Deliberately compact code (two slots per trip, no further unrolling): the min-sum iteration has to stay
// resident in the instruction caches (L0 ~6 KB, L1.5 32 KB) while 6 CTAs per SM run different phases.
__device__ __forceinline__ void check_update(Ctx &c, int p0, int len, int cm, double fpos, double fneg) {
    double *row = c.msg + p0;
    if (len > 32) { check_update_long(row, len, cm, fpos, fneg); return; }
    double m1 = SWD_BIG, m2 = SWD_BIG; int arg = -1;
    u32 neg = 0, dead = 0;
    // rows have an odd number of slots (pad): the first one alone, then two per trip
    check_slot<!SWD_LATE_CLIP>(row[0], 0, m1, m2, arg, neg, dead);
#pragma unroll 1
    for (int k = 1; k < len; k += 2) {
        const double b0 = row[k], b1 = row[k + 1];
        check_slot<!SWD_LATE_CLIP>(b0, k, m1, m2, arg, neg, dead);
        check_slot<!SWD_LATE_CLIP>(b1, k + 1, m1, m2, arg, neg, dead);
    }
    if (SWD_LATE_CLIP) {
        // fewer than two live magnitudes below the 1e308 sentinel (a check of degree 1, or magnitudes that overflowed): the exact
        // slot-by-slot path; else clip the two minima (min of clipped values = clipped min, for both order statistics)
        if (!(m2 < SWD_BIG)) { check_update_long(row, len, cm, fpos, fneg); return; }
        m1 = (m1 > SWD_CLIP) ? SWD_CLIP : m1; m2 = (m2 > SWD_CLIP) ? SWD_CLIP : m2;
    }
    if (m1 == 0.0) neg = check_neg_mask_exact(row, len);
    const u32 par = (u32)cm ^ (__popc(neg) & 1u);
    const double q1 = m1 * fpos, q2 = m2 * fpos;                 // c2b magnitude * alpha (sign applied below)
    // second sweep: every live slot gets +-q1 (sign = row parity ^ own sign), then the argmin slot is patched with +-q2.
    // Masks re-aligned so that slot k sits at bit 31 - k; the row parity is folded into the sign mask.
    const int sh = 32 - len;                                     // 1 <= len <= 31 (odd)
    u32 negA = (neg << sh) ^ (0u - par), deadA = dead << sh;
    const int q1lo = __double2loint(q1), q1hi = __double2hiint(q1);
    if (!(deadA & 0x80000000u)) row[0] = __hiloint2double(q1hi ^ (int)(negA & 0x80000000u), q1lo);
#pragma unroll 1
    for (int k = 1; k < len; k += 2) {
        if (!(deadA & 0x40000000u)) row[k] = __hiloint2double(q1hi ^ (int)((negA << 1) & 0x80000000u), q1lo);
        if (!(deadA & 0x20000000u)) row[k + 1] = __hiloint2double(q1hi ^ (int)((negA << 2) & 0x80000000u), q1lo);
        negA <<= 2; deadA <<= 2;
    }
    if (arg >= 0) row[arg] = flip_sign(q2, par ^ ((neg >> (len - 1 - arg)) & 1u));
}

// one variable-node update (bpgd.cpp:151-182) for a VN of degree d <= DM: returns the posterior, writes the hard
// decision, the parity contributions and the new bit-to-check messages
#ifndef SWD_VNZ
#define SWD_VNZ 0           /* measured -1.7 % (A/B r2): the select per edge costs more than the four predicated selects it removes */
#endif
template <int DM>
__device__ __forceinline__ double vn_update(Ctx &c, const int j, const int e0, const int d, const int dw) {
    double cc[DM], pre[DM]; int pp[DM];
    double t = c.prior[j];
#if SWD_VNZ
    // The loop bound dw is the warp's largest degree; a VN of smaller degree reads a constant +0.0 slot for its missing
    // edges: adding +0.0 changes no partial sum (bpgd.cpp:151-182 skips those edges), so the prefix sums need no
    // per-edge predicate / select - only the store keeps one.
    const int zslot = c.zslot;
#pragma unroll
    for (int k = 0; k < DM; k++) { if (k >= dw) break; const int p = c.vpos[e0 + k]; pp[k] = (k < d) ? p : zslot; cc[k] = c.msg[pp[k]]; }
#pragma unroll
    for (int k = 0; k < DM; k++) { if (k >= dw) break; pre[k] = t; t += cc[k]; }
#else
#pragma unroll
    for (int k = 0; k < DM; k++) { if (k >= dw) break; if (k < d) { pp[k] = c.vpos[e0 + k]; cc[k] = c.msg[pp[k]]; } }
#pragma unroll
    for (int k = 0; k < DM; k++) { if (k >= dw) break; if (k < d) { pre[k] = t; t += cc[k]; } }
#endif
    const int hard = (t <= 0.0);
    c.error[j] = (i8)hard;
    if (hard) {
#pragma unroll 1
        for (int k = 0; k < d; k++) atomicXor(&c.upar[c.vrow[e0 + k]], 1u);
    }
    double s = 0.0;
#pragma unroll
    for (int k = DM - 1; k >= 0; k--) if (k < dw) { if (k < d) { c.msg[pp[k]] = pre[k] + s; s += cc[k]; } }
    return t;
}

// The same update when every active lane of the warp holds a VN of degree K (VNs are owned in degree order): no per-edge
// predicates, selects or loop tests.  Same sums in the same order as vn_update.
#ifndef SWD_VN_UNIFORM
#define SWD_VN_UNIFORM 1
#endif
template <int K>
__device__ __forceinline__ double vn_uniform(Ctx &c, const int j, const int e0) {
    double cc[K], b[K]; int pp[K];
#pragma unroll
    for (int k = 0; k < K; k++) { pp[k] = c.vpos[e0 + k]; cc[k] = c.msg[pp[k]]; }
    double t = c.prior[j];
#pragma unroll
    for (int k = 0; k < K; k++) { b[k] = t; t += cc[k]; }
    const int hard = (t <= 0.0);
    c.error[j] = (i8)hard;
    if (hard) {
#pragma unroll 1
        for (int k = 0; k < K; k++) atomicXor(&c.upar[c.vrow[e0 + k]], 1u);
    }
    double s = 0.0;
#pragma unroll
    for (int k = K - 1; k >= 0; k--) { c.msg[pp[k]] = b[k] + s; s += cc[k]; }
    return t;
}

// BPGD::min_sum_log (bpgd.cpp:97-197) on the shortened graph, whole CTA.
// h[i][s]: posterior history of the VN owned as slot i, ring slot s = iteration % 4.
// Two barriers per iteration: the H*error == syndrome test of iteration `it` (bpgd.cpp:185-194;
// decided VNs are folded into cn_mask) is evaluated by the check threads at the start of the next
// check pass and reduced by the barrier that separates the check pass from the variable pass.
// On a converged return the messages may already hold the next check pass; they are never used then.
template <int VPT, int DMAX>
__device__ __forceinline__ int bp_run(Ctx &c, double (&h)[VPT][4], int num_iter, u64 &edge_iters, u32 &vn_iters, u32 &cn_iters,
                                      u64 &slot_iters, int *iters_done = nullptr) {
    const int T = blockDim.x, tid = threadIdx.x;
    const double fpos = c.factor, fneg = -c.factor;
    // ---- active checks of this call, compacted in rank order (cn_mask does not change inside a call; an
    //      inactive check has no undecided neighbour, so its parity / flip flags are never read).  The list
    //      aliases `dec`, which is only live inside select_vn.
    u16 *alist = (u16 *)c.dec;
    int na = 0;
#ifndef SWD_ALIST1
#define SWD_ALIST1 1
#endif
    if (SWD_ALIST1 && T == 128 && c.m <= 256) {
        // small windows: every warp takes the ballots of all <= 8 words of ranks itself, so the offsets need no exchange
        // through shared memory and the list is complete after ONE barrier (same order: rank-ascending)
        const int lane = tid & 31, wid = tid >> 5;
        u32 my0 = 0, my1 = 0; int off0 = 0, off1 = 0, run = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) {
            const int q = w * 32 + lane;
            const bool act = (q < c.m) && (c.cn_mask[c.cperm[q]] >= 0);
            const u32 b = __ballot_sync(FULLMASK, act);
            if (w == wid) { my0 = b; off0 = run; }
            if (w == 4 + wid) { my1 = b; off1 = run; }
            run += __popc(b);
        }
        const u32 below = (1u << lane) - 1u;
        if ((my0 >> lane) & 1u) alist[off0 + __popc(my0 & below)] = (u16)tid;
        if ((my1 >> lane) & 1u) alist[off1 + __popc(my1 & below)] = (u16)(128 + tid);
        na = run;
        __syncthreads();
    } else {
        const int lane = tid & 31, wid = tid >> 5, nw = (T + 31) >> 5;
        int *wcnt = (int *)c.red_d;                           // [SWD_CPT * nw] <= 128 ints = the 512 bytes of red_d
        u32 bal[SWD_CPT];
#pragma unroll
        for (int i = 0; i < SWD_CPT; i++) {
            const int q = i * T + tid;
            const bool act = (q < c.m) && (c.cn_mask[c.cperm[q]] >= 0);
            bal[i] = __ballot_sync(FULLMASK, act);
            if (lane == 0) wcnt[i * nw + wid] = __popc(bal[i]);
        }
        __syncthreads();
        int run = 0;
#pragma unroll
        for (int i = 0; i < SWD_CPT; i++) {
            int off = run;
#pragma unroll 1
            for (int w = 0; w < nw; w++) { const int cw = wcnt[i * nw + w]; if (w < wid) off += cw; run += cw; }
            if ((bal[i] >> lane) & 1u) alist[off + __popc(bal[i] & ((1u << lane) - 1u))] = (u16)(i * T + tid);
        }
        na = run;
        __syncthreads();
    }
#ifndef SWD_VN_JPACK
#define SWD_VN_JPACK 2      /* 2: (index, first edge, degree) records; 1: indices only; 0: ownership arithmetic per round */
#endif
    u32 jj01 = 0xffffffffu, jj23 = 0xffffffffu;
    u32 vr0 = 0, vr1 = 0, vr2 = 0, vr3 = 0;
    if (SWD_VN_JPACK == 2 && VPT == 4) {
        auto rec = [&](int i) -> u32 {
            const int sl = own_slot(i, tid, T);
            if (sl >= c.nn) return 0u;
            const int j = c.vperm[sl];
            if (c.vn_mask[j] >= 0) return 0u;
            const int e0 = c.voff[j], d = c.voff[j + 1] - e0;
            return (u32)j | ((u32)e0 << 12) | ((u32)d << 27);
        };
        vr0 = rec(0); vr1 = rec(1); vr2 = rec(2); vr3 = rec(3);
    } else
    if (SWD_VN_JPACK && VPT == 4) {
        const int s0 = own_slot(0, tid, T), s1 = own_slot(1, tid, T), s2 = own_slot(2, tid, T), s3 = own_slot(3, tid, T);
        const u32 j0 = s0 < c.nn ? c.vperm[s0] : 0xffffu, j1 = s1 < c.nn ? c.vperm[s1] : 0xffffu;
        const u32 j2 = s2 < c.nn ? c.vperm[s2] : 0xffffu, j3 = s3 < c.nn ? c.vperm[s3] : 0xffffu;
        jj01 = j0 | (j1 << 16); jj23 = j2 | (j3 << 16);
    }
    int it = 0, conv = 0;
#ifndef SWD_MISM_SMEM
#define SWD_MISM_SMEM 1
#endif
    // convergence flag of an iteration: a shared-memory word that any check thread with a mismatching row sets (cleared
    // during the previous variable pass) instead of an OR-reduction barrier over a per-thread accumulator
    // Two words, alternating by iteration parity: the word of iteration `it` is cleared by thread 0 after the barrier of
    // iteration it + 1 - behind every read of it (those precede the variable pass of `it`) and ahead of every set of it + 2.
    if (SWD_MISM_SMEM && tid == 0) { c.misc[5] = 0; c.misc[6] = 0; }     // published by the first barrier of the loop; the first set comes two barriers later
    for (;; it++) {
        // ---- check pass (+ convergence test of the previous iteration)
        int mism = 0;
        const bool last = (it == num_iter);
#pragma unroll 1
        for (int i = 0; i * T < na; i++) {
            const int k = own_slot(i, tid, T);
            if (k >= na) continue;
            const int q = alist[k];
            const int r = c.cperm[q];
            const int cm = c.cn_mask[r];
            if (it > 0) {
                const int f = (c.upar[r] != (u32)cm);
                c.flip[r] = (u8)f;
                if (SWD_MISM_SMEM) { if (f) c.misc[5 + (it & 1)] = 1; } else mism |= f;
            }
            c.upar[r] = 0;
            if (last) continue;
            { const int p0 = c.coff[q]; check_update(c, p0, c.coff[q + 1] - p0, cm, fpos, fneg); }
        }
        if (it > 0) {
            // a check that lost all its columns at reset while its syndrome bit is 1 (bad_rows) can never be satisfied
            if (SWD_MISM_SMEM) {
                __syncthreads();
                if (c.misc[5 + (it & 1)] == 0 && !c.bad_rows) { conv = 1; break; }
                if (tid == 0) c.misc[5 + ((it & 1) ^ 1)] = 0;
            } else if (!__syncthreads_or(mism) && !c.bad_rows) { conv = 1; break; }
        } else __syncthreads();
        if (last) break;
        // ---- variable pass: ordered prefix / suffix sums (bpgd.cpp:151-182); predicated straight-line code per slot.
        //      VNs are owned in degree order, so most warps only hold VNs of degree <= 3 and take the short body.
        const int ring = it & 3;
#pragma unroll 1
        for (int i = 0; i < VPT; i++) {      // rolled: one copy of the update bodies (instruction-cache footprint of the iteration)
            int j = -1, e0 = 0, d = 0;
            if (SWD_VN_JPACK == 2 && VPT == 4) {
                // the thread's four VNs as packed records (index | first edge << 12 | degree << 27; degree 0: decided or none), built
                // once per call - the masks do not change inside a call; the four registers rotate, the current one is vr0
                const u32 w = vr0; vr0 = vr1; vr1 = vr2; vr2 = vr3; vr3 = w;
                d = (int)(w >> 27);
                if (d) { j = (int)(w & 0xfffu); e0 = (int)((w >> 12) & 0x7fffu); }
            } else if (SWD_VN_JPACK && VPT == 4) {
                // the thread's four VNs, packed once per call: no ownership arithmetic / vperm load per round
                const u32 w = (i < 2) ? jj01 : jj23;
                j = (int)((w >> ((i & 1) << 4)) & 0xffffu);
                if (j != 0xffff && c.vn_mask[j] < 0) { e0 = c.voff[j]; d = c.voff[j + 1] - e0; } else j = -1;
            } else {
            const int sl = own_slot(i, tid, T);
            if (sl < c.nn) { j = c.vperm[sl]; if (c.vn_mask[j] < 0) { e0 = c.voff[j]; d = c.voff[j + 1] - e0; } else j = -1; }
            }
            const int dw = __reduce_max_sync(FULLMASK, d);
            const bool uni = SWD_VN_UNIFORM && dw <= 3 && __all_sync(FULLMASK, j < 0 || d == dw);
            if (j >= 0) {
                double t;
                if (uni) {
                    if (dw == 3) t = vn_uniform<3>(c, j, e0);
                    else if (dw == 2) t = vn_uniform<2>(c, j, e0);
                    else t = vn_uniform<1>(c, j, e0);
                } else
                t = vn_update<DMAX>(c, j, e0, d, dw);     // dw: warp-uniform loop bound (VNs are owned in degree order)
                h[i][ring] = t;      // dynamic ring index: the history lives in (L1/L2-backed) local memory, written once per
                                     // iteration and read once per call by select_vn - it does not occupy 32 registers
            }
        }
        __syncthreads();
    }
    // `it` variable passes were executed; check updates: one per variable pass, plus one more when the call converged
    // before the last iteration (the messages of that extra pass are never used)
    // work counters: the active sets do not change inside a call, so count them once (not per iteration) - and after the
    // loop, so that they do not occupy registers inside it
    u32 my_vn = 0, my_edges = 0, my_cn = 0;
    // (only while profiling is on, swd_set_profiling: the counting costs 1.7 % of the shots/s - A/B r2b)
    if (c.count_work)
#pragma unroll 1
    for (int i = 0; i < VPT; i++) {
        const int sl = own_slot(i, tid, T);
        if (sl < c.nn) { const int j = c.vperm[sl]; if (c.vn_mask[j] < 0) { my_vn++; my_edges += (u32)(c.voff[j + 1] - c.voff[j]); } }
    }
    u32 my_slots = 0;                                       // message slots (live + dead + pad) of the owned active rows
    if (c.count_work)
    for (int i = 0; i * T < na; i++) {
        const int k = own_slot(i, tid, T);
        if (k < na) { const int q = alist[k]; my_cn++; my_slots += (u32)(c.coff[q + 1] - c.coff[q]); }
    }
    if (c.count_work) {
    const u32 vp = (u32)it, cp = (u32)(conv ? (it < num_iter ? it + 1 : it) : it);
    edge_iters += (u64)my_edges * vp; vn_iters += my_vn * vp; cn_iters += my_cn * cp; slot_iters += (u64)my_slots * cp;
    }
    if (iters_done) *iters_done = conv ? it : (num_iter > 0 ? num_iter : 0);
    return conv;
}

// BPGD::select_vn (bpgd.cpp:288-351), whole CTA.  Returns favor (0/1) or -1; guess = -1 if no
// candidate.  The scan's aggressive decimations are classified in parallel (classification of a
// VN never depends on earlier decimations of the same scan) and applied per check; a contradiction
// is resolved to the first failing VN in scan order so that `error` matches the reference.
template <int VPT>
__device__ __forceinline__ int select_vn(Ctx &c, const double (&h)[VPT][4], int depth, int &guess) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    double best = SWD_MAX_PM, bestn = SWD_MAX_PM; int bi = 0x7fffffff, bni = 0x7fffffff;
    int any_dec = 0;
    if (tid == 0) c.misc[0] = 0x7fffffff;                    // failpos
#pragma unroll 1
    for (int i = 0; i < VPT; i++) {
        const int sl = own_slot(i, tid, T);
        if (sl < c.nn) {
            const int j = c.vperm[sl];
            int action = -1;
            if (c.vn_mask[j] < 0) {
                const int e0 = c.voff[j], d = c.voff[j + 1] - e0;
                if (d > 2) {
                    int nf = 0;
#pragma unroll 1
                    for (int k = 0; k < d; k++) nf += c.flip[c.vrow[e0 + k]];
                    bool geC = true, geD = true, leA = true, neg = true; double sum = 0.0;
#pragma unroll
                    for (int s = 0; s < 4; s++) {
                        const double l = h[i][s]; sum += l;
                        if (l < (double)c.C) geC = false;
                        if (l < (double)c.D) geD = false;
                        if (l > (double)c.A) leA = false;
                        if (l > 0.0) neg = false;
                    }
                    if (!c.low_error && geC && depth < 4) action = 0;
                    else if (!c.low_error && nf >= 3 && geD) action = 0;
                    else if (!c.low_error && leA && sum < (double)c.A_sum) action = 1;
                    else {
                        if (sum < best || (sum == best && j < bi)) { best = sum; bi = j; }      // sum < MAX_PM is implied
                        if (neg && (sum < bestn || (sum == bestn && j < bni))) { bestn = sum; bni = j; }
                    }
                }
            }
            c.dec[j] = (i8)action;
            any_dec |= (action >= 0);
        }
    }
    any_dec = __syncthreads_or(any_dec);
    if (any_dec) {
        // per check: how many of its undecided VNs were decimated and with which parity.  The decimated VNs (few) add
        // (1 | value << 8) to their checks' parity words - `upar` is zero for every active check between two min-sum
        // calls (the check pass clears it, bp_run) and is cleared again by the next call's first check pass - so no
        // thread scans whole rows here (and `cvn` is only touched on the contradiction path below).
#pragma unroll 1
        for (int i = 0; i < VPT; i++) {
            const int sl = own_slot(i, tid, T);
            if (sl < c.nn) {
                const int j = c.vperm[sl];
                const int a = c.dec[j];
                if (a >= 0) {
#pragma unroll 1
                    for (int e = c.voff[j]; e < c.voff[j + 1]; e++) atomicAdd(&c.upar[c.vrow[e]], 1u | ((u32)a << 8));
                }
            }
        }
        __syncthreads();
        int ndg[SWD_CPT], nmk[SWD_CPT];                      // SWD_CPT checks per thread (m <= SWD_CPT*T)
#pragma unroll
        for (int i = 0; i < SWD_CPT; i++) {
            const int q = own_slot(i, tid, T);
            ndg[i] = -1; nmk[i] = 0;
            if (q >= c.m) continue;
            const int r = c.cperm[q];
            const int cm = c.cn_mask[r];
            if (cm < 0) continue;
            const u32 w = c.upar[r];
            const int cnt = (int)(w & 0xffu), par = (int)((w >> 8) & 1u);        // row weight <= 255
            if (cnt) {
                const int nd = (int)c.cn_deg[r] - cnt, nm = cm ^ par;
                if (nd == 0 && nm != 0) {                    // contradiction (rare): last decimated VN of the row in scan order
                    int last = -1;
                    const int p0 = c.coff[q], p1 = c.coff[q + 1];
#pragma unroll 1
                    for (int p = p0; p < p1; p++) {
                        const int j = c.cvn[p];
                        if (j != 0xffff && c.dec[j] >= 0) last = max(last, j);
                    }
                    atomicMin(&c.misc[0], last);
                }
                ndg[i] = nd; nmk[i] = (nd == 0) ? -1 : nm;
            }
        }
        __syncthreads();
        const int failpos = c.misc[0];
        if (failpos != 0x7fffffff) {                         // contradiction: branch is dead
#pragma unroll 1
            for (int i = 0; i < VPT; i++) {
                const int sl = own_slot(i, tid, T);
                if (sl < c.nn) {
                    const int j = c.vperm[sl];
                    if (c.dec[j] >= 0 && j <= failpos) { c.vn_mask[j] = c.dec[j]; c.error[j] = c.dec[j]; }
                }
            }
            __syncthreads();
            guess = -1;
            return -1;
        }
#pragma unroll
        for (int i = 0; i < SWD_CPT; i++) {
            const int q = own_slot(i, tid, T);
            if (q < c.m && ndg[i] >= 0) { const int r = c.cperm[q]; c.cn_deg[r] = (u8)ndg[i]; c.cn_mask[r] = (i8)nmk[i]; }
        }
#pragma unroll 1
        for (int i = 0; i < VPT; i++) {
            const int sl = own_slot(i, tid, T);
            if (sl < c.nn) {
                const int j = c.vperm[sl];
                if (c.dec[j] >= 0) {
                    c.vn_mask[j] = c.dec[j]; c.error[j] = c.dec[j];
#pragma unroll 1
                    for (int e = c.voff[j]; e < c.voff[j + 1]; e++) c.msg[c.vpos[e]] = dnan();
                }
            }
        }
    }
    block_argmin(best, bi, c.red_d, c.red_i);                // contains the barriers that publish the updates
    block_argmin(bestn, bni, c.red_d, c.red_i);
    if (wid == 0) {
        int st = peel_warp<true>(c, lane);
        if (lane == 0) c.misc[1] = st;
    }
    __syncthreads();
    if (c.misc[1] < 0) { guess = -1; return -1; }
    if (bni != 0x7fffffff) { guess = bni; return 1; }
    guess = (bi == 0x7fffffff) ? -1 : bi;
    return (best > 0.0) ? 0 : 1;
}

// vn_set_value(guess, value) followed by peel (bpgd.cpp:485-486, :665), whole CTA. 0 ok / -1.
__device__ __forceinline__ int set_and_peel(Ctx &c, int vn, int val) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (wid == 0) {
        int st = set_warp<true>(c, vn, val, lane);
        if (st == 0) st = peel_warp<true>(c, lane);
        if (lane == 0) c.misc[1] = st;
    }
    __syncthreads();
    return c.misc[1];
}
