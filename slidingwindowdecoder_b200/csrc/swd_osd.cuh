// swd_osd.cuh — window OSD on the device (osd_window.pyx:201-284 + mod2sparse_extra.cpp:78-376).
//
// The reference runs a sparse LU with fill-in on linked lists, then k + w(w-1)/2 (CS) or 2^w (E)
// triangular re-solves.  Here one CTA per shot keeps the m x m row-transform T bit-packed in shared
// memory (64-bit words, column-major), scans the columns in LLR order, and for each new column c
// computes the reduced column v = T h_c as the XOR of <= 16 words-vectors, picks the first free row
// as pivot and applies the rank-1 update T += (v - e_i) (e_i^T T).  The syndrome rides along as an
// extra column, so OSD-0 is read off directly; every higher-order candidate is y0 ^ v_t1 ^ v_t2 ...
// and its path metric is an ordered fp64 sum (ascending column index, as the reference).
#pragma once
#include <stdlib.h>
#include "swd_kernels.cuh"

#define SWD_OSD_0  0
#define SWD_OSD_E  1
#define SWD_OSD_CS 2

struct OsdSmem {
    int np2, W64, k;
    int off_key, off_idx, off_tcol, off_vt, off_colinfo, off_ent, off_vbuf, off_piv, off_scan, off_wt, off_red, off_misc, off_ybest, off_pend, off_prow;
    int total;
    int big;                    // T does not fit next to the sort keys: key aliases tcol, vt / scan live in a per-CTA HBM scratch
    long long big_stride;       // bytes of that scratch per CTA
};

struct OsdWork {
    // outputs of the last batch (device), for the osd_window read-only properties
    u8 *bp_dec = nullptr, *osd0 = nullptr, *osdw = nullptr;
    double *lpr = nullptr;
    int *bp_iter = nullptr;
    long long out_cap = 0;
    // per-chunk scratch (inside the workspace block)
    u8 *need_osd = nullptr;         // [cap] 1 if slot must run OSD
    u8 *big_scratch = nullptr;      // [grid5][big_stride] (OsdSmem::big)
};

static inline size_t osd_bytes_per_shot(int m, int n) { return 2; }   // need_osd[cap] + in_list[cap]
static inline void osd_bind(OsdWork *ow, unsigned char *base, long long cap, int m, int n) { ow->need_osd = base; }

// ----------------------------------------------------------------------------------------------
// post-BP on the shortened graph (osd_window.pyx:187-192): one CTA per non-converged shot
// ----------------------------------------------------------------------------------------------
template <int VPT, int DMAX, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
post_bp_kernel(Workspace ws, SubLayout LG, SubLayout L, PathSmem S, GdgDev P, int n, OsdWork ow, long long chunk_base, int tier, int capA,
               const u8 *__restrict__ dec_in) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    unsigned char *blob = smem;
    unsigned char *st = smem + L.blob_bytes;
    Ctx c;
    c.m = L.m; c.nn = L.nn; c.factor = P.factor; c.low_error = 0; c.count_work = P.count_work;
    c.prior = (const double *)(blob + L.off_prior);
    c.voff = (const u16 *)(blob + L.off_voff); c.coff = (const u16 *)(blob + L.off_coff);
    c.crank = (const u16 *)(blob + L.off_crank);
    c.vrow = (const u16 *)(blob + L.off_vrow); c.vpos = (const u16 *)(blob + L.off_vpos); c.cvn = (const u16 *)(blob + L.off_cvn);
    c.vperm = (const u16 *)(blob + L.off_vperm); c.cperm = (const u16 *)(blob + L.off_cperm);
    c.synd = blob + L.off_synd;
    c.msg = (double *)(st + S.off_msg);
    c.vn_mask = (i8 *)(st + S.off_vnmask); c.error = (i8 *)(st + S.off_error); c.dec = (i8 *)(st + S.off_dec);
    c.cn_mask = (i8 *)(st + S.off_cnmask); c.cn_deg = st + S.off_cndeg; c.flip = st + S.off_flip;
    c.upar = (u32 *)(st + S.off_upar);
    c.red_d = (double *)(st + S.off_red); c.red_i = (int *)(c.red_d + 64); c.misc = (int *)(st + S.off_misc);
    c.zslot = (int)((double *)(st + S.off_misc + 48) - c.msg);      // misc[12..13]: the constant +0.0 of vn_update
    if (threadIdx.x == 0) *(double *)(st + S.off_misc + 48) = 0.0;
    u64 *bar = (u64 *)(st + S.off_bar);
#if !SWD_DIET
    const i8 *snap_vn = (const i8 *)(blob + L.off_vnmask), *snap_cn = (const i8 *)(blob + L.off_cnmask);
    const u8 *snap_deg = blob + L.off_cndeg;
#endif
    c.A = 0; c.A_sum = 0; c.C = 0; c.D = 0;
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    u32 mphase = 0;
    const int count = (tier == 1 && ws.counters[8] == 0) ? 0 : ws.counters[0];
    u64 edge_iters = 0, bp_calls = 0, paths_run = 0, slot_iters = 0; u32 vn_iters = 0, cn_iters = 0;
    for (;;) {
        __syncthreads();
        if (tid == 0) c.misc[2] = atomicAdd(&ws.counters[1 + 3 * tier], 1);
        __syncthreads();
        const int slot = c.misc[2];
        if (slot >= count) break;
        const unsigned char *gblob = ws.blob + (size_t)slot * LG.blob_bytes;
        const BlobHeader gh = *(const BlobHeader *)gblob;
        if ((gh.es > capA) != (tier == 1)) continue;
        if (tid == 0) ow.need_osd[slot] = 0;
        if (gh.status != 0) continue;
        if (tid == 0) {
            fence_proxy_async();
            const u32 vb = (u32)((gh.es * 2 + 15) & ~15);
            mbar_expect_tx(bar, (u32)L.fixed_bytes + (SWD_DIET ? 2 : 3) * vb);
            bulk_g2s(blob, gblob, (u32)L.fixed_bytes, bar);
            if (vb) {
                bulk_g2s(blob + L.off_vrow, gblob + LG.off_vrow, vb, bar);
                bulk_g2s(blob + L.off_vpos, gblob + LG.off_vpos, vb, bar);
#if !SWD_DIET
                bulk_g2s(blob + L.off_cvn, gblob + LG.off_cvn, vb, bar);
#endif
            }
        }
#if SWD_DIET
        c.cvn = (const u16 *)(gblob + LG.off_cvn);
        const i8 *snap_vn = (const i8 *)(gblob + LG.off_vnmask), *snap_cn = (const i8 *)(gblob + LG.off_cnmask);
        const u8 *snap_deg = gblob + LG.off_cndeg;
#endif
        mbar_wait(bar, mphase);
        mphase ^= 1;
        c.es = gh.es; c.bad_rows = gh.bad_rows;
        const u16 *col = (const u16 *)(gblob + LG.off_col);                 // only in the global blob (not staged)
        // undecided VNs start from the pre-BP hard decision (bp_decoding persists across the two BP stages,
        // osd_window.pyx:381-485; visible when post_max_iter = 0 or the first iteration converges nothing)
        for (int j = tid; j < c.nn; j += T) { const i8 v = snap_vn[j]; c.vn_mask[j] = v; c.error[j] = v < 0 ? (i8)dec_in[(size_t)gh.shot * n + col[j]] : v; }
        for (int r = tid; r < c.m; r += T) { c.cn_mask[r] = snap_cn[r]; c.cn_deg[r] = snap_deg[r]; c.flip[r] = 0; }
        __syncthreads();
        init_msgs<VPT>(c);                                                  // bp_init, osd_window.pyx:370-379
        // the history ring continues from the pre-BP (osd_window.pyx:458 re-uses log_prob_ratios)
        double h[VPT][4];
        const double *hg = ws.hist + (size_t)slot * n * 4;
#pragma unroll
        for (int i = 0; i < VPT; i++) {
            const int sl = own_slot(i, tid, T);
            const int j = (sl < c.nn) ? (int)c.vperm[sl] : -1;
#pragma unroll
            for (int s = 0; s < 4; s++) h[i][s] = (j >= 0) ? hg[(size_t)col[j] * 4 + s] : 0.0;
        }
        __syncthreads();
        paths_run++;
        int iters = 0;
        const int conv = bp_run<VPT, DMAX>(c, h, P.post_max_iter, edge_iters, vn_iters, cn_iters, slot_iters, &iters); bp_calls++;
        const long long shot = gh.shot;
        // outputs: bp_decoding, log_prob_ratios, bp_iteration; sort keys for OSD (osd_window.pyx:205-213)
        double *key = ws.sum + (size_t)slot * n;
        double *lpr = ow.lpr + ((size_t)(chunk_base + shot) * n) * 4;
        u8 *bpd = ow.bp_dec + (size_t)(chunk_base + shot) * n;
        for (int v = tid; v < n; v += T) bpd[v] = 0;                        // dropped columns were decimated to 0
        __syncthreads();
#pragma unroll
        for (int i = 0; i < VPT; i++) {
            const int sl = own_slot(i, tid, T);
            if (sl < c.nn) {
                const int j = c.vperm[sl];
                const int cj = col[j];
                const int vm = c.vn_mask[j];
                double k;
                if (vm == 1) k = -1000.0; else if (vm == 0) k = 1000.0;
                else {
                    k = ((h[i][0] + h[i][1]) + h[i][2]) + h[i][3];
#pragma unroll
                    for (int s = 0; s < 4; s++) lpr[(size_t)cj * 4 + s] = h[i][s];
                }
                key[cj] = k;
                bpd[cj] = (u8)(c.error[j] != 0);
            }
        }
        if (tid == 0) { ow.bp_iter[chunk_base + shot] += iters; ow.need_osd[slot] = conv ? 0 : 1; }
        record_result(c, ws.rec + (size_t)slot * P.n_rec * P.rec_stride, conv);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) edge_iters += __shfl_xor_sync(FULLMASK, edge_iters, o);
    if (lane == 0 && edge_iters) atomicAdd(&ws.stats[1], edge_iters);
    u64 vi = vn_iters, ci = cn_iters;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { vi += __shfl_xor_sync(FULLMASK, vi, o); ci += __shfl_xor_sync(FULLMASK, ci, o); }
    if (lane == 0) { if (vi) atomicAdd(&ws.stats[6], vi); if (ci) atomicAdd(&ws.stats[7], ci); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) slot_iters += __shfl_xor_sync(FULLMASK, slot_iters, o);
    if (lane == 0 && slot_iters) atomicAdd(&ws.stats[8], slot_iters);
    if (tid == 0) { if (paths_run) atomicAdd(&ws.stats[2], paths_run); if (bp_calls) atomicAdd(&ws.stats[3], bp_calls); }
}

// ----------------------------------------------------------------------------------------------
// OSD: one CTA per shot that needs it
// ----------------------------------------------------------------------------------------------
// SHOT = true: path metrics from the shot's row of g.llr_shot
template <bool SHOT = false>
__global__ void __launch_bounds__(1024, 1)
osd_kernel(GraphDev g, const u8 *__restrict__ synd, Workspace ws, SubLayout L, GdgDev P, OsdSmem S, OsdWork ow,
           int method, int order_w, int rank, u8 *__restrict__ dec_out, double *__restrict__ pm_out, long long chunk_base) {
    extern __shared__ __align__(16) unsigned char smem[];
    double *key = (double *)(smem + S.off_key);
    u16 *idx = (u16 *)(smem + S.off_idx);               // after the sort: scan order of the columns
    u64 *tcol = (u64 *)(smem + S.off_tcol);             // [(m+1)][W64]; column m carries T*syndrome
    u64 *vt = S.big ? (u64 *)(ow.big_scratch + (size_t)blockIdx.x * S.big_stride) : (u64 *)(smem + S.off_vt);   // [k][W64] reduced non-pivot columns
    u16 *colinfo = S.big ? (u16 *)(ow.big_scratch + (size_t)blockIdx.x * S.big_stride + (size_t)S.off_colinfo) : (u16 *)(smem + S.off_colinfo);   // per column: 0xffff none | pivot row | 0x8000 + T index
    u32 *ent = (u32 *)(smem + S.off_ent);               // [nn'] (col << 16 | info), ascending col
    u64 *pivmask = (u64 *)(smem + S.off_piv);           // [W64]
    u32 *scan = S.big ? (u32 *)(ow.big_scratch + (size_t)blockIdx.x * S.big_stride + (size_t)S.off_scan) : (u32 *)(smem + S.off_scan);   // [n+1]
    u32 *wt = (u32 *)(smem + S.off_wt);
    double *red_d = (double *)(smem + S.off_red); int *red_i = (int *)(red_d + 64);
    int *misc = (int *)(smem + S.off_misc);
    u64 *ybest = (u64 *)(smem + S.off_ybest);           // [W64]
    u64 *pend = (u64 *)(smem + S.off_pend);             // [32][W64] pending pivots in composed form
    int *prow = (int *)(smem + S.off_prow);             // [32] their pivot rows
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int m = g.m, n = g.n, nn = L.nn, W64 = S.W64, NP2 = S.np2, k = S.k;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const int count = ws.counters[0];
    u64 osd_shots = 0, osd_cols = 0, osd_piv = 0;

    for (;;) {
        __syncthreads();
        if (tid == 0) misc[2] = atomicAdd(&ws.counters[3], 1);
        __syncthreads();
        const int slot = misc[2];
        if (slot >= count) break;
        if (!ow.need_osd[slot]) continue;
        const int shot = ws.gdg_list[slot];
        osd_shots++;
        // ---- order the columns (osd_window.pyx:205-215)
        const bool regsort = (NP2 == 8 * T);                     // osd_setup sizes the CTA for this whenever it can
        if (!regsort) {
            for (int i = tid; i < NP2; i += T) {
                key[i] = (i < n) ? ws.sum[(size_t)slot * n + i] : inf;
                idx[i] = (i < n) ? (u16)i : (u16)0xffff;
            }
        }
        // big: the sort keys alias T, so T is set up after the sort
        for (int pass = 0; pass < 2; pass++) {
            if ((pass == 0) == (S.big == 0)) {
                if (S.big) __syncthreads();
                for (int i = tid; i < (m + 1) * W64; i += T) tcol[i] = 0;
                for (int i = tid; i < n; i += T) colinfo[i] = 0xffff;
                for (int i = tid; i < W64; i += T) pivmask[i] = 0;
                __syncthreads();
                for (int r = tid; r < m; r += T) {
                    tcol[r * W64 + (r >> 6)] = 1ull << (r & 63);
                    if (synd[(size_t)shot * m + r]) atomicOr(&tcol[m * W64 + (r >> 6)], 1ull << (r & 63));
                }
            }
            if (pass == 0) {
                if (S.big) __syncthreads();
                if (regsort) block_bitonic_sort_regs<8>(key, idx, NP2, ws.sum + (size_t)slot * n, n);
                else block_bitonic_sort(key, idx, NP2);
            }
        }
        if (tid == 0) { misc[0] = 0; }
        __syncthreads();
        // ---- greedy independent columns in scan order, Gauss-Jordan on T (mod2sparse_extra.cpp:113-376).
        // A column has to be reduced by all earlier pivots, but only a column that yields a pivot changes the state, and deep
        // in the scan (the last pivots of a full-rank window sit thousands of columns down the order) almost none does.
        // So the scan takes a block of one column per warp: every warp gathers its column against the last *applied* T and
        // resolves it against up to 32 *pending* pivots kept in composed form
        //   M = U_p ... U_1 = I + sum_j w_j e_{pr_j}^T,   appending U = I + a e_s^T:  w_j += a * w_j[s],  w_new = a,
        // (one gather of the bits x[pr_j], all tests on the original x).  The first column of the block with a free row
        // becomes the next pivot (its warp appends it), the columns before it are dependent and done, the columns after it
        // take the one new elementary step in registers and the block goes round again; a block without a free row costs one
        // barrier for all its columns.  The whole CTA folds the pending pivots into T every 32 pivots.  Pivots, their order
        // and the final T are exactly those of the column-at-a-time elimination (ncu r1h, C4: 76 % of the samples were the
        // other 18 warps waiting for the one scanning warp).
        int found = 0, pos = 0, pcount = 0, rnd = 0;
        const int nw = T >> 5;
        for (;;) {
            const int ci = pos + wid;
            bool valid = (ci < n);
            int cidx = 0; u64 x = 0;
            if (valid) {
                cidx = idx[ci];
                const int e0 = g.cp[cidx], d = g.cp[cidx + 1] - e0;
                if (lane < W64) for (int e = 0; e < d; e++) x ^= tcol[(int)g.cr[e0 + e] * W64 + lane];
                const int myprow = (lane < pcount) ? prow[lane] : 0;
                const u64 xw = __shfl_sync(FULLMASK, x, myprow >> 6);
                u32 hm = __ballot_sync(FULLMASK, (lane < pcount) && ((xw >> (myprow & 63)) & 1ull));
                while (hm) { const int jj = __ffs(hm) - 1; hm &= hm - 1; if (lane < W64) x ^= pend[jj * W64 + lane]; }
            }
            int cur = 0;
            bool stop = false;
            for (;;) {
                int *flags = red_i + 32 * (rnd & 1); rnd++;
                const u64 free_bits = (valid && lane < W64) ? (x & ~pivmask[lane]) : 0ull;
                const u32 bsel = __ballot_sync(FULLMASK, free_bits != 0);
                if (lane == 0) flags[wid] = bsel ? 1 : 0;
                __syncthreads();
                const u32 fm = __ballot_sync(FULLMASK, lane < nw && lane >= cur && flags[lane] != 0);
                if (!fm) break;                                  // the rest of the block depends on the pivots so far
                const int first = __ffs(fm) - 1;
                if (wid == first) {
                    const int fl = __ffs(bsel) - 1;
                    const u64 fb = __shfl_sync(FULLMASK, free_bits, fl);
                    const int pr = fl * 64 + (__ffsll((long long)fb) - 1);
                    u64 av = x; if (lane == fl) av &= ~(1ull << (pr & 63));
                    u32 tm = __ballot_sync(FULLMASK, (lane < pcount) && ((pend[lane * W64 + (pr >> 6)] >> (pr & 63)) & 1ull));
                    __syncwarp();
                    while (tm) { const int jj = __ffs(tm) - 1; tm &= tm - 1; if (lane < W64) pend[jj * W64 + lane] ^= av; }
                    if (lane < W64) pend[pcount * W64 + lane] = av;
                    if (lane == fl) pivmask[lane] |= 1ull << (pr & 63);
                    if (lane == 0) { colinfo[cidx] = (u16)pr; prow[pcount] = pr; }
                }
                if (wid <= first) valid = false;
                pcount++; found++;
                __syncthreads();
                if (valid) {                                     // later columns of the block: the one new elementary step
                    const int pr = prow[pcount - 1];
                    const u64 xw = __shfl_sync(FULLMASK, x, pr >> 6);
                    if (((xw >> (pr & 63)) & 1ull) && lane < W64) x ^= pend[(pcount - 1) * W64 + lane];
                }
                cur = first + 1;
                if (found >= rank) { stop = true; break; }
                if (pcount == 32) {
                    __syncthreads();
                    for (int r = tid; r <= m; r += T) {
                        u64 *tc = tcol + r * W64;
                        u32 hits = 0;
                        for (int jj = 0; jj < 32; jj++) { const int pr = prow[jj]; hits |= (u32)((tc[pr >> 6] >> (pr & 63)) & 1ull) << jj; }
                        while (hits) {
                            const int jj = __ffs(hits) - 1; hits &= hits - 1;
                            for (int w = 0; w < W64; w++) tc[w] ^= pend[jj * W64 + w];
                        }
                    }
                    pcount = 0;
                    __syncthreads();
                }
            }
            pos += nw;
            if (stop || pos >= n) break;
        }
        osd_cols += (u64)min(pos, n); osd_piv += (u64)found;
        __syncthreads();
        if (pcount > 0) {
            for (int r = tid; r <= m; r += T) {
                u64 *tc = tcol + r * W64;
                u32 hits = 0;
                for (int jj = 0; jj < pcount; jj++) { const int pr = prow[jj]; hits |= (u32)((tc[pr >> 6] >> (pr & 63)) & 1ull) << jj; }
                while (hits) {
                    const int jj = __ffs(hits) - 1; hits &= hits - 1;
                    for (int w = 0; w < W64; w++) tc[w] ^= pend[jj * W64 + w];
                }
            }
        }
        __syncthreads();
        // ---- the non-pivot columns that may be flipped: first k of order[0..nn) \ pivots (osd_window.pyx:243-258)
        if (wid == 0) {
            int cnt = 0;
            for (int base = 0; base < nn && cnt < k; base += 32) {
                const int pos = base + lane;
                int cidx = -1; bool np_ = false;
                if (pos < nn) { cidx = idx[pos]; np_ = (colinfo[cidx] == 0xffff); }
                const u32 b = __ballot_sync(FULLMASK, np_);
                const int my = cnt + __popc(b & ((1u << lane) - 1));
                if (np_ && my < k) colinfo[cidx] = (u16)(0x8000 | my);
                cnt += __popc(b);
            }
        }
        __syncthreads();
        // ---- entries (pivot or flippable column) in ascending column index
        for (int cI = tid; cI < n; cI += T) scan[cI] = (colinfo[cI] != 0xffff) ? 1u : 0u;
        if (tid == 0) scan[n] = 0;
        __syncthreads();
        block_excl_scan(scan, n + 1, wt);
        const int nent = (int)scan[n];
        for (int cI = tid; cI < n; cI += T) if (colinfo[cI] != 0xffff) ent[scan[cI]] = ((u32)cI << 16) | colinfo[cI];
        // reduced flippable columns vt[t] = T h_t
        for (int cI = tid; cI < n; cI += T) {
            const u16 ci = colinfo[cI];
            if (ci != 0xffff && (ci & 0x8000)) {
                const int t = ci & 0x7fff;
                for (int w = 0; w < W64; w++) {
                    u64 v = 0;
                    for (int e = g.cp[cI]; e < g.cp[cI + 1]; e++) v ^= tcol[(int)g.cr[e] * W64 + w];
                    vt[t * W64 + w] = v;
                }
            }
        }
        __syncthreads();
        const u64 *y0 = tcol + m * W64;
        // ---- candidates: id 0 = OSD-0; CS: singles 1..k, then pairs i<j<w; E: patterns 0..2^w-1 as id+... (see below)
        long long ncand;
        if (order_w <= 0 || method == SWD_OSD_0) ncand = 1;
        else if (method == SWD_OSD_CS) ncand = 1 + (long long)k + (long long)order_w * (order_w - 1) / 2;
        else ncand = 1 + (1ll << order_w);
        double best = inf; int besti = 0x7fffffff;
        double pm0 = 0.0;
        for (long long cand = tid; cand < ncand; cand += T) {
            // flipped T indices of this candidate
            int t1 = -1, t2 = -1; u32 emask = 0;
            if (cand > 0) {
                const long long l = cand - 1;
                if (method == SWD_OSD_CS) {
                    if (l < k) t1 = (int)l;
                    else {
                        long long q = l - k; int i = 0;
                        while (q >= order_w - 1 - i) { q -= order_w - 1 - i; i++; }
                        t1 = i; t2 = i + 1 + (int)q;
                    }
                } else emask = (u32)l;
            }
            double pm = 0.0;
            for (int q = 0; q < nent; q++) {
                const u32 en = ent[q];
                const int info = en & 0xffff, cI = en >> 16;
                bool on;
                if (info & 0x8000) {
                    const int t = info & 0x7fff;
                    on = (t == t1) || (t == t2) || (t < 32 && ((emask >> t) & 1u));
                } else {
                    const int w = info >> 6;
                    u64 y = y0[w];
                    if (t1 >= 0) y ^= vt[t1 * W64 + w];
                    if (t2 >= 0) y ^= vt[t2 * W64 + w];
                    if (emask) { u32 e2 = emask; while (e2) { const int t = __ffs(e2) - 1; e2 &= e2 - 1; y ^= vt[t * W64 + w]; } }
                    on = (y >> (info & 63)) & 1ull;
                }
                if (on) pm += SHOT ? g.llr_shot[(size_t)shot * n + cI] : g.llr[cI];
            }
            if (cand == 0) pm0 = pm;
            else if (pm < best) { best = pm; besti = (int)cand; }       // candidates visited in ascending id per thread
        }
        // OSD-0 path metric broadcast, then strict-min over higher-order candidates (first wins)
        if (tid == 0) red_d[63] = pm0;
        block_argmin(best, besti, red_d, red_i);
        pm0 = red_d[63];
        const bool use_w = (besti != 0x7fffffff) && (best < pm0);         // osd_window.pyx:276
        // ---- materialise osd0 and osdw
        int t1 = -1, t2 = -1; u32 emask = 0;
        if (use_w) {
            const long long l = (long long)besti - 1;
            if (method == SWD_OSD_CS) {
                if (l < k) t1 = (int)l;
                else { long long q = l - k; int i = 0; while (q >= order_w - 1 - i) { q -= order_w - 1 - i; i++; } t1 = i; t2 = i + 1 + (int)q; }
            } else emask = (u32)l;
        }
        if (tid < W64) {
            u64 y = y0[tid];
            if (t1 >= 0) y ^= vt[t1 * W64 + tid];
            if (t2 >= 0) y ^= vt[t2 * W64 + tid];
            u32 e2 = emask; while (e2) { const int t = __ffs(e2) - 1; e2 &= e2 - 1; y ^= vt[t * W64 + tid]; }
            ybest[tid] = y;
        }
        __syncthreads();
        const size_t row = (size_t)(shot) * n, orow = (size_t)(chunk_base + shot) * n;
        for (int cI = tid; cI < n; cI += T) {
            const u16 info = colinfo[cI];
            u8 b0 = 0, bw = 0;
            if (info != 0xffff) {
                if (info & 0x8000) { const int t = info & 0x7fff; bw = (u8)((t == t1) || (t == t2) || (t < 32 && ((emask >> t) & 1u))); }
                else { b0 = (u8)((y0[info >> 6] >> (info & 63)) & 1ull); bw = (u8)((ybest[info >> 6] >> (info & 63)) & 1ull); }
            }
            dec_out[row + cI] = bw;
            ow.osd0[orow + cI] = b0;
            ow.osdw[orow + cI] = bw;
        }
        if (tid == 0 && pm_out) pm_out[shot] = use_w ? best : pm0;
    }
    if (tid == 0 && osd_shots) { atomicAdd(&ws.stats[4], osd_shots); atomicAdd(&ws.stats[9], osd_cols); atomicAdd(&ws.stats[10], osd_piv); }
}

// ----------------------------------------------------------------------------------------------
// finish: scatter post-BP results of converged shots, converge flags (BP only, osd_window.pyx:189)
// ----------------------------------------------------------------------------------------------
__global__ void osd_finish_kernel(Workspace ws, SubLayout L, GdgDev P, OsdWork ow, int n, u8 *__restrict__ dec_out,
                                  u8 *__restrict__ conv_out, long long chunk_base, int no_osd) {
    const int T = blockDim.x, tid = threadIdx.x;
    const int count = ws.counters[0];
    for (int slot = blockIdx.x; slot < count; slot += gridDim.x) {
        const unsigned char *gblob = ws.blob + (size_t)slot * L.blob_bytes;
        const BlobHeader gh = *(const BlobHeader *)gblob;
        const u16 *col = (const u16 *)(gblob + L.off_col);
        // no_osd (osd_order = -1, "BP only", osd_window.pyx:192,199): a shot whose post-BP did not converge returns its
        // bp_decoding with converge = 0
        if (gh.status == 0 && (no_osd || !ow.need_osd[slot])) {
            const u8 *rec = ws.rec + (size_t)slot * P.n_rec * P.rec_stride;
            const u32 *bits = (const u32 *)(rec + sizeof(RecHeader));
            for (int j = tid; j < L.nn; j += T) dec_out[(size_t)gh.shot * n + col[j]] = (u8)((bits[j >> 5] >> (j & 31)) & 1u);
            if (tid == 0 && !ow.need_osd[slot]) conv_out[gh.shot] = 1;
        } else if (gh.status != 0) {
            // decimation / peeling contradiction: bp_decoding is what decode() returned (osd_window.pyx:179-186)
            for (int v = tid; v < n; v += T) ow.bp_dec[(size_t)(chunk_base + gh.shot) * n + v] = dec_out[(size_t)gh.shot * n + v];
        }
    }
}

// min_pm of BP-converged shots: ordered fp64 sum over ascending column (osd_window.pyx:168-170,190-191);
// also mirrors bp_decoding for shots that never left the BP stages.  One warp per shot.  SHOT = true: llr is [B][n], row b.
template <bool SHOT = false>
__global__ void osd_pm_kernel(const double *__restrict__ llr, int n, const u8 *__restrict__ dec, const u8 *__restrict__ conv,
                              long long B, double *__restrict__ pm_out, OsdWork ow, long long chunk_base, const u8 *__restrict__ in_list) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (long long b = (long long)blockIdx.x * wpb + (threadIdx.x >> 5); b < B; b += (long long)gridDim.x * wpb) {
        const u8 *row = dec + b * n;
        const bool cv = conv[b] != 0;
        double pm = 0.0;
        for (int base = 0; base < n; base += 32) {
            const int v = base + lane;
            const u8 bit = (v < n) ? row[v] : 0;
            if (!in_list[b] && v < n) ow.bp_dec[(size_t)(chunk_base + b) * n + v] = bit;
            u32 bm = __ballot_sync(FULLMASK, bit != 0);
            if (SHOT) { if (cv) while (bm) { const int kk = __ffs(bm) - 1; bm &= bm - 1; pm += llr[(size_t)b * n + base + kk]; } }
            else if (cv) while (bm) { const int kk = __ffs(bm) - 1; bm &= bm - 1; pm += llr[base + kk]; }
        }
        if (cv && lane == 0 && pm_out) pm_out[b] = pm;
    }
}

__global__ void osd_mark_list_kernel(const Workspace ws, u8 *in_list) {
    const int count = ws.counters[0];
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < count; s += gridDim.x * blockDim.x) in_list[ws.gdg_list[s]] = 1;
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
static inline int osd_r16(int x) { return (x + 15) & ~15; }

static inline int osd_setup(int m, int n, int nn, int rank, int method, int order_w, int num_sm, OsdSmem *S, int *T5, int *grid5) {
    int np2 = 64; while (np2 < n) np2 <<= 1;
    S->np2 = np2; S->W64 = (m + 1 + 63) / 64; if (S->W64 < (m + 63) / 64) S->W64 = (m + 63) / 64;
    S->W64 = (m + 63) / 64;
    S->k = nn - rank;
    int o = 0;
    S->off_key = o; o += 8 * np2;
    S->off_idx = o; o += 2 * np2; o = osd_r16(o);
    S->off_tcol = o; o += 8 * (m + 1) * S->W64; o = osd_r16(o);
    S->off_vt = o; o += 8 * (S->k > 0 ? S->k : 1) * S->W64; o = osd_r16(o);
    S->off_colinfo = o; o += 2 * n; o = osd_r16(o);
    S->off_ent = o; o += 4 * (nn + rank + 1); o = osd_r16(o);
    S->off_vbuf = o; o += 8 * S->W64; o = osd_r16(o);
    S->off_piv = o; o += 8 * S->W64; o = osd_r16(o);
    S->off_scan = o; o += 4 * (n + 1); o = osd_r16(o);
    S->off_wt = o; o += 4 * 64;
    S->off_red = o; o += 64 * 8 + 64 * 4; o = osd_r16(o);
    S->off_misc = o; o += 64;
    S->off_ybest = o; o += 8 * S->W64; o = osd_r16(o);
    S->off_pend = o; o += 8 * 32 * S->W64; o = osd_r16(o);
    S->off_prow = o; o += 4 * 32; o = osd_r16(o);
    S->total = o;
    S->big = 0; S->big_stride = 0;
    if (S->W64 > 32) return -2;                          // one word of a T column per lane of the scanning warp
    if (S->total > 227 * 1024 || getenv("SWD_FORCE_BIG_OSD")) {
        // large window: key[] (dead after the sort) aliases T, the reduced flippable columns and the scan array go to HBM
        S->big = 1;
        const int ta = 8 * (m + 1) * S->W64, ka = 8 * np2;
        o = 0;
        S->off_key = 0; S->off_tcol = 0; o = osd_r16(ta > ka ? ta : ka);
        S->off_idx = o; o += 2 * np2; o = osd_r16(o);
        S->off_ent = o; o += 4 * (nn + rank + 1); o = osd_r16(o);
        S->off_vbuf = o; o += 8 * S->W64; o = osd_r16(o);
        S->off_piv = o; o += 8 * S->W64; o = osd_r16(o);
        S->off_wt = o; o += 4 * 64;
        S->off_red = o; o += 64 * 8 + 64 * 4; o = osd_r16(o);
        S->off_misc = o; o += 64;
        S->off_ybest = o; o += 8 * S->W64; o = osd_r16(o);
        S->off_pend = o; o += 8 * 32 * S->W64; o = osd_r16(o);
        S->off_prow = o; o += 4 * 32; o = osd_r16(o);
        S->total = o;
        long long q = (long long)8 * (S->k > 0 ? S->k : 1) * S->W64; q = (q + 255) & ~255ll;
        S->off_vt = 0; S->off_scan = (int)q;               // offsets inside the per-CTA HBM scratch
        q += (long long)4 * (n + 1); q = (q + 255) & ~255ll;
        S->off_colinfo = (int)q; q += (long long)2 * n; q = (q + 255) & ~255ll;
        S->big_stride = q;
        if (S->total > 227 * 1024) return -2;
    }
    int t = ((m + 1 + 31) / 32) * 32; if (t < 128) t = 128; if (t > 1024) t = 1024;
    if (np2 / 8 >= t && np2 / 8 <= 1024) t = np2 / 8;     // 8 sort keys per thread in registers; more warps for the block scan
    *T5 = t;
    if (cudaFuncSetAttribute(osd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -3;
    if (cudaFuncSetAttribute(osd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -3;
    int occ = 0, occ_shot = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, osd_kernel<false>, t, S->total) != cudaSuccess || occ < 1) return -2;
    // the per-shot twin runs on the same grid (the CTAs draw shots from a ticket counter, any grid size is correct)
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_shot, osd_kernel<true>, t, S->total) != cudaSuccess || occ_shot < 1) return -2;
    *grid5 = num_sm * occ;
    return 0;
}

typedef void (*post_fn_t)(Workspace, SubLayout, SubLayout, PathSmem, GdgDev, int, OsdWork, long long, int, int, const u8 *);
static inline post_fn_t pick_post_kernel(int dmax, int T) {
    if (dmax == 6) {
        if (T <= 128) return post_bp_kernel<4, 6, 128, 5>;
#ifndef SWD_MINB320
#define SWD_MINB320 3      /* 64 registers, three CTAs per SM: C4 post-BP -4.5 % (A/B r2) */
#endif
        if (T <= 320) return post_bp_kernel<4, 6, 320, SWD_MINB320>;
        if (T <= 512) return post_bp_kernel<4, 6, 512, 1>;
        return post_bp_kernel<4, 6, 1024, 1>;
    }
    if (T <= 128) return post_bp_kernel<4, 16, 128, 3>;
    return post_bp_kernel<4, 16, 1024, 1>;
}

// everything after sort_reset for the osd_window kind
static inline int osd_launch(const GraphDev &g, const u8 *d_synd, const Workspace &ws, const SubLayout &L, const SubLayout &LsA,
                             const SubLayout &LsB, const PathSmem &PS, const PathSmem &PSB, int capA, int grid3B, size_t smem3B,
                             const GdgDev &P, const OsdSmem &OS, const OsdWork &ow, int dmax, int T3, int grid3, size_t smem3,
                             int T5, int grid5, int method, int order_w, int rank, u8 *d_corr, u8 *d_conv, double *d_pm,
                             long long B, long long chunk_base, cudaStream_t s, uint64_t *launches, u8 *in_list, int stage) {
    if (stage == 0) {        // post-BP on the shortened graph
        post_fn_t post = pick_post_kernel(dmax, T3);
        if (cudaFuncSetAttribute(post, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -3;
        post<<<grid3, T3, smem3, s>>>(ws, L, LsA, PS, P, g.n, ow, chunk_base, 0, capA, d_corr);
        *launches += 1;
        if (capA < L.es_max) { post<<<grid3B, T3, smem3B, s>>>(ws, L, LsB, PSB, P, g.n, ow, chunk_base, 1, capA, d_corr); *launches += 1; }
        return cudaGetLastError() == cudaSuccess ? 0 : -3;
    }
    if (order_w >= 0) {
        if (g.llr_shot) osd_kernel<true><<<grid5, T5, OS.total, s>>>(g, d_synd, ws, L, P, OS, ow, method, order_w, rank, d_corr, d_pm, chunk_base);
        else osd_kernel<false><<<grid5, T5, OS.total, s>>>(g, d_synd, ws, L, P, OS, ow, method, order_w, rank, d_corr, d_pm, chunk_base);
    }
    osd_finish_kernel<<<grid5, 128, 0, s>>>(ws, L, P, ow, g.n, d_corr, d_conv, chunk_base, order_w < 0 ? 1 : 0);
    cudaMemsetAsync(in_list, 0, (size_t)B, s);
    osd_mark_list_kernel<<<64, 256, 0, s>>>(ws, in_list);
    const unsigned gpm = (unsigned)((B + 7) / 8 < 1 ? 1 : ((B + 7) / 8 > 65535 ? 65535 : (B + 7) / 8));
    if (g.llr_shot) osd_pm_kernel<true><<<gpm, 256, 0, s>>>(g.llr_shot, g.n, d_corr, d_conv, B, d_pm, ow, chunk_base, in_list);
    else osd_pm_kernel<false><<<gpm, 256, 0, s>>>(g.llr, g.n, d_corr, d_conv, B, d_pm, ow, chunk_base, in_list);
    *launches += 4;
    return cudaGetLastError() == cudaSuccess ? 0 : -3;
}
