// swd_kernels.cuh — the kernels of the GDG / GD / post-BP pipeline.
//
//   pre_bp_kernel      full-window min-sum (bp_guessing_decoder.pyx:48-139), one CTA per shot,
//                      messages in shared memory, early exit, appends non-converged shots to the
//                      GDG list together with their posterior-history sums
//   sort_reset_kernel  index_sort (bpgd.cpp:384-389) + BPGD::reset (bpgd.cpp:199-239): builds the
//                      shortened graph of one shot ("blob") and its post-reset state
//   path_kernel        one CTA per (shot, branch path): main / tree(+backup) / side branches of
//                      BPGD_main_thread::do_work (bpgd.cpp:435-688), bpgd_decoder.gd (pyx:517-560)
//   select_kernel      min path-metric selection + scatter through `cols` (pyx:246-251)
#pragma once
#include "swd_device.cuh"

#define SWD_KIND_BPGDG       0
#define SWD_KIND_BPGD        1
#define SWD_KIND_OSD_WINDOW  2

// ----------------------------------------------------------------------------------------------
// K1: full-window BP
// ----------------------------------------------------------------------------------------------
struct PreSmem { int off_msg, off_upar, off_synd, off_dec, off_misc, total; int off_fwd; int off_vrec, off_cpos, off_prow; };
// off_fwd: product-sum forward products; off_vrec / off_cpos: staged copies of the static per-slot records and CSC->CSR map

#ifndef SWD_PRE_MINB
#define SWD_PRE_MINB 3
#endif
// one variable-node update of the full-window BP (bp_guessing_decoder.pyx:98-127): ordered prefix / suffix sums; the
// hard decision goes to s_dec[sl] (ownership-slot order), parity contributions to upar
template <int DM>
__device__ __forceinline__ double pre_vn_update(double *msg, u32 *upar, const u16 *cpj_sl, const int (&jb)[17], const u16 *__restrict__ cr,
                                                const double prior, const int e0, const int d, const int dw, u8 *dec_slot) {
    double cc[DM], pre[DM]; int pp[DM];
    double t = prior;
#pragma unroll
    for (int k = 0; k < DM; k++) { if (k >= dw) break; if (k < d) { pp[k] = cpj_sl[jb[k]]; cc[k] = msg[pp[k]]; } }
#pragma unroll
    for (int k = 0; k < DM; k++) { if (k >= dw) break; if (k < d) { pre[k] = t; t += cc[k]; } }
    const int hard = (t <= 0.0);
    *dec_slot = (u8)hard;
    if (hard) {
#pragma unroll 1
        for (int k = 0; k < d; k++) atomicXor(&upar[cr[e0 + k]], 1u);
    }
    double s = 0.0;
#pragma unroll
    for (int k = DM - 1; k >= 0; k--) if (k < dw) { if (k < d) { msg[pp[k]] = pre[k] + s; s += cc[k]; } }
    return t;
}

// The same update for a warp whose 32 columns all have degree K (the columns are owned in degree order, so that is nearly every
// warp): no per-edge predicates, selects or loop tests - load, K-term prefix chain, store.  Same sums in the same order.
template <int K>
__device__ __forceinline__ double pre_vn_uniform(double *msg, const u16 *cpj_sl, const int (&jb)[17], const double prior, double (&b2c)[K], int (&pp)[K]) {
    double cc[K];
#pragma unroll
    for (int k = 0; k < K; k++) { pp[k] = cpj_sl[jb[k]]; cc[k] = msg[pp[k]]; }
    double t = prior;
#pragma unroll
    for (int k = 0; k < K; k++) { b2c[k] = t; t += cc[k]; }
    double s = 0.0;
#pragma unroll
    for (int k = K - 1; k >= 0; k--) { b2c[k] = b2c[k] + s; s += cc[k]; }
    return t;
}
template <int K>
__device__ __forceinline__ double pre_vn_uniform_apply(double *msg, u32 *upar, const u16 *cpj_sl, const int (&jb)[17], const u16 *__restrict__ cr,
                                                       const double prior, const int e0, u8 *dec_slot) {
    double b2c[K]; int pp[K];
    const double t = pre_vn_uniform<K>(msg, cpj_sl, jb, prior, b2c, pp);
    const int hard = (t <= 0.0);
    *dec_slot = (u8)hard;
    if (hard) {
#pragma unroll 1
        for (int k = 0; k < K; k++) atomicXor(&upar[cr[e0 + k]], 1u);
    }
#pragma unroll
    for (int k = 0; k < K; k++) msg[pp[k]] = b2c[k];
    return t;
}

// MAXT = 256: several CTAs per SM (small windows).  MAXT = 1024: windows whose messages leave room for one CTA per
// SM only (e.g. 576 x 4896, 136 KB) get one large CTA instead of eight warps per SM.
// PS = true: product-sum check update (tanh products, forward / backward) instead of normalised min-sum.
// STAGED = true: the per-slot records (first edge, degree) and the CSC->CSR map live in shared memory (copied once per
// persistent CTA): the variable pass then chases vrec -> cpos -> msg through shared memory instead of
// vord -> cp -> cpos through L1 (ncu r1g: long_scoreboard was the second largest stall of this kernel).
// SHOT = true: per-shot priors (g.llr_shot, row `shot`).  Iteration 1 computes its check pass instead of reading the static
// table c2b1 (which was built to be bit-identical to that pass), and the shot's priors are gathered once into slot order
// in a fifth row of the CTA's hscratch (stride 5 n instead of 4 n): the variable pass reads them as coalesced as llr_s.
template <int DMAX, int MAXT, int MINB, bool PS, bool STAGED, bool SHOT = false>
__global__ void __launch_bounds__(MAXT, MINB)
pre_bp_kernel(GraphDev g, const u8 *__restrict__ synd, long long B, int max_iter, double alpha,
              u8 *__restrict__ dec_out, u8 *__restrict__ conv_out, Workspace ws, double *hscratch,
              int full_hist, PreSmem S, int *iter_out, double *lpr_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    double *msg = pinned_smem<double>(smem + S.off_msg);
    u32 *upar = pinned_smem<u32>(smem + S.off_upar);
    u8 *s_synd = pinned_smem<u8>(smem + S.off_synd);
    u8 *s_dec = pinned_smem<u8>(smem + S.off_dec);                 // hard decisions in ownership-slot order
    int *misc = (int *)(smem + S.off_misc);
    const int T = blockDim.x, tid = threadIdx.x;
    const int m = g.m, n = g.n;
    double *hs = hscratch + (size_t)blockIdx.x * (SHOT ? 5 : 4) * n;   // last four posteriors, ownership-slot order (coalesced)
    double *hl = hs + (size_t)4 * n;                               // SHOT: the shot's priors in ownership-slot order
    const double fpos = alpha;
    u64 edge_iters = 0;
    const u32 *vrec = g.vrec; const u16 *cpj = g.cpj; const u32 *prow = g.prow;
    if (STAGED) {
        u32 *sv = pinned_smem<u32>(smem + S.off_vrec); u16 *sc = pinned_smem<u16>(smem + S.off_cpos);
        u32 *sr = pinned_smem<u32>(smem + S.off_prow);
        for (int i = tid; i < n; i += T) sv[i] = g.vrec[i];
        for (int i = tid; i < g.nnz; i += T) sc[i] = g.cpj[i];
        for (int i = tid; i < m; i += T) sr[i] = g.prow[i];
        vrec = sv; cpj = sc; prow = sr;
        __syncthreads();
    }

    for (long long shot = blockIdx.x; shot < B; shot += gridDim.x) {
        for (int r = tid; r < m; r += T) s_synd[r] = synd[shot * m + r];
        const bool table1 = !PS && !SHOT && g.c2b1 != nullptr;        // iteration 1's check pass comes from the static table
        if (table1) {
            __syncthreads();
            for (int r = tid; r < m; r += T) upar[r] = 0;
#pragma unroll 4
            for (int p = tid; p < g.nphys; p += T) msg[p] = flip_sign(g.c2b1[p], (u32)s_synd[g.rowof[p]]);
            for (int sl = tid; sl < n; sl += T) s_dec[sl] = 0;
        } else
        for (int sl = tid; sl < n; sl += T) {                  // pyx:55-60
            const u32 vr = vrec[sl];
            const int d = (int)(vr >> 16);
            double l;
            if (SHOT) { l = g.llr_shot[(size_t)shot * n + g.vord[sl]]; hl[sl] = l; }      // read back by this thread only
            else l = g.llr_s[sl];
#pragma unroll 1
            for (int k = 0; k < d; k++) msg[cpj[g.jb[k] + sl]] = l;
            s_dec[sl] = 0;
        }
        __syncthreads();
        int conv = 0, it = 0;
        for (; it < max_iter; it++) {
            // ---- check pass: min1/min2/argmin/parity with plain compares, sign applied by xor (all edges live)
            if (it == 0 && table1) {
            } else if (PS) {
                // product-sum (restated from the published ldpc BpOsdDecoder algorithm, parity unpinned): forward products
                // in `fwd`, backward sweep writes c2b = s * log((1 + P) / (1 - P)), P saturated to +-(1 - 2^-52)
                double *fwd = (double *)(smem + S.off_fwd);
                const double PMAX = 1.0 - 2.220446049250313e-16;
                for (int r = tid; r < m; r += T) {
                    upar[r] = 0;
                    const u32 pr = prow[r];
                    const int p0 = (int)(pr & 0xffffu), p1 = p0 + (int)(pr >> 16);
                    double tmp = 1.0;
                    for (int p = p0; p < p1; p++) { fwd[p] = tmp; tmp *= tanh(msg[p] * 0.5); }
                    tmp = 1.0;
                    const double sg = s_synd[r] ? -1.0 : 1.0;
                    for (int p = p1 - 1; p >= p0; p--) {
                        const double b = msg[p];
                        double P = fwd[p] * tmp;
                        P = (P > PMAX) ? PMAX : ((P < -PMAX) ? -PMAX : P);
                        msg[p] = sg * log((1.0 + P) / (1.0 - P));
                        tmp *= tanh(b * 0.5);
                    }
                }
            } else
            for (int r = tid; r < m; r += T) {
                upar[r] = 0;
                const u32 pr = prow[r];
                const int p0 = (int)(pr & 0xffffu), p1 = p0 + (int)(pr >> 16);
                double m1 = SWD_BIG, m2 = SWD_BIG; int arg = -1; u32 par = s_synd[r];
                // the +-50 clip (pyx:74-76) is monotone: the two smallest clipped magnitudes are the clipped two smallest
                // magnitudes, so it is applied to min1 / min2 once per row ...
#pragma unroll 4
                for (int p = p0; p < p1; p++) {
                    const double b = msg[p];
                    const double a = fabs(b);
                    const bool lt = a < m1;
                    const double hi = lt ? m1 : a;
                    m2 = (hi < m2) ? hi : m2;
                    m1 = lt ? a : m1;
                    arg = lt ? p : arg;
                    par ^= (u32)(b <= 0.0);
                }
                if (m2 < SWD_BIG) { m1 = (m1 > SWD_CLIP) ? SWD_CLIP : m1; m2 = (m2 > SWD_CLIP) ? SWD_CLIP : m2; }
                else {
                    // ... unless fewer than two magnitudes lie below the 1e308 sentinel (a row of weight 1, or sums that
                    // overflowed): slot-by-slot clip as the reference writes it
                    m1 = SWD_BIG; m2 = SWD_BIG; arg = -1;
                    for (int p = p0; p < p1; p++) {
                        double a = fabs(msg[p]);
                        a = (a > SWD_CLIP) ? SWD_CLIP : a;
                        const bool lt = a < m1;
                        const double hi = lt ? m1 : a;
                        m2 = (hi < m2) ? hi : m2;
                        m1 = lt ? a : m1;
                        arg = lt ? p : arg;
                    }
                }
                const double q1 = m1 * fpos, q2 = m2 * fpos;
#ifndef SWD_PRE_SWEEP2
#define SWD_PRE_SWEEP2 1
#endif
                if (SWD_PRE_SWEEP2 && m1 != 0.0) {
                    // no message of the row is an exact zero, so "b <= 0" is the sign bit: every slot gets +-q1 (only the sign bit of
                    // the old message is used), then the argmin slot is patched with +-q2 of the sign just written
                    const int q1lo = __double2loint(q1), q1hi = __double2hiint(q1) ^ (int)(par << 31);
#pragma unroll 8
                    for (int p = p0; p < p1; p++) msg[p] = __hiloint2double(q1hi ^ (__double2hiint(msg[p]) & (int)0x80000000), q1lo);
                    if (arg >= 0) {
                        const int x = (__double2hiint(msg[arg]) ^ __double2hiint(q1)) & (int)0x80000000;
                        msg[arg] = __hiloint2double(__double2hiint(q2) ^ x, __double2loint(q2));
                    }
                } else
                for (int p = p0; p < p1; p++) {
                    const double b = msg[p];
                    msg[p] = flip_sign((p == arg) ? q2 : q1, par ^ (u32)(b <= 0.0));
                }
            }
            __syncthreads();
            const bool keep = full_hist || (it >= max_iter - 4);
            double *hs_it = hs + (size_t)(it & 3) * n;
            // ---- variable pass: columns are owned in degree order, so a warp's loop bound is uniform
            for (int base = 0; base < n; base += T) {
                const int sl = base + tid;
                int e0 = 0, d = 0;
                if (sl < n) { const u32 vr = vrec[sl]; e0 = (int)(vr & 0xffffu); d = (int)(vr >> 16); }
                const int dw = __reduce_max_sync(FULLMASK, d);
#ifndef SWD_PRE_UNIFORM
#define SWD_PRE_UNIFORM 1
#endif
                const bool uni = SWD_PRE_UNIFORM && dw >= 1 && dw <= 6 && __all_sync(FULLMASK, d == dw);     // implies sl < n in every lane
                if (uni) {
                    double t;
                    const double pr = SHOT ? hl[sl] : g.llr_s[sl];
                    switch (dw) {
                        case 1: t = pre_vn_uniform_apply<1>(msg, upar, cpj + sl, g.jb, g.cr, pr, e0, s_dec + sl); break;
                        case 2: t = pre_vn_uniform_apply<2>(msg, upar, cpj + sl, g.jb, g.cr, pr, e0, s_dec + sl); break;
                        case 3: t = pre_vn_uniform_apply<3>(msg, upar, cpj + sl, g.jb, g.cr, pr, e0, s_dec + sl); break;
                        case 4: t = pre_vn_uniform_apply<4>(msg, upar, cpj + sl, g.jb, g.cr, pr, e0, s_dec + sl); break;
                        case 5: t = pre_vn_uniform_apply<5>(msg, upar, cpj + sl, g.jb, g.cr, pr, e0, s_dec + sl); break;
                        default: t = pre_vn_uniform_apply<6>(msg, upar, cpj + sl, g.jb, g.cr, pr, e0, s_dec + sl); break;
                    }
                    if (keep) hs_it[sl] = t;
                } else
                if (sl < n) {
                    const double t = pre_vn_update<DMAX>(msg, upar, cpj + sl, g.jb, g.cr, SHOT ? hl[sl] : g.llr_s[sl], e0, d, dw, s_dec + sl);
                    if (keep) hs_it[sl] = t;
                }
            }
            edge_iters += 1;
            __syncthreads();
            int mism = 0;
            for (int r = tid; r < m; r += T) mism |= (upar[r] != (u32)s_synd[r]);
            if (!__syncthreads_or(mism)) { conv = 1; it++; break; }
        }
        for (int sl = tid; sl < n; sl += T) dec_out[shot * n + g.vord[sl]] = s_dec[sl];
        if (tid == 0) {
            conv_out[shot] = (u8)conv;
            if (iter_out) iter_out[shot] = it;
            if (!conv) { int slot = atomicAdd(&ws.counters[0], 1); ws.gdg_list[slot] = (int)shot; misc[0] = slot; }
        }
        __syncthreads();
        if (!conv || lpr_out) {
            const int slot = misc[0];
            for (int sl = tid; sl < n; sl += T) {
                const int v = g.vord[sl];
                double h4[4];
#pragma unroll
                for (int s = 0; s < 4; s++) {
                    // slots never written in this call are 0 (fresh ring); `it` iterations were executed
                    // (with full_hist all of them were stored, otherwise only the last four of max_iter).
                    const bool written = (s < it);
                    h4[s] = written ? hs[(size_t)s * n + sl] : 0.0;
                }
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
        __syncthreads();
    }
    if (tid == 0 && edge_iters) atomicAdd(&ws.stats[0], edge_iters * (u64)g.nnz);
}

// ----------------------------------------------------------------------------------------------
// K2: sort + reset
// ----------------------------------------------------------------------------------------------
struct SortSmem { int off_key, off_idx, off_posof, off_blob, off_u32a, off_u32b, off_u32c, off_wt, off_error, off_misc, off_bins, total; int np2;
                  int cap_sel;        // > 0: select + sort the cap_sel smallest keys instead of sorting all n
                  int big;            // n beyond the register sort: block_select_sort_big only (key / idx hold cap_sel entries)
                  int key_bytes; };

// SHOT = true: the kept columns' priors come from the shot's row of g.llr_shot
template <bool SHOT = false>
__global__ void __launch_bounds__(1024, 1)
sort_reset_kernel(GraphDev g, const u8 *__restrict__ synd, Workspace ws, SubLayout L, GdgDev P, SortSmem S,
                  u8 *__restrict__ dec_out, int capA) {
    extern __shared__ __align__(16) unsigned char smem[];
    double *key = (double *)(smem + S.off_key);
    u16 *idx = (u16 *)(smem + S.off_idx);
    u16 *posof = (u16 *)(smem + S.off_posof);
    unsigned char *blob = smem + S.off_blob;
    u32 *ua = (u32 *)(smem + S.off_u32a);         // [nn+1]
    u32 *ub = (u32 *)(smem + S.off_u32b);         // [m+1]
    u32 *uc = (u32 *)(smem + S.off_u32c);         // [m+1]
    u32 *wt = (u32 *)(smem + S.off_wt);
    i8 *s_error = (i8 *)(smem + S.off_error);
    int *misc = (int *)(smem + S.off_misc);
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int m = g.m, n = g.n, nn = L.nn, NP2 = S.np2;

    BlobHeader *hdr = (BlobHeader *)blob;
    double *prior = (double *)(blob + L.off_prior);
    u16 *col = (u16 *)(blob + L.off_col);
    u16 *voff = (u16 *)(blob + L.off_voff);
    u16 *coff = (u16 *)(blob + L.off_coff);
    u16 *crank = (u16 *)(blob + L.off_crank);
    u8 *s_synd = blob + L.off_synd;
    i8 *vn_mask = (i8 *)(blob + L.off_vnmask);
    i8 *cn_mask = (i8 *)(blob + L.off_cnmask);
    u8 *cn_deg = blob + L.off_cndeg;
    u16 *vrow = (u16 *)(blob + L.off_vrow);
    u16 *vpos = (u16 *)(blob + L.off_vpos);
    u16 *cvn = (u16 *)(blob + L.off_cvn);
    u16 *vperm = (u16 *)(blob + L.off_vperm);
    u16 *cperm = (u16 *)(blob + L.off_cperm);
    u32 *bins = (u32 *)(smem + S.off_bins);       // [17 + 256]

    const int count = ws.counters[0];
    for (int slot = blockIdx.x; slot < count; slot += gridDim.x) {
        const int shot = ws.gdg_list[slot];
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        bool partial = false;                                       // only idx[0..nn) is ordered, posof = 0xffff for the rest
        if (S.big) { block_select_sort_big(key, idx, wt, misc, ws.sum + (size_t)slot * n, n, nn, S.cap_sel); partial = true; }
        else if (S.cap_sel > 0 && NP2 == 8 * T)
            partial = block_select_sort<8>(key, idx, wt, misc, ws.sum + (size_t)slot * n, n, nn, S.cap_sel);
        if (partial) {
            for (int cI = tid; cI < n; cI += T) posof[cI] = (u16)0xffff;
            __syncthreads();
        } else if (NP2 == 8 * T) {
            block_bitonic_sort_regs<8>(key, idx, NP2, ws.sum + (size_t)slot * n, n);      // 8 keys per thread in registers
        } else {
            for (int i = tid; i < NP2; i += T) {
                key[i] = (i < n) ? ws.sum[(size_t)slot * n + i] : inf;
                idx[i] = (i < n) ? (u16)i : (u16)0xffff;
            }
            __syncthreads();
            block_bitonic_sort(key, idx, NP2);
        }
        for (int j = tid; j < (partial ? nn : n); j += T) posof[idx[j]] = (u16)j;
        for (int j = tid; j < nn; j += T) {
            const int c = idx[j];
            col[j] = (u16)c; prior[j] = SHOT ? g.llr_shot[(size_t)shot * n + c] : g.llr[c];
            ua[j] = (u32)(g.cp[c + 1] - g.cp[c]);
            vn_mask[j] = -1; s_error[j] = 0;
        }
        if (tid == 0) ua[nn] = 0;
        __syncthreads();
        block_excl_scan(ua, nn + 1, wt);
        const int es = (int)ua[nn];
        for (int j = tid; j <= nn; j += T) voff[j] = (u16)ua[j];
        for (int j = tid; j < nn; j += T) {
            const int c = col[j], e0 = g.cp[c], d = g.cp[c + 1] - e0, o = (int)ua[j];
            for (int k = 0; k < d; k++) vrow[o + k] = g.cr[e0 + k];
        }
        for (int r = tid; r < m; r += T) {
            int cnt = 0;
            for (int q = g.rp[r]; q < g.rp[r + 1]; q++) cnt += (posof[g.rc[q]] < nn);
            ub[r] = (u32)cnt;
        }
        __syncthreads();
        // kept-row lengths are in ub[0..m): rank the checks by length (descending); message slots are laid out
        // row after row in rank order, each row padded to an odd number of slots (bank-conflict-free warps)
        for (int i = tid; i < 17 + 256; i += T) bins[i] = 0;
        __syncthreads();
        for (int j = tid; j < nn; j += T) atomicAdd(&bins[16 - (int)(ua[j + 1] - ua[j])], 1u);
        for (int r = tid; r < m; r += T) atomicAdd(&bins[17 + 255 - (int)ub[r]], 1u);
        __syncthreads();
        if (tid == 0) { u32 a = 0; for (int i = 0; i < 17; i++) { u32 t = bins[i]; bins[i] = a; a += t; } }
        if (tid == 32) { u32 a = 0; for (int i = 17; i < 17 + 256; i++) { u32 t = bins[i]; bins[i] = a; a += t; } }
        __syncthreads();
        for (int j = tid; j < nn; j += T) vperm[atomicAdd(&bins[16 - (int)(ua[j + 1] - ua[j])], 1u)] = (u16)j;
        int bad = 0;
        for (int r = tid; r < m; r += T) {
            const int d = (int)ub[r];
            const int q = (int)atomicAdd(&bins[17 + 255 - d], 1u);
            cperm[q] = (u16)r; crank[r] = (u16)q;
            const int s = synd[(size_t)shot * m + r];
            s_synd[r] = (u8)s;
            cn_deg[r] = (u8)d;
            cn_mask[r] = (d == 0) ? (i8)-1 : (i8)s;          // bpgd.cpp:210-217
            bad |= (d == 0 && s);
        }
        if (tid == 0) misc[0] = 0x7fffffff;
        bad = __syncthreads_or(bad);
        for (int q = tid; q < m; q += T) { const u32 d = ub[cperm[q]]; uc[q] = (d > 0 && !(d & 1u)) ? d + 1 : d; }
        if (tid == 0) uc[m] = 0;
        __syncthreads();
        block_excl_scan(uc, m + 1, wt);
        const int nslots = (int)uc[m];
        for (int q = tid; q <= m; q += T) coff[q] = (u16)uc[q];
        // message slot of every kept edge: the row pass notes the slot under the edge's CSR position (in the `key` area,
        // dead after the sort), the column pass picks it up through the static CSC -> CSR map
        u16 *slot_of = (u16 *)key;
        const bool via_table = (2 * g.nnz <= S.key_bytes);
        for (int r = tid; r < m; r += T) {
            const int q = crank[r];
            int p = (int)uc[q];
            for (int qq = g.rp[r]; qq < g.rp[r + 1]; qq++) {
                const int j = posof[g.rc[qq]];
                if (j < nn) {
                    cvn[p] = (u16)j;
                    if (via_table) slot_of[qq] = (u16)p;
                    else for (int e = voff[j]; e < voff[j + 1]; e++) if (vrow[e] == r) vpos[e] = (u16)p;
                    p++;
                }
            }
            if (p < (int)uc[q + 1]) cvn[p] = (u16)0xffff;      // pad slot
        }
        __syncthreads();
        if (via_table) {
            for (int j = tid; j < nn; j += T) {
                const int cI = col[j], e0 = g.cp[cI], d = g.cp[cI + 1] - e0, o = (int)voff[j];
                for (int k = 0; k < d; k++) vpos[o + k] = slot_of[g.cpos[e0 + k]];
            }
            __syncthreads();
        }

        int status = 0;
        if (P.kind == SWD_KIND_OSD_WINDOW && bad) {
            // osd_window.pyx:178-181: decimating the dropped columns in sorted order hits a check whose every VN is dropped
            // while its syndrome bit is 1; the failure is at the last column of that check in the scan order, and the
            // dropped columns up to there have been set to 0.  The scan order is the stable (key, index) order, so no
            // ranks are needed: M_r = the largest (key, index) pair of bad row r, F = the smallest M_r, and a dropped
            // column was reached iff its pair is <= F.  (Before the dropped columns' keys are overwritten below.)
            const double *ksrc = ws.sum + (size_t)slot * n;
            u64 *fkey = (u64 *)wt;
            if (tid == 0) { *fkey = ~0ull; misc[0] = 0x7fffffff; }
            __syncthreads();
            u64 mk = 0; int mi = -1;
            for (int r = tid; r < m; r += T) {          // at most one bad row per thread matters: keep the smallest M_r
                if (ub[r] == 0 && s_synd[r]) {
                    u64 rk = 0; int ri = -1;
                    for (int q = g.rp[r]; q < g.rp[r + 1]; q++) {
                        const int cI = g.rc[q]; const u64 kk = ordered_key(ksrc[cI]);
                        if (ri < 0 || kk > rk || (kk == rk && cI > ri)) { rk = kk; ri = cI; }
                    }
                    if (ri >= 0 && (mi < 0 || rk < mk || (rk == mk && ri < mi))) { mk = rk; mi = ri; }
                }
            }
            if (mi >= 0) atomicMin(fkey, mk);
            __syncthreads();
            const u64 fk = *fkey;
            if (mi >= 0 && mk == fk) atomicMin(&misc[0], mi);
            __syncthreads();
            const int fi = misc[0];
            for (int cI = tid; cI < n; cI += T) {
                if (posof[cI] >= nn) {
                    const u64 kk = ordered_key(ksrc[cI]);
                    if (kk < fk || (kk == fk && cI <= fi)) dec_out[(size_t)shot * n + cI] = 0;
                }
            }
            status = -2;
            __syncthreads();
        }
        if (P.kind == SWD_KIND_OSD_WINDOW) {
            // decided-0 key of the dropped columns (osd_window.pyx:208-209)
            if (partial) { for (int cI = tid; cI < n; cI += T) if (posof[cI] >= nn) ws.sum[(size_t)slot * n + cI] = 1000.0; }
            else for (int j = nn + tid; j < n; j += T) ws.sum[(size_t)slot * n + idx[j]] = 1000.0;
        }
        if (status == 0) {
            if (partial) { for (int cI = tid; cI < n; cI += T) if (posof[cI] >= nn) dec_out[(size_t)shot * n + cI] = 0; }
            else for (int j = nn + tid; j < n; j += T) dec_out[(size_t)shot * n + idx[j]] = 0;   // pyx:250-251 / :270-271
            Ctx c;
            c.m = m; c.nn = nn; c.es = es; c.msg = nullptr; c.prior = prior; c.voff = voff; c.vrow = vrow; c.vpos = vpos;
            c.coff = coff; c.crank = crank; c.cvn = cvn; c.vperm = vperm; c.cperm = cperm; c.synd = s_synd; c.vn_mask = vn_mask; c.error = s_error; c.cn_mask = cn_mask;
            c.cn_deg = cn_deg;
            if (wid == 0) {
                int st = peel_warp<false>(c, lane);                                          // bpgd.cpp:236
                if (lane == 0) misc[1] = st;
            }
            __syncthreads();
            status = misc[1];
            if (status < 0 && P.kind == SWD_KIND_OSD_WINDOW) {
                // osd_window.pyx:184-186: bp_decoding keeps the values peeled so far
                for (int j = tid; j < nn; j += T) if (vn_mask[j] >= 0) dec_out[(size_t)shot * n + col[j]] = (u8)vn_mask[j];
            }
        }
        if (tid == 0) {
            hdr->es = nslots; hdr->status = status; hdr->bad_rows = bad; hdr->shot = shot;
            if (nslots > capA) atomicAdd(&ws.counters[8], 1);
            if (status == 0) wl_push(ws, nslots > capA ? 1 : 0, wl_pack(slot, nslots, bad, 0));
        }
        __syncthreads();
        // publish the blob (16-byte vectors): fixed part + the three es-sized arrays
        {
            uint4 *dst = (uint4 *)(ws.blob + (size_t)slot * L.blob_bytes);
            const uint4 *src = (const uint4 *)blob;
            const int nfix = L.fixed_bytes >> 4, nvar = (nslots * 2 + 15) >> 4;
            for (int i = tid; i < nfix; i += T) dst[i] = src[i];
            for (int i = tid; i < nvar; i += T) {
                dst[(L.off_vrow >> 4) + i] = src[(L.off_vrow >> 4) + i];
                dst[(L.off_vpos >> 4) + i] = src[(L.off_vpos >> 4) + i];
                dst[(L.off_cvn >> 4) + i] = src[(L.off_cvn >> 4) + i];
            }
        }
        // clear result records and side snapshots' valid flags
        {
            u32 *rec = (u32 *)(ws.rec + (size_t)slot * P.n_rec * P.rec_stride);
            for (int i = tid; i < (P.n_rec * P.rec_stride) >> 2; i += T) rec[i] = 0;
            for (int j = tid; j < P.n_side; j += T) *(int *)(ws.side + ((size_t)slot * P.n_side + j) * P.side_stride) = 0;
            for (int j = tid; j < P.n_nodes; j += T) *(int *)(ws.node + ((size_t)slot * P.n_nodes + j) * P.node_stride) = 0;
        }
        __syncthreads();
    }
}

// ----------------------------------------------------------------------------------------------
// K3: branch paths
// ----------------------------------------------------------------------------------------------
struct RecHeader { double pm; int status; int pad; };          // 16 bytes, followed by error bit words
struct SideHeader { int valid, vn, value, depth; };            // 16 bytes, followed by vn_mask, cn_mask, cn_deg
struct NodeHeader { int alive, guess, favor, pad; };           // 16 bytes, followed by masks, messages, history

// write (status, pm, error bits) of the current path
// path metric of the current `error`, broadcast to the whole CTA (contains barriers)
__device__ __forceinline__ double block_pm(Ctx &c) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (wid == 0) { const double pm = pm_warp(c, lane); if (lane == 0) c.red_d[62] = pm; }
    __syncthreads();
    return c.red_d[62];
}

__device__ __forceinline__ void record_result(Ctx &c, u8 *rec, int converged, const double *pm_known = nullptr) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (wid == 0) {
        double pm = pm_known ? *pm_known : (converged ? pm_warp(c, lane) : SWD_MAX_PM);
        if (lane == 0) { RecHeader *h = (RecHeader *)rec; h->pm = pm; h->status = converged ? 1 : 2; }
    }
    u32 *bits = (u32 *)(rec + sizeof(RecHeader));
    const int nwords = (c.nn + 31) >> 5;
#pragma unroll 1
    for (int w = wid; w < nwords; w += nw) {
        const int j = w * 32 + lane;
        u32 b = __ballot_sync(FULLMASK, j < c.nn && c.error[j] != 0);
        if (lane == 0) bits[w] = b;
    }
}

// 16-byte vector copy of a small state array (both sides 16-byte aligned, allocations padded to 16 bytes)
__device__ __forceinline__ void copy_vec16(void *dst, const void *src, int nbytes, int tid, int T) {
    const int nv = (nbytes + 15) >> 4;
#pragma unroll 1
    for (int i = tid; i < nv; i += T) ((uint4 *)dst)[i] = ((const uint4 *)src)[i];
}

template <int VPT, int DMAX, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
path_kernel(Workspace ws, SubLayout LG, SubLayout L, PathSmem S, GdgDev P, int phase, int tier, int capA) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    unsigned char *blob = smem;
    unsigned char *st = smem + L.blob_bytes;
    Ctx c;
    c.m = L.m; c.nn = L.nn; c.factor = P.factor; c.low_error = P.low_error; c.count_work = P.count_work;
    c.prior = pinned_smem<const double>(blob + L.off_prior);
    c.voff = pinned_smem<const u16>(blob + L.off_voff); c.coff = pinned_smem<const u16>(blob + L.off_coff);
    c.crank = (const u16 *)(blob + L.off_crank);
    c.vrow = pinned_smem<const u16>(blob + L.off_vrow); c.vpos = pinned_smem<const u16>(blob + L.off_vpos); c.cvn = (const u16 *)(blob + L.off_cvn);   // SWD_DIET: re-pointed per item
    c.vperm = pinned_smem<const u16>(blob + L.off_vperm); c.cperm = pinned_smem<const u16>(blob + L.off_cperm);
    c.synd = blob + L.off_synd;
    c.msg = pinned_smem<double>(st + S.off_msg);
    c.vn_mask = pinned_smem<i8>(st + S.off_vnmask); c.error = pinned_smem<i8>(st + S.off_error); c.dec = pinned_smem<i8>(st + S.off_dec);
    c.cn_mask = pinned_smem<i8>(st + S.off_cnmask); c.cn_deg = st + S.off_cndeg; c.flip = pinned_smem<u8>(st + S.off_flip);
    c.upar = pinned_smem<u32>(st + S.off_upar);
    c.red_d = (double *)(st + S.off_red); c.red_i = (int *)(c.red_d + 64); c.misc = (int *)(st + S.off_misc);
    c.zslot = (int)((double *)(st + S.off_misc + 48) - c.msg);      // misc[12..13]: the constant +0.0 of vn_update
    if (threadIdx.x == 0) *(double *)(st + S.off_misc + 48) = 0.0;
#if !SWD_DIET
    i8 *bvn = (i8 *)(st + S.off_bvn); i8 *bcn = (i8 *)(st + S.off_bcn); u8 *bdeg = st + S.off_bdeg;
#endif
    u64 *bar = (u64 *)(st + S.off_bar);
#if !SWD_DIET
    const i8 *snap_vn = (const i8 *)(blob + L.off_vnmask), *snap_cn = (const i8 *)(blob + L.off_cnmask);
    const u8 *snap_deg = blob + L.off_cndeg;
#endif

    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    u32 mphase = 0;
    const int node_level = (phase >= 2) ? phase - 2 : -1;          // >= 0: shared-prefix node of that depth
    const int sT = P.shared_T;
    const int npaths = (phase == 0 && sT == 0 && P.kind == SWD_KIND_BPGDG && P.multi_thread) ? 1 + P.n_tree : 1;
    // input lists of this launch (see swd_device.cuh): l1 is drawn `npaths` times (path-major), then l2
    int l1, l2 = -1;
    if (node_level >= 0) l1 = 2 * node_level + tier;
    else if (phase == 0) { if (sT > 0) { l1 = 2 * sT + tier; l2 = 2 * sT + 2 + tier; } else l1 = tier; }
    else l1 = 2 * sT + 4 + tier;
    // list lengths live in shared memory (misc[8..10]): they are only needed once per item
    if (tid == T - 1) {          // the thread that draws the tickets (it reads these back before the first barrier)
        const int n1 = ws.counters[SWD_WL_CNT + l1], n2 = (l2 >= 0) ? ws.counters[SWD_WL_CNT + l2] : 0;
        c.misc[8] = n1; c.misc[9] = npaths * n1; c.misc[10] = npaths * n1 + n2;
    }
    const int ticket = (node_level >= 0) ? 16 + 2 * node_level + tier : 1 + phase + 3 * tier;
    u64 edge_iters = 0, bp_calls = 0, paths_run = 0, slot_iters = 0;
    u32 vn_iters = 0, cn_iters = 0;

#ifndef SWD_CLAIM_AHEAD
#define SWD_CLAIM_AHEAD 0     /* measured -3..4 % (A/B r2, as in round 1): kept for the record */
#endif
    // (SWD_CLAIM_AHEAD = 1, measured and rejected) One item ahead: while the CTA works on an item, its last thread has already drawn the next ticket, read that item
    // (shared memory: misc[2] = ticket, misc[14..15] = item - no registers are held across the item) and asked L2 for the
    // item's graph, parent messages and parent state, so the next set-up starts without a global round trip and its TMA
    // copies come from L2 instead of HBM.
    auto claim = [&]() {
        const int ntk = atomicAdd(&ws.counters[ticket], 1);
        c.misc[2] = ntk;
        if (ntk >= c.misc[10]) return;
        const int n1c = c.misc[8], t1c = c.misc[9];
        const u64 it = (ntk < t1c) ? ws.wl[(size_t)l1 * ws.wl_stride + (npaths > 1 ? ntk % n1c : ntk)]
                                   : ws.wl[(size_t)l2 * ws.wl_stride + (ntk - t1c)];
        *(u64 *)&c.misc[14] = it;
        if (SWD_CLAIM_AHEAD) {
            const int nslot = (int)(it & 0xfffffffu), nes = (int)((it >> 28) & 0xffffu);
            const int npath = (npaths > 1) ? ntk / n1c : (int)(it >> 48);
            const unsigned char *nb = ws.blob + (size_t)nslot * LG.blob_bytes;
            const u32 vb = (u32)((nes * 2 + 15) & ~15);
            bulk_prefetch_l2(nb, (u32)L.fixed_bytes);
            if (vb) { bulk_prefetch_l2(nb + LG.off_vrow, vb); bulk_prefetch_l2(nb + LG.off_vpos, vb); }
            if (sT > 0 && (node_level > 0 || phase == 0)) {
                const int plevel = (node_level > 0) ? node_level - 1 : sT - 1;
                const unsigned char *pn = ws.node + ((size_t)nslot * P.n_nodes + ((1 << plevel) - 1) + (npath >> 1)) * P.node_stride;
                bulk_prefetch_l2(pn, (u32)P.node_off_msg);                                   // header + masks
                bulk_prefetch_l2(pn + P.node_off_msg, (u32)((nes * 8 + 15) & ~15));             // messages
                bulk_prefetch_l2(pn + P.node_off_hist, (u32)(8 * 16 * T));                     // posterior history
            }
        }
    };
    if (SWD_CLAIM_AHEAD && tid == T - 1) claim();
    for (;;) {
        __syncthreads();
        if (!SWD_CLAIM_AHEAD) { if (tid == T - 1) claim(); __syncthreads(); }
        const int tk = c.misc[2];
        if (tk >= c.misc[10]) break;
        const int n1 = c.misc[8];
        const u64 item = *(const u64 *)&c.misc[14];
        if (SWD_CLAIM_AHEAD) { __syncthreads(); if (tid == T - 1) claim(); }       // everyone holds the current item: draw the next
        const int slot = (int)(item & 0xfffffffu), es = (int)((item >> 28) & 0xffffu);
        const int path = (npaths > 1) ? tk / n1 : (int)(item >> 48);
        const unsigned char *gblob = ws.blob + (size_t)slot * LG.blob_bytes;
        // parent node of the shared-prefix tree (if this item continues from one)
        const unsigned char *pnode = nullptr;
        if (sT > 0 && (node_level > 0 || phase == 0)) {
            const int plevel = (node_level > 0) ? node_level - 1 : sT - 1;
            pnode = ws.node + ((size_t)slot * P.n_nodes + ((1 << plevel) - 1) + (path >> 1)) * P.node_stride;
        }
        // ---- stage the shot's shortened graph into shared memory with TMA bulk copies
        if (tid == 0) {
            fence_proxy_async();
            const u32 vb = (u32)((es * 2 + 15) & ~15);
            const u32 mb = pnode ? (u32)((es * 8 + 15) & ~15) : 0u;
            mbar_expect_tx(bar, (u32)L.fixed_bytes + (SWD_DIET ? 2 : 3) * vb + mb);
            bulk_g2s(blob, gblob, (u32)L.fixed_bytes, bar);
            if (vb) {
                bulk_g2s(blob + L.off_vrow, gblob + LG.off_vrow, vb, bar);
                bulk_g2s(blob + L.off_vpos, gblob + LG.off_vpos, vb, bar);
#if !SWD_DIET
                bulk_g2s(blob + L.off_cvn, gblob + LG.off_cvn, vb, bar);
#endif
            }
            if (mb) bulk_g2s(c.msg, pnode + P.node_off_msg, mb, bar);       // messages of the parent node
        }
#if SWD_DIET
        c.cvn = (const u16 *)(gblob + LG.off_cvn);
        const i8 *snap_vn = (const i8 *)(gblob + LG.off_vnmask), *snap_cn = (const i8 *)(gblob + LG.off_cnmask);
        const u8 *snap_deg = gblob + LG.off_cndeg;
#define SWD_BAK_PTRS i8 *bvn = (i8 *)(ws.bak + ((size_t)slot * max(1, P.n_tree) + (size_t)max(0, path - 1)) * P.bak_stride); \
                     i8 *bcn = bvn + ((c.nn + 15) & ~15); u8 *bdeg = (u8 *)(bcn + ((c.m + 15) & ~15));
#else
#define SWD_BAK_PTRS
#endif
        // ---- meanwhile: headers and the start state that comes from HBM (parent node / side snapshot)
        const SideHeader *sh = nullptr;
        SideHeader shv = {0, -1, 0, 0};
        if (phase == 1) { sh = (const SideHeader *)(ws.side + ((size_t)slot * P.n_side + path) * P.side_stride); shv = *sh; }
        NodeHeader ph = {0, -1, 0, 0};
        if (pnode) ph = *(const NodeHeader *)pnode;
        c.es = es; c.bad_rows = (int)((item >> 44) & 1u);
        c.C = 30; c.D = 3;
        double h[VPT][4];
        if (pnode) {
            const i8 *nvn = (const i8 *)(pnode + sizeof(NodeHeader)), *ner = (const i8 *)(pnode + P.node_off_err);
            const i8 *ncn = (const i8 *)(pnode + P.node_off_cn);
            const u8 *ndg = pnode + P.node_off_deg, *nfl = pnode + P.node_off_flip;
            const double *nh = (const double *)(pnode + P.node_off_hist);
            copy_vec16(c.vn_mask, nvn, c.nn, tid, T); copy_vec16(c.error, ner, c.nn, tid, T);
            copy_vec16(c.cn_mask, ncn, c.m, tid, T); copy_vec16(c.cn_deg, ndg, c.m, tid, T); copy_vec16(c.flip, nfl, c.m, tid, T);
#pragma unroll
            for (int i = 0; i < VPT; i++)
#pragma unroll
                for (int q = 0; q < 4; q++) h[i][q] = nh[(size_t)(i * 4 + q) * T + tid];
        } else if (phase == 1) {
            const i8 *svn = (const i8 *)(sh + 1); const i8 *scn = svn + c.nn; const u8 *sdg = (const u8 *)(scn + c.m);
#pragma unroll 1
            for (int j = tid; j < c.nn; j += T) { const i8 v = svn[j]; c.vn_mask[j] = v; c.error[j] = v; }   // bpgd.cpp:541
#pragma unroll 1
            for (int r = tid; r < c.m; r += T) { c.cn_mask[r] = scn[r]; c.cn_deg[r] = sdg[r]; c.flip[r] = 0; }
        }
#if SWD_DIET
        else {      // the post-reset state, from the global blob
#pragma unroll 1
            for (int j = tid; j < c.nn; j += T) { const i8 v = snap_vn[j]; c.vn_mask[j] = v; c.error[j] = v < 0 ? 0 : v; }
#pragma unroll 1
            for (int r = tid; r < c.m; r += T) { c.cn_mask[r] = snap_cn[r]; c.cn_deg[r] = snap_deg[r]; c.flip[r] = 0; }
        }
#endif
        mbar_wait(bar, mphase);
        mphase ^= 1;
        if (pnode) __syncthreads();
        else {
#if !SWD_DIET
        if (phase != 1) {
#pragma unroll 1
            for (int j = tid; j < c.nn; j += T) { const i8 v = snap_vn[j]; c.vn_mask[j] = v; c.error[j] = v < 0 ? 0 : v; }
#pragma unroll 1
            for (int r = tid; r < c.m; r += T) { c.cn_mask[r] = snap_cn[r]; c.cn_deg[r] = snap_deg[r]; c.flip[r] = 0; }
        }
#endif
        __syncthreads();
        init_msgs<VPT>(c);
#pragma unroll
        for (int i = 0; i < VPT; i++) { h[i][0] = 0.0; h[i][1] = 0.0; h[i][2] = 0.0; h[i][3] = 0.0; }
        __syncthreads();
        }
        paths_run++;

        u8 *recbase = ws.rec + (size_t)slot * P.n_rec * P.rec_stride;

        // ---- one interpreter loop for every kind of branch, so that bp_run / select_vn /
        //      set_and_peel are instantiated once (registers, code size)
        enum { R_MAIN = 0, R_TREE = 1, R_SIDE = 2, R_GD = 3, R_ST = 4, R_NODE = 5 };
        int role, limit, depth = 0, pend_vn = -1, pend_val = 0;
        u8 *rec = recbase;
        bool mainlike = false, node_alive = false; int node_guess = -1, node_favor = 0;
        // single-thread schedule (pyx:254-338): guess stack lives in this slot's side-snapshot area
        int st_used = 0, st_i = 0, st_min_depth = P.max_step, st_conv = 0; double st_min_pm = SWD_MAX_PM;
        if (P.kind == SWD_KIND_BPGD) { role = R_GD; limit = P.max_step; }
        else if (!P.multi_thread) { role = R_ST; limit = P.max_step; c.A = -3; c.A_sum = -16; }
        else if (node_level >= 0) {
            // shared-prefix node: ONE decimation step for every branch path whose first node_level decisions equal
            // `path` (bit k of the prefix = decision at depth k flipped, bpgd.cpp:464-470)
            role = R_NODE; limit = 1; depth = node_level; mainlike = (path == 0);
            rec = recbase + (size_t)(path << (P.shared_T - node_level)) * P.rec_stride;     // lowest branch id with this prefix
            if (path == 0) { c.A = -3; c.A_sum = (depth == 0) ? -16 : -12; } else { c.A = 0; c.A_sum = -10; }
            if (pnode) { pend_vn = ph.guess; pend_val = ph.favor ^ (path & 1); }
        }
        else if (phase == 1) {                                  // side branch j (bpgd.cpp:527-570)
            role = R_SIDE; limit = P.side_step; rec = recbase + (size_t)(1 + P.n_tree + path) * P.rec_stride;
            c.A = 0; c.A_sum = -10; depth = shv.depth; pend_vn = shv.vn; pend_val = shv.value;
        } else if (path == 0) { role = R_MAIN; mainlike = true; limit = P.max_step; c.A = -3; c.A_sum = -16; }   // bpgd.cpp:623-683
        else {                                                  // tree branch id (bpgd.cpp:435-525)
            role = R_TREE; limit = P.tree_step + P.T + 1; rec = recbase + (size_t)path * P.rec_stride;
            c.A = -3; c.A_sum = -16;
        }
        int stage = 0, steps = 0, on_side = 0, saved = 0, bvar = -1, bval = 0, conv = 0;
        if (pnode && node_level < 0) {
            // continue from the last shared node: decision of depth shared_T-1 with this path's own bit, then depth shared_T
            depth = P.shared_T; steps = P.shared_T;
            pend_vn = ph.guess; pend_val = ph.favor ^ (path & 1);
            if (role == R_TREE) { on_side = 1; c.A = 0; c.A_sum = -10; }      // every tree id has taken a flip by now
        }
        for (;;) {
            bool stage_end = false;
            if (pend_vn >= 0) {
                const int r = set_and_peel(c, pend_vn, pend_val);
                pend_vn = -1;
                if (r < 0) stage_end = true;
            }
            if (!stage_end && steps >= limit) stage_end = true;
            if (!stage_end) {
                if (role == R_MAIN) c.A_sum = (depth == 0) ? -16 : -12;                          // :631
                if (role == R_ST) {                                                               // pyx:341-343
                    c.A = stage ? 0 : -3; c.A_sum = stage ? -10 : -12;
                    if (depth == 0) c.A_sum = -16;
                }
                if (role == R_TREE && stage == 0 && depth > 0 && !on_side) c.A_sum = -12;         // :450
                conv = bp_run<VPT, DMAX>(c, h, P.num_iter, edge_iters, vn_iters, cn_iters, slot_iters); bp_calls++;
                steps++;
                if (role == R_GD) {
                    // bpgd_decoder.gd (pyx:540-553) with decimate_vn_reliable (bpgd.cpp:258-286)
                    if (conv) break;
                    double best = 0.0; int bi = 0x7fffffff;   // argmax |h[3]|, first wins
#pragma unroll
                    for (int i = 0; i < VPT; i++) {
                        const int sl = own_slot(i, tid, T);
                        if (sl < c.nn) {
                            const int j = c.vperm[sl];
                            if (c.vn_mask[j] < 0) { const double a = -fabs(h[i][3]); if (a < best || (a == best && a < 0.0 && j < bi)) { best = a; bi = j; } }
                        }
                    }
                    block_argmin(best, bi, c.red_d, c.red_i);
                    if (bi == 0x7fffffff) break;
#pragma unroll
                    for (int i = 0; i < VPT; i++) { const int sl = own_slot(i, tid, T); if (sl < c.nn && c.vperm[sl] == bi) c.misc[3] = (h[i][3] > 0.0) ? 0 : 1; }
                    __syncthreads();
                    pend_vn = bi; pend_val = c.misc[3]; depth++;
                    continue;
                }
                if (role == R_ST && conv) {                                                       // pyx:284-292, :320-330
                    const double pm = block_pm(c);
                    st_conv = 1;
                    if (stage == 0) { st_min_depth = depth; st_min_pm = pm; record_result(c, rec, 1, &pm); }
                    else if (pm < st_min_pm) {
                        if (depth < st_min_depth) st_min_depth = depth;
                        st_min_pm = pm; record_result(c, rec, 1, &pm);
                    }
                    stage_end = true;
                }
                if (role == R_ST && !stage_end && stage == 1 && depth > st_min_depth + 2) stage_end = true;   // pyx:331
                if (conv && !mainlike && role != R_ST) break;                                     // :452-459, :552-559
                if (!stage_end) {
                int guess = -1;
                int favor = select_vn<VPT>(c, h, depth, guess);
                if (conv) break;                                                                  // main: :633-649
                if (favor == -1 || guess == -1) stage_end = true;
                else {
                    if (role == R_NODE) { node_alive = true; node_guess = guess; node_favor = favor; break; }
                    if (role == R_ST) {                                                           // pyx:416-433
                        bool do_guess = !(depth > st_min_depth);
                        if (stage == 0 && depth >= P.S) do_guess = false;
                        if (stage == 1 && depth > P.T) do_guess = false;
                        if (do_guess && st_used < P.n_side) {
                            unsigned char *sp = ws.side + ((size_t)slot * P.n_side + st_used) * P.side_stride;
                            i8 *svn = (i8 *)(sp + sizeof(SideHeader)); i8 *scn = svn + c.nn; u8 *sdg = (u8 *)(scn + c.m);
#pragma unroll 1
                            for (int j = tid; j < c.nn; j += T) svn[j] = c.vn_mask[j];
#pragma unroll 1
                            for (int r = tid; r < c.m; r += T) { scn[r] = c.cn_mask[r]; sdg[r] = c.cn_deg[r]; }
                            if (tid == 0) { SideHeader *q = (SideHeader *)sp; q->vn = guess; q->value = 1 - favor; q->depth = depth + 1; q->valid = 1; }
                            st_used++;
                        }
                    }
                    if (role == R_MAIN && depth >= P.T && depth < P.S) {                          // :651-664
                        unsigned char *sp = ws.side + ((size_t)slot * P.n_side + (depth - P.T)) * P.side_stride;
                        i8 *svn = (i8 *)(sp + sizeof(SideHeader)); i8 *scn = svn + c.nn; u8 *sdg = (u8 *)(scn + c.m);
#pragma unroll 1
                        for (int j = tid; j < c.nn; j += T) svn[j] = c.vn_mask[j];
#pragma unroll 1
                        for (int r = tid; r < c.m; r += T) { scn[r] = c.cn_mask[r]; sdg[r] = c.cn_deg[r]; }
                        if (tid == 0) {
                            SideHeader *q = (SideHeader *)sp; q->vn = guess; q->value = 1 - favor; q->depth = depth + 1; q->valid = 1;
                            wl_push(ws, 2 * sT + 4 + tier, wl_pack(slot, c.es, c.bad_rows, depth - P.T));
                        }
                    }
                    if (role == R_TREE && stage == 0) {
                        if (depth < P.T) {                                                        // :464-470
                            if ((path >> (P.T - 1 - depth)) & 1) { on_side = 1; c.A = 0; c.A_sum = -10; favor = 1 - favor; }
                        } else if (depth == P.T) {                                                // :476-484
                            SWD_BAK_PTRS
#pragma unroll 1
                            for (int j = tid; j < c.nn; j += T) bvn[j] = c.vn_mask[j];
#pragma unroll 1
                            for (int r = tid; r < c.m; r += T) { bcn[r] = c.cn_mask[r]; bdeg[r] = c.cn_deg[r]; }
                            bvar = guess; bval = 1 - favor; saved = 1;
                        }
                    }
                    pend_vn = guess; pend_val = favor; depth++;
                    continue;
                }
                }
            }
            // ---- the current stage ended without convergence
            if (role == R_ST) {
                if (stage == 0 && !st_conv) record_result(c, rec, 0);                             // pyx:295-298
                bool again = false;
                while (st_i < st_used) {                                                          // pyx:302-335
                    const unsigned char *sp = ws.side + ((size_t)slot * P.n_side + st_i) * P.side_stride;
                    st_i++;
                    const SideHeader q = *(const SideHeader *)sp;
                    if (q.depth > st_min_depth) continue;                                         // pyx:304
                    const i8 *svn = (const i8 *)(sp + sizeof(SideHeader)); const i8 *scn = svn + c.nn; const u8 *sdg = (const u8 *)(scn + c.m);
                    __syncthreads();
#pragma unroll 1
                    for (int j = tid; j < c.nn; j += T) { const i8 v = svn[j]; c.vn_mask[j] = v; c.error[j] = v; }   // set_masks, bpgd.cpp:241-248
#pragma unroll 1
                    for (int r = tid; r < c.m; r += T) { c.cn_mask[r] = scn[r]; c.cn_deg[r] = sdg[r]; }
                    __syncthreads();
                    init_msgs<VPT>(c);
                    stage = 1; steps = 0; limit = P.side_step; depth = q.depth; pend_vn = q.vn; pend_val = q.value;
                    again = true;
                    break;
                }
                if (again) continue;
                conv = 0;
                break;
            }
            if (role == R_TREE && stage == 0 && saved) {                                          // :490-503
                __syncthreads();
                SWD_BAK_PTRS
#pragma unroll 1
                for (int j = tid; j < c.nn; j += T) { const i8 v = bvn[j]; c.vn_mask[j] = v; c.error[j] = v; }
#pragma unroll 1
                for (int r = tid; r < c.m; r += T) { c.cn_mask[r] = bcn[r]; c.cn_deg[r] = bdeg[r]; }
                __syncthreads();
                init_msgs<VPT>(c);
                stage = 1; steps = 0; limit = P.tree_step; depth = P.T + 1; pend_vn = bvar; pend_val = bval;
                continue;
            }
            break;
        }
        if (node_alive) {
            // publish the node: state after select_vn of this depth, before the decision is applied
            unsigned char *nd = ws.node + ((size_t)slot * P.n_nodes + ((1 << node_level) - 1) + path) * P.node_stride;
            i8 *nvn = (i8 *)(nd + sizeof(NodeHeader)), *ner = (i8 *)(nd + P.node_off_err), *ncn = (i8 *)(nd + P.node_off_cn);
            u8 *ndg = nd + P.node_off_deg, *nfl = nd + P.node_off_flip;
            double *nm = (double *)(nd + P.node_off_msg), *nh = (double *)(nd + P.node_off_hist);
            __syncthreads();
            copy_vec16(nvn, c.vn_mask, c.nn, tid, T); copy_vec16(ner, c.error, c.nn, tid, T);
            copy_vec16(ncn, c.cn_mask, c.m, tid, T); copy_vec16(ndg, c.cn_deg, c.m, tid, T); copy_vec16(nfl, c.flip, c.m, tid, T);
            copy_vec16(nm, c.msg, 8 * c.es, tid, T);
#pragma unroll
            for (int i = 0; i < VPT; i++)
#pragma unroll
                for (int q = 0; q < 4; q++) nh[(size_t)(i * 4 + q) * T + tid] = h[i][q];
            if (tid == 0) {
                NodeHeader *hd = (NodeHeader *)nd; hd->guess = node_guess; hd->favor = node_favor; hd->alive = 1;
                // the two continuations of this prefix: next node level, or (after the last level) the branch paths - the
                // main path has its own list, drawn first (it is the longest item of the launch)
                const bool lastlv = (node_level + 1 >= sT);
                const int lnext = lastlv ? 2 * sT + 2 + tier : 2 * (node_level + 1) + tier;
                wl_push(ws, (lastlv && path == 0) ? 2 * sT + tier : lnext, wl_pack(slot, c.es, c.bad_rows, 2 * path));
                wl_push(ws, lnext, wl_pack(slot, c.es, c.bad_rows, 2 * path + 1));
            }
        } else if (role != R_ST && (conv || mainlike || role == R_GD)) record_result(c, rec, conv);
    }
    // ---- work counters
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
// K4: pick the branch with the smallest path metric (first wins ties; order main, tree ids, sides)
// ----------------------------------------------------------------------------------------------
__global__ void select_kernel(Workspace ws, SubLayout L, GdgDev P, int n, u8 *__restrict__ dec_out,
                              u8 *__restrict__ conv_out, double *__restrict__ pm_out) {
    const int T = blockDim.x, tid = threadIdx.x;
    const int count = ws.counters[0];
    for (int slot = blockIdx.x; slot < count; slot += gridDim.x) {
        const unsigned char *gblob = ws.blob + (size_t)slot * L.blob_bytes;
        const BlobHeader gh = *(const BlobHeader *)gblob;
        const u16 *col = (const u16 *)(gblob + L.off_col);
        const u8 *recbase = ws.rec + (size_t)slot * P.n_rec * P.rec_stride;
        int best = -1; double pm = SWD_MAX_PM;
        if (gh.status == 0) {
            for (int r = 0; r < P.n_rec; r++) {
                const RecHeader *h = (const RecHeader *)(recbase + (size_t)r * P.rec_stride);
                if (h->status == 1 && h->pm < pm) { pm = h->pm; best = r; }
            }
        }
        const int conv = (P.kind == SWD_KIND_BPGDG && P.multi_thread) ? (pm < 9999.0) : (best >= 0);   // pyx:247
        const size_t row = (size_t)gh.shot * n;
        if (gh.status == 0) {
            const u32 *bits = (const u32 *)(recbase + (size_t)(best < 0 ? 0 : best) * P.rec_stride + sizeof(RecHeader));
            for (int j = tid; j < L.nn; j += T) dec_out[row + col[j]] = (u8)((bits[j >> 5] >> (j & 31)) & 1u);
        } else if (P.kind == SWD_KIND_BPGDG && P.multi_thread) {
            for (int j = tid; j < L.nn; j += T) dec_out[row + col[j]] = 0;      // fresh min_pm_error (see DESIGN.md)
        }
        if (tid == 0) { conv_out[gh.shot] = (u8)conv; if (pm_out) pm_out[gh.shot] = pm; }
    }
}

// min_pm for BP-converged shots is not defined by the GDG decoders; fill with MAX_PM.
__global__ void fill_pm_kernel(double *pm_out, long long B, double v) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) pm_out[i] = v;
}
