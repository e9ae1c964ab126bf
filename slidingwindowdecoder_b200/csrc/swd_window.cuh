// swd_window.cuh — sliding-window bookkeeping kernels (guessing.py:204-227, osd.py:170-179):
// window syndrome extraction, commit of the first F rounds with the sparse syndrome update
// new_det = det + e_hat @ chk.T (the reference does a dense float GEMM), failure counters, DEM, code-capacity and circuit-level samplers.
#pragma once
#include "swd_device.cuh"

__global__ void accumulate_count_kernel(const int *counters, u64 *stats) { stats[5] += (u64)counters[0]; }

__global__ void window_extract_kernel(const u8 *__restrict__ det, long long B, int num_det, int row0, int m, u8 *__restrict__ synd) {
    const long long total = B * m;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / m; const int r = (int)(i - b * m);
        synd[i] = det[b * num_det + row0 + r];
    }
}

// one warp per shot: lanes scan 32 committed columns at a time (coalesced), every set bit's
// detector / observable rows are XORed by the first lanes (rows of one column are distinct).
__global__ void window_commit_kernel(const u8 *__restrict__ corr, long long B, int n_win, int col0, int ncommit,
                                     const int *__restrict__ chk_cp, const int *__restrict__ chk_ri, int num_det, u8 *det,
                                     const int *__restrict__ obs_cp, const int *__restrict__ obs_ri, int num_obs, u8 *obs) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (long long b = (long long)blockIdx.x * wpb + (threadIdx.x >> 5); b < B; b += (long long)gridDim.x * wpb) {
        const u8 *row = corr + b * n_win;
        for (int base = 0; base < ncommit; base += 32) {
            const int j = base + lane;
            u32 bits = __ballot_sync(FULLMASK, j < ncommit && row[j] != 0);
            while (bits) {
                const int k = __ffs(bits) - 1; bits &= bits - 1;
                const int c = col0 + base + k;
                for (int e = chk_cp[c] + lane; e < chk_cp[c + 1]; e += 32) det[b * num_det + chk_ri[e]] ^= 1;
                if (obs && num_obs > 0) for (int e = obs_cp[c] + lane; e < obs_cp[c + 1]; e += 32) obs[b * num_obs + obs_ri[e]] ^= 1;
                __syncwarp();
            }
        }
    }
}

__global__ void window_count_kernel(const u8 *__restrict__ det, int num_det, const u8 *__restrict__ obs, int num_obs, long long B, u64 *out2) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    u64 nflag = 0, nfail = 0;
    for (long long b = (long long)blockIdx.x * wpb + (threadIdx.x >> 5); b < B; b += (long long)gridDim.x * wpb) {
        int f = 0, l = 0;
        for (int r = lane; r < num_det; r += 32) f |= det[b * num_det + r];
        if (obs) for (int r = lane; r < num_obs; r += 32) l |= obs[b * num_obs + r];
        f = __any_sync(FULLMASK, f); l = __any_sync(FULLMASK, l);
        nflag += f ? 1 : 0; nfail += (f || l) ? 1 : 0;
    }
    if (lane == 0) { if (nflag) atomicAdd(&out2[0], nflag); if (nfail) atomicAdd(&out2[1], nfail); }
}

// ----------------------------------------------------------------------------------------------
// DEM sampling on the device: what stim's CompiledDemSampler.sample draws (guessing.py:129-130,
// build_circuit.py:271-288) - an independent Bernoulli(prior[c]) per DEM column, det = chk . e,
// obs = obs_mat . e (mod 2) - so that large runs never touch the host (SURVEY.md 8(f)-1).
// Counter-based generator: Philox4x32-10 keyed by the seed, counter = (shot, column block), four
// columns per call; a column fires when its 32-bit draw is below floor(p * 2^32).  One warp per
// shot; detector / observable parities are accumulated in shared-memory bit words.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(u32 c0, u32 c1, u32 c2, u32 c3, u32 k0, u32 k1, u32 (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const u32 hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const u32 hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const u32 n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__global__ void window_sample_kernel(const u32 *__restrict__ thr, int num_col, const int *__restrict__ chk_cp, const int *__restrict__ chk_ri,
                                     int num_det, const int *__restrict__ obs_cp, const int *__restrict__ obs_ri, int num_obs,
                                     unsigned long long seed, long long shot0, long long B, u8 *__restrict__ det, u8 *__restrict__ obs,
                                     u8 *__restrict__ err) {
    extern __shared__ u32 s_bits[];                           // per warp: ceil(num_det/32) + ceil(num_obs/32) words
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int wd = (num_det + 31) >> 5, wo = (num_obs + 31) >> 5;
    u32 *dbits = s_bits + (size_t)wid * (wd + wo), *obits = dbits + wd;
    const int nblk = (num_col + 3) >> 2;
    for (long long b = (long long)blockIdx.x * wpb + wid; b < B; b += (long long)gridDim.x * wpb) {
        for (int i = lane; i < wd + wo; i += 32) dbits[i] = 0;
        __syncwarp();
        const unsigned long long shot = (unsigned long long)(shot0 + b);
        for (int blk = lane; blk < nblk; blk += 32) {
            u32 r[4];
            philox4x32_10((u32)blk, 0u, (u32)shot, (u32)(shot >> 32), (u32)seed, (u32)(seed >> 32), r);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int c = blk * 4 + q;
                if (c >= num_col) break;
                const bool fire = r[q] < thr[c];
                if (err) err[b * num_col + c] = (u8)fire;
                if (fire) {
                    for (int e = chk_cp[c]; e < chk_cp[c + 1]; e++) { const int row = chk_ri[e]; atomicXor(&dbits[row >> 5], 1u << (row & 31)); }
                    if (num_obs > 0) for (int e = obs_cp[c]; e < obs_cp[c + 1]; e++) { const int row = obs_ri[e]; atomicXor(&obits[row >> 5], 1u << (row & 31)); }
                }
            }
        }
        __syncwarp();
        for (int i = lane; i < num_det; i += 32) det[b * num_det + i] = (u8)((dbits[i >> 5] >> (i & 31)) & 1u);
        if (obs) for (int i = lane; i < num_obs; i += 32) obs[b * num_obs + i] = (u8)((obits[i >> 5] >> (i & 31)) & 1u);
        __syncwarp();
    }
}

// ----------------------------------------------------------------------------------------------
// Code-capacity Pauli sampling: depolarizing noise with heralded erasures on n data qubits, as a plan over 2n columns
// (column v = X part of qubit v, column n + v = its Z part).  One Philox call per qubit pair k with counter (k, 1, shot) -
// the 1 keeps this stream apart from window_sample_kernel's - whose words 2j / 2j+1 are the erasure / Pauli draws of qubit
// 2k + j, both always drawn.  Erased (w_e < t_erase): Pauli = w_p >> 30 (0 I, 1 X, 2 Y, 3 Z: exactly uniform); otherwise X,
// Y, Z below the cumulative thresholds thr3[v], thr3[n + v], thr3[2n + v], else I.  e_x = X or Y, e_z = Y or Z; the chk / obs
// columns of the set bits are XORed into shared-memory parity words as in window_sample_kernel.  channel_llr [5][B][n]
// copies the host-computed rows llr5[5][n] with 0.0 at erased qubits (no log on the device).
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void xor_column(int c, const int *__restrict__ cp, const int *__restrict__ ri, u32 *bits) {
    for (int e = cp[c]; e < cp[c + 1]; e++) { const int row = ri[e]; atomicXor(&bits[row >> 5], 1u << (row & 31)); }
}

__global__ void window_sample_pauli_kernel(const u32 *__restrict__ thr3, u32 t_erase, int n, const double *__restrict__ llr5,
                                           const int *__restrict__ chk_cp, const int *__restrict__ chk_ri, int num_det,
                                           const int *__restrict__ obs_cp, const int *__restrict__ obs_ri, int num_obs,
                                           unsigned long long seed, long long shot0, long long B, u8 *__restrict__ det,
                                           u8 *__restrict__ obs, u8 *__restrict__ err, u8 *__restrict__ erased,
                                           double *__restrict__ channel_llr) {
    extern __shared__ u32 s_bits[];                           // per warp: ceil(num_det/32) + ceil(num_obs/32) words
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int wd = (num_det + 31) >> 5, wo = (num_obs + 31) >> 5;
    u32 *dbits = s_bits + (size_t)wid * (wd + wo), *obits = dbits + wd;
    const int npair = (n + 1) >> 1;
    for (long long b = (long long)blockIdx.x * wpb + wid; b < B; b += (long long)gridDim.x * wpb) {
        for (int i = lane; i < wd + wo; i += 32) dbits[i] = 0;
        __syncwarp();
        const unsigned long long shot = (unsigned long long)(shot0 + b);
        for (int k = lane; k < npair; k += 32) {
            u32 r[4];
            philox4x32_10((u32)k, 1u, (u32)shot, (u32)(shot >> 32), (u32)seed, (u32)(seed >> 32), r);
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int v = 2 * k + j;
                if (v >= n) break;
                const u32 we = r[2 * j], wp = r[2 * j + 1];
                const bool er = we < t_erase;
                const u32 pauli = er ? (wp >> 30) : wp < thr3[v] ? 1u : wp < thr3[n + v] ? 2u : wp < thr3[2 * n + v] ? 3u : 0u;
                const bool ex = pauli == 1u || pauli == 2u, ez = pauli >= 2u;
                if (err) { err[b * 2 * n + v] = (u8)ex; err[b * 2 * n + n + v] = (u8)ez; }
                if (erased) erased[b * n + v] = (u8)er;
                if (channel_llr)
                    for (int q = 0; q < 5; q++) channel_llr[((long long)q * B + b) * n + v] = er ? 0.0 : llr5[q * n + v];
                if (ex) { xor_column(v, chk_cp, chk_ri, dbits); if (num_obs > 0) xor_column(v, obs_cp, obs_ri, obits); }
                if (ez) { xor_column(n + v, chk_cp, chk_ri, dbits); if (num_obs > 0) xor_column(n + v, obs_cp, obs_ri, obits); }
            }
        }
        __syncwarp();
        for (int i = lane; i < num_det; i += 32) det[b * num_det + i] = (u8)((dbits[i >> 5] >> (i & 31)) & 1u);
        if (obs) for (int i = lane; i < num_obs; i += 32) obs[b * num_obs + i] = (u8)((obits[i >> 5] >> (i & 31)) & 1u);
        __syncwarp();
    }
}

// ----------------------------------------------------------------------------------------------
// Circuit-level noise with heralded erasures, sampled per noise location (dem.noise_locations: one per DEPOLARIZE2, one per
// target of X_ERROR / Z_ERROR / DEPOLARIZE1) rather than per merged DEM column.  Location l has n_l <= 15 mechanisms
// mech[m0 .. m0 + n_l - 1] = (DEM column or -1, thr(p)) and uses draws t = 0 .. n_l: draw t is word t & 3 of the Philox call
// with counter (l, 2 + (t >> 2), shot) - tags 0 and 1 belong to window_sample_kernel and window_sample_pauli_kernel.  Draw 0
// is the erasure draw (erased iff w < thr(e_l)); draw 1 + k is mechanism k, which fires iff w < (erased ? 2^31 : thr(p_k)).
// Every draw is made.  Lanes take locations from a work list sorted by n_l, work[i] = (l, m0, n_l, thr(e_l)), so that the
// lanes of a warp make the same number of calls; the result depends on l only.  One warp per shot; a fired mechanism with a
// column XORs that column of chk / obs into the shared-memory parity words (and its bit into the err words when err is
// requested); an erased location ORs its columns into the erased-column words when channel_llr is requested.
// channel_llr [B][num_col] = col_llr with 0.0 at the erased columns (no log on the device).
// ----------------------------------------------------------------------------------------------
__global__ void window_sample_circuit_kernel(const uint4 *__restrict__ work, int num_loc, const uint2 *__restrict__ mech,
                                             const double *__restrict__ col_llr, int num_col,
                                             const int *__restrict__ chk_cp, const int *__restrict__ chk_ri, int num_det,
                                             const int *__restrict__ obs_cp, const int *__restrict__ obs_ri, int num_obs,
                                             unsigned long long seed, long long shot0, long long B, u8 *__restrict__ det,
                                             u8 *__restrict__ obs, u8 *__restrict__ err, u8 *__restrict__ erased,
                                             double *__restrict__ channel_llr) {
    extern __shared__ u32 s_bits[];        // per warp: det, obs, [err], [erased columns] words
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int wd = (num_det + 31) >> 5, wo = (num_obs + 31) >> 5, wc = (num_col + 31) >> 5;
    const int we = err ? wc : 0, wx = channel_llr ? wc : 0, words = wd + wo + we + wx;
    u32 *dbits = s_bits + (size_t)wid * words, *obits = dbits + wd, *ebits = obits + wo, *xbits = ebits + we;
    for (long long b = (long long)blockIdx.x * wpb + wid; b < B; b += (long long)gridDim.x * wpb) {
        for (int i = lane; i < words; i += 32) dbits[i] = 0;
        __syncwarp();
        const unsigned long long shot = (unsigned long long)(shot0 + b);
        for (int i = lane; i < num_loc; i += 32) {
            const uint4 wk = work[i];                   // (l, m0, n_l, thr(e_l))
            const int n = (int)wk.z;
            bool er = false;
            for (int call = 0; 4 * call <= n; call++) {
                u32 r[4];
                philox4x32_10(wk.x, 2u + (u32)call, (u32)shot, (u32)(shot >> 32), (u32)seed, (u32)(seed >> 32), r);
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int t = 4 * call + q;
                    if (t > n) break;
                    if (t == 0) { er = r[0] < wk.w; continue; }
                    const uint2 m = mech[wk.y + t - 1];
                    const int c = (int)m.x;
                    if (c < 0) continue;
                    if (r[q] < (er ? 0x80000000u : m.y)) {
                        xor_column(c, chk_cp, chk_ri, dbits);
                        if (num_obs > 0) xor_column(c, obs_cp, obs_ri, obits);
                        if (err) atomicXor(&ebits[c >> 5], 1u << (c & 31));
                    }
                    if (er && channel_llr) atomicOr(&xbits[c >> 5], 1u << (c & 31));
                }
            }
            if (erased) erased[b * num_loc + wk.x] = (u8)er;
        }
        __syncwarp();
        for (int i = lane; i < num_det; i += 32) det[b * num_det + i] = (u8)((dbits[i >> 5] >> (i & 31)) & 1u);
        if (obs) for (int i = lane; i < num_obs; i += 32) obs[b * num_obs + i] = (u8)((obits[i >> 5] >> (i & 31)) & 1u);
        if (err) for (int i = lane; i < num_col; i += 32) err[b * num_col + i] = (u8)((ebits[i >> 5] >> (i & 31)) & 1u);
        if (channel_llr)
            for (int i = lane; i < num_col; i += 32) channel_llr[b * num_col + i] = ((xbits[i >> 5] >> (i & 31)) & 1u) ? 0.0 : col_llr[i];
        __syncwarp();
    }
}

// ----------------------------------------------------------------------------------------------
// bit-packed shot I/O (SURVEY 7 step 1 / 8(b) "or bit-packed"): row b of `packed` holds ceil(nbits / 64) 64-bit words,
// bit j of the row = (word[j >> 6] >> (j & 63)) & 1 (numpy: packbits(bitorder="little") viewed as uint64).
// One warp per 1024 bits of a row: 32 coalesced 32-byte reads + ballots, one coalesced 128-byte store (and the reverse).
// ----------------------------------------------------------------------------------------------
__global__ void pack_bits_kernel(const u8 *__restrict__ bytes, long long B, int nbits, int words64, u32 *__restrict__ packed) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int segs = (words64 * 2 + 31) / 32;                   // segments of 32 32-bit words per row
    if (warp >= B * segs) return;
    const long long b = warp / segs; const int seg = (int)(warp % segs);
    const u8 *row = bytes + b * nbits;
    u32 mine = 0;
#pragma unroll 4
    for (int k = 0; k < 32; k++) {
        const int j = (seg * 32 + k) * 32 + lane;
        const u32 w = __ballot_sync(FULLMASK, j < nbits && row[j] != 0);
        if (lane == k) mine = w;
    }
    const int wi = seg * 32 + lane;
    if (wi < words64 * 2) packed[b * words64 * 2 + wi] = mine;
}

__global__ void unpack_bits_kernel(const u32 *__restrict__ packed, long long B, int nbits, int words64, u8 *__restrict__ bytes) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int segs = (words64 * 2 + 31) / 32;
    if (warp >= B * segs) return;
    const long long b = warp / segs; const int seg = (int)(warp % segs);
    const int wi = seg * 32 + lane;
    const u32 mine = (wi < words64 * 2) ? packed[b * words64 * 2 + wi] : 0u;
    u8 *row = bytes + b * nbits;
#pragma unroll 4
    for (int k = 0; k < 32; k++) {
        const u32 w = __shfl_sync(FULLMASK, mine, k);
        const int j = (seg * 32 + k) * 32 + lane;
        if (j < nbits) row[j] = (u8)((w >> lane) & 1u);
    }
}
