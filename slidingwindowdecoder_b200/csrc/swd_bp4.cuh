// swd_bp4.cuh — quaternary (X / Y / Z) min-sum BP over the pair (Hx, Hz) of a CSS code: the BP stage of the
// reference's bp4_osd decoder (src/bp4_osd.pyx:425-591).  One CTA per shot; the check-to-bit / bit-to-check messages
// of both graphs live in two shared-memory arrays (in place, as in pre_bp_kernel), the three posterior LLRs per
// qubit go to HBM once per iteration.  The OSD stage re-uses osd_kernel (swd_osd.cuh) once per basis.
#pragma once
#include "swd_device.cuh"

struct Bp4Smem { int off_mx, off_mz, off_ux, off_uz, off_sx, off_sz, total; };

// bpgd.cpp:399-416
__device__ __forceinline__ double b4_log1pexp(double x) {
    if (x > 36.04365338911715) return x + log1p(exp(-x));          // -log(DBL_EPSILON)
    return log1p(exp(x));
}
__device__ __forceinline__ double b4_logaddexp(double x, double y) {
    const double tmp = x - y;
    if (x == y) return x + 0.69314718055994530942;
    if (tmp > 0) return x + b4_log1pexp(-tmp);
    return y + b4_log1pexp(tmp);
}

// bp4_osd.cn_update_all (pyx:483-529) for one check row: min1 / min2 / argmin / parity form of the reference's
// prefix / suffix sweep (identical values, incl. the 1e308 sentinel of a degree-1 check)
__device__ __forceinline__ void b4_row_update(double *msg, int p0, int p1, u32 par, double alpha) {
    double m1 = SWD_BIG, m2 = SWD_BIG; int arg = -1;
    for (int p = p0; p < p1; p++) {
        const double b = msg[p];
        double a = fabs(b);
        a = (a > SWD_CLIP) ? SWD_CLIP : a;
        const bool lt = a < m1;
        const double hi = lt ? m1 : a;
        m2 = (hi < m2) ? hi : m2;
        m1 = lt ? a : m1;
        arg = lt ? p : arg;
        par ^= (u32)(b <= 0.0);
    }
    const double q1 = m1 * alpha, q2 = m2 * alpha;
    for (int p = p0; p < p1; p++) {
        const double b = msg[p];
        msg[p] = flip_sign((p == arg) ? q2 : q1, par ^ (u32)(b <= 0.0));
    }
}

// CAMEL = true: bp4_osd.camel_decode (pyx:223-248) - an item is (shot, value), value = 0..3 = I / X / Z / Y pinned on the last
// qubit (vn_set_value, pyx:389-423): the pinned qubit is skipped by the variable pass, its bit-to-check messages keep their
// initial value, and its contribution to the checks is folded into the syndrome (seed of the check pass = current_cn;
// H.dec == s  <=>  H_rest.dec_rest == s ^ H_fix.dec_fix).  Per item: converge flag, iteration count, hard decision and the
// path metric cal_pm (pyx:250-259, ordered sum); the posteriors of the last run (value 3) go to lpr.
// SHOT = true: per-shot priors.  llrx / llry / llrz are then planes of [B][n] and the shot reads its own rows
// (plane + shot * n) in bp_init, the variable pass and cal_pm; CAMEL's pinned-qubit messages are computed per item.
template <bool CAMEL, bool SHOT = false>
__global__ void __launch_bounds__(256)
bp4_kernel(GraphDev gx, GraphDev gz, const double *__restrict__ llrx, const double *__restrict__ llry, const double *__restrict__ llrz,
           const u8 *__restrict__ synd_x, const u8 *__restrict__ synd_z, long long B, int max_iter, double alpha,
           u8 *__restrict__ bp_dec /*[B][2n]*/, u8 *__restrict__ conv_out, int *__restrict__ iter_out, double *__restrict__ lpr /*[B][n][3]*/,
           double *__restrict__ key_x /*[B][n]*/, double *__restrict__ key_z, Bp4Smem S, double *__restrict__ pm_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    double *mx = (double *)(smem + S.off_mx), *mz = (double *)(smem + S.off_mz);
    u32 *ux = (u32 *)(smem + S.off_ux), *uz = (u32 *)(smem + S.off_uz);
    u8 *sx = smem + S.off_sx, *sz = smem + S.off_sz;
    const int T = blockDim.x, tid = threadIdx.x;
    const int n = gx.n, nmx = gx.m, nmz = gz.m;
    const long long items = CAMEL ? 4 * B : B;
    const int fix = CAMEL ? n - 1 : -1;
    double fix_mx = 0.0, fix_mz = 0.0;
    if (CAMEL && !SHOT) {
        const double lx = llrx[fix], ly = llry[fix], lz = llrz[fix];
        fix_mx = b4_log1pexp(-1. * lx) - b4_logaddexp(-1. * ly, -1. * lz);
        fix_mz = b4_log1pexp(-1. * lz) - b4_logaddexp(-1. * ly, -1. * lz);
    }
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const long long shot = CAMEL ? (item >> 2) : item;
        const int value = CAMEL ? (int)(item & 3) : 0;
        const double *Lx = SHOT ? llrx + (size_t)shot * n : llrx, *Ly = SHOT ? llry + (size_t)shot * n : llry;
        const double *Lz = SHOT ? llrz + (size_t)shot * n : llrz;
        if (CAMEL && SHOT) {
            const double lx = Lx[fix], ly = Ly[fix], lz = Lz[fix];
            fix_mx = b4_log1pexp(-1. * lx) - b4_logaddexp(-1. * ly, -1. * lz);
            fix_mz = b4_log1pexp(-1. * lz) - b4_logaddexp(-1. * ly, -1. * lz);
        }
        for (int r = tid; r < nmx; r += T) sx[r] = synd_x[shot * nmx + r];
        for (int r = tid; r < nmz; r += T) sz[r] = synd_z[shot * nmz + r];
        if (CAMEL) {
            __syncthreads();
            if (value >> 1) for (int e = gx.cp[fix] + tid; e < gx.cp[fix + 1]; e += T) sx[gx.cr[e]] ^= 1;     // z part toggles the Hx checks
            if (value & 1) for (int e = gz.cp[fix] + tid; e < gz.cp[fix + 1]; e += T) sz[gz.cr[e]] ^= 1;      // x part toggles the Hz checks
        }
        for (int v = tid; v < n; v += T) {                                     // bp_init, pyx:425-442
            const double lx = Lx[v], ly = Ly[v], lz = Lz[v];
            const double msg_x = b4_log1pexp(-1. * lx) - b4_logaddexp(-1. * ly, -1. * lz);
            const double msg_z = b4_log1pexp(-1. * lz) - b4_logaddexp(-1. * ly, -1. * lz);     // sic (pyx:438)
            for (int e = gx.cp[v]; e < gx.cp[v + 1]; e++) mx[gx.cpos[e]] = msg_x;
            for (int e = gz.cp[v]; e < gz.cp[v + 1]; e++) mz[gz.cpos[e]] = msg_z;
        }
        __syncthreads();
        int conv = 0, it = 0;
        double *lp = lpr + (size_t)shot * n * 3;
        const bool write_lp = !CAMEL || value == 3;
        u8 *bx = bp_dec + (size_t)item * 2 * n, *bz = bx + n;
        if (CAMEL && tid == 0) {
            bx[fix] = (u8)(value & 1); bz[fix] = (u8)(value >> 1);
            if (write_lp) { lp[3 * fix] = 0.0; lp[3 * fix + 1] = 0.0; lp[3 * fix + 2] = 0.0; }
        }
        for (int iter = 0; iter < max_iter; iter++) {
            it++;
            for (int r = tid; r < nmx + nmz; r += T) {                         // cn_update_all('x'), ('z')
                if (r < nmx) { ux[r] = 0; b4_row_update(mx, gx.rp[r], gx.rp[r + 1], sx[r] == 1, alpha); }
                else { const int q = r - nmx; uz[q] = 0; b4_row_update(mz, gz.rp[q], gz.rp[q + 1], sz[q] == 1, alpha); }
            }
            __syncthreads();
            for (int v = tid; v < n; v += T) {                                 // vn_update, pyx:533-591
                if (CAMEL && v == fix) continue;
                const int x0 = gx.cp[v], x1 = gx.cp[v + 1], z0 = gz.cp[v], z1 = gz.cp[v + 1];
                double llrx_hx = 0.0, llrz_hz = 0.0;
                for (int e = z0; e < z1; e++) llrx_hx += mz[gz.cpos[e]];
                for (int e = x0; e < x1; e++) llrz_hz += mx[gx.cpos[e]];
                const double llry_all = llrx_hx + llrz_hz + Ly[v];
                llrx_hx = llrx_hx + Lx[v];
                llrz_hz = llrz_hz + Lz[v];
                if (write_lp) { lp[3 * v] = llrx_hx; lp[3 * v + 1] = llry_all; lp[3 * v + 2] = llrz_hz; }
                int idx;
                if (0 < llrx_hx && 0 < llry_all && 0 < llrz_hz) idx = 0;
                else if (llrx_hx < llry_all && llrx_hx < llrz_hz) idx = 1;
                else if (llry_all > llrz_hz) idx = 2;
                else idx = 3;
                const int ex = idx & 1, ez = idx >> 1;
                bx[v] = (u8)ex; bz[v] = (u8)ez;
                if (ez) for (int e = x0; e < x1; e++) atomicXor(&ux[gx.cr[e]], 1u);     // Hx . bp_decoding_z
                if (ex) for (int e = z0; e < z1; e++) atomicXor(&uz[gz.cr[e]], 1u);     // Hz . bp_decoding_x
                const double num_hx = b4_log1pexp(-1. * llrx_hx);
                for (int e = x0; e < x1; e++) {
                    const int p = gx.cpos[e];
                    const double msg = mx[p];
                    mx[p] = num_hx - b4_logaddexp(-1. * (llrz_hz - msg), -1. * (llry_all - msg));
                }
                const double num_hz = b4_log1pexp(-1. * llrz_hz);
                for (int e = z0; e < z1; e++) {
                    const int p = gz.cpos[e];
                    const double msg = mz[p];
                    mz[p] = num_hz - b4_logaddexp(-1. * (llrx_hx - msg), -1. * (llry_all - msg));
                }
            }
            if (CAMEL) {                                                       // the pinned qubit keeps its initial messages
                for (int e = gx.cp[fix] + tid; e < gx.cp[fix + 1]; e += T) mx[gx.cpos[e]] = fix_mx;
                for (int e = gz.cp[fix] + tid; e < gz.cp[fix + 1]; e += T) mz[gz.cpos[e]] = fix_mz;
            }
            __syncthreads();
            int mism = 0;
            for (int r = tid; r < nmx + nmz; r += T) mism |= (r < nmx) ? (ux[r] != (u32)sx[r]) : (uz[r - nmx] != (u32)sz[r - nmx]);
            if (!__syncthreads_or(mism)) { conv = 1; break; }
        }
        if (tid == 0) { conv_out[item] = (u8)conv; iter_out[item] = it; }
        if (CAMEL) {
            if (conv && tid == 0) {                                            // cal_pm, pyx:250-259
                double pm = 0.0;
                for (int v = 0; v < n; v++) {
                    const int ex = bx[v], ez = bz[v];
                    if (ex && ez) pm += Ly[v];
                    else if (ex) pm += Lx[v];
                    else if (ez) pm += Lz[v];
                }
                pm_out[item] = pm;
            }
        } else if (!conv) {                                                           // OSD ranking keys, pyx:280,297
            for (int v = tid; v < n; v += T) {
                const double lx = lp[3 * v], ly = lp[3 * v + 1], lz = lp[3 * v + 2];
                key_x[(size_t)shot * n + v] = b4_log1pexp(-1. * lx) - b4_logaddexp(-1. * ly, -1. * lz);
                key_z[(size_t)shot * n + v] = b4_log1pexp(-1. * lz) - b4_logaddexp(-1. * ly, -1. * lx);
            }
        }
        __syncthreads();
    }
}

// camel_decode (pyx:229-245): the converged run with the smallest path metric in the order I, X, Z, Y (strict <, start 10000);
// zeros when no run converged (the reference returns the buffer of an earlier call)
__global__ void bp4_camel_finish_kernel(const u8 *__restrict__ bp_dec /*[4B][2n]*/, const u8 *__restrict__ conv4, const double *__restrict__ pm4,
                                        const int *__restrict__ it4, long long B, int n, u8 *__restrict__ dec, u8 *__restrict__ conv,
                                        double *__restrict__ min_pm, int *__restrict__ iters) {
    const int warps = (gridDim.x * blockDim.x) >> 5, lane = threadIdx.x & 31;
    for (long long b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < B; b += warps) {
        double best = 10000.0; int arg = -1;
        for (int v = 0; v < 4; v++) if (conv4[4 * b + v] && pm4[4 * b + v] < best) { best = pm4[4 * b + v]; arg = v; }
        const u8 *src = bp_dec + (size_t)(4 * b + (arg < 0 ? 0 : arg)) * 2 * n;
        for (int i = lane; i < 2 * n; i += 32) dec[(size_t)b * 2 * n + i] = (arg < 0) ? (u8)0 : src[i];
        if (lane == 0) { conv[b] = (u8)(best < 9999.0); min_pm[b] = best; iters[b] = it4[4 * b + 3]; }
    }
}

// workspace set-up for an OSD-only pass: every shot is a slot; converged shots are skipped
__global__ void bp4_osd_setup_kernel(Workspace ws, u8 *need_osd, const double *__restrict__ keys, const u8 *__restrict__ conv, long long B, int n) {
    const long long total = B * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) ws.sum[i] = keys[i];
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        ws.gdg_list[b] = (int)b; need_osd[b] = conv[b] ? 0 : 1;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) ws.counters[0] = (int)B;
}

// final assembly (pyx:204-219): converged shots return the BP decoding (osd0 = BP decoding), the others the OSD results
// of the opposite basis: osd('x') on Hx gives the z part, osd('z') on Hz the x part
__global__ void bp4_finish_kernel(const u8 *__restrict__ bp_dec, const u8 *__restrict__ conv, const u8 *__restrict__ osdw_from_x,
                                  const u8 *__restrict__ osd0_from_x, const u8 *__restrict__ osdw_from_z, const u8 *__restrict__ osd0_from_z,
                                  long long B, int n, u8 *__restrict__ dec, u8 *__restrict__ osd0) {
    const long long total = B * 2 * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / (2 * n); const int c = (int)(i - b * 2 * n);
        u8 d, o;
        if (conv[b]) { d = bp_dec[i]; o = d; }
        else if (c < n) { d = osdw_from_z[b * n + c]; o = osd0_from_z[b * n + c]; }
        else { d = osdw_from_x[b * n + (c - n)]; o = osd0_from_x[b * n + (c - n)]; }
        dec[i] = d;
        if (osd0) osd0[i] = o;
    }
}
