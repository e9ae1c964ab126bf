// swd_api.cu — host side of libswd_b200.so: the C-ABI declared in include/swd_b200.h.
// Builds the flat graph, sizes the per-batch workspace, launches the kernel pipeline.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <vector>
#include <string>
#include <mutex>

#include "../../include/swd_b200.h"
#include "swd_kernels.cuh"
#include "swd_stream.cuh"
#include "swd_osd.cuh"
#include "swd_window.cuh"
#include "swd_bp4.cuh"

static thread_local std::string g_last_error;
static void set_err(const std::string &s) { g_last_error = s; }
#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) {                                                                          \
            set_err(std::string(#call) + ": " + cudaGetErrorString(e_));                                  \
            return SWD_ERR_CUDA;                                                                          \
        }                                                                                                 \
    } while (0)

// Owns one device allocation of T[cap], freed on destruction (on the current device: the destroy entry points select the
// handle's).  reserve() only grows it and discards the old contents; the raw-pointer views that kernels take by value
// (GraphDev, Workspace, StreamWs, OsdWork) are re-pointed after it.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
    ~DevBuf() { release(); }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    // A refused allocation leaves the buffer empty and clears the runtime's last error, which would otherwise fail the next
    // cudaGetLastError check of this or any other handle.
    int reserve(size_t count) {
        if (count <= cap) return SWD_OK;
        release();
        const size_t bytes = std::max<size_t>(16, count * sizeof(T));
        const cudaError_t e = cudaMalloc((void **)&p, bytes);
        if (e != cudaSuccess) {
            p = nullptr;
            cudaGetLastError();
            set_err("cudaMalloc(" + std::to_string(bytes) + " bytes): " + cudaGetErrorString(e));
            return SWD_ERR_NOMEM;
        }
        cap = count;
        return SWD_OK;
    }
    // a fresh allocation holding v; an empty v still gets one (a table pointer is never null)
    int upload(const std::vector<T> &v) {
        release();
        const int st = reserve(std::max<size_t>(1, v.size()));
        if (st) return st;
        CK(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
        return SWD_OK;
    }
};

static inline int r16(int x) { return (x + 15) & ~15; }
static inline int r32up(int x) { return (x + 31) & ~31; }

typedef void (*path_fn_t)(Workspace, SubLayout, SubLayout, PathSmem, GdgDev, int, int, int);
static path_fn_t pick_path_kernel(int dmax, int T) {
    if (dmax == 6) {
#ifndef SWD_MINB
#define SWD_MINB (SWD_DIET ? 8 : 7)
#endif
        if (T <= 128) return path_kernel<4, 6, 128, SWD_MINB>;
#ifndef SWD_MINB320
#define SWD_MINB320 3      /* 64 registers, three CTAs per SM: C4 post-BP -4.5 % (A/B r2) */
#endif
        if (T <= 320) return path_kernel<4, 6, 320, SWD_MINB320>;          // e.g. 576 x 4896 windows (new_n = 1152): two CTAs per SM
        if (T <= 512) return path_kernel<4, 6, 512, 1>;
        return path_kernel<4, 6, 1024, 1>;
    }
    if (T <= 128) return path_kernel<4, 16, 128, 3>;
    return path_kernel<4, 16, 1024, 1>;
}

typedef void (*pre_fn_t)(GraphDev, const u8 *, long long, int, double, u8 *, u8 *, Workspace, double *, int, PreSmem, int *, double *);
struct PreFns { pre_fn_t f, f_llr; };     // a pre-BP instantiation and its per-shot-prior twin
struct swd_decoder {
    swd_config cfg;
    path_fn_t path_fn = nullptr;
    pre_fn_t pre_fn = nullptr;
    pre_fn_t pre_fn_llr = nullptr; int grid1_llr = 0;     // per-shot priors (the *_llr entry points)
    int m = 0, n = 0, nnz = 0, nn = 0, max_col_deg = 0, max_row_deg = 0, es_max = 0, rank = -1;
    bool osd_only = false;
    int device = 0, num_sm = 0;
    GraphDev g{};               // views of the graph arrays below
    DevBuf<int> g_rp, g_cp;
    DevBuf<u16> g_rc, g_cr, g_cpos, g_vord, g_rowof, g_cpj;
    DevBuf<u32> g_vrec, g_prow;
    DevBuf<double> g_llr, g_llr_s, g_c2b1;
    int nphys = 0;              // message slots of the pre-BP kernel's physical layout (>= nnz)
    SubLayout L{}, LsA{}, LsB{};
    PathSmem PS{}, PSB{};
    int es_capA = 0, grid3B = 0;
    // latency configuration (tiny batches): a branch path spread over one VN per thread
    path_fn_t path_fn_lat = nullptr; int T3lat = 0, grid3lat = 0;
    PreSmem PRE{};
    // graphs whose messages exceed one SM's shared memory: HBM-streamed full-window BP (swd_stream.cuh)
    bool stream_mode = false; int Ts = 256; size_t stream_smem = 0; StreamWs sw{}; DevBuf<unsigned char> sw_block; long long sw_G = 0;
    DevBuf<double> sw_llrT;     // per-shot priors of a tile, [n][G] (allocated by the first per-shot call)
    SortSmem SS{};
    OsdSmem OS{};
    GdgDev P{};
    GdgDev Plat{};            // the same with the node-snapshot stride of the latency configuration (T3lat threads of history)
    int T1 = 0, T2 = 0, T3 = 0, T5 = 0, dmax = 8;
    int grid1 = 0, grid2 = 0, grid3 = 0, grid5 = 0;
    // workspace
    long long cap = 0;            // shots per chunk
    Workspace ws{};             // views of ws_block
    DevBuf<double> hscratch;
    OsdWork ow{};               // views of the osd_* buffers and of ws_block
    DevBuf<unsigned char> ws_block;
    DevBuf<u8> osd_bp_dec, osd_osd0, osd_osdw, osd_scratch;
    DevBuf<double> osd_lpr;
    DevBuf<int> osd_bp_iter;
    // staging for the host and packed entry points
    DevBuf<u8> d_synd, d_corr, d_conv; DevBuf<double> d_pm; DevBuf<u64> d_psynd, d_pcorr;
    DevBuf<double> d_llr;       // one chunk of host per-shot priors (swd_decode_batch_host*_llr)
    cudaStream_t stream = nullptr;
    // accumulated counters
    swd_counters ctr{};
    long long last_B = 0;
    // optional per-kernel event timing
    bool profiling = false;
    struct EvPair { cudaEvent_t a, b; int k; };
    std::vector<EvPair> ev_used;
    std::vector<cudaEvent_t> ev_free;
    cudaEvent_t ev_get() {
        if (!ev_free.empty()) { cudaEvent_t e = ev_free.back(); ev_free.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    ~swd_decoder() {
        for (auto &e : ev_used) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
        for (auto &e : ev_free) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
};

struct KTimer {     // brackets one launch with events when profiling is on
    swd_decoder *d; cudaStream_t s; int k; cudaEvent_t a = nullptr;
    KTimer(swd_decoder *d_, cudaStream_t s_, int k_) : d(d_), s(s_), k(k_) {
        if (d->profiling) { a = d->ev_get(); cudaEventRecord(a, s); }
    }
    ~KTimer() {
        if (d->profiling) { cudaEvent_t b = d->ev_get(); cudaEventRecord(b, s); d->ev_used.push_back({a, b, k}); }
    }
};

extern "C" const char *swd_version(void) { return "swd_b200 0.1 (sm_100a)"; }
extern "C" const char *swd_last_error(void) { return g_last_error.c_str(); }
extern "C" const char *swd_strerror(int s) {
    switch (s) {
        case SWD_OK: return "ok";
        case SWD_ERR_INVALID: return "invalid argument";
        case SWD_ERR_UNSUPPORTED: return "unsupported configuration";
        case SWD_ERR_CUDA: return "CUDA error";
        case SWD_ERR_NOMEM: return "out of memory";
    }
    return "unknown";
}

// GF(2) rank of the pcm (what mod2sparse_rank returns, mod2sparse_extra.cpp:32-76), dense bit-packed.
static int host_rank(int m, int n, const std::vector<int> &cp, const std::vector<int> &cr) {
    const int W = (m + 63) / 64;
    std::vector<std::vector<uint64_t>> basis;
    std::vector<int> prow;
    std::vector<uint64_t> v(W);
    for (int c = 0; c < n && (int)basis.size() < std::min(m, n); c++) {
        std::fill(v.begin(), v.end(), 0);
        for (int e = cp[c]; e < cp[c + 1]; e++) v[cr[e] >> 6] ^= 1ull << (cr[e] & 63);
        for (size_t i = 0; i < basis.size(); i++)
            if ((v[prow[i] >> 6] >> (prow[i] & 63)) & 1) for (int w = 0; w < W; w++) v[w] ^= basis[i][w];
        int pr = -1;
        for (int w = 0; w < W && pr < 0; w++) if (v[w]) pr = w * 64 + __builtin_ctzll(v[w]);
        if (pr >= 0) { basis.push_back(v); prow.push_back(pr); }
    }
    return (int)basis.size();
}

// The flat graph of a CSC parity-check matrix whose rows may come in any order inside a column: the CSC with ascending rows,
// the CSR with ascending columns (mod2sparse.c:358-432), the CSR position of every CSC entry, and the columns in descending
// degree order (stable).
struct FlatGraph {
    std::vector<int> cp, cr, rp, rc, cpos;
    std::vector<u16> vord;
    int max_col_deg = 0, max_row_deg = 0;
};
// Returns nullptr, or what is malformed.  The caller has checked colptr[0] == 0 and 0 <= colptr[n] <= 65535.
static const char *flat_graph(int m, int n, const int32_t *colptr, const int32_t *rowidx, FlatGraph &G) {
    const int nnz = colptr[n];
    G.cp.assign(colptr, colptr + n + 1); G.cr.assign(nnz, 0); G.rp.assign(m + 1, 0); G.rc.assign(nnz, 0); G.cpos.assign(nnz, 0);
    for (int c = 0; c < n; c++) {
        if (G.cp[c + 1] < G.cp[c]) return "colptr not monotone";
        std::vector<int> rows(rowidx + G.cp[c], rowidx + G.cp[c + 1]);
        std::sort(rows.begin(), rows.end());
        for (size_t k = 0; k < rows.size(); k++) {
            if (rows[k] < 0 || rows[k] >= m || (k && rows[k] == rows[k - 1])) return "bad row index";
            G.cr[G.cp[c] + k] = rows[k]; G.rp[rows[k] + 1]++;
        }
        G.max_col_deg = std::max(G.max_col_deg, (int)rows.size());
    }
    for (int r = 0; r < m; r++) { G.max_row_deg = std::max(G.max_row_deg, G.rp[r + 1]); G.rp[r + 1] += G.rp[r]; }
    std::vector<int> fill(G.rp.begin(), G.rp.end() - 1);
    for (int c = 0; c < n; c++) for (int e = G.cp[c]; e < G.cp[c + 1]; e++) { const int p = fill[G.cr[e]]++; G.rc[p] = c; G.cpos[e] = p; }
    std::vector<int> idx(n);
    for (int c = 0; c < n; c++) idx[c] = c;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return G.cp[a + 1] - G.cp[a] > G.cp[b + 1] - G.cp[b]; });
    G.vord.assign(idx.begin(), idx.end());
    return nullptr;
}

static int setup_kernels(swd_decoder *d);
static int alloc_workspace(swd_decoder *d, long long want_cap, cudaStream_t s);

static int create_impl(const swd_config *cfg, int m, int n, const int32_t *colptr, const int32_t *rowidx,
                       const double *channel_llr, swd_decoder **out, bool osd_only);

extern "C" int swd_create(const swd_config *cfg, int m, int n, const int32_t *colptr, const int32_t *rowidx,
                          const double *channel_llr, swd_decoder **out) {
    return create_impl(cfg, m, n, colptr, rowidx, channel_llr, out, false);
}

// Physical message layout of the pre-BP kernel (GraphDev::prow / cpj / c2b1 / rowof).  Static graph -> solved once per decoder:
//  * row starts: inside every aligned group of 16 rows (the rows a half-warp of the check pass owns) the starts fall on 16
//    distinct 8-byte banks - a few pad slots between rows;
//  * slot order inside a row (free: the check update does not depend on it): local search (pair swaps inside a row, non-worsening
//    moves accepted) on the number of extra shared-memory wavefronts of the variable pass, where the 16 ownership slots of a
//    half-warp touch their k-th edges together.  [[144,12,12]] (3,1) window: 3040 -> ~1570 wavefronts per iteration (ideal 1538).
// optimize = false: slots in CSR order without pads (SWD_PRE_NO_LAYOUT=1, for A/B runs).
struct PreLayout { int nphys = 0; std::vector<int> pstart, phys; int jb[17]; std::vector<u16> cpj; long long excess0 = 0, excess = 0; };
static void pre_layout(int m, int n, int nnz, const std::vector<int> &cp, const std::vector<int> &cr, const std::vector<int> &rp,
                       const std::vector<int> &cpos, const std::vector<u16> &vord, bool optimize, PreLayout &L) {
    L.pstart.assign(m + 1, 0); L.phys.assign(std::max(nnz, 1), 0);
    {
        int pos = 0; unsigned used = 0;
        for (int r = 0; r < m; r++) {
            if ((r & 15) == 0) used = 0;
            if (optimize) while (used & (1u << (pos & 15))) pos++;
            used |= 1u << (pos & 15);
            L.pstart[r] = pos; pos += rp[r + 1] - rp[r];
        }
        L.pstart[m] = pos; L.nphys = pos;
    }
    if (L.nphys > 65535) {      // 16-bit slots: fall back to the unpadded order
        optimize = false;
        for (int r = 0; r <= m; r++) L.pstart[r] = rp[r];
        L.nphys = nnz;
    }
    std::vector<int> deg(n), gid(std::max(nnz, 1)), tpos(std::max(nnz, 1)), epos(std::max(nnz, 1));
    for (int sl = 0; sl < n; sl++) deg[sl] = cp[vord[sl] + 1] - cp[vord[sl]];            // descending
    int ng = 0;
    for (int h = 0; h * 16 < n; h++) {
        const int gb = ng; ng += deg[h * 16];
        for (int sl = h * 16; sl < std::min(n, h * 16 + 16); sl++) for (int k = 0; k < deg[sl]; k++) gid[cp[vord[sl]] + k] = gb + k;
    }
    for (int e = 0; e < nnz; e++) { epos[cpos[e]] = e; tpos[e] = cpos[e] - rp[cr[e]]; }
    std::vector<unsigned char> cnt((size_t)std::max(ng, 1) * 16, 0);
    for (int e = 0; e < nnz; e++) cnt[(size_t)gid[e] * 16 + ((L.pstart[cr[e]] + tpos[e]) & 15)]++;
    auto excess = [&]() { long long x = 0; for (unsigned char c : cnt) x += c > 1 ? c - 1 : 0; return x; };
    L.excess0 = L.excess = excess();
    if (optimize) {
        unsigned long long rng = 0x9e3779b97f4a7c15ull;
        long long best = L.excess0; int stale = 0;
        for (int sweep = 0; sweep < 64 && best > 0 && stale < 6; sweep++) {
            for (int r = 0; r < m; r++) {
                const int S = L.pstart[r], len = rp[r + 1] - rp[r];
                const int *E = &epos[rp[r]];
                for (int i = 0; i < len; i++) {
                    const int e = E[i], b = (S + tpos[e]) & 15, g = gid[e];
                    if (cnt[(size_t)g * 16 + b] <= 1) continue;
                    int bf_best = -1, bestd = 1, nzero = 0;
                    for (int j = 0; j < len; j++) {
                        const int f = E[j], bf = (S + tpos[f]) & 15, gf = gid[f];
                        if (bf == b || gf == g) continue;
                        const int d = -1 + (cnt[(size_t)g * 16 + bf] >= 1) - (cnt[(size_t)gf * 16 + bf] > 1) + (cnt[(size_t)gf * 16 + b] >= 1);
                        if (d < 0) { if (d < bestd) { bestd = d; bf_best = j; } }
                        else if (d == 0 && bestd >= 0) {            // no improving swap so far: keep one of the neutral ones at random
                            rng = rng * 6364136223846793005ull + 1442695040888963407ull;
                            if ((rng >> 33) % (unsigned)(++nzero) == 0) { bestd = 0; bf_best = j; }
                        }
                    }
                    if (bf_best >= 0 && bestd <= 0) {
                        const int f = E[bf_best], bf = (S + tpos[f]) & 15, gf = gid[f];
                        cnt[(size_t)g * 16 + b]--; cnt[(size_t)g * 16 + bf]++; cnt[(size_t)gf * 16 + bf]--; cnt[(size_t)gf * 16 + b]++;
                        std::swap(tpos[e], tpos[f]);
                    }
                }
            }
            const long long x = excess();
            if (x < best) { best = x; stale = 0; } else stale++;
        }
        L.excess = best;
    }
    for (int e = 0; e < nnz; e++) L.phys[e] = L.pstart[cr[e]] + tpos[e];
    // jagged-diagonal map in ownership-slot order
    L.cpj.assign(std::max(nnz, 1), 0);
    int o = 0;
    for (int k = 0; k < 17; k++) {
        L.jb[k] = o;
        if (k == 16) break;
        for (int sl = 0; sl < n && deg[sl] > k; sl++) L.cpj[o + sl] = (u16)L.phys[cp[vord[sl]] + k];
        int nk = 0; while (nk < n && deg[nk] > k) nk++;
        o += nk;
    }
}

// osd_only: the graph is used by osd_kernel alone (bp4_osd runs its own BP kernel) - no pre-BP / sort / path set-up and no
// column- or row-weight limit (CAMEL codes tie every check to the last qubit)
static int create_impl(const swd_config *cfg, int m, int n, const int32_t *colptr, const int32_t *rowidx,
                       const double *channel_llr, swd_decoder **out, bool osd_only) {
    if (!cfg || !colptr || !rowidx || !channel_llr || !out || m <= 0 || n <= 0) { set_err("swd_create: null/empty argument"); return SWD_ERR_INVALID; }
    if (cfg->kind < 0 || cfg->kind > 2) { set_err("swd_create: bad kind"); return SWD_ERR_INVALID; }
    if (cfg->bp_method != SWD_BP_MIN_SUM && cfg->bp_method != SWD_BP_PRODUCT_SUM) { set_err("swd_create: bad bp_method"); return SWD_ERR_INVALID; }
    const int nnz = colptr[n];
    if (colptr[0] != 0 || nnz < 0) { set_err("swd_create: bad colptr"); return SWD_ERR_INVALID; }
    if (n > 65534 || m > 65534 || nnz > 65535) { set_err("swd_create: graph too large for 16-bit indices"); return SWD_ERR_UNSUPPORTED; }
    FlatGraph G;
    if (const char *why = flat_graph(m, n, colptr, rowidx, G)) { set_err(std::string("swd_create: ") + why); return SWD_ERR_INVALID; }
    const std::vector<int> &cp = G.cp, &cr = G.cr, &rp = G.rp, &rc = G.rc, &cpos = G.cpos;
    const std::vector<u16> &vord = G.vord;
    swd_decoder *d = new swd_decoder();
    d->cfg = *cfg; d->m = m; d->n = n; d->nnz = nnz; d->device = cfg->device; d->osd_only = osd_only;
    d->max_col_deg = G.max_col_deg; d->max_row_deg = G.max_row_deg;
    if (osd_only && cfg->kind != SWD_KIND_OSD_WINDOW) { delete d; set_err("swd_create: bad kind"); return SWD_ERR_INVALID; }
    if (!osd_only && d->max_col_deg > 16) { delete d; set_err("swd_create: column weight > 16 unsupported"); return SWD_ERR_UNSUPPORTED; }
    if (!osd_only && d->max_row_deg > 255) { delete d; set_err("swd_create: row weight > 255 unsupported"); return SWD_ERR_UNSUPPORTED; }
    d->dmax = d->max_col_deg <= 8 ? 8 : 16;
    d->nn = (cfg->new_n <= 0) ? std::min(n, 2 * m) : std::min(cfg->new_n, n);
    {   // worst-case edge count of a shortened graph: the nn heaviest columns
        std::vector<int> deg(n);
        for (int c = 0; c < n; c++) deg[c] = cp[c + 1] - cp[c];
        std::sort(deg.begin(), deg.end(), std::greater<int>());
        long long s = 0; for (int j = 0; j < d->nn; j++) s += deg[j];
        d->es_max = (int)s;
    }
    if (cfg->kind == SWD_KIND_OSD_WINDOW) {
        d->rank = host_rank(m, n, cp, cr);
        int method = cfg->osd_method, order = cfg->osd_order;
        if (method == SWD_OSD_0) order = 0;
        if (order == -1 && method != SWD_OSD_0) { /* BP only: no OSD stage (osd_window.pyx:86,192) */ }
        else if (order < 0 || order > d->nn - d->rank) {     // osd_window.pyx:88-92
            delete d; set_err("swd_create: osd_order out of range 0..new_n-rank"); return SWD_ERR_INVALID;
        }
        if (method == SWD_OSD_E && order > 20) { delete d; set_err("swd_create: osd_e order > 20 unsupported"); return SWD_ERR_UNSUPPORTED; }
        d->cfg.osd_order = order;
    }
    if (cudaSetDevice(d->device) != cudaSuccess) { delete d; set_err("cudaSetDevice failed"); return SWD_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, d->device) != cudaSuccess) { delete d; set_err("cudaGetDeviceProperties failed"); return SWD_ERR_CUDA; }
    d->num_sm = prop.multiProcessorCount;
    std::vector<u16> cr16(cr.begin(), cr.end()), rc16(rc.begin(), rc.end()), cpos16(cpos.begin(), cpos.end());
    std::vector<double> llr(channel_llr, channel_llr + n);
    std::vector<u32> vrec(n);          // per ownership slot of the pre-BP kernel: first CSC entry | degree << 16
    std::vector<double> llr_s(n);
    for (int sl = 0; sl < n; sl++) {
        const int v = vord[sl];
        vrec[sl] = (u32)cp[v] | ((u32)(cp[v + 1] - cp[v]) << 16);
        llr_s[sl] = llr[v];
    }
    PreLayout PL;
    std::vector<u32> prow(std::max(m, 1));
    if (!osd_only) {
        pre_layout(m, n, nnz, cp, cr, rp, cpos, vord, !getenv("SWD_PRE_NO_LAYOUT"), PL);
        for (int r = 0; r < m; r++) prow[r] = (u32)PL.pstart[r] | ((u32)(rp[r + 1] - rp[r]) << 16);
        if (getenv("SWD_DEBUG")) fprintf(stderr, "[swd] pre-BP layout: nnz=%d slots=%d extra VN-pass wavefronts %lld -> %lld\n", nnz, PL.nphys, PL.excess0, PL.excess);
    } else { PL.nphys = nnz; PL.cpj.assign(std::max(nnz, 1), 0); for (int k = 0; k < 17; k++) PL.jb[k] = 0; }
    d->nphys = PL.nphys;
    int st;
    if ((st = d->g_prow.upload(prow)) || (st = d->g_cpj.upload(PL.cpj))) { swd_destroy(d); return st; }
    if ((st = d->g_rp.upload(rp)) || (st = d->g_rc.upload(rc16)) || (st = d->g_cp.upload(cp)) ||
        (st = d->g_cr.upload(cr16)) || (st = d->g_cpos.upload(cpos16)) || (st = d->g_llr.upload(llr)) ||
        (st = d->g_vord.upload(vord)) || (st = d->g_vrec.upload(vrec)) || (st = d->g_llr_s.upload(llr_s))) {
        swd_destroy(d); return st;
    }
    if (!osd_only && cfg->bp_method == SWD_BP_MIN_SUM && !getenv("SWD_NO_FIRST_PASS_TABLE")) {
        // the check pass of iteration 1 for syndrome 0, with the kernel's own arithmetic (osd / bpgd pyx:62-96)
        std::vector<double> t(std::max(PL.nphys, 1), 0.0); std::vector<u16> ro(std::max(PL.nphys, 1), 0);     // physical slot order
        std::vector<int> physof(std::max(nnz, 1));                                                          // CSR position -> physical slot
        for (int e = 0; e < nnz; e++) physof[cpos[e]] = PL.phys[e];
        const double alpha = cfg->ms_scaling_factor;
        for (int r = 0; r < m; r++) {
            double m1 = SWD_BIG, m2 = SWD_BIG; int arg = -1; unsigned par = 0;
            for (int p = rp[r]; p < rp[r + 1]; p++) {
                const double b = llr[rc[p]];
                double a = fabs(b); a = (a > SWD_CLIP) ? SWD_CLIP : a;
                const bool lt = a < m1; const double hi = lt ? m1 : a;
                m2 = (hi < m2) ? hi : m2; m1 = lt ? a : m1; arg = lt ? p : arg;
                par ^= (unsigned)(b <= 0.0);
            }
            const double q1 = m1 * alpha, q2 = m2 * alpha;
            for (int p = rp[r]; p < rp[r + 1]; p++) {
                const double b = llr[rc[p]];
                const double q = (p == arg) ? q2 : q1;
                t[physof[p]] = ((par ^ (unsigned)(b <= 0.0)) & 1u) ? -q : q;
                ro[physof[p]] = (u16)r;
            }
        }
        if ((st = d->g_c2b1.upload(t)) || (st = d->g_rowof.upload(ro))) { swd_destroy(d); return st; }
    }
    d->g.c2b1 = d->g_c2b1.p; d->g.rowof = d->g_rowof.p;     // nullptr without the first-pass table
    d->g.m = m; d->g.n = n; d->g.nnz = nnz;
    d->g.nphys = PL.nphys; d->g.prow = d->g_prow.p; d->g.cpj = d->g_cpj.p;
    for (int k = 0; k < 17; k++) d->g.jb[k] = PL.jb[k];
    d->g.rp = d->g_rp.p; d->g.rc = d->g_rc.p; d->g.cp = d->g_cp.p; d->g.cr = d->g_cr.p; d->g.cpos = d->g_cpos.p; d->g.llr = d->g_llr.p;
    d->g.vord = d->g_vord.p; d->g.vrec = d->g_vrec.p; d->g.llr_s = d->g_llr_s.p;
    if (cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) != cudaSuccess) { swd_destroy(d); set_err("stream create failed"); return SWD_ERR_CUDA; }
    if ((st = setup_kernels(d)) != SWD_OK) { swd_destroy(d); return st; }
    *out = d;
    return SWD_OK;
}

extern "C" void swd_destroy(swd_decoder *d) {
    if (!d) return;
    cudaSetDevice(d->device);
    delete d;
}

template <typename K>
static int occupancy(K kernel, int threads, size_t smem, int *out) {
    // opt in to the full 227 KB once: several decoders with different footprints share each kernel
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    int nb = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem));
    *out = nb;
    return SWD_OK;
}

// with_col = false: shared-memory image of the blob; `col` (needed only for the final scatter) stays in HBM
static void make_layout(SubLayout &L, int nn, int m, int es, int lcap, bool with_col = true) {
    // with_col = false: the shared-memory image.  With SWD_DIET it is a prefix of the global blob's fixed part (what the
    // min-sum iteration reads) plus vrow / vpos; the reset snapshot, col and cvn are read from the global blob.
    const bool image = !with_col;
    L.nn = nn; L.m = m; L.es_max = es; L.lcap = lcap;
    int o = 16;
    L.off_prior = o; o += 8 * nn; o = r16(o);
    L.off_voff = o; o += 2 * (nn + 1); o = r16(o);
    L.off_coff = o; o += 2 * (m + 1); o = r16(o);
    L.off_crank = o; o += 2 * m; o = r16(o);
    L.off_synd = o; o += m; o = r16(o);
    L.off_vperm = o; o += 2 * nn; o = r16(o);
    L.off_cperm = o; o += 2 * m; o = r16(o);
    const int prefix = o;
    L.off_vnmask = o; o += nn; o = r16(o);
    L.off_cnmask = o; o += m; o = r16(o);
    L.off_cndeg = o; o += m; o = r16(o);
    if (image && SWD_DIET) o = prefix;
    L.off_col = o; if (with_col) { o += 2 * nn; o = r16(o); }
    L.fixed_bytes = o;
    L.off_vrow = o; o += r16(2 * es);
    L.off_vpos = o; o += r16(2 * es);
    L.off_cvn = o; if (!(image && SWD_DIET)) o += r16(2 * es);
    L.blob_bytes = o;
}

static void make_path_smem(PathSmem &S3, int nn, int m, int es) {
    int o = 0;
    S3.off_msg = o; o += 8 * es; o = r16(o);
    S3.off_vnmask = o; o += nn; o = r16(o);
    S3.off_error = o; o += nn; o = r16(o);
    S3.off_dec = o; o += std::max(nn, 2 * m); o = r16(o);      // select_vn actions (i8[nn]) / active-check list of bp_run (u16[m])
    S3.off_cnmask = o; o += m; o = r16(o);
    S3.off_cndeg = o; o += m; o = r16(o);
    S3.off_flip = o; o += m; o = r16(o);
    S3.off_upar = o; o += 4 * m; o = r16(o);
    S3.off_bvn = o; if (!SWD_DIET) { o += nn; o = r16(o); }
    S3.off_bcn = o; if (!SWD_DIET) { o += m; o = r16(o); }
    S3.off_bdeg = o; if (!SWD_DIET) { o += m; o = r16(o); }
    S3.off_red = o; o += 64 * 8 + 64 * 4; o = r16(o);
    S3.off_misc = o; o += 64;
    S3.off_bar = o; o += 16;
    S3.total = o;
}

static int setup_kernels(swd_decoder *d) {
    const int m = d->m, n = d->n, nn = d->nn, es = std::max(d->es_max, 1);
    const bool osd_only = d->osd_only;
    const swd_config &c = d->cfg;
    // ---- GDG parameters
    GdgDev &P = d->P;
    P.kind = c.kind; P.multi_thread = c.multi_thread; P.low_error = (c.kind == SWD_KIND_BPGD) ? 0 : c.low_error_mode;
    P.num_iter = c.max_iter_per_step; P.max_step = c.max_step; P.T = c.max_tree_depth; P.S = c.max_side_depth;
    P.tree_step = c.max_tree_branch_step; P.side_step = c.max_side_branch_step; P.factor = c.gdg_factor;
    P.post_max_iter = c.post_max_iter;
    if (c.kind == SWD_KIND_BPGDG && c.multi_thread) {
        if (P.T < 0 || P.T > 10) { set_err("max_tree_depth out of range"); return SWD_ERR_UNSUPPORTED; }
        P.n_tree = (1 << P.T) - 1; P.n_side = std::max(0, P.S - P.T); P.n_rec = 1 + P.n_tree + P.n_side;
    } else if (c.kind == SWD_KIND_BPGDG) {
        // single-thread schedule: the side-snapshot area holds the guess stack (max_guess entries, pyx:181)
        if (P.T < 0 || P.T > 10) { set_err("max_tree_depth out of range"); return SWD_ERR_UNSUPPORTED; }
        P.n_tree = 0; P.n_side = std::max(0, ((1 << P.T) - 1) * 2 + P.S - P.T); P.n_rec = 1;
    } else { P.n_tree = 0; P.n_side = 0; P.n_rec = 1; }
    if (c.kind == SWD_KIND_OSD_WINDOW) { P.factor = c.ms_scaling_factor; P.low_error = 0; }
    P.rec_stride = r16((int)sizeof(RecHeader) + 4 * ((nn + 31) / 32));
    P.side_stride = r16((int)sizeof(SideHeader) + nn + 2 * m);
    P.shared_T = 0; P.n_nodes = 0; P.node_stride = 16; P.count_work = d->profiling ? 1 : 0;
    P.bak_stride = SWD_DIET ? r16(nn) + 2 * r16(m) : 16;
    // ---- blob layouts: global (worst case), shared-memory tier A (typical shots), tier B (worst case)
    const int lcap = std::min(255, d->max_row_deg);
    const int es_slots = es + m;      // every row may carry one pad slot
    make_layout(d->L, nn, m, osd_only ? 8 : es_slots, lcap);
    if (osd_only) {
        int st;
        if ((st = osd_setup(d->m, d->n, d->nn, d->rank, d->cfg.osd_method, d->cfg.osd_order, d->num_sm, &d->OS, &d->T5, &d->grid5))) {
            set_err("osd kernel does not fit in shared memory"); return st;
        }
        return SWD_OK;
    }
    // ---- K1
    d->T1 = std::min(256, std::max(64, r32up((n + 3) / 4)));
    if (const char *e = getenv("SWD_T1")) d->T1 = std::min(256, std::max(32, r32up(atoi(e))));
    PreSmem &S1 = d->PRE;
    int o = 0; S1.off_msg = o; o += 8 * std::max(d->nphys, 1); o = r16(o);
    S1.off_upar = o; o += 4 * m; o = r16(o);
    S1.off_synd = o; o += m; o = r16(o);
    S1.off_dec = o; o += n; o = r16(o);
    S1.off_misc = o; o += 64;
    S1.off_fwd = o;
    const bool ps = (c.bp_method == SWD_BP_PRODUCT_SUM);
    if (ps) { o = r16(o); S1.off_fwd = o; o += 8 * std::max(d->nphys, 1); }
    S1.total = o; S1.off_vrec = o; S1.off_cpos = o; S1.off_prow = o;
    if (S1.total > 227 * 1024 || getenv("SWD_FORCE_STREAM")) {
        // messages streamed from HBM, one thread per shot (swd_stream.cuh); syndrome + parity bit words per thread in shared memory
        if (ps) { set_err("product-sum BP: window graph does not fit in shared memory (nnz too large)"); return SWD_ERR_UNSUPPORTED; }
        const int MW = (m + 31) / 32;
        // shared memory per thread: the cp.async ring (SWD_SK doubles) + parity bit words; two CTAs per SM
        int ts = 256; while (ts > 32 && (size_t)(4 * MW + 8 * SWD_SK) * ts > (SWD_STREAM_MINB >= 3 ? 72 : 110) * 1024) ts -= 32;
        if ((size_t)(4 * MW + 8 * SWD_SK) * ts > 110 * 1024) { set_err("window graph has too many checks for the streamed BP kernel"); return SWD_ERR_UNSUPPORTED; }
        d->stream_mode = true; d->Ts = ts; d->stream_smem = (size_t)(4 * MW + 8 * SWD_SK) * ts;
        S1.total = 0;
    }
    // staged static graph info (per-slot records + CSC->CSR map) if it still fits next to the messages
    bool staged = false;
    {
        int q = r16(o); const int ov = q; q += 4 * n; q = r16(q); const int oc = q; q += 2 * std::max(d->nnz, 1); q = r16(q);
        const int opr = q; q += 4 * m; q = r16(q);
        // staging must not cost occupancy: 256-thread CTAs are register limited to 3 per SM, so compare at that count
        const int occ_unstaged = std::min(3, (int)(233472 / (S1.total + 1024))), occ_staged = std::min(3, (int)(233472 / (q + 1024)));
        if (q <= 227 * 1024 && occ_staged >= occ_unstaged && !getenv("SWD_PRE_UNSTAGED")) { staged = true; S1.off_vrec = ov; S1.off_cpos = oc; S1.off_prow = opr; S1.total = q; }
    }
    int occ = 0, st;
    if (!d->stream_mode) {
#define SWD_PRE_PICK(D, MT, MB, SH) (ps ? (staged ? pre_bp_kernel<D, MT, MB, true, true, SH> : pre_bp_kernel<D, MT, MB, true, false, SH>) \
                                        : (staged ? pre_bp_kernel<D, MT, MB, false, true, SH> : pre_bp_kernel<D, MT, MB, false, false, SH>))
#define SWD_PRE_BOTH(D, MT, MB) PreFns{SWD_PRE_PICK(D, MT, MB, false), SWD_PRE_PICK(D, MT, MB, true)}
    PreFns pf;
    if (ps) pf = d->max_col_deg <= 8 ? SWD_PRE_BOTH(8, 256, 2) : SWD_PRE_BOTH(16, 256, 2);
    else pf = d->max_col_deg <= 6 ? SWD_PRE_BOTH(6, 256, SWD_PRE_MINB) : (d->max_col_deg <= 8 ? SWD_PRE_BOTH(8, 256, SWD_PRE_MINB) : SWD_PRE_BOTH(16, 256, 2));
    st = occupancy(pf.f, d->T1, S1.total, &occ);
    if (st) return st;
    if (!ps && d->max_col_deg <= 8 && (int)(233472 / (S1.total + 1024)) > occ && !getenv("SWD_T1")) {
        // small windows: shared memory would allow more CTAs than the 3-per-SM register budget (85) of the default instantiation -
        // take the 64-register one when it raises the number of resident warps ([[72,12,6]] windows: 4 instead of 3 CTAs of 224 threads)
        PreFns f4 = d->max_col_deg <= 6 ? SWD_PRE_BOTH(6, 256, 4) : SWD_PRE_BOTH(8, 256, 4);
        int occ4 = 0;
        if ((st = occupancy(f4.f, d->T1, S1.total, &occ4))) return st;
        if (occ4 > occ) { pf = f4; occ = occ4; }
    }
    if (occ * d->T1 < 512 && !getenv("SWD_T1")) {
        // shared memory allows fewer than 16 warps per SM with 256-thread CTAs: use one large CTA per SM instead
        const int want = std::min(1024, std::max(256, r32up(std::max((n + 3) / 4, m))));
        PreFns big = d->max_col_deg <= 6 && !ps ? SWD_PRE_BOTH(6, 1024, 1) : (d->max_col_deg <= 8 ? SWD_PRE_BOTH(8, 1024, 1) : SWD_PRE_BOTH(16, 1024, 1));
        int occ_big = 0;
        if ((st = occupancy(big.f, want, S1.total, &occ_big))) return st;
        if (occ_big * want > occ * d->T1) { pf = big; d->T1 = want; occ = occ_big; }
    }
#undef SWD_PRE_BOTH
#undef SWD_PRE_PICK
    if (occ < 1) { set_err("pre_bp_kernel does not fit"); return SWD_ERR_UNSUPPORTED; }
    d->pre_fn = pf.f; d->pre_fn_llr = pf.f_llr;
    d->grid1 = d->num_sm * occ;
    // the per-shot twin: same CTA size and shared memory; its grid never exceeds grid1 (hscratch is sized for grid1 CTAs)
    int occ_llr = 0;
    if ((st = occupancy(pf.f_llr, d->T1, S1.total, &occ_llr))) return st;
    if (occ_llr < 1) { set_err("pre_bp_kernel (per-shot priors) does not fit"); return SWD_ERR_UNSUPPORTED; }
    d->grid1_llr = d->num_sm * std::min(occ, occ_llr);
    } else d->grid1 = d->num_sm;
    // ---- K2
    SortSmem &S2 = d->SS;
    int np2 = 64; while (np2 < n) np2 <<= 1;
    S2.np2 = np2;
    S2.cap_sel = 0;
    if (np2 >= 2048 && !getenv("SWD_FULL_SORT")) {
        int cap = 64; while (cap < nn + 64) cap <<= 1;
        if (cap <= np2 / 4) S2.cap_sel = cap;
    }
    d->T2 = std::min(1024, std::max(128, np2 / 8));
    if (const char *e = getenv("SWD_T2")) d->T2 = std::min(1024, std::max(64, r32up(atoi(e))));
    // n beyond the register sort (8 keys x 1024 threads): radix-select from global memory only, no full-sort fall-back, so
    // key / idx hold cap_sel entries instead of np2 (the un-windowed [[144,12,12]] DEM has n = 8784)
    S2.big = (np2 > 8192 || getenv("SWD_FORCE_BIG_SORT")) ? 1 : 0;
    int idx_entries = np2;
    S2.key_bytes = 8 * np2;
    if (S2.big) {
        int cap = 64; while (cap < nn + 64) cap <<= 1;
        S2.cap_sel = cap; idx_entries = cap;
        S2.key_bytes = r16(std::max(8 * cap, 4 * 2052));
    }
    auto sort_layout = [&](int key_bytes) {
        int o = 0; S2.off_key = o; o += key_bytes; S2.off_idx = o; o += 2 * idx_entries; o = r16(o);
        S2.off_posof = o; o += 2 * n; o = r16(o);
        S2.off_blob = o; o += d->L.blob_bytes;
        S2.off_u32a = o; o += 4 * (nn + 1); o = r16(o);
        S2.off_u32b = o; o += 4 * (m + 1); o = r16(o);
        S2.off_u32c = o; o += 4 * (m + 1); o = r16(o);
        S2.off_wt = o; o += 4 * 64;
        S2.off_error = o; o += nn; o = r16(o);
        S2.off_misc = o; o += 64;
        S2.off_bins = o; o += 4 * (17 + 256); o = r16(o);
        S2.total = o;
    };
    sort_layout(S2.key_bytes);
    if (S2.big && 2 * d->nnz > S2.key_bytes) {       // room for the CSR-position -> message-slot table (else: per-edge search)
        const int kb = r16(2 * d->nnz);
        sort_layout(kb);
        if (S2.total <= 227 * 1024) S2.key_bytes = kb; else sort_layout(S2.key_bytes);
    }
    if (S2.total > 227 * 1024) { set_err("sort/reset kernel does not fit in shared memory"); return SWD_ERR_UNSUPPORTED; }
    {   // the per-shot twin runs on the same grid (persistent CTAs stride over the work list)
        int occ_llr = 0;
        if ((st = occupancy(sort_reset_kernel<true>, d->T2, S2.total, &occ_llr))) return st;
        if (occ_llr < 1) { set_err("sort_reset_kernel (per-shot priors) does not fit"); return SWD_ERR_UNSUPPORTED; }
    }
    if ((st = occupancy(sort_reset_kernel<false>, d->T2, S2.total, &occ))) return st;
    if (occ < 1) { set_err("sort_reset_kernel does not fit"); return SWD_ERR_UNSUPPORTED; }
    d->grid2 = d->num_sm * occ;
    // ---- K3
    d->T3 = std::max(32, std::max(r32up((nn + 3) / 4), r32up((m + SWD_CPT - 1) / SWD_CPT)));
    if (d->T3 > 1024) { set_err("new_n > 4096 unsupported"); return SWD_ERR_UNSUPPORTED; }
    d->dmax = d->max_col_deg <= 6 ? 6 : (d->max_col_deg <= 8 ? 8 : 16);
    d->path_fn = pick_path_kernel(d->dmax, d->T3);
    // Tier A capacity: the largest that still allows the best occupancy, provided it covers the typical shortened
    // graph (the nn most error-prone columns are lighter than average: ~0.8 x mean degree measured on BB windows;
    // oversized shots fall to tier B, same kernel with the worst-case footprint, so this only affects speed).
    auto path_smem = [&](int cap) {
        SubLayout a; PathSmem b;
        make_layout(a, nn, m, cap, lcap, false); make_path_smem(b, nn, m, cap);
        return (size_t)a.blob_bytes + b.total;
    };
    const int typ = std::min(es_slots, (int)((double)nn * d->nnz / n * 0.85) + m / 2 + 16);
    int max_occ_threads = 1;                                   // limit set by registers / threads alone
    if ((st = occupancy(d->path_fn, d->T3, path_smem(8), &max_occ_threads))) return st;
    max_occ_threads = std::max(1, max_occ_threads);
    int capA = es_slots;
    for (int occ = max_occ_threads; occ >= 1; occ--) {
        const size_t budget = (size_t)233472 / occ - 1024;
        if (path_smem(8) > budget) continue;
        int lo = 8, hi = es_slots;
        while (lo < hi) { const int mid = (lo + hi + 1) / 2; if (path_smem(mid) <= budget) lo = mid; else hi = mid - 1; }
        const int cap = (lo == es_slots) ? lo : (lo & ~7);
        if (cap >= typ) { capA = std::min(es_slots, cap); break; }
    }
    if (const char *e = getenv("SWD_ES_TIER_A")) capA = std::min(es_slots, std::max(8, atoi(e)));
    d->es_capA = capA;
    make_layout(d->LsA, nn, m, capA, lcap, false);
    make_layout(d->LsB, nn, m, es_slots, lcap, false);
    make_path_smem(d->PS, nn, m, capA);
    make_path_smem(d->PSB, nn, m, es_slots);
    if (getenv("SWD_DEBUG")) fprintf(stderr, "[swd] m=%d n=%d nn=%d es_slots=%d typ=%d capA=%d smemA=%zu smemB=%zu\n", m, n, nn, es_slots, typ, capA,
                                     (size_t)d->LsA.blob_bytes + d->PS.total, (size_t)d->LsB.blob_bytes + d->PSB.total);
    const size_t smemB = (size_t)d->LsB.blob_bytes + d->PSB.total;
    if (smemB > 227 * 1024) { set_err("shortened graph does not fit in shared memory"); return SWD_ERR_UNSUPPORTED; }
    // the per-call VN records of bp_run pack (index < 4096, first edge < 32768, degree < 32) into one word; the shared-memory bound above
    // keeps es_slots far below that, this only states the invariant
    if (es_slots > 32767 || nn > 4096) { set_err("shortened graph too large for the packed VN records"); return SWD_ERR_UNSUPPORTED; }
    const size_t smemA = (size_t)d->LsA.blob_bytes + d->PS.total;
    if ((st = occupancy(d->path_fn, d->T3, smemA, &occ))) return st;
    if (occ < 1) { set_err("path_kernel does not fit"); return SWD_ERR_UNSUPPORTED; }
    d->grid3 = d->num_sm * occ;
    if ((st = occupancy(d->path_fn, d->T3, smemB, &occ))) return st;
    d->grid3B = d->num_sm * std::max(1, occ);
    // Latency configuration: with a handful of shots every branch path has an SM to itself, and what counts is the length of
    // one min-sum iteration on one CTA (tools/latency_probe.py: ~5 us with 128 threads, 97 % of the window latency is kernel
    // execution).  One VN per thread (one variable round instead of four, one check round) shortens it several times.
    d->T3lat = 0;
    if (c.kind != SWD_KIND_OSD_WINDOW && !getenv("SWD_NO_LATENCY_MODE")) {
        const int tl = std::min(1024, std::max(d->T3, r32up(nn)));
        if (tl > d->T3) {
            path_fn_t f = pick_path_kernel(d->dmax, tl);
            int occl = 0;
            if (occupancy(f, tl, smemB, &occl) == SWD_OK && occl >= 1) { d->path_fn_lat = f; d->T3lat = tl; d->grid3lat = d->num_sm * occl; }
        }
    }
    d->Plat = P;
    // shared-prefix tree (multi-thread GDG): depths 0..T-1 are computed once per decision prefix
    if (c.kind == SWD_KIND_BPGDG && c.multi_thread && P.T >= 1 && P.T <= 6 && P.max_step >= P.T && !getenv("SWD_NO_SHARED_PREFIX")) {
        P.shared_T = P.T; P.n_nodes = (1 << P.T) - 1;
        int q = (int)sizeof(NodeHeader);
        q += nn; q = r16(q); P.node_off_err = q;
        q += nn; q = r16(q); P.node_off_cn = q;
        q += m; q = r16(q); P.node_off_deg = q;
        q += m; q = r16(q); P.node_off_flip = q;
        q += m; q = r16(q); P.node_off_msg = q;
        q += 8 * es_slots; q = r16(q); P.node_off_hist = q;
        const int q_hist = q;
        q += 8 * 16 * d->T3; q = r16(q);
        P.node_stride = q;
        d->Plat = P;
        d->Plat.node_stride = r16(q_hist + 8 * 16 * std::max(d->T3, d->T3lat));
    }
    // ---- K5 (OSD)
    if (c.kind == SWD_KIND_OSD_WINDOW) {
        if ((st = osd_setup(d->m, d->n, d->nn, d->rank, d->cfg.osd_method, d->cfg.osd_order, d->num_sm, &d->OS, &d->T5, &d->grid5))) {
            set_err("osd kernel does not fit in shared memory"); return st;
        }
    }
    return SWD_OK;
}

static int alloc_workspace(swd_decoder *d, long long want, cudaStream_t s) {
    if (want <= d->cap) return SWD_OK;
    CK(cudaSetDevice(d->device));
    size_t budget = (size_t)16 << 30;     // per decoder; 180 GB of HBM3e per GPU
    if (const char *e = getenv("SWD_WS_BYTES")) budget = (size_t)atoll(e);
    const int n = d->n;
    const bool osd = d->cfg.kind == SWD_KIND_OSD_WINDOW;
    size_t per = (size_t)n * 8 + d->L.blob_bytes + (size_t)d->P.n_rec * d->P.rec_stride + (size_t)d->P.n_side * d->P.side_stride + 4 + 64 +
                 (size_t)d->P.n_nodes * d->P.node_stride + (size_t)std::max(1, std::max(d->P.n_tree + 1, d->P.n_side)) * SWD_WL_MAX * sizeof(u64) +
                 (size_t)std::max(1, d->P.n_tree) * d->P.bak_stride;
    if (osd) per += (size_t)n * 32 + osd_bytes_per_shot(d->m, n);
    long long cap = std::max<long long>(1, std::min<long long>(want, (long long)(budget / per)));
    if (cap <= d->cap) return SWD_OK;
    // growing the workspace: the accumulated work counters (ws.stats) survive the re-allocation
    u64 keep_stats[16];
    const bool have_stats = d->ws_block.p != nullptr;
    if (have_stats) {
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(keep_stats, d->ws.stats, sizeof(keep_stats), cudaMemcpyDeviceToHost));
    }
    d->cap = 0;
    auto a256 = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t o = 0;
    size_t o_cnt = o; o += a256(64 * sizeof(int));
    size_t o_stats = o; o += a256(16 * sizeof(u64));
    size_t o_list = o; o += a256((size_t)cap * 4);
    size_t o_sum = o; o += a256((size_t)cap * n * 8);
    size_t o_hist = o; if (osd) o += a256((size_t)cap * n * 32);
    size_t o_blob = o; o += a256((size_t)cap * d->L.blob_bytes);
    size_t o_rec = o; o += a256((size_t)cap * d->P.n_rec * d->P.rec_stride);
    size_t o_side = o; o += a256((size_t)cap * std::max(1, d->P.n_side) * d->P.side_stride);
    size_t o_node = o; o += a256(std::max((size_t)cap * std::max(1, d->P.n_nodes) * d->P.node_stride,
                                          (size_t)std::min<long long>(cap, 8) * std::max(1, d->P.n_nodes) * d->Plat.node_stride));
    size_t o_osd = o; if (osd) o += a256((size_t)cap * osd_bytes_per_shot(d->m, n));
    const long long wl_stride = cap * std::max(1, std::max(d->P.n_tree + 1, d->P.n_side));
    size_t o_bak = o; o += a256((size_t)cap * std::max(1, d->P.n_tree) * d->P.bak_stride);
    size_t o_wl = o; o += a256((size_t)wl_stride * SWD_WL_MAX * sizeof(u64));
    int st = d->ws_block.reserve(o);
    if (st) { d->ws = Workspace{}; return st; }
    // counters / stats / work list zeroed on the caller's stream (the kernels that use them are launched there)
    CK(cudaMemsetAsync(d->ws_block.p, 0, o_list, s));
    unsigned char *b = d->ws_block.p;
    d->ws.counters = (int *)(b + o_cnt); d->ws.stats = (u64 *)(b + o_stats); d->ws.gdg_list = (int *)(b + o_list);
    d->ws.sum = (double *)(b + o_sum); d->ws.hist = osd ? (double *)(b + o_hist) : nullptr;
    d->ws.blob = b + o_blob; d->ws.rec = b + o_rec; d->ws.side = b + o_side; d->ws.node = b + o_node;
    d->ws.wl = (u64 *)(b + o_wl); d->ws.wl_stride = wl_stride; d->ws.bak = b + o_bak;
    if (have_stats) CK(cudaMemcpyAsync(d->ws.stats, keep_stats, sizeof(keep_stats), cudaMemcpyHostToDevice, s));
    if (have_stats) CK(cudaStreamSynchronize(s));          // keep_stats is a stack buffer
    if (osd) osd_bind(&d->ow, b + o_osd, cap, d->m, n);
    if (osd && d->OS.big) {
        if ((st = d->osd_scratch.reserve((size_t)d->grid5 * d->OS.big_stride))) return st;
        d->ow.big_scratch = d->osd_scratch.p;
    }
    // four posterior rows per CTA, and a fifth for the per-shot twin's slot-ordered priors
    if (!d->stream_mode && (st = d->hscratch.reserve((size_t)d->grid1 * 5 * n))) return st;
    d->cap = cap;
    return SWD_OK;
}

static int pull_stats(swd_decoder *d, cudaStream_t s) {
    u64 h[16];
    CK(cudaMemcpyAsync(h, d->ws.stats, sizeof(h), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    d->ctr.pre_bp_edge_iters = h[0]; d->ctr.path_edge_iters = h[1]; d->ctr.paths_run = h[2]; d->ctr.bp_calls = h[3];
    d->ctr.osd_shots = h[4]; d->ctr.gdg_shots = h[5]; d->ctr.path_vn_iters = h[6]; d->ctr.path_cn_iters = h[7];
    d->ctr.path_slot_iters = h[8]; d->ctr.osd_cols_scanned = h[9]; d->ctr.osd_pivots = h[10];
    return SWD_OK;
}

// HBM-streamed full-window BP (graphs beyond one SM's shared memory): tiles of G = grid * Ts shots, one thread per shot
static int stream_pre_bp(swd_decoder *d, const GraphDev &g, const u8 *d_synd, long long B, u8 *d_corr, u8 *d_conv, int full_hist, int *iter_out,
                         double *lpr_out, cudaStream_t s) {
    const int Ts = d->Ts, n = d->n;
    size_t budget = (size_t)48 << 30;
    if (const char *e = getenv("SWD_STREAM_BYTES")) budget = (size_t)atoll(e);
    const size_t per_shot = (size_t)8 * (d->nnz + 4 * (size_t)n) + 4 * (size_t)((n + 31) / 32) + 4 * (size_t)((d->m + 31) / 32) + 8;
    typedef void (*sfn_t)(GraphDev, const u8 *, long long, long long, int, double, StreamWs, int, u64 *);
    const bool shot_llr = g.llr_shot != nullptr;
    sfn_t fn = shot_llr ? (d->max_col_deg <= 6 ? pre_bp_stream_kernel<6, true> : (d->max_col_deg <= 8 ? pre_bp_stream_kernel<8, true> : pre_bp_stream_kernel<16, true>))
                        : (d->max_col_deg <= 6 ? pre_bp_stream_kernel<6> : (d->max_col_deg <= 8 ? pre_bp_stream_kernel<8> : pre_bp_stream_kernel<16>));
    int socc = 0;
    { int st = occupancy(fn, Ts, d->stream_smem, &socc); if (st) return st; }
    if (socc < 1) { set_err("pre_bp_stream_kernel does not fit"); return SWD_ERR_UNSUPPORTED; }
    long long Gmax = (long long)d->num_sm * Ts * socc;                            // a tile = one resident wave
    Gmax = std::max<long long>(Ts, std::min<long long>(Gmax, (long long)(budget / per_shot) / Ts * Ts));
    const long long want = std::min<long long>(Gmax, (B + Ts - 1) / Ts * Ts);
    if (want > d->sw_G) {
        CK(cudaStreamSynchronize(s));
        d->sw_G = 0;
        auto a256 = [](size_t x) { return (x + 255) & ~(size_t)255; };
        size_t o = 0;
        const size_t o_msg = o; o += a256((size_t)8 * d->nnz * want);
        const size_t o_hs = o; o += a256((size_t)32 * n * want);
        const size_t o_dec = o; o += a256((size_t)4 * ((n + 31) / 32) * want);
        const size_t o_sy = o; o += a256((size_t)4 * ((d->m + 31) / 32) * want);
        const size_t o_it = o; o += a256((size_t)4 * want);
        const size_t o_cv = o; o += a256((size_t)want);
        if (int st = d->sw_block.reserve(o)) return st;
        unsigned char *b = d->sw_block.p;
        d->sw.msg = (double *)(b + o_msg); d->sw.hs = (double *)(b + o_hs); d->sw.decw = (u32 *)(b + o_dec);
        d->sw.itdone = (int *)(b + o_it); d->sw.conv = b + o_cv; d->sw.syndw = (u32 *)(b + o_sy);
        d->sw_G = want;
    }
    if (shot_llr && d->sw_llrT.cap < (size_t)n * d->sw_G) {
        CK(cudaStreamSynchronize(s));
        if (int st = d->sw_llrT.reserve((size_t)n * d->sw_G)) return st;
    }
    for (long long t0 = 0; t0 < B; t0 += d->sw_G) {
        const long long nb = std::min<long long>(d->sw_G, B - t0);
        StreamWs sw = d->sw; sw.G = (nb + Ts - 1) / Ts * Ts;
        if (shot_llr) {
            sw.llrT = d->sw_llrT.p;
            llr_transpose_kernel<<<dim3((unsigned)((n + 31) / 32), (unsigned)((nb + 31) / 32)), 256, 0, s>>>(g.llr_shot, B, t0, n, sw.G, d->sw_llrT.p);
            d->ctr.kernel_launches++;
        }
        fn<<<(unsigned)(sw.G / Ts), Ts, d->stream_smem, s>>>(g, d_synd, B, t0, d->cfg.max_iter, d->cfg.ms_scaling_factor, sw, full_hist, d->ws.stats);
        pre_bp_stream_finish_kernel<<<(unsigned)std::min<long long>((nb + 7) / 8, 8 * (long long)d->num_sm), 256, 0, s>>>(g, B, t0, sw, d_corr, d_conv, d->ws,
                                                                                                              iter_out, lpr_out);
        d->ctr.kernel_launches += 2;
    }
    CK(cudaGetLastError());
    return SWD_OK;
}

// one chunk (B <= cap), everything asynchronous on `s`.  d_llr: the chunk's per-shot priors [B][n] (device) or nullptr
static int launch_chunk(swd_decoder *d, const u8 *d_synd, long long B, u8 *d_corr, u8 *d_conv, double *d_pm, cudaStream_t s,
                        long long chunk_base, const double *d_llr) {
    const swd_config &c = d->cfg;
    GraphDev g = d->g;
    g.llr_shot = d_llr;
    CK(cudaMemsetAsync(d->ws.counters, 0, 64 * sizeof(int), s));
    const int g1 = (int)std::min<long long>(B, d_llr ? d->grid1_llr : d->grid1);
    const int full_hist = (c.kind == SWD_KIND_OSD_WINDOW) ? 1 : 0;
    int *iter_out = (c.kind == SWD_KIND_OSD_WINDOW) ? d->ow.bp_iter + chunk_base : nullptr;
    double *lpr_out = (c.kind == SWD_KIND_OSD_WINDOW) ? d->ow.lpr + (size_t)chunk_base * d->n * 4 : nullptr;
    if (d->stream_mode) {
        KTimer kt(d, s, SWD_K_PRE_BP);
        int st = stream_pre_bp(d, g, d_synd, B, d_corr, d_conv, full_hist, iter_out, lpr_out, s);
        if (st) return st;
    } else {
    KTimer kt(d, s, SWD_K_PRE_BP);
    (d_llr ? d->pre_fn_llr : d->pre_fn)<<<g1, d->T1, d->PRE.total, s>>>(g, d_synd, B, c.max_iter, c.ms_scaling_factor, d_corr, d_conv, d->ws,
                                                                     d->hscratch.p, full_hist, d->PRE, iter_out, lpr_out);
    d->ctr.kernel_launches++;
    }
    if (d_pm) {
        const double fillv = (c.kind == SWD_KIND_OSD_WINDOW) ? 0.0 : SWD_MAX_PM;
        fill_pm_kernel<<<(unsigned)((B + 255) / 256), 256, 0, s>>>(d_pm, B, fillv);
        d->ctr.kernel_launches++;
    }
    if (c.kind == SWD_KIND_BPGD && c.max_iter <= -1) return SWD_OK;   // pyx:506
    const int g2 = (int)std::min<long long>(B, d->grid2);
    // Latency mode: with so few shots that every work item gets its own CTA even at the worst-case footprint, run one
    // tier (worst-case shared memory) instead of two - five launches less per window (p50 per-window latency at batch 1).
    const bool lat = d->T3lat > 0 && B <= 8 && (B * (long long)std::max(1, d->P.n_rec) <= (long long)d->grid3lat / 2);     // <= 8: the node region holds 8 slots at the latency stride
    const bool one_tier = lat || ((d->es_capA < d->L.es_max) && (B * (long long)std::max(1, d->P.n_rec) <= (long long)d->grid3B));
    const int capA = one_tier ? d->L.es_max : d->es_capA;
    const SubLayout &LsA = one_tier ? d->LsB : d->LsA;
    const PathSmem &PSA = one_tier ? d->PSB : d->PS;
    { KTimer kt(d, s, SWD_K_SORT_RESET);
      if (d_llr) sort_reset_kernel<true><<<g2, d->T2, d->SS.total, s>>>(g, d_synd, d->ws, d->L, lat ? d->Plat : d->P, d->SS, d_corr, capA);
      else sort_reset_kernel<false><<<g2, d->T2, d->SS.total, s>>>(g, d_synd, d->ws, d->L, lat ? d->Plat : d->P, d->SS, d_corr, capA); }
    d->ctr.kernel_launches++;
    const size_t smem3 = (size_t)LsA.blob_bytes + PSA.total;
    const size_t smem3B = (size_t)d->LsB.blob_bytes + d->PSB.total;
    const bool two_tier = capA < d->L.es_max;
    int g3 = one_tier ? d->grid3B : d->grid3;
    path_fn_t pfn = d->path_fn; int T3 = d->T3;
    if (lat) { pfn = d->path_fn_lat; T3 = d->T3lat; g3 = d->grid3lat; }
    const int phases = (c.kind == SWD_KIND_BPGDG && c.multi_thread && d->P.n_side > 0) ? 2 : 1;
    if (c.kind == SWD_KIND_OSD_WINDOW) {
        for (int stage = 0; stage < 2; stage++) {
            KTimer kt(d, s, stage == 0 ? SWD_K_POST_BP : SWD_K_OSD);
            int st = osd_launch(g, d_synd, d->ws, d->L, LsA, d->LsB, PSA, d->PSB, capA, d->grid3B, smem3B, d->P, d->OS, d->ow, d->dmax, d->T3, g3, smem3, d->T5, d->grid5,
                                c.osd_method, c.osd_order, d->rank, d_corr, d_conv, d_pm, B, chunk_base, s, &d->ctr.kernel_launches,
                                d->ow.need_osd + d->cap, stage);
            if (st) { set_err("osd launch failed"); return st; }
        }
    } else {
        for (int lv = 0; lv < d->P.shared_T; lv++) {       // shared-prefix nodes, level by level
            KTimer kt(d, s, SWD_K_PATH_TRUNK);
            pfn<<<g3, T3, smem3, s>>>(d->ws, d->L, LsA, PSA, lat ? d->Plat : d->P, 2 + lv, 0, capA);
            d->ctr.kernel_launches++;
            if (two_tier) {
                d->path_fn<<<d->grid3B, d->T3, smem3B, s>>>(d->ws, d->L, d->LsB, d->PSB, d->P, 2 + lv, 1, capA);
                d->ctr.kernel_launches++;
            }
        }
        for (int ph = 0; ph < phases; ph++) {
            KTimer kt(d, s, ph == 0 ? SWD_K_PATH_MAIN : SWD_K_PATH_SIDE);
            pfn<<<g3, T3, smem3, s>>>(d->ws, d->L, LsA, PSA, lat ? d->Plat : d->P, ph, 0, capA);
            d->ctr.kernel_launches++;
            if (two_tier) {      // shots whose shortened graph exceeds tier A (rare): same kernel, worst-case footprint
                d->path_fn<<<d->grid3B, d->T3, smem3B, s>>>(d->ws, d->L, d->LsB, d->PSB, d->P, ph, 1, capA);
                d->ctr.kernel_launches++;
            }
        }
        { KTimer kt(d, s, SWD_K_SELECT);
          select_kernel<<<std::max(1, std::min<int>((int)B, d->num_sm * 8)), 128, 0, s>>>(d->ws, d->L, lat ? d->Plat : d->P, d->n, d_corr, d_conv, d_pm); }
        d->ctr.kernel_launches++;
    }
    CK(cudaGetLastError());
    return SWD_OK;
}

// The outputs of the last batch of an osd_window-kind decoder (swd_osd_last_outputs), grown with B.  The zero fill runs on the
// caller's stream: the kernels that write these buffers run there (a legacy-stream memset would not be ordered against a
// non-blocking stream).
static int reserve_osd_outputs(swd_decoder *d, long long B, cudaStream_t s) {
    if (B <= d->ow.out_cap) return SWD_OK;
    const size_t n = d->n;
    OsdWork &ow = d->ow;
    ow.out_cap = 0;
    int st;
    if ((st = d->osd_bp_dec.reserve(B * n)) || (st = d->osd_osd0.reserve(B * n)) || (st = d->osd_osdw.reserve(B * n)) ||
        (st = d->osd_lpr.reserve(B * n * 4)) || (st = d->osd_bp_iter.reserve(B)))
        d->last_B = 0;          // the last batch's outputs may be gone
    ow.bp_dec = d->osd_bp_dec.p; ow.osd0 = d->osd_osd0.p; ow.osdw = d->osd_osdw.p; ow.lpr = d->osd_lpr.p; ow.bp_iter = d->osd_bp_iter.p;
    if (st) return st;
    CK(cudaMemsetAsync(ow.osd0, 0, B * n, s)); CK(cudaMemsetAsync(ow.osdw, 0, B * n, s)); CK(cudaMemsetAsync(ow.bp_dec, 0, B * n, s));
    ow.out_cap = B;
    return SWD_OK;
}

// llr: per-shot priors [B][n] or nullptr; llr_host: llr is a host array, copied one workspace chunk at a time into d->d_llr
static int decode_device_impl(swd_decoder *d, const uint8_t *d_synd, int64_t B, uint8_t *d_corr, uint8_t *d_conv, double *d_pm,
                              cudaStream_t s, const double *llr, bool llr_host) {
    int st = alloc_workspace(d, B, s);
    if (st) return st;
    if (d->cfg.kind == SWD_KIND_OSD_WINDOW && (st = reserve_osd_outputs(d, B, s))) return st;
    if (llr_host && d->d_llr.cap < (size_t)d->n * d->cap) {
        CK(cudaStreamSynchronize(s));
        if ((st = d->d_llr.reserve((size_t)d->n * d->cap))) return st;
    }
    for (long long b0 = 0; b0 < B; b0 += d->cap) {
        const long long nb = std::min<long long>(d->cap, B - b0);
        const double *cl = llr ? llr + (size_t)b0 * d->n : nullptr;
        if (llr_host) {     // the buffer is reused chunk after chunk: stream order puts each copy after the previous chunk's kernels
            CK(cudaMemcpyAsync(d->d_llr.p, cl, (size_t)8 * nb * d->n, cudaMemcpyHostToDevice, s));
            cl = d->d_llr.p;
        }
        st = launch_chunk(d, d_synd + b0 * d->m, nb, d_corr + b0 * d->n, d_conv + b0, d_pm ? d_pm + b0 : nullptr, s, b0, cl);
        if (st) return st;
        // fold the per-chunk GDG count into the running statistics (device side, no sync)
        accumulate_count_kernel<<<1, 1, 0, s>>>(d->ws.counters, d->ws.stats);
        d->ctr.kernel_launches++;
    }
    d->ctr.shots += (uint64_t)B;
    d->last_B = B;
    return SWD_OK;
}

// ---- bit-packed shot I/O ------------------------------------------------------------------------------------------
static int launch_pack(const u8 *d_bytes, long long B, int nbits, u64 *d_packed, cudaStream_t s) {
    const int w64 = (nbits + 63) / 64; const long long warps = B * ((w64 * 2 + 31) / 32);
    if (warps > 0) pack_bits_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, s>>>(d_bytes, B, nbits, w64, (u32 *)d_packed);
    CK(cudaGetLastError());
    return SWD_OK;
}
static int launch_unpack(const u64 *d_packed, long long B, int nbits, u8 *d_bytes, cudaStream_t s) {
    const int w64 = (nbits + 63) / 64; const long long warps = B * ((w64 * 2 + 31) / 32);
    if (warps > 0) unpack_bits_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, s>>>((const u32 *)d_packed, B, nbits, w64, d_bytes);
    CK(cudaGetLastError());
    return SWD_OK;
}
extern "C" int swd_pack_bits(int device, const uint8_t *d_bytes, int64_t B, int nbits, uint64_t *d_packed, void *stream) {
    if (B < 0 || nbits <= 0 || (B > 0 && (!d_bytes || !d_packed))) { set_err("pack: bad argument"); return SWD_ERR_INVALID; }
    CK(cudaSetDevice(device));
    return launch_pack(d_bytes, B, nbits, (u64 *)d_packed, (cudaStream_t)stream);
}
extern "C" int swd_unpack_bits(int device, const uint64_t *d_packed, int64_t B, int nbits, uint8_t *d_bytes, void *stream) {
    if (B < 0 || nbits <= 0 || (B > 0 && (!d_bytes || !d_packed))) { set_err("unpack: bad argument"); return SWD_ERR_INVALID; }
    CK(cudaSetDevice(device));
    return launch_unpack((const u64 *)d_packed, B, nbits, d_bytes, (cudaStream_t)stream);
}

// the staging buffers of the host and packed entry points: byte and packed images of B shots' syndromes and corrections
static int ensure_stage(swd_decoder *d, long long B) {
    const size_t ws = (d->m + 63) / 64, wc = (d->n + 63) / 64;
    int st;
    if ((st = d->d_synd.reserve((size_t)B * d->m)) || (st = d->d_corr.reserve((size_t)B * d->n)) || (st = d->d_conv.reserve(B)) ||
        (st = d->d_pm.reserve(B)) || (st = d->d_psynd.reserve((size_t)B * ws)) || (st = d->d_pcorr.reserve((size_t)B * wc))) return st;
    return SWD_OK;
}

// The eight swd_decode_batch_* entry points.  host: syndromes, outputs and per-shot priors in host memory, on the decoder's
// own stream, synchronised before returning; otherwise device pointers on `stream`.  packed: syndromes and corrections
// bit-packed (8x fewer bytes over PCIe for a host call), unpacked and packed through the staging buffers, so calls on one
// decoder must be stream-ordered.  llr: per-shot priors [B][n] or nullptr; llr_ok is false when an _llr entry point got none.
static int decode_impl(swd_decoder *d, bool host, bool packed, const void *synd, int64_t B, void *corr, uint8_t *conv, double *pm,
                       const double *llr, bool llr_ok, void *stream) {
    if (!d || B < 0 || !llr_ok || (B > 0 && (!synd || !corr || !conv))) { set_err("decode: null argument"); return SWD_ERR_INVALID; }
    if (d->osd_only) { set_err("decode: not a window decoder"); return SWD_ERR_INVALID; }
    if (B == 0) return SWD_OK;
    CK(cudaSetDevice(d->device));
    int st;
    if ((host || packed) && (st = ensure_stage(d, B))) return st;
    cudaStream_t s = host ? d->stream : (cudaStream_t)stream;
    // the device images of the syndromes and corrections in the call's format, and of conv and pm: the caller's, or staging
    // buffers for a host call
    const void *d_in = synd;
    void *d_out = corr;
    u8 *d_conv = conv;
    double *d_pm = pm;
    if (host) {
        void *stage_in = packed ? (void *)d->d_psynd.p : d->d_synd.p;
        CK(cudaMemcpyAsync(stage_in, synd, packed ? (size_t)B * ((d->m + 63) / 64) * 8 : (size_t)B * d->m, cudaMemcpyHostToDevice, s));
        d_in = stage_in; d_out = packed ? (void *)d->d_pcorr.p : d->d_corr.p;
        d_conv = d->d_conv.p; d_pm = d->d_pm.p;
    }
    if (packed && (st = launch_unpack((const u64 *)d_in, B, d->m, d->d_synd.p, s))) return st;
    const u8 *d_synd = packed ? d->d_synd.p : (const u8 *)d_in;
    u8 *d_corr = packed ? d->d_corr.p : (u8 *)d_out;
    if ((st = decode_device_impl(d, d_synd, B, d_corr, d_conv, d_pm, s, llr, host && llr))) return st;
    if (packed) {
        d->ctr.kernel_launches += 2;
        if ((st = launch_pack(d_corr, B, d->n, (u64 *)d_out, s))) return st;
    }
    if (host) {
        CK(cudaMemcpyAsync(corr, d_out, packed ? (size_t)B * ((d->n + 63) / 64) * 8 : (size_t)B * d->n, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(conv, d_conv, (size_t)B, cudaMemcpyDeviceToHost, s));
        if (pm) CK(cudaMemcpyAsync(pm, d_pm, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    }
    return SWD_OK;
}

extern "C" int swd_decode_batch_host(swd_decoder *d, const uint8_t *synd, int64_t B, uint8_t *corr, uint8_t *conv, double *pm) {
    return decode_impl(d, true, false, synd, B, corr, conv, pm, nullptr, true, nullptr);
}
extern "C" int swd_decode_batch_host_llr(swd_decoder *d, const uint8_t *synd, int64_t B, uint8_t *corr, uint8_t *conv, double *pm,
                                         const double *channel_llr) {
    return decode_impl(d, true, false, synd, B, corr, conv, pm, channel_llr, channel_llr != nullptr, nullptr);
}
extern "C" int swd_decode_batch_device(swd_decoder *d, const uint8_t *d_synd, int64_t B, uint8_t *d_corr, uint8_t *d_conv,
                                       double *d_pm, void *stream) {
    return decode_impl(d, false, false, d_synd, B, d_corr, d_conv, d_pm, nullptr, true, stream);
}
extern "C" int swd_decode_batch_device_llr(swd_decoder *d, const uint8_t *d_synd, int64_t B, uint8_t *d_corr, uint8_t *d_conv,
                                           double *d_pm, const double *d_channel_llr, void *stream) {
    return decode_impl(d, false, false, d_synd, B, d_corr, d_conv, d_pm, d_channel_llr, d_channel_llr != nullptr, stream);
}
extern "C" int swd_decode_batch_host_packed(swd_decoder *d, const uint64_t *synd_packed, int64_t B, uint64_t *corr_packed, uint8_t *conv,
                                            double *pm) {
    return decode_impl(d, true, true, synd_packed, B, corr_packed, conv, pm, nullptr, true, nullptr);
}
extern "C" int swd_decode_batch_host_packed_llr(swd_decoder *d, const uint64_t *synd_packed, int64_t B, uint64_t *corr_packed, uint8_t *conv,
                                                double *pm, const double *channel_llr) {
    return decode_impl(d, true, true, synd_packed, B, corr_packed, conv, pm, channel_llr, channel_llr != nullptr, nullptr);
}
extern "C" int swd_decode_batch_device_packed(swd_decoder *d, const uint64_t *d_synd_packed, int64_t B, uint64_t *d_corr_packed,
                                              uint8_t *d_conv, double *d_pm, void *stream) {
    return decode_impl(d, false, true, d_synd_packed, B, d_corr_packed, d_conv, d_pm, nullptr, true, stream);
}
extern "C" int swd_decode_batch_device_packed_llr(swd_decoder *d, const uint64_t *d_synd_packed, int64_t B, uint64_t *d_corr_packed,
                                                  uint8_t *d_conv, double *d_pm, const double *d_channel_llr, void *stream) {
    return decode_impl(d, false, true, d_synd_packed, B, d_corr_packed, d_conv, d_pm, d_channel_llr, d_channel_llr != nullptr, stream);
}

extern "C" int swd_is_streamed(swd_decoder *d) { return d ? (d->stream_mode ? 1 : 0) : -1; }

// Host-only diagnostic (no CUDA call): the physical message layout swd_create picks for the pre-BP kernel of this graph.
extern "C" int swd_pre_bp_layout(int m, int n, const int32_t *colptr, const int32_t *rowidx, int optimize,
                                 int32_t *slot_of_entry, int32_t *row_start, int64_t *stats) {
    if (!colptr || !rowidx || m <= 0 || n <= 0 || colptr[0] != 0) { set_err("swd_pre_bp_layout: bad argument"); return SWD_ERR_INVALID; }
    const int nnz = colptr[n];
    if (n > 65534 || m > 65534 || nnz > 65535 || nnz < 0) { set_err("swd_pre_bp_layout: graph too large for 16-bit indices"); return SWD_ERR_UNSUPPORTED; }
    FlatGraph G;
    if (const char *why = flat_graph(m, n, colptr, rowidx, G)) { set_err(std::string("swd_pre_bp_layout: ") + why); return SWD_ERR_INVALID; }
    PreLayout L;
    pre_layout(m, n, nnz, G.cp, G.cr, G.rp, G.cpos, G.vord, optimize != 0, L);
    if (slot_of_entry) for (int e = 0; e < nnz; e++) slot_of_entry[e] = L.phys[e];     // CSC entry (rows ascending inside a column) -> slot
    if (row_start) for (int r = 0; r <= m; r++) row_start[r] = L.pstart[r];
    if (stats) { stats[0] = L.nphys; stats[1] = L.excess0; stats[2] = L.excess; }
    return SWD_OK;
}

extern "C" int swd_osd_last_outputs(swd_decoder *d, int64_t B, uint8_t *bp_dec, uint8_t *osd0, uint8_t *osdw,
                                    double *lpr, int32_t *bp_iteration) {
    if (!d || d->cfg.kind != SWD_KIND_OSD_WINDOW) { set_err("not an osd_window decoder"); return SWD_ERR_INVALID; }
    if (B > d->last_B) { set_err("B exceeds last batch"); return SWD_ERR_INVALID; }
    CK(cudaSetDevice(d->device));
    CK(cudaDeviceSynchronize());
    const size_t n = d->n;
    if (bp_dec) CK(cudaMemcpy(bp_dec, d->ow.bp_dec, (size_t)B * n, cudaMemcpyDeviceToHost));
    if (osd0) CK(cudaMemcpy(osd0, d->ow.osd0, (size_t)B * n, cudaMemcpyDeviceToHost));
    if (osdw) CK(cudaMemcpy(osdw, d->ow.osdw, (size_t)B * n, cudaMemcpyDeviceToHost));
    if (lpr) CK(cudaMemcpy(lpr, d->ow.lpr, (size_t)B * n * 32, cudaMemcpyDeviceToHost));
    if (bp_iteration) CK(cudaMemcpy(bp_iteration, d->ow.bp_iter, (size_t)B * 4, cudaMemcpyDeviceToHost));
    return SWD_OK;
}

extern "C" int swd_set_profiling(swd_decoder *d, int enable) {
    if (!d) return SWD_ERR_INVALID;
    d->profiling = enable != 0;
    d->P.count_work = d->Plat.count_work = d->profiling ? 1 : 0;      // the work counters of the min-sum calls (swd_get_counters)
    return SWD_OK;
}
extern "C" int swd_get_kernel_times(swd_decoder *d, double *ms, uint64_t *launches) {
    if (!d || !ms || !launches) return SWD_ERR_INVALID;
    CK(cudaSetDevice(d->device));
    CK(cudaDeviceSynchronize());
    for (int k = 0; k < SWD_K_COUNT; k++) { ms[k] = 0.0; launches[k] = 0; }
    for (auto &e : d->ev_used) {
        float t = 0.f;
        CK(cudaEventElapsedTime(&t, e.a, e.b));
        ms[e.k] += t; launches[e.k]++;
        d->ev_free.push_back(e.a); d->ev_free.push_back(e.b);
    }
    d->ev_used.clear();
    return SWD_OK;
}

extern "C" int swd_get_counters(swd_decoder *d, swd_counters *out) {
    if (!d || !out) return SWD_ERR_INVALID;
    CK(cudaSetDevice(d->device));
    if (d->ws.stats) { CK(cudaDeviceSynchronize()); int st = pull_stats(d, d->stream); if (st) return st; }
    *out = d->ctr;
    return SWD_OK;
}
extern "C" int swd_reset_counters(swd_decoder *d) {
    if (!d) return SWD_ERR_INVALID;
    CK(cudaSetDevice(d->device));
    memset(&d->ctr, 0, sizeof(d->ctr));
    if (d->ws.stats) { CK(cudaDeviceSynchronize()); CK(cudaMemset(d->ws.stats, 0, 16 * sizeof(u64))); }
    return SWD_OK;
}
extern "C" int swd_rank(swd_decoder *d) { return d ? d->rank : -1; }
extern "C" int swd_new_n(swd_decoder *d) { return d ? d->nn : -1; }

// ------------------------------------------------------------------------------------------------
// sliding-window bookkeeping
// ------------------------------------------------------------------------------------------------
struct swd_window {
    int device, num_det, num_col, num_obs;
    DevBuf<int> chk_cp, chk_ri, obs_cp, obs_ri;
    DevBuf<u32> thr;             // floor(prior * 2^32) per DEM column (set by swd_window_set_priors)
    DevBuf<u32> pauli_thr;       // code capacity (swd_window_set_pauli_priors): thr(px) | thr(px + py) | thr(px + py + pz), n each
    u32 pauli_t_erase = 0;       // thr(erasure_rate)
    int pauli_n = 0;             // 0 until swd_window_set_pauli_priors
    DevBuf<double> pauli_llr5;   // static LLR rows [5][n] copied into the per-shot planes, or empty
    DevBuf<uint4> circ_work;     // circuit noise (swd_window_set_circuit_noise): (l, m0, n_l, thr(e_l)) sorted by n_l
    DevBuf<uint2> circ_mech;     // (DEM column or -1, thr(p)) per mechanism
    DevBuf<double> circ_llr;     // static LLR row [num_col], or empty
    int circ_num_loc = 0;        // 0 until swd_window_set_circuit_noise
    std::vector<uint4> circ_work_h;   // host copies of circ_work and of the mechanisms' columns (readout set-up reads them)
    std::vector<int> circ_col_h;
    struct Readout {             // soft readout (swd_window_set_circuit_readout); a new circuit-noise set-up clears it
        DevBuf<uint4> work;      // circ_work with z = 1 | (r + 1) << 4 at readout r
        DevBuf<u32> thr;         // thr(w_0 + .. + w_{k-1}) for k = 1 .. K-1, then thr(q_k) for k = 0 .. K-1
        DevBuf<int> col;         // [num_col] readout location whose mechanism is in column c, or -1
        DevBuf<double> llr;      // class_llr [num_readout][K], or empty
        int num = 0, K = 0;      // 0 until swd_window_set_circuit_readout
    } ro;
};

extern "C" int swd_window_create(int device, int num_det, int num_col, const int32_t *chk_cp, const int32_t *chk_ri, int num_obs,
                                 const int32_t *obs_cp, const int32_t *obs_ri, swd_window **out) {
    if (!chk_cp || !chk_ri || !out || num_det <= 0 || num_col <= 0 || num_obs < 0 || (num_obs > 0 && (!obs_cp || !obs_ri))) {
        set_err("swd_window_create: bad argument"); return SWD_ERR_INVALID;
    }
    CK(cudaSetDevice(device));
    swd_window *w = new swd_window();
    w->device = device; w->num_det = num_det; w->num_col = num_col; w->num_obs = num_obs;
    std::vector<int> a(chk_cp, chk_cp + num_col + 1), b(chk_ri, chk_ri + chk_cp[num_col]);
    int st;
    if ((st = w->chk_cp.upload(a)) || (st = w->chk_ri.upload(b))) { swd_window_destroy(w); return st; }
    if (num_obs > 0) {
        std::vector<int> c(obs_cp, obs_cp + num_col + 1), e(obs_ri, obs_ri + obs_cp[num_col]);
        if ((st = w->obs_cp.upload(c)) || (st = w->obs_ri.upload(e))) { swd_window_destroy(w); return st; }
    }
    *out = w;
    return SWD_OK;
}
extern "C" void swd_window_destroy(swd_window *w) {
    if (!w) return;
    cudaSetDevice(w->device);
    delete w;
}
static u32 prob_threshold(double p) {          // the samplers' rule: floor(p * 2^32), clamped to 0xffffffff
    const double x = p * 4294967296.0;
    return x >= 4294967295.0 ? 0xffffffffu : (u32)x;
}
// Launches a sampler kernel with one warp per shot and warp_bytes of dynamic shared memory per warp (parity words, and the
// circuit sampler's column words and class bytes): up to 8 warps per block within 200 KB.  A shot's draws depend only on
// (seed, shot index), so the warps per block do not change the results.
template <typename... P, typename... A>
static int launch_sampler(void (*kernel)(P...), const swd_window *w, size_t warp_bytes, int64_t B, void *stream, const char *who,
                          A... args) {
    CK(cudaSetDevice(w->device));
    const size_t limit = 200 * 1024;
    if (warp_bytes > limit) { set_err(std::string(who) + ": one warp's parity and column words exceed the shared-memory limit"); return SWD_ERR_UNSUPPORTED; }
    const int wpb = (int)std::min<size_t>(8, limit / warp_bytes);
    const size_t smem = (size_t)wpb * warp_bytes;
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<(unsigned)std::min<long long>((B + wpb - 1) / wpb, 148 * 16), wpb * 32, smem, (cudaStream_t)stream>>>(args...);
    CK(cudaGetLastError());
    return SWD_OK;
}
// bytes of one shot's det and obs parity words
static size_t parity_bytes(const swd_window *w) { return (size_t)(((w->num_det + 31) >> 5) + ((w->num_obs + 31) >> 5)) * sizeof(u32); }

extern "C" int swd_window_set_priors(swd_window *w, const double *priors) {
    if (!w || !priors) { set_err("swd_window_set_priors: bad argument"); return SWD_ERR_INVALID; }
    std::vector<u32> t(w->num_col);
    for (int c = 0; c < w->num_col; c++) {
        const double p = priors[c];
        if (!(p >= 0.0 && p <= 1.0)) { set_err("swd_window_set_priors: prior outside [0, 1]"); return SWD_ERR_INVALID; }
        t[c] = prob_threshold(p);
    }
    CK(cudaSetDevice(w->device));
    return w->thr.upload(t);
}
extern "C" int swd_window_set_pauli_priors(swd_window *w, int n, const double *px, const double *py, const double *pz,
                                           double erasure_rate, const double *llr5) {
    if (!w || !px || !py || !pz || n <= 0 || w->num_col != 2 * n) { set_err("swd_window_set_pauli_priors: bad argument (num_col must be 2n)"); return SWD_ERR_INVALID; }
    if (!(erasure_rate >= 0.0 && erasure_rate <= 1.0)) { set_err("swd_window_set_pauli_priors: erasure_rate outside [0, 1]"); return SWD_ERR_INVALID; }
    std::vector<u32> t(3 * (size_t)n);
    for (int v = 0; v < n; v++) {
        if (!(px[v] >= 0.0 && py[v] >= 0.0 && pz[v] >= 0.0)) { set_err("swd_window_set_pauli_priors: negative or NaN probability"); return SWD_ERR_INVALID; }
        const double xy = px[v] + py[v], xyz = xy + pz[v];
        if (xyz > 1.0) { set_err("swd_window_set_pauli_priors: px + py + pz > 1"); return SWD_ERR_INVALID; }
        t[v] = prob_threshold(px[v]); t[n + v] = prob_threshold(xy); t[2 * n + v] = prob_threshold(xyz);
    }
    CK(cudaSetDevice(w->device));
    w->pauli_llr5.release();
    w->pauli_n = 0;
    int st;
    if ((st = w->pauli_thr.upload(t))) return st;
    if (llr5 && (st = w->pauli_llr5.upload(std::vector<double>(llr5, llr5 + 5 * (size_t)n)))) return st;
    w->pauli_t_erase = prob_threshold(erasure_rate);
    w->pauli_n = n;
    return SWD_OK;
}
extern "C" int swd_window_sample_pauli(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det, uint8_t *d_obs,
                                       uint8_t *d_err, uint8_t *d_erased, double *d_channel_llr, void *stream) {
    if (!w || !d_det || B < 0 || shot_offset < 0 || (w->num_obs > 0 && !d_obs)) { set_err("swd_window_sample_pauli: bad argument"); return SWD_ERR_INVALID; }
    if (!w->pauli_n) { set_err("swd_window_sample_pauli: call swd_window_set_pauli_priors first"); return SWD_ERR_INVALID; }
    if (d_channel_llr && !w->pauli_llr5.p) { set_err("swd_window_sample_pauli: channel_llr needs the llr5 rows of swd_window_set_pauli_priors"); return SWD_ERR_INVALID; }
    if (B == 0) return SWD_OK;
    return launch_sampler(window_sample_pauli_kernel, w, parity_bytes(w), B, stream, "swd_window_sample_pauli",
        w->pauli_thr.p, w->pauli_t_erase, w->pauli_n, w->pauli_llr5.p, w->chk_cp.p, w->chk_ri.p, w->num_det, w->obs_cp.p, w->obs_ri.p,
        w->num_obs, (unsigned long long)seed, (long long)shot_offset, (long long)B, d_det, d_obs, d_err, d_erased, d_channel_llr);
}
extern "C" int swd_window_set_circuit_noise(swd_window *w, int num_loc, const int32_t *mech_ptr, const int32_t *mech_col,
                                            const double *mech_prob, const double *erasure_rate, const double *col_llr) {
    if (!w || num_loc <= 0 || !mech_ptr || !mech_col || !mech_prob || !erasure_rate) { set_err("swd_window_set_circuit_noise: bad argument"); return SWD_ERR_INVALID; }
    if (mech_ptr[0] != 0) { set_err("swd_window_set_circuit_noise: mech_ptr[0] must be 0"); return SWD_ERR_INVALID; }
    std::vector<uint4> work(num_loc);
    for (int l = 0; l < num_loc; l++) {
        const int n = mech_ptr[l + 1] - mech_ptr[l];
        if (n < 1 || n > 15) { set_err("swd_window_set_circuit_noise: a location needs 1 to 15 mechanisms"); return SWD_ERR_INVALID; }
        const double e = erasure_rate[l];
        if (!(e >= 0.0 && e <= 1.0)) { set_err("swd_window_set_circuit_noise: erasure_rate outside [0, 1]"); return SWD_ERR_INVALID; }
        work[l] = make_uint4((u32)l, (u32)mech_ptr[l], (u32)n, prob_threshold(e));
    }
    const int M = mech_ptr[num_loc];
    std::vector<uint2> mech(M);
    for (int k = 0; k < M; k++) {
        const double p = mech_prob[k];
        if (mech_col[k] < -1 || mech_col[k] >= w->num_col) { set_err("swd_window_set_circuit_noise: mech_col outside [-1, num_col)"); return SWD_ERR_INVALID; }
        if (!(p >= 0.0 && p <= 0.5)) { set_err("swd_window_set_circuit_noise: mech_prob outside [0, 1/2]"); return SWD_ERR_INVALID; }
        mech[k] = make_uint2((u32)mech_col[k], prob_threshold(p));
    }
    // lanes of a warp take consecutive work items: equal mechanism counts give them equal numbers of Philox calls
    std::stable_sort(work.begin(), work.end(), [](const uint4 &a, const uint4 &b) { return a.z > b.z; });
    CK(cudaSetDevice(w->device));
    w->circ_llr.release();
    w->ro = {};
    w->circ_num_loc = 0;
    int st;
    if ((st = w->circ_work.upload(work)) || (st = w->circ_mech.upload(mech))) return st;
    if (col_llr && (st = w->circ_llr.upload(std::vector<double>(col_llr, col_llr + w->num_col)))) return st;
    w->circ_work_h = work;
    w->circ_col_h.assign(mech_col, mech_col + M);
    w->circ_num_loc = num_loc;
    return SWD_OK;
}
extern "C" int swd_window_set_circuit_readout(swd_window *w, int num_readout, const int32_t *readout_loc, int num_classes,
                                              const double *class_weight, const double *flip_prob, const double *class_llr) {
    if (!w || num_readout <= 0 || !readout_loc || !class_weight || !flip_prob) { set_err("swd_window_set_circuit_readout: bad argument"); return SWD_ERR_INVALID; }
    if (!w->circ_num_loc) { set_err("swd_window_set_circuit_readout: call swd_window_set_circuit_noise first"); return SWD_ERR_INVALID; }
    const int K = num_classes, L = w->circ_num_loc;
    if (K < 1 || K > 256) { set_err("swd_window_set_circuit_readout: num_classes outside 1 .. 256"); return SWD_ERR_INVALID; }
    std::vector<u32> thr(2 * K - 1);
    double sum = 0.0;
    for (int k = 0; k < K; k++) {
        const double x = class_weight[k], q = flip_prob[k];
        if (!(x >= 0.0)) { set_err("swd_window_set_circuit_readout: a class weight is negative or NaN"); return SWD_ERR_INVALID; }
        if (!(q >= 0.0 && q <= 0.5)) { set_err("swd_window_set_circuit_readout: flip_prob outside [0, 1/2]"); return SWD_ERR_INVALID; }
        if (k > 0) thr[k - 1] = prob_threshold(sum);
        sum += x;
        thr[K - 1 + k] = prob_threshold(q);
    }
    if (!(std::fabs(sum - 1.0) <= 1e-9)) { set_err("swd_window_set_circuit_readout: class weights do not sum to 1"); return SWD_ERR_INVALID; }
    std::vector<int> slot(L, -1), col_ro(w->num_col, -1);       // slot[l]: position of location l in circ_work
    for (int i = 0; i < L; i++) slot[w->circ_work_h[i].x] = i;
    std::vector<uint4> work = w->circ_work_h;
    for (int r = 0; r < num_readout; r++) {
        const int l = readout_loc[r];
        if (l < 0 || l >= L) { set_err("swd_window_set_circuit_readout: readout_loc outside [0, num_loc)"); return SWD_ERR_INVALID; }
        uint4 &wk = work[slot[l]];
        if (wk.z >> 4) { set_err("swd_window_set_circuit_readout: a location is listed twice"); return SWD_ERR_INVALID; }
        if (wk.z != 1) { set_err("swd_window_set_circuit_readout: a readout location needs exactly one mechanism"); return SWD_ERR_INVALID; }
        const int c = w->circ_col_h[wk.y];
        if (c >= 0) {
            if (col_ro[c] >= 0) { set_err("swd_window_set_circuit_readout: two readout locations share a DEM column"); return SWD_ERR_INVALID; }
            col_ro[c] = r;
        }
        wk.z = 1u | (u32)(r + 1) << 4;
    }
    // readout items last among the single-mechanism locations, so that fewer warps mix the two paths
    std::stable_sort(work.begin(), work.end(), [](const uint4 &a, const uint4 &b) {
        return (a.z & 15u) != (b.z & 15u) ? (a.z & 15u) > (b.z & 15u) : (a.z >> 4 == 0) && (b.z >> 4 != 0);
    });
    CK(cudaSetDevice(w->device));
    w->ro = {};
    int st;
    if ((st = w->ro.work.upload(work)) || (st = w->ro.thr.upload(thr)) || (st = w->ro.col.upload(col_ro)) ||
        (class_llr && (st = w->ro.llr.upload(std::vector<double>(class_llr, class_llr + (size_t)num_readout * K))))) {
        w->ro = {}; return st;
    }
    w->ro.num = num_readout;
    w->ro.K = K;
    return SWD_OK;
}
// the per-warp words are the parity words, the optional err and LLR column words, and the readout class bytes
template <bool READOUT>
static int launch_sample_circuit(swd_window *w, const uint4 *work, const CircuitReadout &ro, uint64_t seed, int64_t shot_offset,
                                 int64_t B, uint8_t *d_det, uint8_t *d_obs, uint8_t *d_err, uint8_t *d_erased, double *d_channel_llr,
                                 void *stream, const char *who) {
    const int wc = (w->num_col + 31) >> 5;
    const size_t warp_bytes = parity_bytes(w) + (size_t)((d_err ? wc : 0) + (d_channel_llr ? wc : 0) +
                                                         (READOUT && d_channel_llr ? (ro.num_readout + 3) >> 2 : 0)) * sizeof(u32);
    return launch_sampler(window_sample_circuit_kernel<READOUT>, w, warp_bytes, B, stream, who,
        work, w->circ_num_loc, w->circ_mech.p, w->circ_llr.p, w->num_col, w->chk_cp.p, w->chk_ri.p, w->num_det, w->obs_cp.p, w->obs_ri.p,
        w->num_obs, (unsigned long long)seed, (long long)shot_offset, (long long)B, d_det, d_obs, d_err, d_erased, d_channel_llr, ro);
}
extern "C" int swd_window_sample_circuit(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det, uint8_t *d_obs,
                                         uint8_t *d_err, uint8_t *d_erased, double *d_channel_llr, void *stream) {
    if (!w || !d_det || B < 0 || shot_offset < 0 || (w->num_obs > 0 && !d_obs)) { set_err("swd_window_sample_circuit: bad argument"); return SWD_ERR_INVALID; }
    if (!w->circ_num_loc) { set_err("swd_window_sample_circuit: call swd_window_set_circuit_noise first"); return SWD_ERR_INVALID; }
    if (d_channel_llr && !w->circ_llr.p) { set_err("swd_window_sample_circuit: channel_llr needs the col_llr row of swd_window_set_circuit_noise"); return SWD_ERR_INVALID; }
    if (B == 0) return SWD_OK;
    return launch_sample_circuit<false>(w, w->circ_work.p, CircuitReadout{}, seed, shot_offset, B, d_det, d_obs, d_err, d_erased,
                                        d_channel_llr, stream, "swd_window_sample_circuit");
}
extern "C" int swd_window_sample_circuit_readout(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det,
                                                 uint8_t *d_obs, uint8_t *d_err, uint8_t *d_erased, uint8_t *d_readout,
                                                 double *d_channel_llr, void *stream) {
    if (!w || !d_det || B < 0 || shot_offset < 0 || (w->num_obs > 0 && !d_obs)) { set_err("swd_window_sample_circuit_readout: bad argument"); return SWD_ERR_INVALID; }
    if (!w->ro.num) { set_err("swd_window_sample_circuit_readout: call swd_window_set_circuit_readout first"); return SWD_ERR_INVALID; }
    if (d_channel_llr && (!w->circ_llr.p || !w->ro.llr.p)) {
        set_err("swd_window_sample_circuit_readout: channel_llr needs the col_llr row and the class_llr table"); return SWD_ERR_INVALID;
    }
    if (B == 0) return SWD_OK;
    const CircuitReadout ro{w->ro.thr.p, w->ro.thr.p + (w->ro.K - 1), w->ro.col.p, w->ro.llr.p, d_readout, w->ro.K, w->ro.num};
    return launch_sample_circuit<true>(w, w->ro.work.p, ro, seed, shot_offset, B, d_det, d_obs, d_err, d_erased, d_channel_llr, stream,
                                       "swd_window_sample_circuit_readout");
}
extern "C" int swd_window_sample(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det, uint8_t *d_obs,
                                 uint8_t *d_err, void *stream) {
    if (!w || !d_det || B < 0 || shot_offset < 0 || (w->num_obs > 0 && !d_obs)) { set_err("swd_window_sample: bad argument"); return SWD_ERR_INVALID; }
    if (!w->thr.p) { set_err("swd_window_sample: call swd_window_set_priors first"); return SWD_ERR_INVALID; }
    if (B == 0) return SWD_OK;
    return launch_sampler(window_sample_kernel, w, parity_bytes(w), B, stream, "swd_window_sample",
        w->thr.p, w->num_col, w->chk_cp.p, w->chk_ri.p, w->num_det, w->obs_cp.p, w->obs_ri.p, w->num_obs, (unsigned long long)seed,
        (long long)shot_offset, (long long)B, d_det, d_obs, d_err);
}
extern "C" int swd_window_extract(swd_window *w, const uint8_t *d_det, int64_t B, int row0, int m, uint8_t *d_synd, void *stream) {
    if (!w || !d_det || !d_synd || B < 0 || row0 < 0 || m <= 0 || row0 + m > w->num_det) { set_err("swd_window_extract: bad argument"); return SWD_ERR_INVALID; }
    if (B == 0) return SWD_OK;
    CK(cudaSetDevice(w->device));
    const long long total = (long long)B * m;
    window_extract_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, 1 << 20), 256, 0, (cudaStream_t)stream>>>(
        d_det, B, w->num_det, row0, m, d_synd);
    CK(cudaGetLastError());
    return SWD_OK;
}
extern "C" int swd_window_commit(swd_window *w, const uint8_t *d_corr, int64_t B, int n_win, int col0, int ncommit, uint8_t *d_det,
                                 uint8_t *d_obs, void *stream) {
    if (!w || !d_corr || !d_det || B < 0 || col0 < 0 || ncommit < 0 || ncommit > n_win || col0 + ncommit > w->num_col) {
        set_err("swd_window_commit: bad argument"); return SWD_ERR_INVALID;
    }
    if (B == 0 || ncommit == 0) return SWD_OK;
    CK(cudaSetDevice(w->device));
    const int wpb = 8;
    window_commit_kernel<<<(unsigned)std::min<long long>((B + wpb - 1) / wpb, 1 << 20), wpb * 32, 0, (cudaStream_t)stream>>>(
        d_corr, B, n_win, col0, ncommit, w->chk_cp.p, w->chk_ri.p, w->num_det, d_det, w->obs_cp.p, w->obs_ri.p, w->num_obs, d_obs);
    CK(cudaGetLastError());
    return SWD_OK;
}
extern "C" int swd_window_count_failures(swd_window *w, const uint8_t *d_det, const uint8_t *d_obs, int64_t B,
                                         unsigned long long *d_out2, void *stream) {
    if (!w || !d_det || !d_out2 || B < 0) { set_err("swd_window_count_failures: bad argument"); return SWD_ERR_INVALID; }
    CK(cudaSetDevice(w->device));
    CK(cudaMemsetAsync(d_out2, 0, 2 * sizeof(unsigned long long), (cudaStream_t)stream));
    if (B == 0) return SWD_OK;
    const int wpb = 8;
    window_count_kernel<<<(unsigned)std::min<long long>((B + wpb - 1) / wpb, 1 << 20), wpb * 32, 0, (cudaStream_t)stream>>>(
        d_det, w->num_det, d_obs, w->num_obs, B, d_out2);
    CK(cudaGetLastError());
    return SWD_OK;
}

// ------------------------------------------------------------------------------------------------
// bp4_osd: quaternary BP over (Hx, Hz) + one OSD per basis (src/bp4_osd.pyx)
// ------------------------------------------------------------------------------------------------
struct swd_bp4 {
    int device = 0, n = 0, mx = 0, mz = 0, max_iter = 32, num_sm = 0;
    double alpha = 1.0;
    swd_decoder *dx = nullptr, *dz = nullptr;      // osd_window-kind decoders over Hx / Hz: graph upload, rank, OSD machinery
    DevBuf<double> llr;                            // llr_x | llr_y | llr_z, n each
    Bp4Smem S{};
    int grid = 0;
    int grid_llr[2] = {0, 0};                      // per-shot priors: bp4_kernel<false, true>, <true, true> (camel)
    DevBuf<double> d_llr5;                         // host per-shot priors staged on the device, [5][B][n]; first _llr call
    // per-batch device buffers
    DevBuf<u8> synd_x, synd_z, bp_dec, conv, dec, osd0, tmp;
    DevBuf<int> iters;
    DevBuf<double> lpr, key_x, key_z;
    // camel_decode: four runs per shot
    DevBuf<u8> c_synd_x, c_synd_z, c_bp_dec, c_conv4, c_dec, c_conv;
    DevBuf<int> c_it4, c_it;
    DevBuf<double> c_pm4, c_pm, c_lpr;
    cudaStream_t stream = nullptr;
    ~swd_bp4() {
        swd_destroy(dx);
        swd_destroy(dz);
        if (stream) cudaStreamDestroy(stream);
    }
};

extern "C" void swd_bp4_destroy(swd_bp4 *b) {
    if (!b) return;
    cudaSetDevice(b->device);
    delete b;
}

extern "C" int swd_bp4_create(int device, int mx, int mz, int n, const int32_t *hx_colptr, const int32_t *hx_rowidx,
                              const int32_t *hz_colptr, const int32_t *hz_rowidx, const double *llr_x, const double *llr_y,
                              const double *llr_z, const double *prior_llr_x, const double *prior_llr_z, int max_iter,
                              double ms_scaling_factor, int osd_method, int osd_order, swd_bp4 **out) {
    if (!hx_colptr || !hx_rowidx || !hz_colptr || !hz_rowidx || !llr_x || !llr_y || !llr_z || !prior_llr_x || !prior_llr_z || !out ||
        mx <= 0 || mz <= 0 || n <= 0 || max_iter < 0) { set_err("swd_bp4_create: bad argument"); return SWD_ERR_INVALID; }
    swd_bp4 *b = new swd_bp4();
    b->device = device; b->n = n; b->mx = mx; b->mz = mz; b->max_iter = max_iter; b->alpha = ms_scaling_factor;
    swd_config cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.kind = SWD_KIND_OSD_WINDOW; cfg.device = device; cfg.max_iter = 1; cfg.ms_scaling_factor = 1.0; cfg.new_n = n;
    cfg.post_max_iter = 0; cfg.osd_method = osd_method; cfg.osd_order = osd_order; cfg.max_iter_per_step = 6; cfg.max_step = 1;
    int st;
    if ((st = create_impl(&cfg, mx, n, hx_colptr, hx_rowidx, prior_llr_x, &b->dx, true)) != SWD_OK) { swd_bp4_destroy(b); return st; }
    if ((st = create_impl(&cfg, mz, n, hz_colptr, hz_rowidx, prior_llr_z, &b->dz, true)) != SWD_OK) { swd_bp4_destroy(b); return st; }
    b->num_sm = b->dx->num_sm;
    std::vector<double> l(3 * (size_t)n);
    for (int v = 0; v < n; v++) { l[v] = llr_x[v]; l[n + v] = llr_y[v]; l[2 * (size_t)n + v] = llr_z[v]; }
    if ((st = b->llr.upload(l)) != SWD_OK) { swd_bp4_destroy(b); return st; }
    int o = 0;
    b->S.off_mx = o; o += 8 * std::max(1, b->dx->nnz); o = r16(o);
    b->S.off_mz = o; o += 8 * std::max(1, b->dz->nnz); o = r16(o);
    b->S.off_ux = o; o += 4 * mx; o = r16(o);
    b->S.off_uz = o; o += 4 * mz; o = r16(o);
    b->S.off_sx = o; o += mx; o = r16(o);
    b->S.off_sz = o; o += mz; o = r16(o);
    b->S.total = o;
    if (o > 227 * 1024) { swd_bp4_destroy(b); set_err("bp4: the two message arrays do not fit in shared memory"); return SWD_ERR_UNSUPPORTED; }
    int occ = 0;
    if ((st = occupancy(bp4_kernel<true>, 256, b->S.total, &occ)) != SWD_OK || occ < 1 ||
        (st = occupancy(bp4_kernel<false>, 256, b->S.total, &occ)) != SWD_OK || occ < 1) { swd_bp4_destroy(b); if (!st) { set_err("bp4_kernel does not fit"); st = SWD_ERR_UNSUPPORTED; } return st; }
    b->grid = b->num_sm * occ;
    // the per-shot twins get their own grids: their occupancy need not match the static instantiations'
    int occ_llr = 0;
    if ((st = occupancy(bp4_kernel<false, true>, 256, b->S.total, &occ_llr)) != SWD_OK || occ_llr < 1) {
        swd_bp4_destroy(b); if (!st) { set_err("bp4_kernel (per-shot priors) does not fit"); st = SWD_ERR_UNSUPPORTED; } return st;
    }
    b->grid_llr[0] = b->num_sm * occ_llr;
    if ((st = occupancy(bp4_kernel<true, true>, 256, b->S.total, &occ_llr)) != SWD_OK || occ_llr < 1) {
        swd_bp4_destroy(b); if (!st) { set_err("bp4_kernel (camel, per-shot priors) does not fit"); st = SWD_ERR_UNSUPPORTED; } return st;
    }
    b->grid_llr[1] = b->num_sm * occ_llr;
    if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess) { swd_bp4_destroy(b); set_err("stream create failed"); return SWD_ERR_CUDA; }
    *out = b;
    return SWD_OK;
}

extern "C" int swd_bp4_rank(swd_bp4 *b, int which) { return !b ? -1 : (which == 0 ? b->dx->rank : b->dz->rank); }

// OSD-only pass of an osd_window-kind decoder: ranking keys are supplied, converged shots are skipped.
// d_prior: per-shot basis priors [B][n] (plane 3 or 4 of the five) or nullptr for the decoder's static priors
static int bp4_osd_pass(swd_decoder *d, const u8 *d_synd, const double *d_keys, const u8 *d_conv, long long B, u8 *d_tmp, cudaStream_t s,
                        const double *d_prior) {
    int st = alloc_workspace(d, B, s);
    if (st) return st;
    if ((st = reserve_osd_outputs(d, B, s))) return st;
    for (long long b0 = 0; b0 < B; b0 += d->cap) {
        const long long nb = std::min<long long>(d->cap, B - b0);
        CK(cudaMemsetAsync(d->ws.counters, 0, 64 * sizeof(int), s));
        bp4_osd_setup_kernel<<<(unsigned)std::min<long long>((nb * d->n + 255) / 256, 4096), 256, 0, s>>>(d->ws, d->ow.need_osd, d_keys + b0 * d->n, d_conv + b0, nb, d->n);
        if (d_prior) {                                                         // chunk-local rows, as the window decoders
            GraphDev g = d->g; g.llr_shot = d_prior + b0 * d->n;
            osd_kernel<true><<<d->grid5, d->T5, d->OS.total, s>>>(g, d_synd + b0 * d->m, d->ws, d->L, d->P, d->OS, d->ow, d->cfg.osd_method, d->cfg.osd_order,
                                                                  d->rank, d_tmp + b0 * d->n, nullptr, b0);
        } else {
            osd_kernel<false><<<d->grid5, d->T5, d->OS.total, s>>>(d->g, d_synd + b0 * d->m, d->ws, d->L, d->P, d->OS, d->ow, d->cfg.osd_method, d->cfg.osd_order,
                                                                   d->rank, d_tmp + b0 * d->n, nullptr, b0);
        }
        d->ctr.kernel_launches += 2;
    }
    CK(cudaGetLastError());
    return SWD_OK;
}

static int bp4_reserve(swd_bp4 *b, int64_t B) {
    const size_t n = b->n;
    int st;
    if ((st = b->synd_x.reserve((size_t)B * b->mx)) || (st = b->synd_z.reserve((size_t)B * b->mz)) ||
        (st = b->bp_dec.reserve((size_t)B * 2 * n)) || (st = b->conv.reserve(B)) || (st = b->dec.reserve((size_t)B * 2 * n)) ||
        (st = b->osd0.reserve((size_t)B * 2 * n)) || (st = b->tmp.reserve((size_t)B * n)) || (st = b->iters.reserve(B)) ||
        (st = b->lpr.reserve((size_t)B * n * 3)) || (st = b->key_x.reserve((size_t)B * n)) || (st = b->key_z.reserve((size_t)B * n))) return st;
    return SWD_OK;
}

// host per-shot priors [5][B][n] -> b->d_llr5 on `s` (allocated on the first call that needs it, grown with B)
static int bp4_stage_llr(swd_bp4 *b, const double *llr5, int64_t B, cudaStream_t s) {
    if (int st = b->d_llr5.reserve((size_t)5 * B * b->n)) return st;
    CK(cudaMemcpyAsync(b->d_llr5.p, llr5, (size_t)40 * B * b->n, cudaMemcpyHostToDevice, s));
    return SWD_OK;
}

// BP4 + OSD per basis on device-resident syndromes; results are left in the decoder's own buffers (dec, conv, bp_dec, osd0, lpr, iters).
// d_llr5: per-shot priors, five planes [5][B][n] on the device (llr_x, llr_y, llr_z, prior_llr_x, prior_llr_z), or nullptr
static int bp4_run(swd_bp4 *b, const u8 *d_sx, const u8 *d_sz, int64_t B, cudaStream_t s, const double *d_llr5) {
    const size_t n = b->n;
    const size_t P = (size_t)B * n;                                            // plane stride
    if (d_llr5)
        bp4_kernel<false, true><<<(int)std::min<long long>(B, b->grid_llr[0]), 256, b->S.total, s>>>(b->dx->g, b->dz->g, d_llr5, d_llr5 + P, d_llr5 + 2 * P,
            d_sx, d_sz, B, b->max_iter, b->alpha, b->bp_dec.p, b->conv.p, b->iters.p, b->lpr.p, b->key_x.p, b->key_z.p, b->S, nullptr);
    else
        bp4_kernel<false><<<(int)std::min<long long>(B, b->grid), 256, b->S.total, s>>>(b->dx->g, b->dz->g, b->llr.p, b->llr.p + n, b->llr.p + 2 * n, d_sx, d_sz, B,
                                                                                        b->max_iter, b->alpha, b->bp_dec.p, b->conv.p, b->iters.p, b->lpr.p, b->key_x.p, b->key_z.p, b->S, nullptr);
    CK(cudaGetLastError());
    int st;
    if ((st = bp4_osd_pass(b->dx, d_sx, b->key_x.p, b->conv.p, B, b->tmp.p, s, d_llr5 ? d_llr5 + 3 * P : nullptr))) return st;      // osd('x') -> z part
    if ((st = bp4_osd_pass(b->dz, d_sz, b->key_z.p, b->conv.p, B, b->tmp.p, s, d_llr5 ? d_llr5 + 4 * P : nullptr))) return st;      // osd('z') -> x part
    bp4_finish_kernel<<<(unsigned)std::min<long long>((B * 2 * (long long)n + 255) / 256, 8192), 256, 0, s>>>(
        b->bp_dec.p, b->conv.p, b->dx->ow.osdw, b->dx->ow.osd0, b->dz->ow.osdw, b->dz->ow.osd0, B, (int)n, b->dec.p, b->osd0.p);
    CK(cudaGetLastError());
    return SWD_OK;
}

// The argument check of the bp4 batch entry points: a decoder, B >= 0, the per-shot priors of an _llr entry point, and the
// syndromes and the two required outputs when B > 0.
static bool bp4_args_ok(const char *who, const swd_bp4 *b, int64_t B, const void *sx, const void *sz, const void *dec, const void *conv,
                        bool llr_ok = true) {
    if (b && B >= 0 && llr_ok && (B == 0 || (sx && sz && dec && conv))) return true;
    set_err(std::string(who) + ": null argument");
    return false;
}

// A host call stages its syndromes (into buf_x / buf_z) and its per-shot priors (into b->d_llr5) on the decoder's own stream
// and points sx, sz and llr5 at the device copies.
static int bp4_stage_inputs(swd_bp4 *b, u8 *buf_x, u8 *buf_z, const u8 *&sx, const u8 *&sz, const double *&llr5, int64_t B,
                            cudaStream_t s) {
    CK(cudaMemcpyAsync(buf_x, sx, (size_t)B * b->mx, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(buf_z, sz, (size_t)B * b->mz, cudaMemcpyHostToDevice, s));
    sx = buf_x; sz = buf_z;
    if (llr5) {
        int st = bp4_stage_llr(b, llr5, B, s);
        if (st) return st;
        llr5 = b->d_llr5.p;
    }
    return SWD_OK;
}

// Copies the results out of the decoder's buffers into the caller's (a NULL destination is skipped): device-to-host followed
// by a synchronise for a host call, device-to-device on the caller's stream otherwise.
struct Bp4Out { void *dst; const void *src; size_t bytes; };
static int bp4_copy_out(bool host, cudaStream_t s, std::initializer_list<Bp4Out> outs) {
    for (const Bp4Out &o : outs)
        if (o.dst) CK(cudaMemcpyAsync(o.dst, o.src, o.bytes, host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s));
    if (host) CK(cudaStreamSynchronize(s));
    return SWD_OK;
}

// host: syndromes, outputs and llr5 in host memory, on the decoder's own stream, synchronised before returning; otherwise device
// pointers on `stream` with no host synchronisation.  llr5: per-shot priors [5][B][n] or nullptr (static priors).
static int bp4_decode_impl(swd_bp4 *b, bool host, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *conv,
                           uint8_t *bp_dec, uint8_t *osd0, double *lpr, int32_t *bp_iteration, const double *llr5, void *stream) {
    if (B == 0) return SWD_OK;
    CK(cudaSetDevice(b->device));
    const size_t n = b->n;
    int st;
    if ((st = bp4_reserve(b, B))) return st;
    cudaStream_t s = host ? b->stream : (cudaStream_t)stream;
    if (host && (st = bp4_stage_inputs(b, b->synd_x.p, b->synd_z.p, synd_x, synd_z, llr5, B, s))) return st;
    if ((st = bp4_run(b, synd_x, synd_z, B, s, llr5))) return st;
    return bp4_copy_out(host, s, {{dec, b->dec.p, (size_t)B * 2 * n}, {conv, b->conv.p, (size_t)B}, {bp_dec, b->bp_dec.p, (size_t)B * 2 * n},
                                  {osd0, b->osd0.p, (size_t)B * 2 * n}, {lpr, b->lpr.p, (size_t)B * n * 24}, {bp_iteration, b->iters.p, (size_t)B * 4}});
}

extern "C" int swd_bp4_decode_batch_host(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *conv,
                                         uint8_t *bp_dec, uint8_t *osd0, double *lpr, int32_t *bp_iteration) {
    if (!bp4_args_ok(__func__, b, B, synd_x, synd_z, dec, conv)) return SWD_ERR_INVALID;
    return bp4_decode_impl(b, true, synd_x, synd_z, B, dec, conv, bp_dec, osd0, lpr, bp_iteration, nullptr, nullptr);
}

extern "C" int swd_bp4_decode_batch_host_llr(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *conv,
                                             uint8_t *bp_dec, uint8_t *osd0, double *lpr, int32_t *bp_iteration, const double *channel_llr) {
    if (!bp4_args_ok(__func__, b, B, synd_x, synd_z, dec, conv, channel_llr != nullptr)) return SWD_ERR_INVALID;
    return bp4_decode_impl(b, true, synd_x, synd_z, B, dec, conv, bp_dec, osd0, lpr, bp_iteration, channel_llr, nullptr);
}

// the same with device pointers (e.g. torch tensors) on the caller's stream, no host synchronisation
extern "C" int swd_bp4_decode_batch_device(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                           uint8_t *d_conv, uint8_t *d_bp_dec, uint8_t *d_osd0, double *d_lpr, int32_t *d_bp_iteration,
                                           void *stream) {
    if (!bp4_args_ok(__func__, b, B, d_synd_x, d_synd_z, d_dec, d_conv)) return SWD_ERR_INVALID;
    return bp4_decode_impl(b, false, d_synd_x, d_synd_z, B, d_dec, d_conv, d_bp_dec, d_osd0, d_lpr, d_bp_iteration, nullptr, stream);
}

extern "C" int swd_bp4_decode_batch_device_llr(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                               uint8_t *d_conv, uint8_t *d_bp_dec, uint8_t *d_osd0, double *d_lpr, int32_t *d_bp_iteration,
                                               const double *d_channel_llr, void *stream) {
    if (!bp4_args_ok(__func__, b, B, d_synd_x, d_synd_z, d_dec, d_conv, d_channel_llr != nullptr)) return SWD_ERR_INVALID;
    return bp4_decode_impl(b, false, d_synd_x, d_synd_z, B, d_dec, d_conv, d_bp_dec, d_osd0, d_lpr, d_bp_iteration, d_channel_llr, stream);
}

// bp4_osd.camel_decode (src/bp4_osd.pyx:223-248) for a batch: four BP runs per shot with the last qubit pinned to I / X / Z / Y,
// the converged run with the smallest path metric wins.  min_pm: 10000.0 when no run converged (then dec = 0, converge = 0).
// lpr / bp_iteration: those of the last run (Y), as the reference's properties show after the call.
static int bp4_camel_reserve(swd_bp4 *b, int64_t B) {
    const size_t n = b->n;
    int st;
    if ((st = b->c_synd_x.reserve((size_t)B * b->mx)) || (st = b->c_synd_z.reserve((size_t)B * b->mz)) ||
        (st = b->c_bp_dec.reserve((size_t)B * 8 * n)) || (st = b->c_conv4.reserve((size_t)B * 4)) || (st = b->c_dec.reserve((size_t)B * 2 * n)) ||
        (st = b->c_conv.reserve(B)) || (st = b->c_it4.reserve((size_t)B * 4)) || (st = b->c_it.reserve(B)) ||
        (st = b->c_pm4.reserve((size_t)B * 4)) || (st = b->c_pm.reserve(B)) || (st = b->c_lpr.reserve((size_t)B * n * 3))) return st;
    return SWD_OK;
}

// d_llr5: per-shot priors [5][B][n] on the device (planes 0-2 are read) or nullptr
static int bp4_camel_run(swd_bp4 *b, const u8 *d_sx, const u8 *d_sz, int64_t B, cudaStream_t s, const double *d_llr5) {
    const size_t n = b->n;
    const size_t P = (size_t)B * n;
    if (d_llr5)
        bp4_kernel<true, true><<<(int)std::min<long long>(4 * B, b->grid_llr[1]), 256, b->S.total, s>>>(b->dx->g, b->dz->g, d_llr5, d_llr5 + P, d_llr5 + 2 * P,
            d_sx, d_sz, B, b->max_iter, b->alpha, b->c_bp_dec.p, b->c_conv4.p, b->c_it4.p, b->c_lpr.p, nullptr, nullptr, b->S, b->c_pm4.p);
    else
        bp4_kernel<true><<<(int)std::min<long long>(4 * B, b->grid), 256, b->S.total, s>>>(b->dx->g, b->dz->g, b->llr.p, b->llr.p + n, b->llr.p + 2 * n, d_sx, d_sz, B,
                                                                                           b->max_iter, b->alpha, b->c_bp_dec.p, b->c_conv4.p, b->c_it4.p, b->c_lpr.p, nullptr, nullptr, b->S, b->c_pm4.p);
    CK(cudaGetLastError());
    bp4_camel_finish_kernel<<<(unsigned)std::min<long long>((B + 7) / 8, 4096), 256, 0, s>>>(b->c_bp_dec.p, b->c_conv4.p, b->c_pm4.p, b->c_it4.p, B, (int)n,
                                                                                             b->c_dec.p, b->c_conv.p, b->c_pm.p, b->c_it.p);
    CK(cudaGetLastError());
    return SWD_OK;
}

// host / device and llr5 as bp4_decode_impl
static int bp4_camel_impl(swd_bp4 *b, bool host, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *conv,
                          double *min_pm, double *lpr, int32_t *bp_iteration, const double *llr5, void *stream) {
    if (B == 0) return SWD_OK;
    CK(cudaSetDevice(b->device));
    const size_t n = b->n;
    int st;
    if ((st = bp4_camel_reserve(b, B))) return st;
    cudaStream_t s = host ? b->stream : (cudaStream_t)stream;
    if (host && (st = bp4_stage_inputs(b, b->c_synd_x.p, b->c_synd_z.p, synd_x, synd_z, llr5, B, s))) return st;
    if ((st = bp4_camel_run(b, synd_x, synd_z, B, s, llr5))) return st;
    return bp4_copy_out(host, s, {{dec, b->c_dec.p, (size_t)B * 2 * n}, {conv, b->c_conv.p, (size_t)B}, {min_pm, b->c_pm.p, (size_t)B * 8},
                                  {lpr, b->c_lpr.p, (size_t)B * n * 24}, {bp_iteration, b->c_it.p, (size_t)B * 4}});
}

extern "C" int swd_bp4_camel_decode_batch_host(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *conv,
                                               double *min_pm, double *lpr, int32_t *bp_iteration) {
    if (!bp4_args_ok(__func__, b, B, synd_x, synd_z, dec, conv)) return SWD_ERR_INVALID;
    return bp4_camel_impl(b, true, synd_x, synd_z, B, dec, conv, min_pm, lpr, bp_iteration, nullptr, nullptr);
}

extern "C" int swd_bp4_camel_decode_batch_host_llr(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *conv,
                                                   double *min_pm, double *lpr, int32_t *bp_iteration, const double *channel_llr) {
    if (!bp4_args_ok(__func__, b, B, synd_x, synd_z, dec, conv, channel_llr != nullptr)) return SWD_ERR_INVALID;
    return bp4_camel_impl(b, true, synd_x, synd_z, B, dec, conv, min_pm, lpr, bp_iteration, channel_llr, nullptr);
}

extern "C" int swd_bp4_camel_decode_batch_device(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                                 uint8_t *d_conv, double *d_min_pm, double *d_lpr, int32_t *d_bp_iteration, void *stream) {
    if (!bp4_args_ok(__func__, b, B, d_synd_x, d_synd_z, d_dec, d_conv)) return SWD_ERR_INVALID;
    return bp4_camel_impl(b, false, d_synd_x, d_synd_z, B, d_dec, d_conv, d_min_pm, d_lpr, d_bp_iteration, nullptr, stream);
}

extern "C" int swd_bp4_camel_decode_batch_device_llr(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                                     uint8_t *d_conv, double *d_min_pm, double *d_lpr, int32_t *d_bp_iteration,
                                                     const double *d_channel_llr, void *stream) {
    if (!bp4_args_ok(__func__, b, B, d_synd_x, d_synd_z, d_dec, d_conv, d_channel_llr != nullptr)) return SWD_ERR_INVALID;
    return bp4_camel_impl(b, false, d_synd_x, d_synd_z, B, d_dec, d_conv, d_min_pm, d_lpr, d_bp_iteration, d_channel_llr, stream);
}
