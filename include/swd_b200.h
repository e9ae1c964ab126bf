/*
 * swd_b200.h — C-ABI of the B200-native batched window decoder (libswd_b200.so).
 *
 * Drop-in boundary for the hot path of gongaa/SlidingWindowDecoder: one handle
 * replaces one Cython decoder object of the reference and decodes a BATCH of
 * syndromes of the same window on one B200.  Plain pointers and sizes only; no
 * torch / numpy types.  Every entry point returns an int status (0 = OK, <0 =
 * error, see swd_strerror) and never aborts the process (the reference's C
 * layer may exit(1)/abort(), mod2sparse.c:94-97, mod2sparse_extra.cpp:139).
 *
 * Reference interfaces replaced (file:line under the reference's src/):
 *   swd_create            <- bp_history_decoder.__cinit__  bp_guessing_decoder.pyx:6-46
 *                            bpgdg_decoder.__cinit__       bp_guessing_decoder.pyx:161-219
 *                            bpgd_decoder.__cinit__        bp_guessing_decoder.pyx:474-499
 *                            osd_window.__cinit__          osd_window.pyx:8-126
 *                            (numpy2mod2sparse / spmatrix2mod2sparse, mod2sparse.pyx:6-32)
 *   swd_decode_batch_*    <- bpgdg_decoder.decode          bp_guessing_decoder.pyx:221-236
 *                            bpgd_decoder.decode           bp_guessing_decoder.pyx:501-514
 *                            osd_window.decode             osd_window.pyx:158-199
 *                            which in turn replace BPGD_main_thread::do_work (bpgd.cpp:591-688),
 *                            BPGD::{reset,min_sum_log,select_vn,peel,vn_set_value,get_pm}
 *                            (bpgd.cpp:13-351), index_sort (bpgd.cpp:384-389),
 *                            mod2sparse_decomp_osd + LU_forward_backward_solve
 *                            (mod2sparse_extra.cpp:78-376)
 *   swd_destroy           <- __dealloc__                   bp_guessing_decoder.pyx:142-154,444-469
 *   swd_window_*          <- the per-window bookkeeping of guessing.py:141-227 / osd.py:134-179
 *                            (commit first F rounds, syndrome update, flagged / logical counters)
 */
#ifndef SWD_B200_H
#define SWD_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWD_OK               0
#define SWD_ERR_INVALID     -1   /* bad argument (NULL, negative size, length mismatch)            */
#define SWD_ERR_UNSUPPORTED -2   /* graph exceeds a kernel limit (see DESIGN.md "limits")           */
#define SWD_ERR_CUDA        -3   /* CUDA runtime error; text via swd_last_error()                   */
#define SWD_ERR_NOMEM       -4

/* decoder kinds == the reference's three decoder classes */
#define SWD_KIND_BPGDG       0   /* bpgdg_decoder  (GDG)                    */
#define SWD_KIND_BPGD        1   /* bpgd_decoder   (plain guided decimation) */
#define SWD_KIND_OSD_WINDOW  2   /* osd_window     (BP + shortening + OSD)   */

#define SWD_OSD_0  0
#define SWD_OSD_E  1
#define SWD_OSD_CS 2

/* kwargs of the reference constructors, same meaning and defaults
 * (bp_guessing_decoder.pyx:7-9,162-171,475-478; osd_window.pyx:10-16). */
typedef struct swd_config {
    int    kind;
    int    device;                /* CUDA device ordinal                                         */
    /* BP on the full window ("max_iter" / "pre_max_iter") */
    int    max_iter;
    double ms_scaling_factor;
    /* GDG / GD */
    int    max_iter_per_step;
    int    max_step;
    int    max_tree_depth;
    int    max_side_depth;
    int    max_tree_branch_step;
    int    max_side_branch_step;
    double gdg_factor;            /* gdg_factor, or gd_factor for SWD_KIND_BPGD                   */
    int    new_n;                 /* <= 0 : min(n, 2m)                                            */
    int    multi_thread;          /* 1: bpgd.cpp branch tree; 0: single-thread schedule (pyx:254) */
    int    low_error_mode;
    /* osd_window */
    int    post_max_iter;
    int    osd_method;            /* SWD_OSD_*                                                    */
    int    osd_order;
    /* BP flavour of the full-window BP: SWD_BP_MIN_SUM (the reference's own decoders) or SWD_BP_PRODUCT_SUM (what the
     * drivers can ask of ldpc.BpOsdDecoder via bp_method="product_sum", osd.py:142-150; third-party, parity unpinned). */
    int    bp_method;
} swd_config;
#define SWD_BP_MIN_SUM      0
#define SWD_BP_PRODUCT_SUM  1

typedef struct swd_decoder swd_decoder;

/* Work counters accumulated since creation / last reset (for roofline accounting). */
typedef struct swd_counters {
    uint64_t shots;               /* syndromes decoded                                           */
    uint64_t pre_bp_edge_iters;   /* edges x iterations executed by the full-window BP kernel    */
    uint64_t path_edge_iters;     /* active edges x iterations executed inside GDG/GD/post-BP    */
    uint64_t gdg_shots;           /* shots that went past the pre-BP                             */
    uint64_t osd_shots;           /* shots that reached OSD                                      */
    uint64_t kernel_launches;     /* kernels launched by this library                            */
    uint64_t paths_run;           /* branch paths that executed at least one BP call             */
    uint64_t bp_calls;            /* min_sum_log-equivalent calls over all branch paths          */
    uint64_t path_vn_iters;       /* active variable nodes x iterations inside GDG/GD/post-BP    */
    uint64_t path_cn_iters;       /* active check nodes x iterations inside GDG/GD/post-BP       */
    uint64_t path_slot_iters;     /* message slots (live, dead, pad) scanned by those check passes */
    uint64_t osd_cols_scanned;    /* columns gathered against T by osd_kernel's elimination scan */
    uint64_t osd_pivots;          /* pivots found (= rank x OSD shots)                           */
} swd_counters;

/* Kernel classes for swd_get_kernel_times */
#define SWD_K_PRE_BP     0
#define SWD_K_SORT_RESET 1
#define SWD_K_PATH_MAIN  2   /* path_kernel phase 0: main + tree branches (or the single GD / post-BP path) */
#define SWD_K_PATH_SIDE  3   /* path_kernel phase 1: side branches                                         */
#define SWD_K_SELECT     4
#define SWD_K_OSD        5   /* osd_window: osd_kernel + finish / path-metric kernels */
#define SWD_K_PATH_TRUNK 6   /* path_kernel on shared-prefix nodes (decimation depths < max_tree_depth)                 */
#define SWD_K_POST_BP    7   /* osd_window: masked min-sum on the shortened graph (post_bp_kernel)                               */
#define SWD_K_COUNT      8

/* pcm as CSC: colptr[n+1], rowidx[nnz] (any order inside a column; sorted internally, as
 * mod2sparse_insert keeps them).  channel_llr[n] = log((1-p)/p) computed by the caller with libm
 * (bp_guessing_decoder.pyx:46).  All arrays are HOST pointers and are copied. */
int  swd_create(const swd_config *cfg, int m, int n, const int32_t *colptr, const int32_t *rowidx,
                const double *channel_llr, swd_decoder **out);
void swd_destroy(swd_decoder *d);

/* Decode B syndromes. synd[B*m], corr[B*n] one byte per bit (0/1), converge[B];
 * min_pm[B] optional (NULL ok).  _host: host pointers, H2D/D2H copies inside the call,
 * synchronous.  _device: device pointers, asynchronous on `stream` (a cudaStream_t). */
int  swd_decode_batch_host(swd_decoder *d, const uint8_t *synd, int64_t B,
                           uint8_t *corr, uint8_t *converge, double *min_pm);
int  swd_decode_batch_device(swd_decoder *d, const uint8_t *d_synd, int64_t B,
                             uint8_t *d_corr, uint8_t *d_converge, double *d_min_pm, void *stream);

/* Bit-packed shot I/O (8x fewer bytes over PCIe / HBM at the boundary): row b of a packed array holds ceil(nbits / 64)
 * uint64 words, bit j of the row = (word[j >> 6] >> (j & 63)) & 1  (numpy: packbits(bitorder="little").view(uint64)).
 * synd_packed [B, ceil(m/64)], corr_packed [B, ceil(n/64)]; converge / min_pm as above.  Same decode(syndrome) semantics
 * as the byte entry points (bp_guessing_decoder.pyx:221-252, osd_window.pyx:158-199).  The _device variant unpacks into /
 * packs from the decoder's own staging buffers on `stream`: calls on one decoder must be stream-ordered. */
int  swd_decode_batch_host_packed(swd_decoder *d, const uint64_t *synd_packed, int64_t B,
                                  uint64_t *corr_packed, uint8_t *converge, double *min_pm);
int  swd_decode_batch_device_packed(swd_decoder *d, const uint64_t *d_synd_packed, int64_t B,
                                    uint64_t *d_corr_packed, uint8_t *d_converge, double *d_min_pm, void *stream);
/* Per-shot channel priors: the four entry points above with one more argument, channel_llr [B*n] row-major (host pointer for
 * the _host variants, device pointer for the _device variants; B rows of n LLRs, column order of the decoder's pcm).  Row b
 * decodes syndrome b exactly as a decoder created with channel_llr = row b would (corrections, converge, min_pm and the
 * osd_window outputs of swd_osd_last_outputs).  Allowed values are those swd_create accepts: 0.0 (erasure, p = 1/2), +inf
 * (p = 0), negative values (p > 1/2).  NaN is undefined behaviour (the branch-path kernels mark decided variable nodes with
 * NaN messages).  channel_llr == NULL returns SWD_ERR_INVALID.  The _host variants copy the priors one workspace chunk at a
 * time (8 bytes per prior over PCIe: device-resident priors are the intended use); the _device variants read them on
 * `stream`, so calls on one decoder must be stream-ordered. */
int  swd_decode_batch_host_llr(swd_decoder *d, const uint8_t *synd, int64_t B, uint8_t *corr, uint8_t *converge, double *min_pm,
                               const double *channel_llr);
int  swd_decode_batch_device_llr(swd_decoder *d, const uint8_t *d_synd, int64_t B, uint8_t *d_corr, uint8_t *d_converge,
                                 double *d_min_pm, const double *d_channel_llr, void *stream);
int  swd_decode_batch_host_packed_llr(swd_decoder *d, const uint64_t *synd_packed, int64_t B, uint64_t *corr_packed,
                                      uint8_t *converge, double *min_pm, const double *channel_llr);
int  swd_decode_batch_device_packed_llr(swd_decoder *d, const uint64_t *d_synd_packed, int64_t B, uint64_t *d_corr_packed,
                                        uint8_t *d_converge, double *d_min_pm, const double *d_channel_llr, void *stream);
/* the two conversions on their own (device pointers), for callers that keep shot data packed (window driver, samplers) */
int  swd_pack_bits(int device, const uint8_t *d_bytes, int64_t B, int nbits, uint64_t *d_packed, void *stream);
int  swd_unpack_bits(int device, const uint64_t *d_packed, int64_t B, int nbits, uint8_t *d_bytes, void *stream);
/* 1 if the full-window BP of this decoder streams its messages from HBM (graph beyond one SM's shared memory), else 0 */
int  swd_is_streamed(swd_decoder *d);
/* Host-only diagnostic (no CUDA call): the shared-memory message layout swd_create chooses for the full-window BP kernel of
 * this graph (static per decoder: row starts on distinct banks, slot order inside a row chosen so that both passes of
 * bp_decode_llr, bp_guessing_decoder.pyx:62-127, are bank-conflict free).  slot_of_entry [nnz] (per CSC entry, rows ascending
 * inside a column), row_start [m + 1], stats[3] = {slots incl. pads, extra variable-pass wavefronts of the plain CSR order,
 * of the chosen layout}; any pointer may be NULL.  optimize = 0: the plain CSR order. */
int  swd_pre_bp_layout(int m, int n, const int32_t *colptr, const int32_t *rowidx, int optimize,
                       int32_t *slot_of_entry, int32_t *row_start, int64_t *stats);

/* osd_window read-only properties of the LAST batch (osd_window.pyx:487-517), host copies.
 * Any pointer may be NULL.  bp_dec/osd0/osdw: [B*n]; log_prob_ratios: [B*n*4]; bp_iteration: [B]. */
int  swd_osd_last_outputs(swd_decoder *d, int64_t B, uint8_t *bp_dec, uint8_t *osd0, uint8_t *osdw,
                          double *log_prob_ratios, int32_t *bp_iteration);

/* Per-kernel device timing.  When enabled, every kernel launch is bracketed by a pair of CUDA events
 * on the launching stream; swd_get_kernel_times synchronises, sums the elapsed times per kernel class
 * into ms[SWD_K_COUNT] / launches[SWD_K_COUNT] (accumulated since the last call) and recycles the events.
 * The work counters of the branch-path / post-BP min-sum calls (swd_counters: path_edge_iters, path_vn_iters, path_cn_iters,
 * path_slot_iters) accumulate only while profiling is enabled: counting them costs 1.7 % of the decoded shots/s. */
int  swd_set_profiling(swd_decoder *d, int enable);
int  swd_get_kernel_times(swd_decoder *d, double *ms, uint64_t *launches);

int  swd_get_counters(swd_decoder *d, swd_counters *out);
int  swd_reset_counters(swd_decoder *d);
int  swd_rank(swd_decoder *d);          /* GF(2) rank of the pcm (mod2sparse_rank), -1 if n/a      */
int  swd_new_n(swd_decoder *d);

/* ---- sliding-window bookkeeping on the device (guessing.py:204-227, osd.py:170-179) ------------
 * A "window plan" holds the full detector matrix chk (num_det x num_col, CSC) and the observable
 * matrix obs (num_obs x num_col, CSC).  All shot data is one byte per bit, row-major, on device. */
typedef struct swd_window swd_window;
int  swd_window_create(int device, int num_det, int num_col, const int32_t *chk_colptr, const int32_t *chk_rowidx,
                       int num_obs, const int32_t *obs_colptr, const int32_t *obs_rowidx, swd_window **out);
void swd_window_destroy(swd_window *w);
/* copy syndrome columns [row0,row0+m) of d_det[B,num_det] into d_synd[B,m]  (detector_win = new_det_data[:, a0:b0]) */
int  swd_window_extract(swd_window *w, const uint8_t *d_det, int64_t B, int row0, int m, uint8_t *d_synd, void *stream);
/* commit: for every shot XOR chk[:, col0+j] into d_det and obs[:, col0+j] into d_obs for each j < ncommit with
 * d_corr[b, j] == 1 (d_corr has row stride n_win); i.e. new_det = det + e_hat @ chk.T restricted to the commit. */
int  swd_window_commit(swd_window *w, const uint8_t *d_corr, int64_t B, int n_win, int col0, int ncommit,
                       uint8_t *d_det, uint8_t *d_obs, void *stream);
/* counts over shots: flagged = any(det residual), logical = flagged or any(obs residual). out[0]=flagged, out[1]=failed */
int  swd_window_count_failures(swd_window *w, const uint8_t *d_det, const uint8_t *d_obs, int64_t B,
                               unsigned long long *d_out2, void *stream);

/* DEM sampling on the device - what CompiledDemSampler.sample draws in the reference's drivers (guessing.py:129-130):
 * one independent Bernoulli(priors[c]) per DEM column, det = chk . e, obs = obs_mat . e (mod 2).  Philox4x32-10 keyed by
 * `seed`, counter = (shot_offset + b, column block): shot b of a call with offset o equals shot 0 of a call with offset o + b.
 * d_err (optional, [B, num_col]) receives the sampled error vectors. */
int  swd_window_set_priors(swd_window *w, const double *priors /* host, [num_col] */);
int  swd_window_sample(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det, uint8_t *d_obs,
                       uint8_t *d_err, void *stream);

/* Code-capacity sampling on the device: depolarizing noise with heralded erasures on the n data qubits of a CSS code.  The plan
 * has num_col = 2n columns: column v is the X part of qubit v, column n + v its Z part (the [B][2][n] layout of bp4 `dec`).  For
 * a CSS pair build chk = [[0, Hx], [Hz, 0]], so det = [synd_x | synd_z] with synd_x = Hx . e_z and synd_z = Hz . e_x (the
 * convention of swd_bp4_*), and obs = [[lz, 0], [0, lx]]: the X part is tested against the Z logicals and the Z part against
 * the X logicals.  Nothing else is CSS-specific: the sampler XORs the chk / obs columns of the bits it sets.
 * swd_window_set_pauli_priors: per-qubit px, py, pz (host, [n] each; non-negative, px + py + pz <= 1), erasure_rate in
 * [0, 1], optional llr5 (host, [5][n]: the static rows of swd_bp4_create, llr_x, llr_y, llr_z, prior_llr_x, prior_llr_z).
 * Thresholds are those of swd_window_set_priors, floor(x * 2^32) clamped to 0xffffffff, of px, px + py and (px + py) + pz
 * and erasure_rate, computed in double on the host.  SWD_ERR_INVALID if num_col != 2n or a value is out of range.
 * swd_window_sample_pauli draws, for shot s = shot_offset + b, one Philox4x32-10 call per qubit pair k keyed by `seed` with
 * counter (k, 1, s & 0xffffffff, s >> 32); words 2j and 2j + 1 are the erasure draw w_e and the Pauli draw w_p of qubit 2k + j.
 * The qubit is erased iff w_e < thr(erasure_rate); an erased qubit's Pauli is w_p >> 30 (0 I, 1 X, 2 Y, 3 Z), any other qubit
 * is X if w_p < thr(px), else Y if w_p < thr(px + py), else Z if w_p < thr(px + py + pz), else I.  e_x = X or Y, e_z = Y or Z.
 * Outputs (device, one byte per bit): d_det [B][num_det] and d_obs [B][num_obs] required; optional (NULL allowed) d_err
 * [B][2n], d_erased [B][n], d_channel_llr [5][B][n] doubles (plane q row b = llr5[q] with 0.0 at the erased qubits of shot b;
 * needs llr5).  Asynchronous on `stream`; B == 0 is a no-op.  Score decoded shots with swd_window_commit(w, d_dec, B, 2n, 0,
 * 2n, d_det, d_obs, stream) and swd_window_count_failures. */
int  swd_window_set_pauli_priors(swd_window *w, int n, const double *px, const double *py, const double *pz,
                                 double erasure_rate, const double *llr5 /* [5*n] host, may be NULL */);
int  swd_window_sample_pauli(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det, uint8_t *d_obs,
                             uint8_t *d_err, uint8_t *d_erased, double *d_channel_llr, void *stream);

/* Circuit-level sampling with heralded erasures on the device.  The window's columns are the DEM columns of a circuit; a
 * noise location l (one DEPOLARIZE2 instruction, or one target of X_ERROR / Z_ERROR / DEPOLARIZE1: dem.noise_locations) has
 * n_l = mech_ptr[l + 1] - mech_ptr[l] (1 .. 15) independent mechanisms k, each with a probability mech_prob[k] in [0, 1/2]
 * and the DEM column of its symptom mech_col[k] (-1: empty symptom).  Location l is erased with probability
 * erasure_rate[l] in [0, 1]; an erased location's mechanisms fire with probability exactly 1/2 (a uniformly random Pauli).
 * swd_window_set_circuit_noise copies the tables (host arrays) and col_llr (host, [num_col], the static LLR row; NULL if no
 * LLR rows will be asked for).  Thresholds thr(x) = floor(x * 2^32) clamped to 0xffffffff, computed in double on the host.
 * SWD_ERR_INVALID for a NULL table, num_loc <= 0, mech_ptr[0] != 0, a count outside 1 .. 15, a column outside [-1, num_col),
 * a probability outside [0, 1/2] or a rate outside [0, 1] (NaN included).
 * swd_window_sample_circuit: for shot s = shot_offset + b, location l uses draws t = 0 .. n_l; draw t is word t & 3 of
 * Philox4x32-10 keyed by `seed` with counter (l, 2 + (t >> 2), s & 0xffffffff, s >> 32).  Draw 0 is the erasure draw
 * (erased iff w < thr(erasure_rate[l])); draw 1 + k is mechanism k, which fires iff w < (erased ? 0x80000000 : thr(p_k)).
 * Every draw is made.  Outputs (device, one byte per bit): d_det [B][num_det] and d_obs [B][num_obs] required; optional
 * (NULL allowed) d_err [B][num_col] (parity of the fired mechanisms per column: det = chk . err, obs = obs_mat . err),
 * d_erased [B][num_loc], d_channel_llr [B][num_col] doubles (col_llr with 0.0 at every column of an erased location's
 * mechanisms; needs col_llr).  Asynchronous on `stream`; B == 0 is a no-op; SWD_ERR_UNSUPPORTED if one warp's parity and
 * column words do not fit in shared memory. */
int  swd_window_set_circuit_noise(swd_window *w, int num_loc, const int32_t *mech_ptr, const int32_t *mech_col,
                                  const double *mech_prob, const double *erasure_rate /* [num_loc] */,
                                  const double *col_llr /* [num_col] host, may be NULL */);
int  swd_window_sample_circuit(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det, uint8_t *d_obs,
                               uint8_t *d_err, uint8_t *d_erased, double *d_channel_llr, void *stream);

/* Soft measurement readout on top of the circuit noise above.  A readout location is an X_ERROR (Z_ERROR) target whose next
 * instruction on that qubit is M / MR (MX / MRX): dem.readout_locations.  readout_loc [num_readout] lists them (indices into
 * the locations of swd_window_set_circuit_noise, each with exactly one mechanism, no two with the same DEM column).  The K =
 * num_classes (1 .. 256) reliability classes are shared by all of them: a readout location draws class k with probability
 * class_weight[k] (>= 0, summing to 1 within 1e-9) and then flips with probability flip_prob[k] in [0, 1/2] (its own
 * probability in mech_prob is not used).  class_llr [num_readout * K] (host, row r = readout r; NULL if no LLR rows will be
 * asked for) is the LLR of readout r's DEM column when r is in class k; rows of readouts without a column are not read.
 * swd_window_set_circuit_readout copies the tables; SWD_ERR_INVALID for a NULL table, num_readout <= 0, a call before
 * swd_window_set_circuit_noise, a location out of range or listed twice, a location with n_l != 1, K outside 1 .. 256, a
 * negative or NaN weight, weights summing to more than 1e-9 away from 1, a flip_prob outside [0, 1/2] (NaN included), or
 * two readout locations whose mechanisms share a DEM column.  A later swd_window_set_circuit_noise clears it, and
 * swd_window_sample_circuit ignores it.
 * swd_window_sample_circuit_readout: every location draws as in swd_window_sample_circuit except readout locations, which
 * use words 0, 1, 2 of their one Philox call (counter (l, 2, s & 0xffffffff, s >> 32)): word 0 is the erasure draw, word 2
 * the class (the number of k in 1 .. K-1 with w >= thr(class_weight[0] + .. + class_weight[k-1]), sums left to right in
 * double) and word 1 the flip, which fires iff w < (erased ? 0x80000000 : thr(flip_prob[class])).  With K = 1 and flip_prob
 * = {p} it reproduces swd_window_sample_circuit.  Outputs as swd_window_sample_circuit, plus optional d_readout
 * [B][num_readout] (the classes, in readout_loc order); d_channel_llr [B][num_col] is col_llr with class_llr[r][class_r] at
 * readout r's column and 0.0 at every column of an erased location (needs col_llr and class_llr).  SWD_ERR_INVALID before
 * swd_window_set_circuit_readout and for the pointer / size errors of swd_window_sample_circuit; SWD_ERR_UNSUPPORTED if one
 * warp's words and class bytes do not fit in shared memory. */
int  swd_window_set_circuit_readout(swd_window *w, int num_readout, const int32_t *readout_loc, int num_classes,
                                    const double *class_weight /* [K] */, const double *flip_prob /* [K] */,
                                    const double *class_llr /* [num_readout * K] host, may be NULL */);
int  swd_window_sample_circuit_readout(swd_window *w, uint64_t seed, int64_t shot_offset, int64_t B, uint8_t *d_det,
                                       uint8_t *d_obs, uint8_t *d_err, uint8_t *d_erased, uint8_t *d_readout,
                                       double *d_channel_llr, void *stream);

/* ---- bp4_osd (src/bp4_osd.pyx:6-684): quaternary min-sum BP over the pair (Hx, Hz) of a CSS code under depolarizing
 * noise, then one OSD per basis for shots whose BP did not converge.  Replaces bp4_osd.__cinit__ / decode (pyx:8-221);
 * swd_bp4_camel_decode_batch_host replaces camel_decode (pyx:223-248).  The two graphs have no column- / row-weight limit
 * (CAMEL codes tie every check to the last qubit).  llr_*: log((1-px-py-pz)/p_*) per qubit, prior_llr_x / _z:
 * log((1-(px+py))/(px+py)) and log((1-(pz+py))/(pz+py)) (pyx:123-133), computed by the caller with libm.
 * decode: synd_x[B*mx] (syndrome of Hx, i.e. of the Z part), synd_z[B*mz]; dec[B*2n] = x part then z part per shot
 * (stackchar2numpy); optional bp_dec / osd0 [B*2n], log_prob_ratios [B*n*3] (x, y, z), bp_iteration [B]. */
typedef struct swd_bp4 swd_bp4;
int  swd_bp4_create(int device, int mx, int mz, int n, const int32_t *hx_colptr, const int32_t *hx_rowidx,
                    const int32_t *hz_colptr, const int32_t *hz_rowidx, const double *llr_x, const double *llr_y,
                    const double *llr_z, const double *prior_llr_x, const double *prior_llr_z, int max_iter,
                    double ms_scaling_factor, int osd_method, int osd_order, swd_bp4 **out);
void swd_bp4_destroy(swd_bp4 *b);
int  swd_bp4_rank(swd_bp4 *b, int which /* 0: Hx, 1: Hz */);
int  swd_bp4_decode_batch_host(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec, uint8_t *converge,
                               uint8_t *bp_dec, uint8_t *osd0, double *log_prob_ratios, int32_t *bp_iteration);
/* camel_decode (pyx:223-248): four BP runs per shot with the last qubit pinned to I / X / Z / Y (vn_set_value, pyx:389-423), the
 * converged run with the smallest path metric (cal_pm, pyx:250-259) wins, ties to the earlier value.  dec[B*2n], converge[B];
 * optional min_pm[B] (10000.0 and dec = 0 when no run converged - the reference returns an earlier call's buffer there),
 * log_prob_ratios [B*n*3] and bp_iteration [B] of the last run, as the reference's properties hold after the call. */
int  swd_bp4_camel_decode_batch_host(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec,
                                     uint8_t *converge, double *min_pm, double *log_prob_ratios, int32_t *bp_iteration);
/* The same two calls with device pointers (e.g. torch tensors) on the caller's stream, without host synchronisation; the
 * optional outputs may be NULL.  Results pass through the decoder's own buffers: calls on one swd_bp4 must be stream-ordered. */
int  swd_bp4_decode_batch_device(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                 uint8_t *d_converge, uint8_t *d_bp_dec, uint8_t *d_osd0, double *d_log_prob_ratios,
                                 int32_t *d_bp_iteration, void *stream);
int  swd_bp4_camel_decode_batch_device(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                       uint8_t *d_converge, double *d_min_pm, double *d_log_prob_ratios, int32_t *d_bp_iteration,
                                       void *stream);
/* Per-shot channel priors: the four bp4 calls above with one more argument, channel_llr = five planes [5][B][n] of float64,
 * row-major (a host pointer for the _host variants, a device pointer on `stream` for the _device variants).  Plane k, row b
 * is the k-th LLR array of swd_bp4_create for shot b, in the order llr_x, llr_y, llr_z, prior_llr_x, prior_llr_z.  Row b
 * decodes syndrome b exactly as a swd_bp4 created with those five rows would, in every output (dec, converge, bp_dec, osd0,
 * log_prob_ratios, bp_iteration, min_pm).  The camel variants read planes 0-2 only; they take the same layout so that both
 * calls can share one array.  Allowed values are finite doubles of either sign; an erased qubit (a uniformly random Pauli,
 * px = py = pz = 1/4) is 0.0 in all five planes.  +-inf and NaN are undefined behaviour.  channel_llr == NULL returns
 * SWD_ERR_INVALID.  The _host variants stage the priors in a device buffer of 5*B*n doubles, allocated on the first such
 * call; the static calls never allocate it. */
int  swd_bp4_decode_batch_host_llr(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec,
                                   uint8_t *converge, uint8_t *bp_dec, uint8_t *osd0, double *log_prob_ratios,
                                   int32_t *bp_iteration, const double *channel_llr);
int  swd_bp4_decode_batch_device_llr(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B, uint8_t *d_dec,
                                     uint8_t *d_converge, uint8_t *d_bp_dec, uint8_t *d_osd0, double *d_log_prob_ratios,
                                     int32_t *d_bp_iteration, const double *d_channel_llr, void *stream);
int  swd_bp4_camel_decode_batch_host_llr(swd_bp4 *b, const uint8_t *synd_x, const uint8_t *synd_z, int64_t B, uint8_t *dec,
                                         uint8_t *converge, double *min_pm, double *log_prob_ratios, int32_t *bp_iteration,
                                         const double *channel_llr);
int  swd_bp4_camel_decode_batch_device_llr(swd_bp4 *b, const uint8_t *d_synd_x, const uint8_t *d_synd_z, int64_t B,
                                           uint8_t *d_dec, uint8_t *d_converge, double *d_min_pm, double *d_log_prob_ratios,
                                           int32_t *d_bp_iteration, const double *d_channel_llr, void *stream);

const char *swd_strerror(int status);
const char *swd_last_error(void);
const char *swd_version(void);

#ifdef __cplusplus
}
#endif
#endif
