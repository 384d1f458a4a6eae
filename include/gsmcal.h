/* gsmcal.h - C ABI of the B200-native GSM sync/calibration hot path.
 *
 * Each entry point replaces one MATLAB function (or inline call site) of
 * JiaoXianjun/multi-rtl-sdr-calibration; the reference has no FFI of its own, its boundary is the
 * MATLAB function call, so a same-named MEX gateway (multi-rtl-sdr-calibration_b200/mex/) binds
 * these symbols and shadows the .m file.  Citations are file:line into the reference.
 *
 * Conventions (all entry points)
 *   - plain pointers + sizes; HOST memory unless a parameter says otherwise; caller allocates outputs.  Host buffers may be
 *     pageable (an mxArray, a NumPy array): transfers above 32 MB then go through the library's own multi-threaded pinned staging
 *     ring (~4x the rate of cudaMemcpy from pageable memory); pinned / registered buffers are used directly.
 *   - matrices are column-major as MATLAB holds them; one stream (dongle / scanned frequency) per column.
 *   - complex128 is interleaved (re,im) pairs of doubles ("double[2]").
 *   - positions / indices are 1-based doubles exactly as the reference returns them.
 *   - return value: GSMCAL_OK or a negative error code; gsmcal_last_error() gives the text.
 *     The reference's own failure *sentinels* (-1 / [-1,-1] / inf) are NOT errors: they are reported
 *     through the count/length outputs (-1 means "the scalar -1") so a gateway can rebuild them.
 *   - every compute call runs hand-written sm_100a kernels; there is no CPU fallback: without a CUDA
 *     device the call fails with GSMCAL_ERR_CUDA.
 *
 * Limits that the reference (MATLAB, unbounded) does not have; every one is checked and reported as GSMCAL_ERR_ARG:
 *   - oversampling_ratio 1..8 in FCCH_fine_correction / SCH_corr_rate_correction / carrier_correct_post_SCH / calibrate_batch
 *     (shared-memory windows are sized for 148*8 samples; the reference scripts only ever use 8);
 *   - fft_len <= 128 in the moving-FFT functions (FCCH_coarse_position uses 16);
 *   - n_taps <= 128 (GSMCAL_MAX_TAPS: the numerator lives in constant memory; the reference uses 47 / 31 / 64 / 60 / 30);
 *   - at most 65,535 streams (columns) per call (CUDA grid y dimension);
 *   - calls are serialised by one process-wide mutex (the MEX entry is single-threaded anyway); _collect / _cancel wait outside it.
 */
#ifndef GSMCAL_H
#define GSMCAL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSMCAL_OK            0
#define GSMCAL_ERR_ARG      -1   /* malformed argument */
#define GSMCAL_ERR_CUDA     -2   /* CUDA runtime failure / no device */
#define GSMCAL_ERR_CAPACITY -3   /* caller-provided output too small */
#define GSMCAL_ERR_RANGE    -4   /* the reference would raise an index-out-of-bounds error here */

#define GSMCAL_ABI_VERSION 1

int         gsmcal_abi_version(void);
const char *gsmcal_last_error(void);
int         gsmcal_device_count(void);          /* 0 when no CUDA device is usable */
int         gsmcal_set_device(int device);      /* device used by the calling thread's later calls */
void        gsmcal_release(void);               /* frees cached device workspaces (mexAtExit) */

/* ---- K1  b = raw2iq(a)                                             raw2iq.m:5-8 ------------------
 * a: (2*n_iq) x n_col, I at odd rows; b: n_iq x n_col complex128.  uint8 (what rtl_tcp delivers,
 * multi_rtl_sdr_split_scanner.m:70) or double holding 0..255 (fread, gsm_sync_demod.m:96). */
int gsmcal_raw2iq_u8 (const uint8_t *a, int64_t n_iq, int64_t n_col, double *b);
int gsmcal_raw2iq_f64(const double  *a, int64_t n_iq, int64_t n_col, double *b);

/* ---- K2  r = filter(coef,1,s); r = r(1:decim:end,:)   gsm_sync_demod.m:34,110,117;
 *          multi_rtl_sdr_gsm_FCCH_scanner.m:53,133,135; multi_rtl_sdr_split_scanner.m:54,155-156 ----
 * s: n x n_col complex128, coef: n_taps real (<=128), r: ceil(n/decim) x n_col complex128. */
int gsmcal_fir1(int order, double wn, double *coef /* order+1 */);      /* MATLAB fir1(order, wn) */
int gsmcal_fir_filter(const double *coef, int n_taps, const double *s, int64_t n, int64_t n_col,
                      int decim, double *r);
/* fused raw2iq -> filter -> decimate straight from the uint8 wire format (same result as the two calls) */
int gsmcal_raw2iq_fir_u8(const uint8_t *a, int64_t n_iq, int64_t n_col, const double *coef, int n_taps,
                         int decim, double *r);
/* r = chn_filter_8x_4x(s)  chn_filter_8x_4x.m:5-15 (60-tap Num, keep rows 1:2:end);
 * r = chn_filter_4x(s)     chn_filter_4x.m:5-13   (30-tap Num).  Num recovered from the .fda sessions. */
int gsmcal_chn_filter_8x_4x(const double *s, int64_t n, int64_t n_col, double *r /* ceil(n/2) x n_col */);
int gsmcal_chn_filter_4x   (const double *s, int64_t n, int64_t n_col, double *r /* n x n_col */);
int gsmcal_chn_filter_taps (int which /* 8 or 4 */, double *coef /* >=60 */, int *n_taps);

/* ---- scanners: mean(abs(r(1:decim:end,:)).^2,1) after raw2iq [+ filter]
 *      scan_band_power_spectrum.m:80-85 (coef NULL, decim 1); multi_rtl_sdr_split_scanner.m:154-156 ---- */
int gsmcal_band_power_u8(const uint8_t *a, int64_t n_iq, int64_t n_col, const double *coef, int n_taps,
                         int decim, double *power /* n_col, linear */);

/* diversity scanner, multi_rtl_sdr_diversity_scanner.m:150-176: every dongle scans the same band.
 * s_all: (2*n_iq) x n_freq x n_dongle uint8 as the script holds it (:118-131).  power_spectrum: n_dongle x n_freq (column-major),
 * power_spectrum(i,:) = mean(abs(r_flt(1:decim:end,:)).^2, 1) of dongle i (:152-156); power_spectrum_combine: 1 x n_freq =
 * mean(power_spectrum, 1) (:172), linear units.  The combination runs on the device (one kernel after the per-column means). */
int gsmcal_diversity_power_u8(const uint8_t *s_all, int64_t n_iq, int64_t n_freq, int64_t n_dongle, const double *coef, int n_taps,
                              int decim, double *power_spectrum, double *power_spectrum_combine);

/* ---- K3  [hit_flag,hit_idx,hit_avg_snr,hit_snr] = move_fft_snr_runtime_avg(s,mv_len,fft_len,th)
 *          move_fft_snr_runtime_avg.m:5-50.   No hit: 0, -1, inf, inf.  fft_len <= 128. ---- */
int gsmcal_move_fft_snr_runtime_avg(const double *s, int64_t len, int mv_len, int fft_len, double th,
                                    int *hit_flag, double *hit_idx, double *hit_avg_snr, double *hit_snr);
/* the per-window SNR trace the reference computes and discards (move_fft_snr_runtime_avg.m:15,28), all
 * len-fft_len+1 windows, no early exit: the "moving-FFT SNR scan" of BASELINE config 4 */
int gsmcal_move_fft_snr_trace(const double *s, int64_t len, int fft_len, double *snr);
/* [hit_flag,hit_idx,hit_snr] = specific_fft_snr_fix_avg(s,target_set,fft_len,th,avg_snr)
 * specific_fft_snr_fix_avg.m:5-34 */
int gsmcal_specific_fft_snr_fix_avg(const double *s, int64_t len, int64_t target_first, int64_t target_last,
                                    int fft_len, double th, double avg_snr,
                                    int *hit_flag, double *hit_idx, double *hit_snr);

/* ---- K4  [position,snr] = FCCH_coarse_position(s,decimation_ratio)   FCCH_coarse_position.m:5-94 ----
 * *n_out = -1 -> position = snr = -1 (scalars); else 1 x n_out rows.  cap >= gsmcal_max_bursts(). */
int gsmcal_FCCH_coarse_position(const double *s, int64_t len, int decimation_ratio,
                                double *position, double *snr, int64_t cap, int64_t *n_out);
int64_t gsmcal_max_bursts(int64_t len_decimated, int decimation_ratio);   /* FCCH_coarse_position.m:38 */

/* ---- K5-K8  [FCCH_pos,r,sampling_ppm,carrier_ppm] = FCCH_fine_correction(s,base_position,osr,carrier_freq)
 *             FCCH_fine_correction.m:5-197 ----
 * *n_pos = -1 -> FCCH_pos is the scalar -1, else 1 x n_pos.  *r_len = -1 -> r is the scalar -1, else r holds
 * r_len complex128 (r_cap >= n).  ppm = +inf on the sentinel paths (SURVEY.md Appendix A). */
int gsmcal_FCCH_fine_correction(const double *s, int64_t n, const double *base_position, int64_t n_base,
                                int oversampling_ratio, double carrier_freq,
                                double *FCCH_pos, int64_t pos_cap, int64_t *n_pos,
                                double *r, int64_t r_cap, int64_t *r_len,
                                double *sampling_ppm, double *carrier_ppm);

/* ---- T1  s = gsm_SCH_training_sequence_gen(osr)   gsm_SCH_training_sequence_gen.m:5-45 ----
 * 64*osr complex128.  GMSK per GSM 05.04 (BT 0.3, L 4, h 0.5); not a bit match of comm.GMSKModulator. */
int gsmcal_SCH_training_sequence_gen(int oversampling_ratio, double *s);

/* ---- K9-K10  [pos_info,r,sampling_ppm] = SCH_corr_rate_correction(s,FCCH_pos,sch_training_sequence,osr)
 *              SCH_corr_rate_correction.m:5-182 ----
 * *n_rows = -1 -> pos_info = [-1,-1] (1x2); else n_rows x 2 (column-major: n_rows positions then n_rows
 * types), possibly all -1 (the 3H x 2 sentinel).  rows_cap >= 6*n_fcch. */
int gsmcal_SCH_corr_rate_correction(const double *s, int64_t n, const double *FCCH_pos, int64_t n_fcch,
                                    const double *sch_training_sequence, int oversampling_ratio,
                                    double *pos_info, int64_t rows_cap, int64_t *n_rows,
                                    double *r, int64_t r_cap, int64_t *r_len, double *sampling_ppm);

/* ---- K8/K7  [r,carrier_ppm] = carrier_correct_post_SCH(s,pos_info,osr,carrier_freq)
 *             carrier_correct_post_SCH.m:5-83 ---- */
int gsmcal_carrier_correct_post_SCH(const double *s, int64_t n, const double *pos_info, int64_t n_rows,
                                    int oversampling_ratio, double carrier_freq,
                                    double *r, int64_t r_cap, int64_t *r_len, double *carrier_ppm);

/* ---- K11  ppm_out = total_ppm_calculation(ppm_in)   total_ppm_calculation.m:5-21 ---- */
int gsmcal_total_ppm_calculation(const double *ppm_in, int64_t n, double *ppm_out);

/* ---- SURVEY 8(f) rows 2 and 4: the consumers of r_correct / pos_info (gsm_sync_demod.m:143-146) -------------
 * The reference functions have no outputs (they disp / plot); these entry points return the quantities they compute.
 *
 * s = gsm_normal_training_sequence_gen(oversampling_ratio)   gsm_normal_training_sequence_gen.m:5-59
 *   s: (26*osr) x 8 complex128, column q = GMSK of training sequence code q (same modulator caveat as T1). */
int gsmcal_normal_training_sequence_gen(int oversampling_ratio, double *s);

/* FCCH_demod(s, pos_info, oversampling_ratio, carrier_freq)   FCCH_demod.m:5-66
 *   per FCCH row of pos_info: freq (:41), snr (:57-63), max_idx - (fft_len/2+1) (:66); mean_freq (:43), carrier_ppm (:47).
 *   *n_fcch = -1 on the `pos_info==-1` path (:7-10), else the number of FCCH rows (<= cap). */
int gsmcal_FCCH_demod(const double *s, int64_t n, const double *pos_info, int64_t n_rows, int oversampling_ratio,
                      double carrier_freq, double *freq, double *snr, double *max_idx, int64_t cap,
                      int64_t *n_fcch, double *mean_freq, double *carrier_ppm);

/* BCCH_demod(s, pos_info, training_sequence, oversampling_ratio)   BCCH_demod.m:5-106
 *   The reference reads `carrier_freq` and `normal_training_sequence` without defining them (:68,:91); here they are
 *   arguments (nts = the (26*osr) x 8 matrix above).  carrier_ppm (:68); nts_idx = 1..8 when the first four BCCH bursts
 *   agree on the best-correlating normal training sequence (:91-97), -1 otherwise (:99-102); both -1 on the early
 *   returns (:6-16).  corr_abs (optional): abs(corr_val), 8 x 4 column-major (:91-93). */
int gsmcal_BCCH_demod(const double *s, int64_t n, const double *pos_info, int64_t n_rows, const double *nts,
                      int oversampling_ratio, double carrier_freq, double *carrier_ppm, int *nts_idx, double *corr_abs);

/* SCH_demod(s, pos_info, training_sequence, oversampling_ratio)   SCH_demod.m:5-121
 *   per SCH row of pos_info: frequency-domain equalisation on the 64-symbol training sequence (:79-90), GMSK MLSE
 *   demodulation (comm.GMSKDemodulator, TracebackDepth 30 - closed source, restated as a 32-state Viterbi over the
 *   modulator of T1: parity unpinned), the 148 burst bits (:94-95), their differential decoding (:97) and the
 *   +-1 correlation with the training bits over 85 lags (:103-110).
 *   demod_bits, bits_to_decoder: 148 x cap uint8 (column per burst); corr_val: 85 x cap double.
 *   *n_sch = -1 on the `pos_info==-1` path (:8-11).  GSMCAL_ERR_RANGE where `x = s(sp:ep)` (:81) would fail. */
int gsmcal_SCH_demod(const double *s, int64_t n, const double *pos_info, int64_t n_rows, const double *sch_training_sequence,
                     int oversampling_ratio, int64_t cap, int64_t *n_sch, uint8_t *demod_bits, uint8_t *bits_to_decoder,
                     double *corr_val);

/* ---- batched pipeline: gsm_sync_demod.m:107-124 for many dongle streams in one call ------------------
 * raw: n_streams rows of 2*n_iq uint8 (row d == column d of the reference's 2N x D matrix `s`).
 * Returns exactly what the function-by-function chain returns per stream (positions, pos_info, ppm),
 * but never materialises the intermediate N-sample complex streams: every stage evaluates the samples
 * it needs from the uint8 input on the fly (see DESIGN.md). */
typedef struct gsmcal_stream_result {
    int32_t n_coarse;            /* FCCH_coarse_position: -1 -> position = -1 */
    int32_t n_fcch;              /* FCCH_fine_correction: -1 -> FCCH_pos = -1 */
    int32_t n_pos_info;          /* SCH_corr_rate_correction: -1 -> pos_info = [-1,-1] */
    int32_t flags;               /* GSMCAL_FLAG_* */
    int64_t r_len[3];            /* length of r after fine / SCH / post-SCH; -1 -> scalar -1 */
    double  sampling_ppm[2];     /* FCCH stage, SCH stage (inf on sentinel paths) */
    double  carrier_ppm[2];      /* FCCH stage, post-SCH stage */
    double  total_sampling_ppm;  /* total_ppm_calculation of the two */
    double  total_carrier_ppm;
} gsmcal_stream_result;

#define GSMCAL_FLAG_FINE_SPACING   1   /* FCCH_fine_correction.m:95-102 */
#define GSMCAL_FLAG_FINE_LOW_SNR   2   /* FCCH_fine_correction.m:192-196 */
#define GSMCAL_FLAG_SCH_EDGE       4   /* SCH_corr_rate_correction.m:59-63 */
#define GSMCAL_FLAG_SCH_SPACING    8   /* SCH_corr_rate_correction.m:106-112 */
#define GSMCAL_FLAG_POST_FEW_BCCH 16   /* carrier_correct_post_SCH.m:15-19 */
#define GSMCAL_FLAG_FINE_FALLBACK 32   /* informational: a burst needed the all-bin fine search */

#define GSMCAL_MEM_HOST   0
#define GSMCAL_MEM_DEVICE 1

/* B = gsmcal_max_bursts(ceil(n_iq/(osr*coarse_dr)), coarse_dr).  Optional outputs may be NULL.
 * coarse_pos/coarse_snr/fcch_pos: [n_streams][B]; pos_info: [n_streams][6*B][2] (row-major rows of
 * {position,type}).  raw_mem says where `raw` lives; results are always written to HOST memory.
 * cuda_stream: a cudaStream_t (NULL = default stream); the call returns after the stream has drained. */
int gsmcal_calibrate_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_streams,
                           double carrier_freq, const double *sch_training_sequence,
                           const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                           gsmcal_stream_result *results,
                           double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info,
                           void *cuda_stream);

/* The same call that also MATERIALISES r_correct, the corrected stream gsm_sync_demod.m:120 hands to SCH_demod (:145):
 *   filter(coef,1,raw2iq(a)) -> interp1 by (1+e1) -> .*exp(1i*n*dphi1) -> interp1 by (1+e2) -> .*exp(1i*n*dphi2)
 * (FCCH_fine_correction.m:125,165; SCH_corr_rate_correction.m:127; carrier_correct_post_SCH.m:83), written in one fused pass from
 * the uint8 capture: 2 bytes in, 16 bytes out per sample.  r_correct: n_streams rows of r_stride complex128 (r_stride >= n_iq), in
 * HOST or DEVICE memory (r_mem); row d holds results[d].r_len[2] samples, nothing is written when that is -1 (r = -1). */
int gsmcal_calibrate_batch_r(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_streams,
                             double carrier_freq, const double *sch_training_sequence,
                             const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                             gsmcal_stream_result *results,
                             double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info,
                             void *cuda_stream, double *r_correct, int r_mem, int64_t r_stride);

/* The same call followed by the two demodulators gsm_sync_demod.m:144-145 hands r_correct to, for every stream, without materialising
 * r_correct: SCH_demod(r_correct, pos_info, ...) (SCH_demod.m:65-110) and FCCH_demod (FCCH_demod.m:21-66) on the samples
 * filter -> interp1(1+e1) -> .*exp(1i*n*dphi1) -> interp1(1+e2) -> .*exp(1i*n*dphi2) evaluated from the uint8 capture where each burst
 * reads them.  results, coarse_*, fcch_pos and pos_info are those of gsmcal_calibrate_batch.
 * Row i of stream d (B = gsmcal_max_bursts(...) as above) is the i-th row of that type in the stream's pos_info.  Per-row outputs may be
 * NULL (not copied back):
 *   sch_ok [n_streams][B]: 1 when the 194*osr-sample equaliser window x = r_correct(pos-8*osr : ...) lies inside r_correct (where the
 *     reference would raise, SCH_demod.m:79-81, the row gets sch_ok = 0 and zero bits / correlations);
 *   demod_bits, bits_to_decoder [n_streams][B][148] (SCH_demod.m:94-97); corr_val [n_streams][B][85] (:103-110);
 *   fcch_freq, fcch_snr, fcch_max_idx [n_streams][B] (FCCH_demod.m:41,57-66; NaN for a window outside r_correct).
 * The per-stream record tells which rows are valid and why a demodulator did not run. */
typedef struct gsmcal_demod_result {
    int32_t n_sch;            /* type-1 rows of pos_info, in pos_info order; -1: SCH_demod not run (flags say why) */
    int32_t n_sch_ok;         /* of those, rows whose 194*osr-sample equaliser window lies inside r_correct */
    int32_t n_fcch;           /* type-0 rows; -1 like n_sch */
    int32_t flags;            /* GSMCAL_DEMOD_* */
    double  fcch_mean_freq;   /* FCCH_demod.m:43; NaN unless every FCCH window lies inside r_correct */
    double  fcch_carrier_ppm; /* FCCH_demod.m:46-47; NaN likewise */
} gsmcal_demod_result;        /* 32 bytes */

#define GSMCAL_DEMOD_NO_POS_INFO  1  /* pos_info == -1 in the all-elements sense (SCH_demod.m:8-11, FCCH_demod.m:7-10) */
#define GSMCAL_DEMOD_NO_R_CORRECT 2  /* pos_info valid but r_correct = -1 (results.r_len[2] == -1): the reference would fail at SCH_demod.m:81 */
#define GSMCAL_DEMOD_SCH_RANGE    4  /* some SCH window leaves r_correct (the reference raises at :79-81); those rows have sch_ok = 0 */
#define GSMCAL_DEMOD_FCCH_RANGE   8  /* some FCCH window leaves r_correct; mean / ppm are NaN */

int gsmcal_calibrate_demod_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_streams,
                                 double carrier_freq, const double *sch_training_sequence,
                                 const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                                 gsmcal_stream_result *results,
                                 double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info,
                                 void *cuda_stream,
                                 gsmcal_demod_result *demod /* [n_streams], required */, uint8_t *sch_ok,
                                 uint8_t *demod_bits, uint8_t *bits_to_decoder, double *corr_val,
                                 double *fcch_freq, double *fcch_snr, double *fcch_max_idx);

/* gsmcal_calibrate_demod_batch (every output as there, byte for byte) followed by BCCH_demod (gsm_sync_demod.m:146, BCCH_demod.m:5-106)
 * on every stream's r_correct, again without materialising it.  BCCH_demod's carrier ppm is that of carrier_correct_post_SCH on
 * r_correct: the FCCH rows' tone-frequency mean, i.e. gsmcal_demod_result.fcch_carrier_ppm (copied bit for bit).  The training windows
 * r_bcch(p+61*osr : p+61*osr+26*osr-1) of the first four BCCH rows, r_bcch(j) = r_correct(j)*exp(1i*(j-1)*comp) with
 * comp = (fs_sym/4 - mean_freq)*2*pi/fs (:72-73, :85-89), are correlated with the eight normal training sequences (:91).
 * normal_training_sequence: (26*osr) x 8 complex128, column-major (gsmcal_normal_training_sequence_gen).  One record per stream;
 * the first flag that applies decides, in this order:
 *   GSMCAL_BCCH_NO_POS_INFO  pos_info == -1 (:9-11):                 carrier_ppm -1,  nts_idx -1, corr_abs NaN
 *   GSMCAL_BCCH_FEW_BCCH     fewer than four BCCH rows (:13-17):      carrier_ppm -1,  nts_idx -1, corr_abs NaN
 *                            (also every stream whose pos_info is valid but r_correct = -1: that happens only with too few BCCH rows)
 *   GSMCAL_BCCH_FCCH_RANGE   no FCCH mean (no FCCH row, or an FCCH window leaves r_correct; gsmcal_BCCH_demod returns GSMCAL_ERR_RANGE):
 *                            carrier_ppm NaN, nts_idx -1, corr_abs NaN
 *   GSMCAL_BCCH_TRAIN_RANGE  a training window leaves r_correct (the reference would raise): that burst's column NaN, nts_idx -1
 *   0                        nts_idx 1..8 when the first maxima of the four columns agree (:93-102), else -1. */
typedef struct gsmcal_bcch_result {
    double  carrier_ppm;      /* BCCH_demod.m:68 on r_correct (== gsmcal_demod_result.fcch_carrier_ppm); -1 / NaN per the flags */
    int32_t nts_idx;          /* 1..8, or -1 */
    int32_t flags;            /* GSMCAL_BCCH_* */
    double  corr_abs[32];     /* abs(corr_val), 8 x 4 column-major (:91-93) */
} gsmcal_bcch_result;         /* 272 bytes */

#define GSMCAL_BCCH_NO_POS_INFO  1
#define GSMCAL_BCCH_FEW_BCCH     2
#define GSMCAL_BCCH_FCCH_RANGE   4
#define GSMCAL_BCCH_TRAIN_RANGE  8

int gsmcal_calibrate_demod_bcch_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_streams,
                                      double carrier_freq, const double *sch_training_sequence,
                                      const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                                      gsmcal_stream_result *results,
                                      double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info,
                                      void *cuda_stream,
                                      gsmcal_demod_result *demod /* [n_streams], required */, uint8_t *sch_ok,
                                      uint8_t *demod_bits, uint8_t *bits_to_decoder, double *corr_val,
                                      double *fcch_freq, double *fcch_snr, double *fcch_max_idx,
                                      const double *normal_training_sequence /* (26*osr) x 8 complex128, column-major */,
                                      gsmcal_bcch_result *bcch /* [n_streams], required */);

/* gsmcal_calibrate_batch (every output as there, byte for byte) followed by sub-sample timing of every SCH burst and a least-squares
 * line through the burst times: each dongle's sample clock measured from the burst positions themselves instead of the integer
 * lattice of sampling_ppm, and the time of its bursts in its own capture.  Only oversampling_ratio 8.  For stream d, with
 * e1 = sampling_ppm[0]*1e-6, e2 = sampling_ppm[1]*1e-6, r = r_correct (1-based, the samples gsmcal_calibrate_batch_r writes) and
 * p_i the position of the i-th SCH row (type 1) of pos_info:
 *   g_i = p_i + 42*8 (training start); c_i(l) = |sum_{n=0..511} conj(t_n) r(g_i+l+n)|^2 (fp64, abs then square) for l = -64..24
 *   (the 89 lags of SCH_corr_rate_correction.m:36,45-48), l* = the first maximum;
 *   GSMCAL_TIMING_RANGE: the 600-sample window leaves r, GSMCAL_TIMING_EDGE: l* is the first or last lag; both give tau_i = NaN;
 *   delta = 0.5*(y- - y+)/(y- - 2*y0 + y+) of y = c_i(l*-1, l*, l*+1) (0 when the denominator is 0), tau_i = g_i + l* + delta;
 *   x_i = ((tau_i - 1)*(1 + e2))*(1 + e1): tau_i in 0-based samples of the uint8 capture (r(j) sits at raw time (j-1)(1+e2)(1+e1));
 *   over the n_fit rows with finite x_i, m_i = p_i - p_first: b = sum (m-mean m)(x-mean x) / sum (m-mean m)^2 (row order),
 *   a = mean x - b*mean m, t0 = a, fit_ppm = (b - 1)*1e6, rms = sqrt(sum (x - a - b*m)^2 / n_fit); n_fit < 3: GSMCAL_TIMING_FEW, NaN.
 * sch_tau, sch_x [n_streams][B] (B as above; NULL = not copied): tau_i and x_i by SCH row, NaN where excluded. */
typedef struct gsmcal_sch_timing_result {
    int32_t n_sch;        /* type-1 rows of pos_info; -1 when the step did not run (flags say why) */
    int32_t n_fit;        /* rows with a finite tau */
    int32_t flags;        /* GSMCAL_TIMING_* */
    int32_t reserved;
    double  t0;           /* fit intercept, raw-capture samples (0-based): the raw time of the first SCH row's training start */
    double  fit_ppm;      /* (slope - 1) * 1e6 */
    double  rms;          /* fit residual RMS, raw-capture samples */
} gsmcal_sch_timing_result;   /* 40 bytes */

#define GSMCAL_TIMING_NO_POS_INFO  1   /* pos_info == -1: nothing to time */
#define GSMCAL_TIMING_NO_R_CORRECT 2   /* pos_info valid but results.r_len[2] == -1 */
#define GSMCAL_TIMING_RANGE        4   /* some row's 600-sample correlation window leaves r_correct */
#define GSMCAL_TIMING_EDGE         8   /* some row's maximum sits on the first or last lag */
#define GSMCAL_TIMING_FEW         16   /* fewer than 3 rows with a finite tau: t0, fit_ppm, rms NaN */

int gsmcal_calibrate_sch_timing_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_streams,
                                      double carrier_freq, const double *sch_training_sequence,
                                      const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                                      gsmcal_stream_result *results,
                                      double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info,
                                      void *cuda_stream,
                                      gsmcal_sch_timing_result *timing /* [n_streams], required */,
                                      double *sch_tau, double *sch_x);

/* gsmcal_calibrate_demod_batch (every output as there, byte for byte; with normal_training_sequence and bcch, both set or both NULL,
 * gsmcal_calibrate_demod_bcch_batch's) followed by SCH channel decoding: the BSIC and the TDMA frame number (FN) each SCH burst carries,
 * and each dongle's capture start on the cell's frame clock.  Per type-1 row of pos_info, in row order (the rows SCH_demod
 * demodulates), with m = its demod_bits and k* = the first maximum of its corr_val (0..84):
 *   1. skip: sch_ok = 0 -> GSMCAL_SCHDEC_ROW_WINDOW; k* < 39 or k* > 45 (the coded bits would leave the 148) -> GSMCAL_SCHDEC_ROW_ALIGN.
 *   2. burst bits: m_i = 1 exactly when b_i = b_(i-1) (demod_bits are differentially encoded; bits_to_decoder is not used).  With
 *      b_(k*+j) = SCH training bit j (j = 0..63): b_i = b_(i+1) xor (1 - m_(i+1)) for i = k*-1 down to k*-39, b_i = b_(i-1) xor (1 - m_i)
 *      for i = k*+64 up to k*+102.  Coded bits e(0..38) = b(k*-39 .. k*-1), e(39..77) = b(k*+64 .. k*+102) (TS 45.002 5.2.5, k* = 42).
 *   3. convolutional code (TS 45.003 4.7): e(2k) = u(k)+u(k-3)+u(k-4), e(2k+1) = u(k)+u(k-1)+u(k-3)+u(k-4) mod 2, k = 0..38, u(k<0) = 0.
 *      Hard-decision Viterbi over the 16 states (u(k), u(k-1), u(k-2), u(k-3)), Hamming branch metrics, from and back to state 0
 *      (u(35..38) = 0 are the tail).  A state keeps the predecessor with the smaller metric, on a tie the one whose dropped (oldest)
 *      bit is 0.  hamming = the final metric of state 0: the number of coded bits the decision disagrees with.
 *   4. CRC (TS 45.003 4.7): d(0)D^34 + ... + d(24)D^10 + p(0)D^9 + ... + p(9), u(0..24) = d, u(25..34) = p, divided by
 *      D^10 + D^8 + D^6 + D^5 + D^4 + D^2 + 1 must leave 1 + D + ... + D^9, else GSMCAL_SCHDEC_ROW_CRC.
 *   5. fields (TS 44.018 9.1.30, d(0) = bit 1 of octet 1, OsmocomBB's packing): d(0), d(1) = T1 bits 9, 10; d(2..7) = BSIC bits 0..5;
 *      d(8..15) = T1 bits 1..8; d(16), d(17) = T3' bits 1, 2; d(18..22) = T2 bits 0..4; d(23) = T1 bit 0; d(24) = T3' bit 0.
 *      T3 = 10*T3' + 1, FN = 51*((T3 - T2) mod 26) + T3 + 1326*T1 (TS 45.002 3.3.2.2).  T2 > 25 or T3' > 4: GSMCAL_SCHDEC_ROW_FIELD.
 *      No recorded capture pins this bit order against a live cell: like the GMSK modulator's, its parity is unverified.
 *   6. vote: with F = 1250*osr samples per frame (10,000 at osr 8) and p_i the SCH rows' pos_info positions (one regridded frame grid,
 *      so f_i = (p_i - p_first)/F is an integer; p_first = the first SCH row's), every row that passes 1-5 votes for
 *      (fn_first = (FN_i - f_i) mod 2,715,648, BSIC_i).  Most votes wins, equal votes: the pair whose earliest voting row comes first.
 *      n_agree = its votes; GSMCAL_SCHDEC_DISAGREE when some valid row voted otherwise; GSMCAL_SCHDEC_NONE when no row passed.
 *   7. frame_clock_start = (fn_first*F - (p_first - 1)) mod (2,715,648*F): the GSM time of raw capture sample 0 in nominal samples since
 *      FN 0 of the hyperframe (r_correct(j) sits at raw time (j-1)(1+e2)(1+e1) and its spacing is nominal).  An integer-valued double,
 *      as accurate as pos_info (a few samples), not sub-sample.
 * sch_fn, sch_bsic [n_streams][B] int32 (-1 where not decoded), sch_hamming, sch_row_flags [n_streams][B] uint8 (B as above); any may be
 * NULL (not copied back).  Rows beyond the record's n_sch hold -1 / -1 / 0 / 0. */
typedef struct gsmcal_sch_decode_result {
    int32_t n_sch;             /* type-1 rows; -1: not run (flags say why: GSMCAL_SCHDEC_NO_POS_INFO / _NO_R_CORRECT only) */
    int32_t n_crc_ok;          /* rows with a valid CRC and valid fields */
    int32_t n_agree;           /* of those, rows that voted for the winning (fn_first, bsic) */
    int32_t flags;             /* GSMCAL_SCHDEC_* */
    int32_t bsic;              /* 0..63 (NCC*8 + BCC), or -1 */
    int32_t fn_first;          /* FN of the frame holding the first SCH row of pos_info, or -1 */
    double  frame_clock_start; /* see 7.; NaN without a winner */
} gsmcal_sch_decode_result;    /* 32 bytes */

#define GSMCAL_SCHDEC_NO_POS_INFO   1  /* as GSMCAL_DEMOD_NO_POS_INFO */
#define GSMCAL_SCHDEC_NO_R_CORRECT  2  /* as GSMCAL_DEMOD_NO_R_CORRECT */
#define GSMCAL_SCHDEC_NONE          4  /* no row passed the CRC and field checks */
#define GSMCAL_SCHDEC_DISAGREE      8  /* some valid row voted for another (fn_first, bsic) */
#define GSMCAL_SCHDEC_ROW_WINDOW    1  /* row flags: sch_ok = 0 */
#define GSMCAL_SCHDEC_ROW_ALIGN     2  /* k* outside 39..45 */
#define GSMCAL_SCHDEC_ROW_CRC       4  /* CRC check failed */
#define GSMCAL_SCHDEC_ROW_FIELD     8  /* T2 > 25 or T3' > 4 */

int gsmcal_calibrate_sch_decode_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_streams,
                                      double carrier_freq, const double *sch_training_sequence,
                                      const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                                      gsmcal_stream_result *results,
                                      double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info,
                                      void *cuda_stream,
                                      gsmcal_demod_result *demod /* [n_streams], required */, uint8_t *sch_ok,
                                      uint8_t *demod_bits, uint8_t *bits_to_decoder, double *corr_val,
                                      double *fcch_freq, double *fcch_snr, double *fcch_max_idx,
                                      const double *normal_training_sequence /* or NULL */, gsmcal_bcch_result *bcch /* or NULL */,
                                      gsmcal_sch_decode_result *dec /* [n_streams], required */,
                                      int32_t *sch_fn, int32_t *sch_bsic, uint8_t *sch_hamming, uint8_t *sch_row_flags);

/* The same pipeline with several batches in flight (continuous captures): _submit enqueues batch `slot` (0..3) on the library's
 * own streams once the caller's `cuda_stream` has produced the DEVICE-resident capture, and returns; _collect waits for that batch
 * and fills the result pointers given to _submit (they must stay valid until then).  Batches are staggered on the device: the
 * burst kernels of batch k+1 start when batch k is done, and the front of batch k+1 - the exact column sums (a one-warp-per-block
 * kernel that brings the bytes in with TMA bulk copies, small enough to sit beside the burst kernels) and the dependent burst chain,
 * both on a high-priority stream - runs underneath the burst kernels of batch k.
 * Results are identical to gsmcal_calibrate_batch.  The capture must not be overwritten before _collect returns. */
int gsmcal_calibrate_batch_submit(int slot, const uint8_t *raw_dev, int64_t n_iq, int64_t n_streams, double carrier_freq,
                                  const double *sch_training_sequence, const double *coef, int n_taps,
                                  int oversampling_ratio, int coarse_decimation_ratio, gsmcal_stream_result *results,
                                  double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream);
int gsmcal_calibrate_batch_collect(int slot);
/* Gives `slot` back without delivering results (waits for the batch; the result pointers passed to _submit are never written).
 * For callers that abandon a submitted batch: the slot would otherwise stay busy and keep pointers into freed memory.
 * _submit, _collect and _cancel of one slot must be called from threads that selected the same device (gsmcal_set_device is
 * per thread; slots belong to the device). */
int gsmcal_calibrate_batch_cancel(int slot);

/* CUDA-event times (ms) of the stages of the last gsmcal_calibrate_batch call on this process:
 * [0] uint8 column sums (+ H2D when raw is on the host) [1] coarse FCCH [2] fine FCCH sliding-DFT peak search
 * [3] fine ppm + tone estimate + gate [4] SCH correlation + pos_info [5] post-SCH tone estimate + result records
 * [6] (gsmcal_calibrate_demod_batch / _demod_bcch_batch / _sch_decode_batch only) SCH_demod (+ SCH decoding) + FCCH_demod (+ BCCH_demod);
 *     (gsmcal_calibrate_sch_timing_batch only) SCH row list, sub-sample SCH timing and the clock fit.  Returns the number of stages written. */
int gsmcal_last_batch_stage_ms(double *ms, int cap);

/* FCCH scanner per-channel processing, multi_rtl_sdr_gsm_FCCH_scanner.m:132-135,163-186, for n_chan
 * captures in one call: raw2iq -> filter(coef) -> r(1:osr*dr:end) -> FCCH_coarse_position -> spacing
 * acceptance.  snr[c]/num_hit[c] as the script computes them (0 when rejected). */
int gsmcal_fcch_scan(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_chan,
                     const double *coef, int n_taps, int oversampling_ratio, int coarse_decimation,
                     double *snr, double *num_hit, double *position /* [n_chan][B] or NULL */,
                     int32_t *n_position /* [n_chan] or NULL */, void *cuda_stream);

/* test / tuning hooks: key 0, value 1 = run the all-bin fine FCCH search for every burst (no band-limited fast path);
 * 3 = stream groups of gsmcal_calibrate_batch; 4 = pretend the tier-1/2 certificates failed; 5 = tier-3 list limit;
 * 6 = burst chain on high-priority streams (default 1); 8 = stream groups inside a submitted batch (default 2); 9, value 1 = the
 * generic tier-1 fine search without the osr-8 fast path and its filtered-window cache (A/B and tests); 10 = passes of 8 tracked bins
 * in the osr-8 tier-1 kernel (1..8, default 8); 11, value 1 = generic tone estimator for every burst (no tone8_kernel); 12, value 1 =
 * plain cudaMemcpyAsync for pageable host buffers instead of the library's multi-threaded pinned staging ring; 13, value 1 = per-phase
 * clock64 counters in fine_core8_kernel / tone8_kernel / coarse_chain_kernel (gsmcal_debug_get 50.. / 150..); 14, value 1 = device
 * timeline of every submitted batch on stderr; 17 = 4 KB ring stages per block of the TMA column-sum kernel of _submit (1..24,
 * default 2); 18 = its blocks per SM (default 3); 24 = the osr-8 SCH correlation: value 0 = fp32 screen of the 89 lags, fp64 only for
 * the lags that can hold the maximum (default), 1 = fp64 correlation of every lag (A/B), 2 = run the screen, then the fp64 fallback as
 * if it had failed (tests).  Any other key: GSMCAL_ERR_ARG */
int gsmcal_debug_set(int key, int value);
/* key 1: number of bursts of the last fine FCCH search whose band certificate failed (all-bin fallback ran); 2: bursts that needed the
 * 64-bin band kernel; 10 + p: bursts the osr-8 tier-1 kernel proved after p passes (p = 0: left open); 30: bytes moved through the
 * pinned staging ring so far; over the last call that ran the SCH stage: 120 = bursts the osr-8 SCH screen decided, 121 = bursts that ran
 * the full fp64 SCH correlation (fallback, or debug key 24 != 0), 121 + c (c = 1..8) = decided bursts with c candidate lags */
int64_t gsmcal_debug_get(int key);

/* kernel-launch counter (all launches since the last reset, this process) - for bench.py's gpu_launches */
int64_t gsmcal_launch_count(int reset);

/* measured FP64 FMA throughput of the current device in TFLOP/s (register-only DFMA kernel, CUDA events): the
 * roofline denominator of the FP64-bound burst stages */
int gsmcal_fp64_peak(double *tflops, void *cuda_stream);

/* measurement helpers used by bench.py for per-stage rooflines on device-resident buffers.
 * stage: 0 colsum_u8, 1 raw2iq, 2 fir c128->c128, 3 fused u8->fir c128, 4 resample, 5 derotate,
 *        6 fused u8->fir->decimate(64).  Buffers are DEVICE pointers sized by the caller. */
int gsmcal_stage_launch(int stage, const void *in, void *out, int64_t n_iq, int64_t n_col,
                        const double *coef, int n_taps, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* GSMCAL_H */
