/* gsmcal_mex.c - thin MEX gateways: one translation unit, one gateway per reference function.
 *
 * Build one MEX file per function, named like the .m file it shadows (a MEX file in the same folder takes
 * precedence over the .m file, so gsm_sync_demod.m etc. call it with no edits):
 *
 *   mex  -R2018a -DGSMCAL_MEX_raw2iq -output raw2iq gsmcal_mex.c -I../../include -L../csrc -lgsmcal      (MATLAB)
 *   mkoctfile --mex -DGSMCAL_MEX_raw2iq -o raw2iq.mex gsmcal_mex.c -I../../include -L../csrc -lgsmcal     (Octave)
 *
 * (see Makefile.mex).  Neither MATLAB nor Octave exists in the build image, so these gateways are compiled
 * and exercised in tests/ against mex/stub/mex.h - a minimal mxArray shim - to keep the marshalling honest.
 *
 * Complex data: with -R2018a MATLAB stores interleaved complex (mxGetComplexDoubles), which is the C ABI's
 * layout, so no copy is needed; the legacy / Octave split layout (mxGetPr/mxGetPi) is converted here.
 * Sentinels: the reference returns -1 / [-1,-1] / inf on its failure paths (SURVEY.md Appendix A); the C ABI
 * reports them as count = -1 and the gateway rebuilds the exact MATLAB shapes.  mexErrMsgIdAndTxt is used only
 * for malformed arguments and CUDA failures.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "mex.h"
#include "gsmcal.h"

#ifndef MX_HAS_INTERLEAVED_COMPLEX
#define MX_HAS_INTERLEAVED_COMPLEX 0
#endif

static void fail_on(int rc, const char *fn) {
    if (rc != GSMCAL_OK) mexErrMsgIdAndTxt("gsmcal:error", "%s: %s (code %d)", fn, gsmcal_last_error(), rc);
}

static int registered = 0;
static void at_exit(void) { gsmcal_release(); }
static void init_once(void) { if (!registered) { mexAtExit(at_exit); registered = 1; } }

/* complex (or real) double matrix -> interleaved buffer the C ABI reads.  *owned tells the caller to mxFree it. */
static const double *get_c128(const mxArray *a, int *owned) {
    size_t n = mxGetNumberOfElements(a);
    *owned = 0;
    if (!mxIsDouble(a)) mexErrMsgIdAndTxt("gsmcal:type", "expected a double array");
#if MX_HAS_INTERLEAVED_COMPLEX
    if (mxIsComplex(a)) return (const double *)mxGetComplexDoubles(a);
    {
        double *buf = (double *)mxMalloc(2 * n * sizeof(double) + 16);
        const double *re = mxGetDoubles(a);
        for (size_t i = 0; i < n; ++i) { buf[2 * i] = re[i]; buf[2 * i + 1] = 0.0; }
        *owned = 1;
        return buf;
    }
#else
    {
        double *buf = (double *)mxMalloc(2 * n * sizeof(double) + 16);
        const double *re = mxGetPr(a), *im = mxIsComplex(a) ? mxGetPi(a) : NULL;
        for (size_t i = 0; i < n; ++i) { buf[2 * i] = re[i]; buf[2 * i + 1] = im ? im[i] : 0.0; }
        *owned = 1;
        return buf;
    }
#endif
}

/* interleaved result -> new complex mxArray (rows x cols) */
static mxArray *put_c128(const double *buf, size_t rows, size_t cols) {
    mxArray *o = mxCreateDoubleMatrix(rows, cols, mxCOMPLEX);
    size_t n = rows * cols;
#if MX_HAS_INTERLEAVED_COMPLEX
    memcpy(mxGetComplexDoubles(o), buf, 2 * n * sizeof(double));
#else
    double *re = mxGetPr(o), *im = mxGetPi(o);
    for (size_t i = 0; i < n; ++i) { re[i] = buf[2 * i]; im[i] = buf[2 * i + 1]; }
#endif
    return o;
}

static mxArray *scalar(double v) { return mxCreateDoubleScalar(v); }
static mxArray *row_vector(const double *v, size_t n) {
    mxArray *o = mxCreateDoubleMatrix(1, n, mxREAL);
    if (n) memcpy(mxGetPr(o), v, n * sizeof(double));
    return o;
}
static const double *real_vector(const mxArray *a, size_t *n) {
    if (!mxIsDouble(a) || mxIsComplex(a)) mexErrMsgIdAndTxt("gsmcal:type", "expected a real double vector");
    *n = mxGetNumberOfElements(a);
    return mxGetPr(a);
}
static void need(int nrhs, int want, const char *usage) {
    if (nrhs != want) mexErrMsgIdAndTxt("gsmcal:nargin", "usage: %s", usage);
}
/* the first four outputs of the batch gateways, as many as asked for: sampling_ppm, carrier_ppm (3 x D), n_pos_info (1 x D) and pos_info
 * ((6B) x 2 x D, NaN beyond n_pos_info(d)), from the D records and pi ([D][6B][2]) of a batch call */
static void batch_outputs(int nlhs, mxArray *plhs[], const gsmcal_stream_result *res, const double *pi, size_t D, size_t B) {
    plhs[0] = mxCreateDoubleMatrix(3, D, mxREAL);
    if (nlhs > 1) plhs[1] = mxCreateDoubleMatrix(3, D, mxREAL);
    if (nlhs > 2) plhs[2] = mxCreateDoubleMatrix(1, D, mxREAL);
    for (size_t d = 0; d < D; ++d) {
        double *sp = mxGetPr(plhs[0]) + 3 * d;
        sp[0] = res[d].sampling_ppm[0]; sp[1] = res[d].sampling_ppm[1]; sp[2] = res[d].total_sampling_ppm;
        if (nlhs > 1) { double *cp = mxGetPr(plhs[1]) + 3 * d; cp[0] = res[d].carrier_ppm[0]; cp[1] = res[d].carrier_ppm[1]; cp[2] = res[d].total_carrier_ppm; }
        if (nlhs > 2) mxGetPr(plhs[2])[d] = res[d].n_pos_info;
    }
    if (nlhs > 3) {
        size_t dims[3] = {6 * B, 2, D};
        plhs[3] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);
        double *o = mxGetPr(plhs[3]);
        for (size_t d = 0; d < D; ++d)
            for (size_t i = 0; i < 6 * B; ++i)
                for (int c = 0; c < 2; ++c)
                    o[d * 12 * B + c * 6 * B + i] = ((int64_t)i < res[d].n_pos_info) ? pi[d * 12 * B + 2 * i + c] : mxGetNaN();
    }
}

/* ------------------------------------------------------------------------------------------------ */
#if defined(GSMCAL_MEX_raw2iq)
/* b = raw2iq(a)                                                                        raw2iq.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    (void)nlhs; init_once(); need(nrhs, 1, "b = raw2iq(a)");
    size_t rows = mxGetM(prhs[0]), cols = mxGetN(prhs[0]);
    if (rows % 2) mexErrMsgIdAndTxt("gsmcal:size", "raw2iq: odd number of rows");
    double *out = (double *)mxMalloc(rows * cols * sizeof(double) + 16);
    if (mxIsUint8(prhs[0])) fail_on(gsmcal_raw2iq_u8((const uint8_t *)mxGetData(prhs[0]), (int64_t)(rows / 2), (int64_t)cols, out), "raw2iq");
    else if (mxIsDouble(prhs[0]) && !mxIsComplex(prhs[0])) fail_on(gsmcal_raw2iq_f64(mxGetPr(prhs[0]), (int64_t)(rows / 2), (int64_t)cols, out), "raw2iq");
    else mexErrMsgIdAndTxt("gsmcal:type", "raw2iq: expected uint8 or real double");
    plhs[0] = put_c128(out, rows / 2, cols);
    mxFree(out);
}

#elif defined(GSMCAL_MEX_fir_filter)
/* r = fir_filter(coef, s [, decim])  - replaces  r = filter(coef,1,s); r = r(1:decim:end,:)   gsm_sync_demod.m:110,117 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    (void)nlhs; init_once();
    if (nrhs < 2 || nrhs > 3) mexErrMsgIdAndTxt("gsmcal:nargin", "usage: r = fir_filter(coef, s [, decim])");
    size_t nt; const double *coef = real_vector(prhs[0], &nt);
    double decim_d = nrhs == 3 ? mxGetScalar(prhs[2]) : 1.0;
    if (!(decim_d >= 1.0 && decim_d <= 1e9) || decim_d != floor(decim_d))      /* before any size is derived from it */
        mexErrMsgIdAndTxt("gsmcal:decim", "fir_filter: decim must be a positive integer");
    int decim = (int)decim_d;
    size_t rows = mxGetM(prhs[1]), cols = mxGetN(prhs[1]);
    int own; const double *s = get_c128(prhs[1], &own);
    size_t n_out = (rows + decim - 1) / decim;
    double *out = (double *)mxMalloc(2 * n_out * cols * sizeof(double) + 16);
    fail_on(gsmcal_fir_filter(coef, (int)nt, s, (int64_t)rows, (int64_t)cols, decim, out), "fir_filter");
    plhs[0] = put_c128(out, n_out, cols);
    mxFree(out); if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_chn_filter_8x_4x) || defined(GSMCAL_MEX_chn_filter_4x)
/* r = chn_filter_8x_4x(s)  chn_filter_8x_4x.m:5 ;  r = chn_filter_4x(s)  chn_filter_4x.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    (void)nlhs; init_once(); need(nrhs, 1, "r = chn_filter_*(s)");
    size_t rows = mxGetM(prhs[0]), cols = mxGetN(prhs[0]);
    int own; const double *s = get_c128(prhs[0], &own);
#if defined(GSMCAL_MEX_chn_filter_8x_4x)
    size_t n_out = (rows + 1) / 2;
    double *out = (double *)mxMalloc(2 * n_out * cols * sizeof(double) + 16);
    fail_on(gsmcal_chn_filter_8x_4x(s, (int64_t)rows, (int64_t)cols, out), "chn_filter_8x_4x");
#else
    size_t n_out = rows;
    double *out = (double *)mxMalloc(2 * n_out * cols * sizeof(double) + 16);
    fail_on(gsmcal_chn_filter_4x(s, (int64_t)rows, (int64_t)cols, out), "chn_filter_4x");
#endif
    plhs[0] = put_c128(out, n_out, cols);
    mxFree(out); if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_move_fft_snr_runtime_avg)
/* [hit_flag, hit_idx, hit_avg_snr, hit_snr] = move_fft_snr_runtime_avg(s, mv_len, fft_len, th)   move_fft_snr_runtime_avg.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "[hit_flag,hit_idx,hit_avg_snr,hit_snr] = move_fft_snr_runtime_avg(s,mv_len,fft_len,th)");
    int own; const double *s = get_c128(prhs[0], &own);
    int flag; double idx, avg, snr;
    fail_on(gsmcal_move_fft_snr_runtime_avg(s, (int64_t)mxGetNumberOfElements(prhs[0]), (int)mxGetScalar(prhs[1]), (int)mxGetScalar(prhs[2]),
                                            mxGetScalar(prhs[3]), &flag, &idx, &avg, &snr), "move_fft_snr_runtime_avg");
    plhs[0] = mxCreateLogicalScalar(flag != 0);
    if (nlhs > 1) plhs[1] = scalar(idx);
    if (nlhs > 2) plhs[2] = scalar(avg);
    if (nlhs > 3) plhs[3] = scalar(snr);
    if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_specific_fft_snr_fix_avg)
/* [hit_flag, hit_idx, hit_snr] = specific_fft_snr_fix_avg(s, target_set, fft_len, th, avg_snr)   specific_fft_snr_fix_avg.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 5, "[hit_flag,hit_idx,hit_snr] = specific_fft_snr_fix_avg(s,target_set,fft_len,th,avg_snr)");
    int own; const double *s = get_c128(prhs[0], &own);
    size_t nt; const double *ts = real_vector(prhs[1], &nt);
    if (nt < 2) mexErrMsgIdAndTxt("gsmcal:size", "target_set needs two elements");
    int flag; double idx, snr;
    fail_on(gsmcal_specific_fft_snr_fix_avg(s, (int64_t)mxGetNumberOfElements(prhs[0]), (int64_t)ts[0], (int64_t)ts[1], (int)mxGetScalar(prhs[2]),
                                            mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), &flag, &idx, &snr), "specific_fft_snr_fix_avg");
    plhs[0] = mxCreateLogicalScalar(flag != 0);
    if (nlhs > 1) plhs[1] = scalar(idx);
    if (nlhs > 2) plhs[2] = scalar(snr);
    if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_FCCH_coarse_position)
/* [position, snr] = FCCH_coarse_position(s, decimation_ratio)                         FCCH_coarse_position.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 2, "[position,snr] = FCCH_coarse_position(s,decimation_ratio)");
    int own; const double *s = get_c128(prhs[0], &own);
    int64_t len = (int64_t)mxGetNumberOfElements(prhs[0]);
    int dr = (int)mxGetScalar(prhs[1]);
    int64_t cap = gsmcal_max_bursts(len, dr), n = 0;
    double *pos = (double *)mxMalloc(cap * sizeof(double)), *snr = (double *)mxMalloc(cap * sizeof(double));
    fail_on(gsmcal_FCCH_coarse_position(s, len, dr, pos, snr, cap, &n), "FCCH_coarse_position");
    if (n < 0) { plhs[0] = scalar(-1); if (nlhs > 1) plhs[1] = scalar(-1); mexPrintf("FCCH coarse: No FCCH found!\n"); }
    else { plhs[0] = row_vector(pos, (size_t)n); if (nlhs > 1) plhs[1] = row_vector(snr, (size_t)n); }
    mxFree(pos); mxFree(snr); if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_FCCH_fine_correction)
/* [FCCH_pos, r, sampling_ppm, carrier_ppm] = FCCH_fine_correction(s, base_position, oversampling_ratio, carrier_freq)   FCCH_fine_correction.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "[FCCH_pos,r,sampling_ppm,carrier_ppm] = FCCH_fine_correction(s,base_position,oversampling_ratio,carrier_freq)");
    int own; const double *s = get_c128(prhs[0], &own);
    int64_t n = (int64_t)mxGetNumberOfElements(prhs[0]);
    size_t nb; const double *base = real_vector(prhs[1], &nb);
    double *pos = (double *)mxMalloc((nb + 1) * sizeof(double));
    double *r = (double *)mxMalloc(2 * (size_t)n * sizeof(double) + 16);
    int64_t n_pos = 0, r_len = 0; double sppm, cppm;
    fail_on(gsmcal_FCCH_fine_correction(s, n, base, (int64_t)nb, (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), pos, (int64_t)nb + 1, &n_pos,
                                        r, n, &r_len, &sppm, &cppm), "FCCH_fine_correction");
    plhs[0] = n_pos < 0 ? scalar(-1) : row_vector(pos, (size_t)n_pos);
    if (nlhs > 1) plhs[1] = r_len < 0 ? scalar(-1) : put_c128(r, (size_t)r_len, 1);
    if (nlhs > 2) plhs[2] = scalar(sppm);
    if (nlhs > 3) plhs[3] = scalar(cppm);
    mxFree(pos); mxFree(r); if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_gsm_SCH_training_sequence_gen)
/* s = gsm_SCH_training_sequence_gen(oversampling_ratio)                       gsm_SCH_training_sequence_gen.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    (void)nlhs; need(nrhs, 1, "s = gsm_SCH_training_sequence_gen(oversampling_ratio)");
    int osr = (int)mxGetScalar(prhs[0]);
    double *buf = (double *)mxMalloc(2 * 64 * (size_t)(osr > 0 ? osr : 1) * sizeof(double));
    fail_on(gsmcal_SCH_training_sequence_gen(osr, buf), "gsm_SCH_training_sequence_gen");
    plhs[0] = put_c128(buf, 64 * (size_t)osr, 1);
    mxFree(buf);
}

#elif defined(GSMCAL_MEX_SCH_corr_rate_correction)
/* [pos_info, r, sampling_ppm] = SCH_corr_rate_correction(s, FCCH_pos, sch_training_sequence, oversampling_ratio)   SCH_corr_rate_correction.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "[pos_info,r,sampling_ppm] = SCH_corr_rate_correction(s,FCCH_pos,sch_training_sequence,oversampling_ratio)");
    int own, own_t; const double *s = get_c128(prhs[0], &own);
    int64_t n = (int64_t)mxGetNumberOfElements(prhs[0]);
    size_t nf; const double *fpos = real_vector(prhs[1], &nf);
    const double *tpl = get_c128(prhs[2], &own_t);
    int osr = (int)mxGetScalar(prhs[3]);
    if (mxGetNumberOfElements(prhs[2]) != (size_t)(64 * osr)) mexErrMsgIdAndTxt("gsmcal:size", "sch_training_sequence must have 64*oversampling_ratio samples");
    int64_t cap = 6 * (int64_t)nf + 1, n_rows = 0, r_len = 0; double sppm;
    double *pi = (double *)mxMalloc(2 * (size_t)cap * sizeof(double));
    double *r = (double *)mxMalloc(2 * (size_t)n * sizeof(double) + 16);
    fail_on(gsmcal_SCH_corr_rate_correction(s, n, fpos, (int64_t)nf, tpl, osr, pi, cap, &n_rows, r, n, &r_len, &sppm), "SCH_corr_rate_correction");
    if (n_rows < 0) { plhs[0] = mxCreateDoubleMatrix(1, 2, mxREAL); mxGetPr(plhs[0])[0] = -1; mxGetPr(plhs[0])[1] = -1; }
    else { plhs[0] = mxCreateDoubleMatrix((size_t)n_rows, 2, mxREAL); memcpy(mxGetPr(plhs[0]), pi, 2 * (size_t)n_rows * sizeof(double)); }
    if (nlhs > 1) plhs[1] = r_len < 0 ? scalar(-1) : put_c128(r, (size_t)r_len, 1);
    if (nlhs > 2) plhs[2] = scalar(sppm);
    mxFree(pi); mxFree(r); if (own) mxFree((void *)s); if (own_t) mxFree((void *)tpl);
}

#elif defined(GSMCAL_MEX_carrier_correct_post_SCH)
/* [r, carrier_ppm] = carrier_correct_post_SCH(s, pos_info, oversampling_ratio, carrier_freq)   carrier_correct_post_SCH.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "[r,carrier_ppm] = carrier_correct_post_SCH(s,pos_info,oversampling_ratio,carrier_freq)");
    int own; const double *s = get_c128(prhs[0], &own);
    int64_t n = (int64_t)mxGetNumberOfElements(prhs[0]);
    if (!mxIsDouble(prhs[1]) || mxIsComplex(prhs[1]) || mxGetN(prhs[1]) != 2) mexErrMsgIdAndTxt("gsmcal:size", "pos_info must be R x 2");
    int64_t r_len = 0; double cppm;
    double *r = (double *)mxMalloc(2 * (size_t)n * sizeof(double) + 16);
    fail_on(gsmcal_carrier_correct_post_SCH(s, n, mxGetPr(prhs[1]), (int64_t)mxGetM(prhs[1]), (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[3]),
                                            r, n, &r_len, &cppm), "carrier_correct_post_SCH");
    plhs[0] = r_len < 0 ? scalar(-1) : put_c128(r, (size_t)r_len, 1);
    if (nlhs > 1) plhs[1] = scalar(cppm);
    mxFree(r); if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_total_ppm_calculation)
/* ppm_out = total_ppm_calculation(ppm_in)                                             total_ppm_calculation.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    (void)nlhs; need(nrhs, 1, "ppm_out = total_ppm_calculation(ppm_in)");
    size_t n; const double *p = real_vector(prhs[0], &n);
    double out;
    fail_on(gsmcal_total_ppm_calculation(p, (int64_t)n, &out), "total_ppm_calculation");
    plhs[0] = scalar(out);
}

#elif defined(GSMCAL_MEX_gsm_calibrate_batch)
/* [sampling_ppm, carrier_ppm, n_pos_info, pos_info, timing] = gsm_calibrate_batch(raw_uint8, carrier_freq, sch_training_sequence, coef)
 * raw_uint8: 2N x D uint8 (one dongle per column) - gsm_sync_demod.m:107-124 for all dongles in one call.
 * sampling_ppm, carrier_ppm: 3 x D ([FCCH stage; SCH/post stage; total]); pos_info: (6B) x 2 x D, rows beyond n_pos_info(d) are NaN.
 * timing (asked for only: with four outputs nothing more runs): 1 x D struct array of the sub-sample SCH timing and clock fit of
 * gsmcal_calibrate_sch_timing_batch: t0 (raw-capture samples, 0-based), fit_ppm, rms, n_fit, flags (1 pos_info == -1, 2 r_correct == -1,
 * 4 a correlation window leaves r_correct, 8 a maximum on the first or last lag, 16 fewer than 3 fitted bursts), tau and x (1 x n_sch:
 * each SCH burst's time in r_correct and in the capture, NaN where excluded; empty when the step did not run).  See include/gsmcal.h. */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once();
    if (nrhs != 4 || nlhs > 5)
        mexErrMsgIdAndTxt("gsmcal:nargin", "usage: [sampling_ppm,carrier_ppm,n_pos_info,pos_info,timing] = "
                          "gsm_calibrate_batch(raw_uint8,carrier_freq,sch_training_sequence,coef)");
    if (!mxIsUint8(prhs[0])) mexErrMsgIdAndTxt("gsmcal:type", "raw must be uint8");
    size_t rows = mxGetM(prhs[0]), D = mxGetN(prhs[0]);
    int own; const double *tpl = get_c128(prhs[2], &own);
    size_t nt; const double *coef = real_vector(prhs[3], &nt);
    int64_t n_iq = (int64_t)(rows / 2);
    int64_t B = gsmcal_max_bursts((n_iq + 63) / 64, 8);
    gsmcal_stream_result *res = (gsmcal_stream_result *)mxMalloc(D * sizeof(*res));
    double *pi = (double *)mxMalloc(D * 12 * (size_t)B * sizeof(double));
    gsmcal_sch_timing_result *tm = NULL;
    double *tau = NULL, *xr = NULL;
    if (nlhs > 4) {
        tm = (gsmcal_sch_timing_result *)mxMalloc(D * sizeof(*tm));
        tau = (double *)mxMalloc(2 * D * (size_t)B * sizeof(double)); xr = tau + D * (size_t)B;
        fail_on(gsmcal_calibrate_sch_timing_batch((const uint8_t *)mxGetData(prhs[0]), GSMCAL_MEM_HOST, n_iq, (int64_t)D, mxGetScalar(prhs[1]), tpl, coef,
                                                  (int)nt, 8, 8, res, NULL, NULL, NULL, pi, NULL, tm, tau, xr), "gsm_calibrate_batch");
    } else
        fail_on(gsmcal_calibrate_batch((const uint8_t *)mxGetData(prhs[0]), GSMCAL_MEM_HOST, n_iq, (int64_t)D, mxGetScalar(prhs[1]), tpl, coef, (int)nt, 8, 8,
                                       res, NULL, NULL, NULL, pi, NULL), "gsm_calibrate_batch");
    batch_outputs(nlhs, plhs, res, pi, D, (size_t)B);
    if (nlhs > 4) {
        const char *f[] = {"t0", "fit_ppm", "rms", "n_fit", "flags", "tau", "x"};
        plhs[4] = mxCreateStructMatrix(1, D, 7, f);
        for (size_t d = 0; d < D; ++d) {
            const size_t n = tm[d].n_sch > 0 ? (size_t)tm[d].n_sch : 0;
            mxArray *ta = mxCreateDoubleMatrix(1, n, mxREAL), *xa = mxCreateDoubleMatrix(1, n, mxREAL);
            if (n) { memcpy(mxGetPr(ta), tau + d * B, n * sizeof(double)); memcpy(mxGetPr(xa), xr + d * B, n * sizeof(double)); }
            mxSetField(plhs[4], d, "t0", scalar(tm[d].t0)); mxSetField(plhs[4], d, "fit_ppm", scalar(tm[d].fit_ppm));
            mxSetField(plhs[4], d, "rms", scalar(tm[d].rms)); mxSetField(plhs[4], d, "n_fit", scalar(tm[d].n_fit));
            mxSetField(plhs[4], d, "flags", scalar(tm[d].flags)); mxSetField(plhs[4], d, "tau", ta); mxSetField(plhs[4], d, "x", xa);
        }
        mxFree(tm); mxFree(tau);
    }
    mxFree(res); mxFree(pi); if (own) mxFree((void *)tpl);
}

#elif defined(GSMCAL_MEX_gsm_calibrate_demod_batch) || defined(GSMCAL_MEX_gsm_calibrate_sch_decode_batch)
/* [sampling_ppm, carrier_ppm, n_pos_info, pos_info, sch, fcch, bcch] =
 *     gsm_calibrate_demod_batch(raw_uint8, carrier_freq, sch_training_sequence, coef [, normal_training_sequence])
 * gsm_calibrate_batch (outputs 1-4 as there) followed by SCH_demod / FCCH_demod on every dongle's r_correct (gsm_sync_demod.m:144-145),
 * and with normal_training_sequence ((26*8) x 8, gsm_normal_training_sequence_gen(8)) BCCH_demod as well (:146).
 * sch, fcch, bcch: 1 x D struct arrays, one element per dongle.
 *   sch(d):  demod_bits, bits_to_decoder (148 x n_sch), corr_val (85 x n_sch), sch_ok (1 x n_sch), flags;
 *   fcch(d): freq, snr, max_idx (1 x n_fcch), mean_freq, carrier_ppm, flags;
 *   bcch(d): carrier_ppm, idx (1..8 or -1), corr_abs (8 x 4, abs(corr_val)), flags.
 * Where the reference would not get that far (pos_info == -1, r_correct == -1: flags 1 / 2) the fields are empty and n_sch = -1 is
 * reported as empty arrays; flags 4 / 8: a window leaves r_correct (sch_ok 0 / NaN rows, NaN mean).  bcch(d).flags: 1 pos_info == -1,
 * 2 fewer than four BCCH rows (carrier_ppm = idx = -1), 4 no FCCH mean (carrier_ppm NaN, idx -1), 8 a training window leaves
 * r_correct (NaN column, idx -1); corr_abs is NaN where it was not computed.  See include/gsmcal.h.
 *
 * [sampling_ppm, carrier_ppm, n_pos_info, pos_info, sch, fcch, cell] = gsm_calibrate_sch_decode_batch(raw_uint8, carrier_freq, sch_training_sequence, coef)
 * (GSMCAL_MEX_gsm_calibrate_sch_decode_batch) is the same call followed by SCH channel decoding (gsmcal_calibrate_sch_decode_batch):
 *   cell(d): bsic (0..63 or -1), ncc, bcc, fn_first (TDMA frame number of the first SCH row of pos_info, or -1), frame_clock_start (GSM
 *   time of capture sample 0 in samples since FN 0 of the hyperframe, NaN without a winner), n_crc_ok, n_agree, flags (1 pos_info == -1,
 *   2 r_correct == -1, 4 no row decoded, 8 rows disagree), and per SCH row fn, bsic (-1 where not decoded), hamming, row_flags
 *   (1 x n_sch; 1 window outside r_correct, 2 training peak too far from bit 42, 4 CRC, 8 invalid T2 / T3'). */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once();
#if defined(GSMCAL_MEX_gsm_calibrate_sch_decode_batch)
    if (nrhs != 4 || nlhs > 7)
        mexErrMsgIdAndTxt("gsmcal:nargin", "usage: [sampling_ppm,carrier_ppm,n_pos_info,pos_info,sch,fcch,cell] = "
                          "gsm_calibrate_sch_decode_batch(raw_uint8,carrier_freq,sch_training_sequence,coef)");
#else
    if (nrhs < 4 || nrhs > 5 || (nlhs > 6 && nrhs < 5))
        mexErrMsgIdAndTxt("gsmcal:nargin", "usage: [sampling_ppm,carrier_ppm,n_pos_info,pos_info,sch,fcch,bcch] = "
                          "gsm_calibrate_demod_batch(raw_uint8,carrier_freq,sch_training_sequence,coef[,normal_training_sequence]) (bcch needs the fifth input)");
#endif
    if (!mxIsUint8(prhs[0])) mexErrMsgIdAndTxt("gsmcal:type", "raw must be uint8");
    size_t rows = mxGetM(prhs[0]), D = mxGetN(prhs[0]);
    int own, own_n = 0; const double *tpl = get_c128(prhs[2], &own), *nts = NULL;
    size_t nt; const double *coef = real_vector(prhs[3], &nt);
    if (nrhs > 4) {
        if (mxGetM(prhs[4]) != 26 * 8 || mxGetN(prhs[4]) != 8) mexErrMsgIdAndTxt("gsmcal:size", "normal_training_sequence must be (26*8) x 8");
        nts = get_c128(prhs[4], &own_n);
    }
    int64_t n_iq = (int64_t)(rows / 2);
    size_t B = (size_t)gsmcal_max_bursts((n_iq + 63) / 64, 8), R = D * B;
    gsmcal_stream_result *res = (gsmcal_stream_result *)mxMalloc(D * sizeof(*res));
    gsmcal_demod_result *dem = (gsmcal_demod_result *)mxMalloc(D * sizeof(*dem));
    gsmcal_bcch_result *bc = nts ? (gsmcal_bcch_result *)mxMalloc(D * sizeof(*bc)) : NULL;
    double *pi = (double *)mxMalloc(D * 12 * B * sizeof(double));
    uint8_t *ok = (uint8_t *)mxMalloc(R * (1 + 2 * 148)), *bits = ok + R, *dec = bits + 148 * R;
    double *corr = (double *)mxMalloc(R * 88 * sizeof(double)), *freq = corr + 85 * R, *snr = freq + R, *idx = snr + R;
#if defined(GSMCAL_MEX_gsm_calibrate_sch_decode_batch)
    gsmcal_sch_decode_result *sd = (gsmcal_sch_decode_result *)mxMalloc(D * sizeof(*sd));
    int32_t *sfn = (int32_t *)mxMalloc(R * 2 * sizeof(int32_t)), *sbs = sfn + R;
    uint8_t *sham = (uint8_t *)mxMalloc(R * 2), *srf = sham + R;
    fail_on(gsmcal_calibrate_sch_decode_batch((const uint8_t *)mxGetData(prhs[0]), GSMCAL_MEM_HOST, n_iq, (int64_t)D, mxGetScalar(prhs[1]), tpl, coef, (int)nt,
                                              8, 8, res, NULL, NULL, NULL, pi, NULL, dem, ok, bits, dec, corr, freq, snr, idx, NULL, NULL,
                                              sd, sfn, sbs, sham, srf), "gsm_calibrate_sch_decode_batch");
#else
    if (nts)
        fail_on(gsmcal_calibrate_demod_bcch_batch((const uint8_t *)mxGetData(prhs[0]), GSMCAL_MEM_HOST, n_iq, (int64_t)D, mxGetScalar(prhs[1]), tpl, coef, (int)nt,
                                                  8, 8, res, NULL, NULL, NULL, pi, NULL, dem, ok, bits, dec, corr, freq, snr, idx, nts, bc),
                "gsm_calibrate_demod_batch");
    else
        fail_on(gsmcal_calibrate_demod_batch((const uint8_t *)mxGetData(prhs[0]), GSMCAL_MEM_HOST, n_iq, (int64_t)D, mxGetScalar(prhs[1]), tpl, coef, (int)nt, 8, 8,
                                             res, NULL, NULL, NULL, pi, NULL, dem, ok, bits, dec, corr, freq, snr, idx), "gsm_calibrate_demod_batch");
#endif
    batch_outputs(nlhs, plhs, res, pi, D, B);
    if (nlhs > 4) {
        const char *f[] = {"demod_bits", "bits_to_decoder", "corr_val", "sch_ok", "flags"};
        plhs[4] = mxCreateStructMatrix(1, D, 5, f);
        for (size_t d = 0; d < D; ++d) {
            size_t k = dem[d].n_sch < 0 ? 0 : (size_t)dem[d].n_sch;
            mxArray *a = mxCreateDoubleMatrix(148, k, mxREAL), *b = mxCreateDoubleMatrix(148, k, mxREAL);
            mxArray *cv = mxCreateDoubleMatrix(85, k, mxREAL), *so = mxCreateDoubleMatrix(1, k, mxREAL);
            for (size_t i = 0; i < 148 * k; ++i) { mxGetPr(a)[i] = bits[148 * d * B + i]; mxGetPr(b)[i] = dec[148 * d * B + i]; }
            if (k) memcpy(mxGetPr(cv), corr + 85 * d * B, 85 * k * sizeof(double));
            for (size_t i = 0; i < k; ++i) mxGetPr(so)[i] = ok[d * B + i];
            mxSetField(plhs[4], d, "demod_bits", a); mxSetField(plhs[4], d, "bits_to_decoder", b); mxSetField(plhs[4], d, "corr_val", cv);
            mxSetField(plhs[4], d, "sch_ok", so); mxSetField(plhs[4], d, "flags", scalar(dem[d].flags));
        }
    }
    if (nlhs > 5) {
        const char *f[] = {"freq", "snr", "max_idx", "mean_freq", "carrier_ppm", "flags"};
        plhs[5] = mxCreateStructMatrix(1, D, 6, f);
        for (size_t d = 0; d < D; ++d) {
            size_t k = dem[d].n_fcch < 0 ? 0 : (size_t)dem[d].n_fcch;
            mxSetField(plhs[5], d, "freq", row_vector(freq + d * B, k)); mxSetField(plhs[5], d, "snr", row_vector(snr + d * B, k));
            mxSetField(plhs[5], d, "max_idx", row_vector(idx + d * B, k)); mxSetField(plhs[5], d, "mean_freq", scalar(dem[d].fcch_mean_freq));
            mxSetField(plhs[5], d, "carrier_ppm", scalar(dem[d].fcch_carrier_ppm)); mxSetField(plhs[5], d, "flags", scalar(dem[d].flags));
        }
    }
#if defined(GSMCAL_MEX_gsm_calibrate_sch_decode_batch)
    if (nlhs > 6) {
        const char *f[] = {"bsic", "ncc", "bcc", "fn_first", "frame_clock_start", "n_crc_ok", "n_agree", "flags", "fn", "bsic_rows", "hamming", "row_flags"};
        plhs[6] = mxCreateStructMatrix(1, D, 12, f);
        for (size_t d = 0; d < D; ++d) {
            const gsmcal_sch_decode_result *c = sd + d;
            const size_t k = c->n_sch < 0 ? 0 : (size_t)c->n_sch;
            mxArray *a[4];
            for (int j = 0; j < 4; ++j) a[j] = mxCreateDoubleMatrix(1, k, mxREAL);
            for (size_t i = 0; i < k; ++i) {
                mxGetPr(a[0])[i] = sfn[d * B + i]; mxGetPr(a[1])[i] = sbs[d * B + i];
                mxGetPr(a[2])[i] = sham[d * B + i]; mxGetPr(a[3])[i] = srf[d * B + i];
            }
            mxSetField(plhs[6], d, "bsic", scalar(c->bsic)); mxSetField(plhs[6], d, "ncc", scalar(c->bsic < 0 ? -1 : c->bsic >> 3));
            mxSetField(plhs[6], d, "bcc", scalar(c->bsic < 0 ? -1 : c->bsic & 7)); mxSetField(plhs[6], d, "fn_first", scalar(c->fn_first));
            mxSetField(plhs[6], d, "frame_clock_start", scalar(c->frame_clock_start)); mxSetField(plhs[6], d, "n_crc_ok", scalar(c->n_crc_ok));
            mxSetField(plhs[6], d, "n_agree", scalar(c->n_agree)); mxSetField(plhs[6], d, "flags", scalar(c->flags));
            mxSetField(plhs[6], d, "fn", a[0]); mxSetField(plhs[6], d, "bsic_rows", a[1]);
            mxSetField(plhs[6], d, "hamming", a[2]); mxSetField(plhs[6], d, "row_flags", a[3]);
        }
    }
    mxFree(sd); mxFree(sfn); mxFree(sham);
#else
    if (nlhs > 6) {
        const char *f[] = {"carrier_ppm", "idx", "corr_abs", "flags"};
        plhs[6] = mxCreateStructMatrix(1, D, 4, f);
        for (size_t d = 0; d < D; ++d) {
            mxArray *ca = mxCreateDoubleMatrix(8, 4, mxREAL);
            memcpy(mxGetPr(ca), bc[d].corr_abs, sizeof bc[d].corr_abs);
            mxSetField(plhs[6], d, "carrier_ppm", scalar(bc[d].carrier_ppm)); mxSetField(plhs[6], d, "idx", scalar(bc[d].nts_idx));
            mxSetField(plhs[6], d, "corr_abs", ca); mxSetField(plhs[6], d, "flags", scalar(bc[d].flags));
        }
    }
#endif
    mxFree(res); mxFree(dem); mxFree(pi); mxFree(ok); mxFree(corr); if (bc) mxFree(bc); if (own) mxFree((void *)tpl); if (own_n) mxFree((void *)nts);
}

#elif defined(GSMCAL_MEX_gsm_normal_training_sequence_gen)
/* s = gsm_normal_training_sequence_gen(oversampling_ratio)                 gsm_normal_training_sequence_gen.m:5 */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    (void)nlhs; need(nrhs, 1, "s = gsm_normal_training_sequence_gen(oversampling_ratio)");
    int osr = (int)mxGetScalar(prhs[0]);
    double *buf = (double *)mxMalloc(2 * 8 * 26 * (size_t)(osr > 0 ? osr : 1) * sizeof(double));
    fail_on(gsmcal_normal_training_sequence_gen(osr, buf), "gsm_normal_training_sequence_gen");
    plhs[0] = put_c128(buf, 26 * (size_t)osr, 8);
    mxFree(buf);
}

#elif defined(GSMCAL_MEX_FCCH_demod)
/* FCCH_demod(s, pos_info, oversampling_ratio, carrier_freq)                                     FCCH_demod.m:5
 * The reference only displays; optional outputs here: [freq, snr, carrier_ppm, max_idx]. */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "FCCH_demod(s,pos_info,oversampling_ratio,carrier_freq)");
    int own; const double *s = get_c128(prhs[0], &own);
    int64_t n = (int64_t)mxGetNumberOfElements(prhs[0]);
    if (!mxIsDouble(prhs[1]) || mxIsComplex(prhs[1]) || mxGetN(prhs[1]) != 2) mexErrMsgIdAndTxt("gsmcal:size", "pos_info must be R x 2");
    size_t rows = mxGetM(prhs[1]), cap = rows ? rows : 1;
    double *freq = (double *)mxMalloc(3 * cap * sizeof(double)), *snr = freq + cap, *idx = snr + cap, mean_freq, cppm;
    int64_t h = 0;
    fail_on(gsmcal_FCCH_demod(s, n, mxGetPr(prhs[1]), (int64_t)rows, (int)mxGetScalar(prhs[2]), mxGetScalar(prhs[3]),
                              freq, snr, idx, (int64_t)cap, &h, &mean_freq, &cppm), "FCCH_demod");
    mexPrintf(" \n");
    if (h < 0) mexPrintf("FCCH demod: Warning! No valid position information!\n");                   /* :8 */
    else {
        mexPrintf("FCCH demod: FCCH freq");  for (int64_t i = 0; i < h; ++i) mexPrintf(" %.5g", freq[i]); mexPrintf("\n");      /* :42 */
        mexPrintf("FCCH demod: mean FCCH freq %.5g\nFCCH demod: carrier error ppm %.5g\n", mean_freq, cppm);                   /* :44,48 */
        mexPrintf("FCCH demod: SNR");        for (int64_t i = 0; i < h; ++i) mexPrintf(" %.5g", snr[i]);  mexPrintf("\n");      /* :65 */
        mexPrintf("FCCH demod: max idx");    for (int64_t i = 0; i < h; ++i) mexPrintf(" %g", idx[i]);    mexPrintf("\n");      /* :66 */
    }
    size_t k = h < 0 ? 0 : (size_t)h;
    if (nlhs > 0) plhs[0] = row_vector(freq, k);
    if (nlhs > 1) plhs[1] = row_vector(snr, k);
    if (nlhs > 2) plhs[2] = scalar(cppm);
    if (nlhs > 3) plhs[3] = row_vector(idx, k);
    mxFree(freq); if (own) mxFree((void *)s);
}

#elif defined(GSMCAL_MEX_BCCH_demod)
/* BCCH_demod(s, pos_info, normal_training_sequence, oversampling_ratio [, carrier_freq])       BCCH_demod.m:5
 * (the reference reads carrier_freq without defining it; default 957.4e6, gsm_sync_demod.m:14).
 * Optional outputs: [carrier_ppm, normal_training_sequence_idx, abs(corr_val)]. */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "BCCH_demod(s,pos_info,normal_training_sequence,oversampling_ratio[,carrier_freq])");
    int own, own_t; const double *s = get_c128(prhs[0], &own);
    int64_t n = (int64_t)mxGetNumberOfElements(prhs[0]);
    if (!mxIsDouble(prhs[1]) || mxIsComplex(prhs[1]) || mxGetN(prhs[1]) != 2) mexErrMsgIdAndTxt("gsmcal:size", "pos_info must be R x 2");
    const double *nts = get_c128(prhs[2], &own_t);
    int osr = (int)mxGetScalar(prhs[3]);
    if (mxGetM(prhs[2]) != (size_t)(26 * osr) || mxGetN(prhs[2]) != 8) mexErrMsgIdAndTxt("gsmcal:size", "normal_training_sequence must be (26*oversampling_ratio) x 8");
    double carrier_freq = nrhs > 4 ? mxGetScalar(prhs[4]) : 957.4e6, cppm, mag[32];
    int idx;
    for (int i = 0; i < 32; ++i) mag[i] = 0.0;
    fail_on(gsmcal_BCCH_demod(s, n, mxGetPr(prhs[1]), (int64_t)mxGetM(prhs[1]), nts, osr, carrier_freq, &cppm, &idx, mag), "BCCH_demod");
    if (idx > 0) mexPrintf("Normal training sequence idx (BCCH) %d\n", idx);                       /* :95 */
    else if (cppm != -1.0) mexPrintf("Fail to identity normal training sequence idx (BCCH).\n");   /* :98 */
    if (nlhs > 0) plhs[0] = scalar(cppm);
    if (nlhs > 1) plhs[1] = scalar((double)idx);
    if (nlhs > 2) { plhs[2] = mxCreateDoubleMatrix(8, 4, mxREAL); memcpy(mxGetPr(plhs[2]), mag, sizeof mag); }
    if (own) mxFree((void *)s); if (own_t) mxFree((void *)nts);
}

#elif defined(GSMCAL_MEX_SCH_demod)
/* SCH_demod(s, pos_info, training_sequence, oversampling_ratio)                                 SCH_demod.m:5
 * Optional outputs: [demod_bits (148 x H), bits_to_decoder (148 x H), corr_val (85 x H)]. */
void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    init_once(); need(nrhs, 4, "SCH_demod(s,pos_info,training_sequence,oversampling_ratio)");
    int own, own_t; const double *s = get_c128(prhs[0], &own);
    int64_t n = (int64_t)mxGetNumberOfElements(prhs[0]);
    if (!mxIsDouble(prhs[1]) || mxIsComplex(prhs[1]) || mxGetN(prhs[1]) != 2) mexErrMsgIdAndTxt("gsmcal:size", "pos_info must be R x 2");
    const double *tpl = get_c128(prhs[2], &own_t);
    int osr = (int)mxGetScalar(prhs[3]);
    if (mxGetNumberOfElements(prhs[2]) != (size_t)(64 * osr)) mexErrMsgIdAndTxt("gsmcal:size", "training_sequence must have 64*oversampling_ratio samples");
    size_t rows = mxGetM(prhs[1]), cap = rows ? rows : 1;
    uint8_t *bits = (uint8_t *)mxMalloc(2 * 148 * cap), *dec = bits + 148 * cap;
    double *corr = (double *)mxMalloc(85 * cap * sizeof(double));
    int64_t h = 0;
    fail_on(gsmcal_SCH_demod(s, n, mxGetPr(prhs[1]), (int64_t)rows, tpl, osr, (int64_t)cap, &h, bits, dec, corr), "SCH_demod");
    mexPrintf(" \n");
    if (h < 0) mexPrintf("SCH demod: Warning! No valid position information!\n");                    /* :9 */
    size_t k = h < 0 ? 0 : (size_t)h;
    for (int o = 0; o < 2 && o < nlhs; ++o) {
        plhs[o] = mxCreateDoubleMatrix(148, k, mxREAL);
        const uint8_t *src = o ? dec : bits;
        for (size_t i = 0; i < 148 * k; ++i) mxGetPr(plhs[o])[i] = (double)src[i];
    }
    if (nlhs > 2) { plhs[2] = mxCreateDoubleMatrix(85, k, mxREAL); memcpy(mxGetPr(plhs[2]), corr, 85 * k * sizeof(double)); }
    mxFree(bits); mxFree(corr); if (own) mxFree((void *)s); if (own_t) mxFree((void *)tpl);
}

#else
#error "define GSMCAL_MEX_<function> (see the header of this file)"
#endif
