// gsmcal_demod.cuh - kernels of the SURVEY 8(f) rows 2 and 4 functions (FCCH_demod.m, BCCH_demod.m, SCH_demod.m): the consumers of
// r_correct / pos_info (gsm_sync_demod.m:143-146).  One thread block per burst, materialised complex128 stream in HBM, fp64.
#pragma once
#include "gsmcal_kernels.cuh"

// ===================================================================================================
// FCCH_demod.m:21-66  per FCCH burst: 148*osr-point power spectrum (fftshift order), tone frequency (same statements as K8)
// and the 5-bin-signal / +-half_noise_len-band SNR.  All N bins are needed (the SNR reads 2*55 of them plus 5 around the peak),
// so the spectrum is evaluated once through the 37 x M row FFT.
// ===================================================================================================
#define FD_THREADS 256
// the arithmetic of one burst, its N = 148*osr samples in u (shared; A, F: N double2, P: N doubles of scratch); thread 0 writes output o
__device__ __forceinline__ void fcch_demod_body(double2 *u, double2 *A, double2 *F, double *P, int osr, const double2 *__restrict__ tw,
                                double *__restrict__ freq_out, double *__restrict__ snr_out, double *__restrict__ idx_out, i64 o) {
    __shared__ double red_v[8];
    __shared__ int red_i[8];
    __shared__ double red_n[32];
    __shared__ double sh_pr;
    const int tid = threadIdx.x;
    const int N = 148 * osr;
    const double sampling_rate = ((1625.0 / 6.0) * 1e3) * (double)osr;
    const double2 *Tm = fft_rows(u, A, F, N, tw);
    double v = -1.0; int j_best = 0x7fffffff;
    for (int j = tid; j < N; j += FD_THREADS) {
        int k = j + N / 2; if (k >= N) k -= N;
        const double p = abs2_ref(dft_col(Tm, k, N, tw));
        P[j] = p;
        argmax_combine(v, j_best, p, j);
    }
    block_argmax(v, j_best, red_v, red_i);                     // first maximum (:33); also orders the P[] writes
    // SNR (:53-63)
    const int hnl = (int)ceil(((double)N * 200e3 / sampling_rate) / 2.0);
    double sn[2] = {0.0, 0.0};
    if (tid < 5) { int j = (j_best - 2 + tid) % N; if (j < 0) j += N; sn[0] = P[j]; }
    for (int j = N / 2 - hnl + tid; j <= N / 2 + hnl - 1; j += FD_THREADS) sn[1] += P[j];
    block_sum_n<2, false>(sn, red_n);
    if (tid == 0) {
        const double noise = sn[1] - sn[0];
        snr_out[o] = 10.0 * log10(sn[0] / noise);
        idx_out[o] = (double)(j_best + 1 - (N / 2 + 1));
    }
    // tone frequency (:35-41): integer-bin derotation, unit phasors, angle of the mean one-sample rotation
    const int jr = j_best + 1 - ((N / 2) + 1);
    const double int_phase_rotate = 2.0 * GSMCAL_PI * (double)jr / (double)N;
    int jm = jr % N; if (jm < 0) jm += N;
    for (int n = tid; n < N; n += FD_THREADS) {
        const double2 w = cmul(u[n], tw[(int)(((i64)n * jm) % N)]);
        const double h = hypot(w.x, w.y);
        A[n] = (h > 0.0) ? make_double2(w.x / h, w.y / h) : make_double2(1.0, 0.0);
    }
    __syncthreads();
    double rri[2] = {0.0, 0.0};
    for (int n = tid; n < N - 1; n += FD_THREADS) {
        const double2 a = A[n + 1], b = A[n];
        const double den = b.x * b.x + b.y * b.y;
        rri[0] += (a.x * b.x + a.y * b.y) / den;
        rri[1] += (a.y * b.x - a.x * b.y) / den;
    }
    block_sum_n<2, false>(rri, red_n);
    if (tid == 0) sh_pr = atan2(rri[1] / (double)(N - 1), rri[0] / (double)(N - 1));
    __syncthreads();
    if (tid == 0) freq_out[o] = sampling_rate * (int_phase_rotate + sh_pr) / (2 * GSMCAL_PI);
}
__global__ void __launch_bounds__(FD_THREADS) fcch_demod_kernel(const double2 *__restrict__ s, const double *__restrict__ pos, int osr,
                                                               const double2 *__restrict__ tw, double *__restrict__ freq_out,
                                                               double *__restrict__ snr_out, double *__restrict__ idx_out) {
    extern __shared__ double2 sm[];
    const int burst = blockIdx.x, tid = threadIdx.x;
    const int N = 148 * osr;
    double2 *u = sm, *A = u + N, *F = A + N;
    double *P = (double *)(F + N);                             // fd_fcch column in fftshift order
    const i64 sp = (i64)pos[burst];
    for (int n = tid; n < N; n += FD_THREADS) u[n] = s[sp - 1 + n];
    __syncthreads();
    fcch_demod_body(u, A, F, P, osr, tw, freq_out, snr_out, idx_out, burst);
}

// ===================================================================================================
// BCCH_demod.m:85-91  zero-lag correlation of the first 4 BCCH bursts with the 8 normal training sequences, on the carrier-
// corrected stream r = s .* exp(1i*(0:len-1)'*comp) (:72-73) evaluated only where it is read.  One block per burst, one warp
// per training sequence.
// ===================================================================================================
__global__ void __launch_bounds__(256) nts_corr_kernel(const double2 *__restrict__ s, double dphi, const double *__restrict__ bpos, int osr,
                                                       const double2 *__restrict__ nts /* (26*osr) x 8 column-major */, double *__restrict__ corr_abs /* 8 x 4 */) {
    const int burst = blockIdx.x, q = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int L = 26 * osr;
    const i64 sp0 = (i64)bpos[burst] + 61 * osr - 1;           // 0-based index of the first training sample (:86)
    double ar = 0.0, ai = 0.0;
    for (int n = lane; n < L; n += 32) {
        double sn, cs; sincos((double)(sp0 + n) * dphi, &sn, &cs);
        const double2 r = cmul(s[sp0 + n], make_double2(cs, sn));
        const double2 t = nts[(i64)q * L + n];
        ar += t.x * r.x + t.y * r.y;                             // conj(t) * r
        ai += t.x * r.y - t.y * r.x;
    }
    ar = warp_sum(ar); ai = warp_sum(ai);
    if (lane == 0) corr_abs[burst * 8 + q] = hypot(ar, ai);
}

// ===================================================================================================
// SCH_demod.m:54-110  per SCH burst: frequency-domain equalisation against the known training sequence, MLSE GMSK demodulation,
// +-1 correlation with the 64 training bits.
//   N = (148 + 2*8 + 30)*osr = 194*osr = 97 * (2*osr): two-stage DFT with direct stages (97 is prime), exact twiddle table.
// ===================================================================================================
template <bool INV>
__device__ void dft_pxm(const double2 *in, double2 *tmp, double2 *out, int N, int P, const double2 *__restrict__ tw) {
    const int M = N / P;
    for (int idx = threadIdx.x; idx < N; idx += blockDim.x) {
        const int n2 = idx % M, k1 = idx / M;
        double ar = 0.0, ai = 0.0;
        int t = 0; const int stp = (M * k1) % N;
#pragma unroll 4
        for (int n1 = 0; n1 < P; ++n1) {
            const double2 x = in[M * n1 + n2];
            double2 w = tw[t]; if (INV) w.y = -w.y;
            ar = fma(x.x, w.x, fma(-x.y, w.y, ar));
            ai = fma(x.x, w.y, fma(x.y, w.x, ai));
            t += stp; if (t >= N) t -= N;
        }
        double2 w = tw[(n2 * k1) % N]; if (INV) w.y = -w.y;
        tmp[idx] = cmul(make_double2(ar, ai), w);
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < N; idx += blockDim.x) {
        const int k1 = idx % P, k2 = idx / P;
        double ar = 0.0, ai = 0.0;
        int t = 0; const int stp = (P * k2) % N;
        const double2 *a = tmp + M * k1;
#pragma unroll 4
        for (int n2 = 0; n2 < M; ++n2) {
            const double2 x = a[n2];
            double2 w = tw[t]; if (INV) w.y = -w.y;
            ar = fma(x.x, w.x, fma(-x.y, w.y, ar));
            ai = fma(x.x, w.y, fma(x.y, w.x, ai));
            t += stp; if (t >= N) t -= N;
        }
        out[k1 + P * k2] = INV ? make_double2(ar / (double)N, ai / (double)N) : make_double2(ar, ai);
    }
    __syncthreads();
}
__device__ __forceinline__ double2 cdiv(double2 a, double2 b) {    // Smith's algorithm (what the oracle's complex division does)
    if (fabs(b.x) >= fabs(b.y)) {
        const double rat = b.y / b.x, scl = 1.0 / (b.x + b.y * rat);
        return make_double2((a.x + a.y * rat) * scl, (a.y - a.x * rat) * scl);
    }
    const double rat = b.x / b.y, scl = 1.0 / (b.y + b.x * rat);
    return make_double2((a.x * rat + a.y) * scl, (a.y * rat - a.x) * scl);
}

#define SD_THREADS 256
#define SD_NSYM 194            // 148 + 2*ex_len + TracebackDepth (SCH_demod.m:54)
#define SD_TB 30               // TracebackDepth (:45)
#define SD_EX 8                // ex_len (:53)
// fd_training_ov = fft(zero-padded training sequence) (:57-59): once per call
__global__ void __launch_bounds__(SD_THREADS) fde_template_kernel(const double2 *__restrict__ tpl, int osr, const double2 *__restrict__ tw,
                                                                 double2 *__restrict__ Ft) {
    extern __shared__ double2 sm[];
    const int N = SD_NSYM * osr, sp_tr = (SD_EX + 42) * osr, L = 64 * osr;
    double2 *x = sm, *tmp = x + N, *out = tmp + N;
    for (int n = threadIdx.x; n < N; n += SD_THREADS) x[n] = (n >= sp_tr && n < sp_tr + L) ? tpl[n - sp_tr] : make_double2(0.0, 0.0);
    __syncthreads();
    dft_pxm<false>(x, tmp, out, N, 97, tw);
    for (int n = threadIdx.x; n < N; n += SD_THREADS) Ft[n] = out[n];
}

// MLSE over the 32-state trellis of the L=4, h=1/2 GMSK: state = 8*p + 4*a(m-1) + 2*a(m-2) + a(m-3) (bits; p = accumulated quarter turns),
// lane == new state.  cb[m*16 + combo] = sum_j x[m*osr+j] * conj(W[combo][j]), combo = 8*a(m) + 4*a(m-1) + 2*a(m-2) + a(m-3).
__device__ void gmsk_viterbi_warp(const double2 *cb, int nsym, unsigned char *bits_out) {
    const int lane = threadIdx.x & 31;
    const int pn = lane >> 3, c1 = (lane >> 2) & 1, c2 = (lane >> 1) & 1, c3 = lane & 1;
    const int p0 = (pn + 1) & 3, p1 = (pn + 3) & 3;             // predecessor phase for a(m-3) = 0 (-1: p = pn + 1) / 1 (+1: p = pn - 1)
    const int pred0 = p0 * 8 + (c2 << 2) + (c3 << 1), pred1 = p1 * 8 + (c2 << 2) + (c3 << 1) + 1;
    const int combo0 = (c1 << 3) + (c2 << 2) + (c3 << 1);
    double metric = 0.0;
    unsigned hist = 0u;
    for (int m = 0; m < nsym; ++m) {
        const double2 v0 = cb[m * 16 + combo0], v1 = cb[m * 16 + combo0 + 1];
        const double bm0 = (p0 == 0) ? v0.x : (p0 == 1) ? v0.y : (p0 == 2) ? -v0.x : -v0.y;
        const double bm1 = (p1 == 0) ? v1.x : (p1 == 1) ? v1.y : (p1 == 2) ? -v1.x : -v1.y;
        const double m0 = __shfl_sync(0xffffffffu, metric, pred0) + bm0;
        const double m1 = __shfl_sync(0xffffffffu, metric, pred1) + bm1;
        const unsigned h0 = __shfl_sync(0xffffffffu, hist, pred0), h1 = __shfl_sync(0xffffffffu, hist, pred1);
        const bool take1 = m1 > m0;                              // first maximum: a(m-3) = 0 wins ties
        metric = take1 ? m1 : m0;
        hist = ((take1 ? h1 : h0) << 1) | (unsigned)c1;
        if (m >= SD_TB) {
            double bv = metric; int bi = lane;
            for (int o = 16; o > 0; o >>= 1) {
                const double v2 = __shfl_xor_sync(0xffffffffu, bv, o);
                const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
                if (v2 > bv || (v2 == bv && i2 < bi)) { bv = v2; bi = i2; }
            }
            const unsigned hb = __shfl_sync(0xffffffffu, hist, bi);
            if (lane == 0) bits_out[m] = (unsigned char)((hb >> SD_TB) & 1u);
        } else if (lane == 0) bits_out[m] = 0;
    }
}

// SCH_demod.m:92-110 on the equalised burst x (shared, 194*osr samples): branch correlations of every symbol interval (the trellis
// then only adds; cb: 194*16 double2 of scratch), MLSE, the 148 burst bits, their differential decoding and the 85-lag correlation
__device__ __forceinline__ void sch_bits_body(const double2 *x, double2 *cb, int osr, const double2 *__restrict__ Wtab, const signed char *dpm /* shared */,
                              unsigned char *bits /* shared, SD_NSYM + 2 */, unsigned char *__restrict__ demod_bits, unsigned char *__restrict__ dec_bits,
                              double *__restrict__ corr_val) {
    const int tid = threadIdx.x;
    for (int i = tid; i < SD_NSYM * 16; i += blockDim.x) {
        const int m = i >> 4, combo = i & 15;
        double ar = 0.0, ai = 0.0;
        for (int j = 0; j < osr; ++j) {
            const double2 v = x[m * osr + j], w = Wtab[combo * osr + j];
            ar += v.x * w.x + v.y * w.y;                         // v * conj(w)
            ai += v.y * w.x - v.x * w.y;
        }
        cb[i] = make_double2(ar, ai);
    }
    __syncthreads();
    if (tid < 32) gmsk_viterbi_warp(cb, SD_NSYM, bits);
    __syncthreads();
    // :94-110
    const unsigned char *db = bits + SD_TB + SD_EX;
    for (int i = tid; i < 148; i += blockDim.x) {
        demod_bits[i] = db[i];
        const int nb = 1 - db[i], pb = (i > 0) ? 1 - db[i - 1] : 0;
        dec_bits[i] = (unsigned char)(nb != pb);
    }
    for (int k = tid; k < 148 - 64 + 1; k += blockDim.x) {
        int acc = 0;
        for (int i = 0; i < 64; ++i) acc += dpm[i] * (2 * (int)db[k + i] - 1);
        corr_val[k] = (double)acc;
    }
}

__global__ void __launch_bounds__(SD_THREADS) sch_demod_kernel(const double2 *__restrict__ s, const double *__restrict__ pos, int osr,
                                                              const double2 *__restrict__ tw, const double2 *__restrict__ Ft,
                                                              const double2 *__restrict__ Wtab /* 16 x osr */, const signed char *__restrict__ data_pm /* 64 */,
                                                              unsigned char *__restrict__ demod_bits /* 148 per burst */,
                                                              unsigned char *__restrict__ dec_bits, double *__restrict__ corr_val /* 85 per burst */) {
    extern __shared__ double2 sm[];
    __shared__ unsigned char bits[SD_NSYM + 2];
    __shared__ signed char dpm[64];
    const int burst = blockIdx.x, tid = threadIdx.x;
    const int N = SD_NSYM * osr, sp_tr = (SD_EX + 42) * osr, L = 64 * osr;
    double2 *x = sm, *tmp = x + N, *fa = tmp + N, *fb = fa + N;
    const i64 sp = (i64)pos[burst] - SD_EX * osr;              // :79
    if (tid < 64) dpm[tid] = data_pm[tid];
    for (int n = tid; n < N; n += SD_THREADS) {
        const double2 v = s[sp - 1 + n];
        x[n] = v;
        fb[n] = (n >= sp_tr && n < sp_tr + L) ? v : make_double2(0.0, 0.0);      // received_training_ov (:83-84)
    }
    __syncthreads();
    dft_pxm<false>(fb, tmp, fa, N, 97, tw);                    // fd_received_training
    for (int n = tid; n < N; n += SD_THREADS) fa[n] = cdiv(fa[n], Ft[n]);       // fd_chn (:86)
    __syncthreads();
    dft_pxm<false>(x, tmp, fb, N, 97, tw);                     // fd_x (:88)
    for (int n = tid; n < N; n += SD_THREADS) fb[n] = cdiv(fb[n], fa[n]);       // :89
    __syncthreads();
    dft_pxm<true>(fb, tmp, x, N, 97, tw);                      // x = ifft(fd_x) (:90)
    sch_bits_body(x, tmp, osr, Wtab, dpm, bits, demod_bits + (i64)burst * 148, dec_bits + (i64)burst * 148, corr_val + (i64)burst * 85);
}

// ===================================================================================================
// Batched SCH_demod / FCCH_demod (gsm_sync_demod.m:144-145) for every stream of gsmcal_calibrate_demod_batch, on the pipeline's own
// r_correct evaluated where it is read: the level-3 loader (filter -> interp1(e1) -> derotation(dphi1) -> interp1(e2)) and then
// r_correct(j) = r(j) * exp(1i*(j-1)*dphi2) (carrier_correct_post_SCH.m:81-83), phasors as materialise_r_kernel forms them.
// ===================================================================================================
struct DemodResultDev {              // mirrors gsmcal_demod_result (include/gsmcal.h)
    int n_sch, n_sch_ok, n_fcch, flags;
    double fcch_mean_freq, fcch_carrier_ppm;
};
#define DM_NO_POS_INFO  1
#define DM_NO_R_CORRECT 2
#define DM_SCH_RANGE    4
#define DM_FCCH_RANGE   8

// One warp per stream: the `pos_info == -1` rule (all elements, SCH_demod.m:8-11, FCCH_demod.m:7-10), r_correct = -1, the split of
// pos_info into SCH (type 1) and FCCH (type 0) rows in pos_info order, and the window range checks against len3 = length(r_correct):
// SCH x = r(sp:ep), sp = pos - 8*osr, 194*osr samples (SCH_demod.m:79-81); FCCH r(pos : pos + 148*osr - 1) (FCCH_demod.m:28).
__global__ void __launch_bounds__(32) demod_compact_kernel(const StreamCtl *__restrict__ ctl, const double *__restrict__ pos_info /* [stream][6*cap][2] */,
                                                           int cap, int osr, DemodResultDev *__restrict__ rec, double *__restrict__ sch_pos,
                                                           unsigned char *__restrict__ sch_ok, double *__restrict__ fcch_pos,
                                                           unsigned char *__restrict__ fcch_ok) {
    const int stream = blockIdx.x, lane = threadIdx.x;
    const StreamCtl c = ctl[stream];
    const double *pi = pos_info + (i64)stream * 6 * cap * 2;
    const int rows = c.n_pos_info;
    bool other = false;
    for (int i = lane; i < 2 * rows; i += 32) other |= (pi[i] != -1.0);
    const bool all_m1 = rows < 0 || (rows > 0 && !__any_sync(0xffffffffu, other));
    DemodResultDev r;
    r.n_sch = r.n_sch_ok = r.n_fcch = -1; r.flags = 0;
    r.fcch_mean_freq = NAN; r.fcch_carrier_ppm = NAN;           // filled by demod_fcch_mean_kernel
    if (all_m1) r.flags = DM_NO_POS_INFO;
    else if (c.len3 < 0) r.flags = DM_NO_R_CORRECT;
    else {
        const double len = (double)c.len3, ns_win = (double)(SD_NSYM * osr), nf_win = (double)(148 * osr);
        const unsigned below = (1u << lane) - 1u;
        int ns = 0, nok = 0, nf = 0; bool f_bad = false;
        for (int i0 = 0; i0 < rows; i0 += 32) {
            const int i = i0 + lane;
            double p = 0.0, t = -1.0;
            if (i < rows) { p = pi[2 * i]; t = pi[2 * i + 1]; }
            const bool is_s = (t == 1.0), is_f = (t == 0.0);
            const double sp = p - SD_EX * osr;
            const bool s_ok = is_s && p == floor(p) && sp >= 1.0 && sp + ns_win - 1.0 <= len;
            const bool f_ok = is_f && p == floor(p) && p >= 1.0 && p + nf_win - 1.0 <= len;
            const unsigned ms = __ballot_sync(0xffffffffu, is_s), mf = __ballot_sync(0xffffffffu, is_f);
            const int ks = ns + __popc(ms & below), kf = nf + __popc(mf & below);
            if (is_s && ks < cap) { sch_pos[(i64)stream * cap + ks] = p; sch_ok[(i64)stream * cap + ks] = s_ok; }
            if (is_f && kf < cap) { fcch_pos[(i64)stream * cap + kf] = p; fcch_ok[(i64)stream * cap + kf] = f_ok; }
            nok += __popc(__ballot_sync(0xffffffffu, s_ok));
            f_bad |= __any_sync(0xffffffffu, is_f && !f_ok);
            ns += __popc(ms); nf += __popc(mf);
        }
        r.n_sch = ns < cap ? ns : cap; r.n_sch_ok = nok; r.n_fcch = nf < cap ? nf : cap;
        r.flags = (nok < ns ? DM_SCH_RANGE : 0) | (f_bad ? DM_FCCH_RANGE : 0);
    }
    if (lane == 0) rec[stream] = r;
}

// N = 97*M point DFT, N = 194*osr, M = 2*osr (n = M*n1 + n2, k = k1 + 97*k2), the same factorisation as dft_pxm:
//   stage 1: the 97-point DFT of every column n2 through its conjugate-pair form: with a_n = v_n + v_(97-n), b_n = v_n - v_(97-n),
//            X(k) = v_0 + A_k + i*B_k and X(97-k) = v_0 + A_k - i*B_k (inverse: i*B_k negated), A_k = sum_n a_n cos, B_k = sum_n b_n Im(W^nk),
//            n = n_lo..48 - real-by-complex products, a quarter of the direct stage's DFMA.  Inputs with v_n = 0 for n < n_lo and
//            48 < 97 - n < n_lo pass n_lo > 1 (the received training sequence occupies outer indices 25..56 only).
//   twiddle W_N^(n2*k1), then stage 2: 97 row DFTs of M points (radix-2 Stockham in shared memory when M is a power of two).
// in and out may alias; t0, t1: N double2 of scratch each; w97[j] = W_97^j, wm[j] = W_M^j (j < M/2), both in shared memory.
#define D97_R 3                        // k values per thread: 16 groups of 3 cover the 48 conjugate pairs
template <bool INV>
__device__ void dft97(const double2 *in, double2 *t0, double2 *t1, double2 *out, int M, int n_lo, const double2 *__restrict__ tw,
                      const double2 *w97, const double2 *wm) {
    const int N = 97 * M, tid = threadIdx.x, nt = blockDim.x;
    for (int task = tid; task < 16 * M; task += nt) {
        const int n2 = task % M, g = task / M, k0 = 1 + D97_R * g;
        double ar[D97_R], ai[D97_R], br[D97_R], bi[D97_R];
        int t[D97_R];
#pragma unroll
        for (int r = 0; r < D97_R; ++r) { ar[r] = ai[r] = br[r] = bi[r] = 0.0; t[r] = (n_lo * (k0 + r)) % 97; }
        double sr = 0.0, si = 0.0;
        for (int n = n_lo; n <= 48; ++n) {
            const double2 p = in[M * n + n2], q = in[M * (97 - n) + n2];
            const double axr = p.x + q.x, axi = p.y + q.y, bxr = p.x - q.x, bxi = p.y - q.y;
            if (g == 0) { sr += axr; si += axi; }
#pragma unroll
            for (int r = 0; r < D97_R; ++r) {
                const double2 w = w97[t[r]];
                ar[r] = fma(axr, w.x, ar[r]); ai[r] = fma(axi, w.x, ai[r]);
                br[r] = fma(bxr, w.y, br[r]); bi[r] = fma(bxi, w.y, bi[r]);
                t[r] += k0 + r; if (t[r] >= 97) t[r] -= 97;
            }
        }
        const double2 v0 = in[n2];
#pragma unroll
        for (int r = 0; r < D97_R; ++r) {
            const int k = k0 + r;
            const double2 xp = make_double2(v0.x + ar[r] - bi[r], v0.y + ai[r] + br[r]), xm = make_double2(v0.x + ar[r] + bi[r], v0.y + ai[r] - br[r]);
            double2 wk = tw[n2 * k], wn = tw[n2 * (97 - k)];
            if (INV) { wk.y = -wk.y; wn.y = -wn.y; }
            t0[k * M + n2] = cmul(INV ? xm : xp, wk);
            t0[(97 - k) * M + n2] = cmul(INV ? xp : xm, wn);
        }
        if (g == 0) t0[n2] = make_double2(v0.x + sr, v0.y + si);
    }
    __syncthreads();
    if ((M & (M - 1)) == 0) {
        const int lm = 31 - __clz(M), half = M / 2;
        const double2 *src = t0; double2 *dst = t1;
        int tsh = lm - 1;
        for (int Ns = 1; Ns < M; Ns <<= 1, --tsh) {
            for (int i = tid; i < 97 * half; i += nt) {
                const int row = i >> (lm - 1), j = i & (half - 1), k = j & (Ns - 1);
                double2 w = wm[k << tsh]; if (INV) w.y = -w.y;
                const double2 x0 = src[row * M + j], x1 = cmul(src[row * M + j + half], w);
                const int o = row * M + ((j - k) << 1) + k;
                dst[o] = make_double2(x0.x + x1.x, x0.y + x1.y);
                dst[o + Ns] = make_double2(x0.x - x1.x, x0.y - x1.y);
            }
            __syncthreads();
            const double2 *sw = src; src = dst; dst = const_cast<double2 *>(sw);
        }
        for (int i = tid; i < N; i += nt) {
            const int k1 = i / M, k2 = i - k1 * M;
            const double2 v = src[i];
            out[k1 + 97 * k2] = INV ? make_double2(v.x / (double)N, v.y / (double)N) : v;
        }
    } else {
        for (int i = tid; i < N; i += nt) {
            const int k1 = i % 97, k2 = i / 97;
            double xr = 0.0, xi = 0.0;
            int tt = 0; const int stp = 97 * k2;
            for (int n2 = 0; n2 < M; ++n2) {
                const double2 x = t0[k1 * M + n2];
                double2 w = tw[tt]; if (INV) w.y = -w.y;
                xr = fma(x.x, w.x, fma(-x.y, w.y, xr));
                xi = fma(x.x, w.y, fma(x.y, w.x, xi));
                tt += stp; if (tt >= N) tt -= N;
            }
            out[i] = INV ? make_double2(xr / (double)N, xi / (double)N) : make_double2(xr, xi);
        }
    }
    __syncthreads();
}

// r_correct(j0+1 : j0+count) = dst .* exp(1i*(j0:j0+count-1)*dphi2) in place; ph0 = exp(1i*j0*dphi2) (exact sincos, one thread)
__device__ __forceinline__ void derotate_post(double2 *dst, int count, double dphi2, double2 ph0) {
    const int tid = threadIdx.x, nt = blockDim.x;
    double sn, cs;
    sincos((double)tid * dphi2, &sn, &cs);
    double2 ph = cmul(ph0, make_double2(cs, sn));
    sincos((double)nt * dphi2, &sn, &cs);
    const double2 st = make_double2(cs, sn);
    for (int i = tid; i < count; i += nt) { dst[i] = cmul(dst[i], ph); ph = cmul(ph, st); }
}

// SCH_demod.m:65-110 for one (SCH row, stream).  320 threads: the 1552-sample level-0 window of the loader is filtered by its unrolled
// 5-outputs-per-thread path.  Shared: x[N] | b1[N] | b2[N] | b3[N] (the loader's scratch and the branch correlations alias b1..b3).
// RESID (sch_demod_resid_kernel): the derotation step is dphi2 - resid, which also rotates the window by exp(-i*resid*n) from its start.
#define SDB_THREADS 320
template <bool RESID>
__device__ __forceinline__ void sch_demod_body(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                               const double *__restrict__ sch_pos, const unsigned char *__restrict__ sch_ok, int cap, int osr,
                                               const double2 *__restrict__ tw, const double2 *__restrict__ Ft,
                                               const double2 *__restrict__ Wtab, const signed char *__restrict__ data_pm,
                                               unsigned char *__restrict__ demod_bits, unsigned char *__restrict__ dec_bits,
                                               double *__restrict__ corr_val, double resid) {
    extern __shared__ double2 sm[];
    __shared__ unsigned char bits[SD_NSYM + 2];
    __shared__ signed char dpm[64];
    __shared__ double2 w97[97], wm[8];
    __shared__ double2 ph0;
    const int row = blockIdx.x, stream = blockIdx.y, tid = threadIdx.x;
    if (row >= rec[stream].n_sch) return;
    const i64 o = (i64)stream * cap + row;
    if (!sch_ok[o]) {                                           // the reference would stop at SCH_demod.m:81: zeros, sch_ok = 0
        for (int i = tid; i < 148; i += SDB_THREADS) { demod_bits[o * 148 + i] = 0; dec_bits[o * 148 + i] = 0; }
        for (int k = tid; k < 85; k += SDB_THREADS) corr_val[o * 85 + k] = 0.0;
        return;
    }
    const StreamCtl c = ctl[stream];
    const int N = SD_NSYM * osr, M = 2 * osr, sp_tr = (SD_EX + 42) * osr, L = 64 * osr;
    double2 *x = sm, *b1 = x + N, *b2 = b1 + N, *b3 = b2 + N;
    const i64 j0 = (i64)sch_pos[o] - SD_EX * osr - 1;           // 0-based first sample of x = s(sp:ep) (:79-81)
    if (tid < 64) dpm[tid] = data_pm[tid];
    for (int j = tid; j < 97; j += SDB_THREADS) w97[j] = tw[M * j];
    if (tid < M / 2) wm[tid] = tw[97 * tid];
    if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); ph0 = make_double2(cs, sn); }
    load_window(src, c, stream, j0, N, x, b1, b1 + GSMCAL_XCAP(N));          // ends with a barrier
    derotate_post(x, N, RESID ? c.dphi2 - resid : c.dphi2, ph0);
    __syncthreads();
    for (int n = tid; n < N; n += SDB_THREADS) b1[n] = (n >= sp_tr && n < sp_tr + L) ? x[n] : make_double2(0.0, 0.0);     // :83-84
    __syncthreads();
    dft97<false>(b1, b2, b3, b1, M, (SD_EX + 42) / 2, tw, w97, wm);          // fd_received_training (outer indices 25..56)
    for (int n = tid; n < N; n += SDB_THREADS) b1[n] = cdiv(b1[n], Ft[n]);  // fd_chn (:86)
    __syncthreads();
    dft97<false>(x, b2, b3, x, M, 1, tw, w97, wm);                           // fd_x (:88)
    for (int n = tid; n < N; n += SDB_THREADS) x[n] = cdiv(x[n], b1[n]);    // :89
    __syncthreads();
    dft97<true>(x, b2, b3, x, M, 1, tw, w97, wm);                            // x = ifft(fd_x) (:90)
    sch_bits_body(x, b1, osr, Wtab, dpm, bits, demod_bits + o * 148, dec_bits + o * 148, corr_val + o * 85);
}
__global__ void __launch_bounds__(SDB_THREADS, 2) sch_demod_batch_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                        const double *__restrict__ sch_pos, const unsigned char *__restrict__ sch_ok, int cap, int osr,
                                                                        const double2 *__restrict__ tw, const double2 *__restrict__ Ft,
                                                                        const double2 *__restrict__ Wtab, const signed char *__restrict__ data_pm,
                                                                        unsigned char *__restrict__ demod_bits, unsigned char *__restrict__ dec_bits,
                                                                        double *__restrict__ corr_val) {
    sch_demod_body<false>(src, ctl, rec, sch_pos, sch_ok, cap, osr, tw, Ft, Wtab, data_pm, demod_bits, dec_bits, corr_val, 0.0);
}

// FCCH_demod.m:21-66 for one (FCCH row, stream): the window comes through the fine search's filtered-window cache where it covers it
// (the windows the post-SCH tone stage reads), then derotation by dphi2 and fcch_demod_body.  A window outside r_correct: NaN.
__global__ void __maxnreg__(80) fcch_demod_batch_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                     const double *__restrict__ fcch_pos, const unsigned char *__restrict__ fcch_ok, int cap, int osr,
                                                                     const double2 *__restrict__ tw, double *__restrict__ freq_out,
                                                                     double *__restrict__ snr_out, double *__restrict__ idx_out) {
    extern __shared__ double2 sm[];
    __shared__ double2 ph0;
    const int row = blockIdx.x, stream = blockIdx.y, tid = threadIdx.x;
    if (row >= rec[stream].n_fcch) return;
    const i64 o = (i64)stream * cap + row;
    if (!fcch_ok[o]) {
        if (tid == 0) { freq_out[o] = NAN; snr_out[o] = NAN; idx_out[o] = NAN; }
        return;
    }
    const StreamCtl c = ctl[stream];
    const int N = 148 * osr;
    double2 *u = sm, *A = u + N, *F = A + N;
    double *P = (double *)(F + N);
    const i64 j0 = (i64)fcch_pos[o] - 1;
    if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); ph0 = make_double2(cs, sn); }
    load_window(src, c, stream, j0, N, u, A, A + GSMCAL_XCAP(N), row);       // ends with a barrier
    derotate_post(u, N, c.dphi2, ph0);
    __syncthreads();
    fcch_demod_body(u, A, F, P, osr, tw, freq_out, snr_out, idx_out, o);
}

// mean(freq) (FCCH_demod.m:43, ascending row order) and carrier_ppm (:46-47) when every FCCH window lies inside r_correct
__global__ void demod_fcch_mean_kernel(DemodResultDev *rec, int n_streams, const double *__restrict__ freq, int cap, double carrier_freq) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_streams) return;
    DemodResultDev r = rec[d];
    if (r.n_fcch <= 0 || (r.flags & DM_FCCH_RANGE)) return;
    double acc = 0.0;
    for (int i = 0; i < r.n_fcch; ++i) acc += freq[(i64)d * cap + i];
    r.fcch_mean_freq = acc / (double)r.n_fcch;
    r.fcch_carrier_ppm = 1e6 * (r.fcch_mean_freq - ((1625.0 / 6.0) * 1e3) / 4.0) / carrier_freq;
    rec[d] = r;
}

// ===================================================================================================
// Batched BCCH_demod (gsm_sync_demod.m:146) for every stream of gsmcal_calibrate_demod_bcch_batch.  Its carrier_correct_post_SCH on
// r_correct (BCCH_demod.m:47-70) runs tone_freq_estimate over the FCCH rows and takes their mean: the statements and windows of
// FCCH_demod.m:36-47, so the carrier ppm is rec.fcch_carrier_ppm and the compensation phase comes from rec.fcch_mean_freq.  Left to do:
// the first four BCCH rows, their training windows r_bcch(p+61*osr : p+61*osr+26*osr-1) with r_bcch(j) = r_correct(j)*exp(1i*(j-1)*comp)
// (:72-73, :85-89), the 8 x 4 correlations with the normal training sequences (:91) and the agreement decision (:93-102).
// ===================================================================================================
struct BcchResultDev {               // mirrors gsmcal_bcch_result (include/gsmcal.h)
    double carrier_ppm;
    int nts_idx, flags;
    double corr_abs[32];             // 8 x 4 column-major
};
#define BC_NO_POS_INFO  1
#define BC_FEW_BCCH     2
#define BC_FCCH_RANGE   4
#define BC_TRAIN_RANGE  8

// One block per stream, one warp per normal training sequence (as nts_corr_kernel).  Shared: window w[26*osr] | the loader's scratch
// X[GSMCAL_XCAP(26*osr)] | Y[26*osr + 8].  Sentinels, in the reference's order: pos_info == -1 (BCCH_demod.m:9-11), fewer than four
// BCCH rows (:13-17), no FCCH mean (no FCCH row, or an FCCH window outside r_correct), then per burst a training window outside
// r_correct (NaN column, nts_idx = -1).
#define BC_THREADS 256
__global__ void __launch_bounds__(BC_THREADS) bcch_demod_batch_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                     const double *__restrict__ pos_info /* [stream][6*cap][2] */, int cap, int osr,
                                                                     const double2 *__restrict__ nts /* (26*osr) x 8 column-major */,
                                                                     BcchResultDev *__restrict__ out) {
    extern __shared__ double2 sm[];
    __shared__ double bpos[4];
    __shared__ int n_bcch;
    __shared__ double mag[32];
    __shared__ double2 ph_a, ph_b;
    const int stream = blockIdx.x, tid = threadIdx.x, q = tid >> 5, lane = tid & 31;
    const int L = 26 * osr;
    const DemodResultDev r = rec[stream];
    BcchResultDev *o = out + stream;
    int flags = 0;
    if (r.flags & DM_NO_POS_INFO) flags = BC_NO_POS_INFO;
    else {
        if (q == 0) {                                           // the first four type-2 rows of pos_info, in pos_info order
            const double *pi = pos_info + (i64)stream * 6 * cap * 2;
            const int rows = ctl[stream].n_pos_info;
            const unsigned below = (1u << lane) - 1u;
            int nb = 0;
            for (int i0 = 0; i0 < rows && nb < 4; i0 += 32) {
                const int i = i0 + lane;
                const bool is_b = i < rows && pi[2 * i + 1] == 2.0;
                const unsigned mb = __ballot_sync(0xffffffffu, is_b);
                const int k = nb + __popc(mb & below);
                if (is_b && k < 4) bpos[k] = pi[2 * i];
                nb += __popc(mb);
            }
            if (lane == 0) n_bcch = nb;
        }
        __syncthreads();
        if (n_bcch < 4) flags = BC_FEW_BCCH;
        else if (isnan(r.fcch_mean_freq)) flags = BC_FCCH_RANGE;
    }
    if (flags) {
        if (tid < 32) o->corr_abs[tid] = NAN;
        if (tid == 0) { o->carrier_ppm = (flags == BC_FCCH_RANGE) ? NAN : -1.0; o->nts_idx = -1; o->flags = flags; }
        return;
    }
    const StreamCtl c = ctl[stream];
    const double symbol_rate = (1625.0 / 6.0) * 1e3, target = symbol_rate / 4.0;
    const double comp = (target - r.fcch_mean_freq) * 2 * GSMCAL_PI / (symbol_rate * osr);      // carrier_correct_post_SCH's comp_phase_rotate
    double2 *w = sm, *X = w + L, *Y = X + GSMCAL_XCAP(L);
    for (int b = 0; b < 4; ++b) {
        const double p = bpos[b];
        if (!(p == floor(p) && p + 61 * osr >= 1.0 && p + 61 * osr + L - 1 <= (double)c.len3)) {       // the reference would raise (:85-89)
            flags = BC_TRAIN_RANGE;
            if (lane == 0) mag[b * 8 + q] = NAN;
            continue;
        }
        const i64 j0 = (i64)p + 61 * osr - 1;                  // 0-based first training sample
        if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); ph_a = make_double2(cs, sn); }
        if (tid == 32) { double sn, cs; sincos((double)j0 * comp, &sn, &cs); ph_b = make_double2(cs, sn); }
        load_window(src, c, stream, j0, L, w, X, Y);           // ends with a barrier
        derotate_post(w, L, c.dphi2, ph_a);                    // r_correct (carrier_correct_post_SCH.m:83)
        derotate_post(w, L, comp, ph_b);                       // r_bcch (BCCH_demod.m:72-73); each thread rotates its own samples twice
        __syncthreads();
        double ar = 0.0, ai = 0.0;
        for (int n = lane; n < L; n += 32) {
            const double2 t = nts[(i64)q * L + n], v = w[n];
            ar += t.x * v.x + t.y * v.y;                         // conj(t) * v
            ai += t.x * v.y - t.y * v.x;
        }
        ar = warp_sum(ar); ai = warp_sum(ai);
        if (lane == 0) mag[b * 8 + q] = hypot(ar, ai);
        __syncthreads();                                       // w is reloaded for the next burst
    }
    __syncthreads();
    if (tid < 32) o->corr_abs[tid] = mag[tid];
    if (tid == 0) {
        int idx[4];
        for (int b = 0; b < 4; ++b) { idx[b] = 0; for (int k = 1; k < 8; ++k) if (mag[b * 8 + k] > mag[b * 8 + idx[b]]) idx[b] = k; }   // first maximum (:93)
        o->carrier_ppm = r.fcch_carrier_ppm;
        o->nts_idx = (!flags && idx[0] == idx[1] && idx[1] == idx[2] && idx[2] == idx[3]) ? idx[0] + 1 : -1;                   // :94-102
        o->flags = flags;
    }
}

// ===================================================================================================
// Sub-sample SCH timing and the per-stream clock fit of gsmcal_calibrate_sch_timing_batch (definition: include/gsmcal.h).  The SCH row
// list is demod_compact_kernel's; its sch_ok is SCH_demod's 194*osr-sample window check, so the 600-sample correlation window is checked
// here.  osr 8 only: the correlation is sch_corr_kernel's register-tiled fp64 one (sch_corr_tiled_fp64, 256 threads, 89 lags of 512).
// ===================================================================================================
struct TimingResultDev {             // mirrors gsmcal_sch_timing_result (include/gsmcal.h)
    int n_sch, n_fit, flags, reserved;
    double t0, fit_ppm, rms;
};
#define TM_NO_POS_INFO  1
#define TM_NO_R_CORRECT 2
#define TM_RANGE        4
#define TM_EDGE         8
#define TM_FEW         16
#define TM_L     512                   // 64 * osr template samples
#define TM_LAG0  64                    // lags -8*osr .. +3*osr (SCH_corr_rate_correction.m:36,45-48)
#define TM_NLAG  89
#define TM_NSMP  (TM_NLAG + TM_L - 1)  // 600
// shared: window [TM_NSMP] | scratch: the loader's X, Y, later the padded window and template and the row sums of sch_corr_tiled_fp64
#define TM_PADW  (TM_NSMP + (TM_NSMP >> 4) + 2)
#define TM_PADT  (TM_L + (TM_L >> 4) + 2)
#define TM_PART  ((2 * (SCH_THREADS >> 5) * SCH_LPG * 9 + 1) / 2 + 1)
#define TM_SCRATCH ((GSMCAL_XCAP(TM_NSMP) + TM_NSMP + 8) > (TM_PADW + TM_PADT + TM_PART) ? (GSMCAL_XCAP(TM_NSMP) + TM_NSMP + 8) : (TM_PADW + TM_PADT + TM_PART))
#define TM_SMEM  ((size_t)(TM_NSMP + TM_SCRATCH) * sizeof(double2))

// One block per (SCH row, stream): c(l) = |sum conj(t) r_correct(g+l : g+l+511)|^2 for the 89 lags, g = p + 42*8, the first maximum
// and the three-point parabola through it.  tau = NaN and row_flag = TM_RANGE / TM_EDGE where the row is excluded.
__global__ void __launch_bounds__(SCH_THREADS) sch_timing_batch_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                      const double *__restrict__ sch_pos, int cap, const double2 *__restrict__ tpl,
                                                                      double *__restrict__ tau, unsigned char *__restrict__ row_flag) {
    extern __shared__ double2 sm[];
    __shared__ double corr[96], corr_i[96];
    __shared__ double2 ph0;
    const int row = blockIdx.x, stream = blockIdx.y, tid = threadIdx.x;
    if (row >= rec[stream].n_sch) return;                      // also n_sch = -1: the step does not run for this stream
    const i64 o = (i64)stream * cap + row;
    const StreamCtl c = ctl[stream];
    const double p = sch_pos[o], g = p + 42.0 * 8.0;
    if (!(p == floor(p) && g - TM_LAG0 >= 1.0 && g + (TM_NLAG - 1 - TM_LAG0) + (TM_L - 1) <= (double)c.len3)) {
        if (tid == 0) { tau[o] = NAN; row_flag[o] = TM_RANGE; }
        return;
    }
    const i64 j0 = (i64)g - TM_LAG0 - 1;                       // 0-based first sample of the window r(g-64 : g+24+511)
    double2 *win = sm, *X = win + TM_NSMP, *Y = X + GSMCAL_XCAP(TM_NSMP);
    if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); ph0 = make_double2(cs, sn); }
    load_window(src, c, stream, j0, TM_NSMP, win, X, Y);        // level 3; ends with a barrier
    derotate_post(win, TM_NSMP, c.dphi2, ph0);                 // r_correct (carrier_correct_post_SCH.m:83)
    __syncthreads();
    double2 *wp = X, *tp = wp + TM_PADW;
    double *part = reinterpret_cast<double *>(tp + TM_PADT);
    for (int i = tid; i < TM_NSMP; i += SCH_THREADS) wp[i + (i >> 4)] = win[i];
    for (int i = tid; i < TM_L; i += SCH_THREADS) tp[i + (i >> 4)] = __ldg(tpl + i);
    __syncthreads();
    sch_corr_tiled_fp64(wp, tp, part, corr, corr_i, TM_NLAG, TM_NSMP);
    __syncthreads();
    if (tid < TM_NLAG) corr[tid] = abs2_ref(make_double2(corr[tid], corr_i[tid]));
    __syncthreads();
    if (tid == 0) {
        int k = 0;
        for (int l = 1; l < TM_NLAG; ++l) if (corr[l] > corr[k]) k = l;      // first maximum, scanning the lags upwards
        if (k == 0 || k == TM_NLAG - 1) { tau[o] = NAN; row_flag[o] = TM_EDGE; return; }
        const double ym = corr[k - 1], y0 = corr[k], yp = corr[k + 1];
        const double den = __dadd_rn(__dsub_rn(ym, 2.0 * y0), yp);
        const double delta = (den == 0.0) ? 0.0 : __ddiv_rn(0.5 * __dsub_rn(ym, yp), den);
        tau[o] = __dadd_rn(g + (double)(k - TM_LAG0), delta);
        row_flag[o] = 0;
    }
}

// One warp per stream: the lanes map tau to raw-capture time, x = ((tau - 1)*(1 + e2))*(1 + e1), and lane 0 fits the line in row
// order (the sums exactly as include/gsmcal.h states them, every product and sum rounded on its own).
__global__ void __launch_bounds__(32) sch_timing_fit_kernel(const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                            const double *__restrict__ sch_pos, const unsigned char *__restrict__ row_flag,
                                                            const double *__restrict__ tau, int cap, double *__restrict__ x_out,
                                                            TimingResultDev *__restrict__ out) {
    const int stream = blockIdx.x, lane = threadIdx.x;
    const DemodResultDev r = rec[stream];
    TimingResultDev t;
    t.n_sch = -1; t.n_fit = 0; t.flags = 0; t.reserved = 0; t.t0 = NAN; t.fit_ppm = NAN; t.rms = NAN;
    if (r.flags & (DM_NO_POS_INFO | DM_NO_R_CORRECT)) {
        t.flags = (r.flags & DM_NO_POS_INFO) ? TM_NO_POS_INFO : TM_NO_R_CORRECT;
        if (lane == 0) out[stream] = t;
        return;
    }
    const StreamCtl c = ctl[stream];
    const double s1 = __dadd_rn(1.0, __dmul_rn(c.sppm1, 1e-6)), s2 = __dadd_rn(1.0, __dmul_rn(c.sppm2, 1e-6));   // sampling_ppm[0], [1] of the record
    const i64 base = (i64)stream * cap;
    const int n = r.n_sch;
    unsigned fl = 0, nf = 0;
    for (int i = lane; i < n; i += 32) {
        const double x = __dmul_rn(__dmul_rn(tau[base + i] - 1.0, s2), s1);
        x_out[base + i] = x;
        fl |= row_flag[base + i];
        nf += isfinite(x) ? 1u : 0u;
    }
    fl = __reduce_or_sync(0xffffffffu, fl);
    nf = __reduce_add_sync(0xffffffffu, nf);
    __syncwarp();                                              // x_out of every lane is visible to lane 0
    if (lane != 0) return;
    t.n_sch = n; t.n_fit = (int)nf; t.flags = (int)fl;
    if (nf < 3) {
        t.flags |= TM_FEW;
        out[stream] = t;
        return;
    }
    double p_first = 0.0, sm = 0.0, sx = 0.0;
    bool first = true;
    for (int i = 0; i < n; ++i) {
        const double x = x_out[base + i];
        if (!isfinite(x)) continue;
        if (first) { p_first = sch_pos[base + i]; first = false; }
        sm = __dadd_rn(sm, sch_pos[base + i] - p_first);
        sx = __dadd_rn(sx, x);
    }
    const double m_bar = sm / (double)nf, x_bar = sx / (double)nf;
    double sxy = 0.0, smm = 0.0;
    for (int i = 0; i < n; ++i) {
        const double x = x_out[base + i];
        if (!isfinite(x)) continue;
        const double dm = __dsub_rn(sch_pos[base + i] - p_first, m_bar), dx = __dsub_rn(x, x_bar);
        sxy = __dadd_rn(sxy, __dmul_rn(dm, dx));
        smm = __dadd_rn(smm, __dmul_rn(dm, dm));
    }
    const double b = sxy / smm, a = __dsub_rn(x_bar, __dmul_rn(b, m_bar));
    double ss = 0.0;
    for (int i = 0; i < n; ++i) {
        const double x = x_out[base + i];
        if (!isfinite(x)) continue;
        const double e = __dsub_rn(__dsub_rn(x, a), __dmul_rn(b, sch_pos[base + i] - p_first));
        ss = __dadd_rn(ss, __dmul_rn(e, e));
    }
    t.t0 = a;
    t.fit_ppm = __dmul_rn(b - 1.0, 1e6);
    t.rms = sqrt(ss / (double)nf);
    out[stream] = t;
}

// ===================================================================================================
// SCH channel decoding of gsmcal_calibrate_sch_decode_batch (definition: include/gsmcal.h) on what sch_demod_batch_kernel wrote: BSIC
// and FN of every SCH row, the per-stream vote and the capture start on the cell's frame clock.
// ===================================================================================================
struct SchDecodeResultDev {          // mirrors gsmcal_sch_decode_result (include/gsmcal.h)
    int n_sch, n_crc_ok, n_agree, flags, bsic, fn_first;
    double frame_clock_start;
};
#define SC_NO_POS_INFO  1
#define SC_NO_R_CORRECT 2
#define SC_NONE         4
#define SC_DISAGREE     8
#define SC_ROW_WINDOW   1
#define SC_ROW_ALIGN    2
#define SC_ROW_CRC      4
#define SC_ROW_FIELD    8
#define SC_FN_MOD 2715648

// one row: the 78 coded bits around the training sequence at k (m: the 148 demodulated symbols), the 16-state Viterbi, CRC and fields.
// Returns the row flag; fn, bsic, ham are written where the steps got that far.
__device__ __forceinline__ int sch_decode_row(const unsigned char *__restrict__ m, int k, int &fn, int &bsic, int &ham) {
    const unsigned long long T = 0xB962040F2D45761Bull;            // SCH training bits 0..63, bit j at position 63 - j (T_0 = MSB)
    unsigned long long e = 0ull;                                   // e(0..63) at bits 63..0
    unsigned e_hi = 0u;                                            // e(64..77) at bits 13..0
    int b = (int)(T >> 63) & 1;                                    // backwards from b(k) = T_0
    for (int i = k - 1; i >= k - 39; --i) {
        b ^= 1 - m[i + 1];
        e |= (unsigned long long)b << (63 - (i - (k - 39)));
    }
    b = (int)T & 1;                                                // forwards from b(k+63) = T_63
    for (int i = k + 64; i <= k + 102; ++i) {
        b ^= 1 - m[i];
        const int j = 39 + i - (k + 64);
        if (j < 64) e |= (unsigned long long)b << (63 - j);
        else e_hi |= (unsigned)b << (77 - j);
    }
    // state s = u(k) | u(k-1) << 1 | u(k-2) << 2 | u(k-3) << 3; survivors: the 39 decided inputs, newest at bit 0
    int metric[16];
    unsigned long long path[16];
#pragma unroll
    for (int s = 0; s < 16; ++s) { metric[s] = (s == 0) ? 0 : 1 << 20; path[s] = 0ull; }
    for (int t = 0; t < 39; ++t) {
        const int c0 = (t < 32) ? (int)(e >> (63 - 2 * t)) & 1 : (int)(e_hi >> (77 - 2 * t)) & 1;      // e(2t), e(2t+1)
        const int c1 = (t < 32) ? (int)(e >> (62 - 2 * t)) & 1 : (int)(e_hi >> (76 - 2 * t)) & 1;
        int nm[16];
        unsigned long long np[16];
#pragma unroll
        for (int s = 0; s < 16; ++s) {
            const int u = s & 1;
            const int p0 = s >> 1, p1 = (s >> 1) | 8;                // predecessors: dropped bit u(k-4) = 0 / 1
            const int a0 = u ^ ((p0 >> 2) & 1) ^ ((p0 >> 3) & 1), a1 = u ^ (p0 & 1) ^ ((p0 >> 2) & 1) ^ ((p0 >> 3) & 1);
            const int m0 = metric[p0] + (a0 ^ c0) + (a1 ^ c1);
            const int m1 = metric[p1] + (a0 ^ 1 ^ c0) + (a1 ^ 1 ^ c1);      // the dropped bit enters both outputs
            const bool take1 = m1 < m0;                              // a tie keeps dropped bit 0
            nm[s] = take1 ? m1 : m0;
            np[s] = ((take1 ? path[p1] : path[p0]) << 1) | (unsigned long long)u;
        }
#pragma unroll
        for (int s = 0; s < 16; ++s) { metric[s] = nm[s]; path[s] = np[s]; }
    }
    ham = metric[0];
    // u(0) at bit 38 ... u(34) at bit 4: the 35-bit word d(0)D^34 + ... + p(9) is path >> 4
    unsigned long long v = path[0] >> 4;
    for (int i = 34; i >= 10; --i)
        if ((v >> i) & 1ull) v ^= 0x575ull << (i - 10);
    if ((v & 0x3FFull) != 0x3FFull) return SC_ROW_CRC;
    const unsigned long long w = path[0] >> 14;                    // d(i) at bit 24 - i
    auto d = [&](int i) { return (int)(w >> (24 - i)) & 1; };
    int bs = 0, t1 = (d(0) << 9) | (d(1) << 10) | d(23), t2 = 0;
    for (int i = 0; i < 6; ++i) bs |= d(2 + i) << i;
    for (int i = 0; i < 8; ++i) t1 |= d(8 + i) << (1 + i);
    for (int i = 0; i < 5; ++i) t2 |= d(18 + i) << i;
    const int t3p = (d(16) << 1) | (d(17) << 2) | d(24);
    if (t2 > 25 || t3p > 4) return SC_ROW_FIELD;
    const int t3 = 10 * t3p + 1;
    fn = 51 * ((t3 - t2 + 26) % 26) + t3 + 1326 * t1;
    bsic = bs;
    return 0;
}

// One warp per stream: each lane decodes whole SCH rows (row = lane, lane + 32, ...), then the warp takes the vote over the rows' keys
// (fn_first * 64 + bsic, -1 for rows that do not vote) and lane 0 writes the record.
__global__ void __launch_bounds__(32) sch_decode_batch_kernel(const DemodResultDev *__restrict__ rec, const double *__restrict__ sch_pos,
                                                              const unsigned char *__restrict__ sch_ok, const unsigned char *__restrict__ bits,
                                                              const double *__restrict__ corr, int cap, int osr, int *__restrict__ key,
                                                              int *__restrict__ fn_out, int *__restrict__ bsic_out,
                                                              unsigned char *__restrict__ ham_out, unsigned char *__restrict__ flag_out,
                                                              SchDecodeResultDev *__restrict__ out) {
    const int stream = blockIdx.x, lane = threadIdx.x;
    const DemodResultDev r = rec[stream];
    const i64 base = (i64)stream * cap;
    const int n = r.n_sch;                                         // -1 when SCH_demod did not run
    const i64 frame = 1250 * (i64)osr;
    const double p_first = (n > 0) ? sch_pos[base] : 0.0;
    int n_ok = 0;
    for (int i = lane; i < cap; i += 32) {
        int fn = -1, bsic = -1, ham = 0, fl = 0, k_vote = -1;
        if (i < n) {
            if (!sch_ok[base + i]) fl = SC_ROW_WINDOW;
            else {
                const double *c = corr + (base + i) * 85;
                int k = 0;
                for (int l = 1; l < 85; ++l) if (c[l] > c[k]) k = l;   // first maximum
                if (k < 39 || k > 45) fl = SC_ROW_ALIGN;
                else fl = sch_decode_row(bits + (base + i) * 148, k, fn, bsic, ham);
                if (fl) { fn = -1; bsic = -1; }
                else {
                    const i64 f = (i64)(sch_pos[base + i] - p_first) / frame;
                    i64 ff = ((i64)fn - f) % SC_FN_MOD; if (ff < 0) ff += SC_FN_MOD;
                    k_vote = (int)ff * 64 + bsic;
                    ++n_ok;
                }
            }
        }
        fn_out[base + i] = fn; bsic_out[base + i] = bsic; ham_out[base + i] = (unsigned char)ham; flag_out[base + i] = (unsigned char)fl;
        key[base + i] = k_vote;
    }
    n_ok = __reduce_add_sync(0xffffffffu, n_ok);
    __syncwarp();                                                  // every lane's keys are visible to the warp
    SchDecodeResultDev o;
    o.n_sch = n; o.n_crc_ok = n_ok; o.n_agree = 0; o.flags = 0; o.bsic = -1; o.fn_first = -1; o.frame_clock_start = NAN;
    if (n < 0) o.flags = (r.flags & DM_NO_POS_INFO) ? SC_NO_POS_INFO : SC_NO_R_CORRECT;
    else if (n_ok == 0) o.flags = SC_NONE;
    else {
        // each lane scores the keys it owns: (votes, first row with that key); the best is the most votes, then the earliest first row
        int best_cnt = 0, best_first = 0x7fffffff, best_key = -1;
        for (int i = lane; i < n; i += 32) {
            const int ki = key[base + i];
            if (ki < 0) continue;
            int cnt = 0, first = i;
            for (int j = 0; j < n; ++j) {
                if (key[base + j] != ki) continue;
                ++cnt;
                if (j < first) first = j;
            }
            if (cnt > best_cnt || (cnt == best_cnt && first < best_first)) { best_cnt = cnt; best_first = first; best_key = ki; }
        }
        for (int o2 = 16; o2 > 0; o2 >>= 1) {
            const int c2 = __shfl_xor_sync(0xffffffffu, best_cnt, o2), f2 = __shfl_xor_sync(0xffffffffu, best_first, o2);
            const int k2 = __shfl_xor_sync(0xffffffffu, best_key, o2);
            if (c2 > best_cnt || (c2 == best_cnt && f2 < best_first)) { best_cnt = c2; best_first = f2; best_key = k2; }
        }
        o.n_agree = best_cnt;
        o.fn_first = best_key >> 6; o.bsic = best_key & 63;
        o.flags = (best_cnt < n_ok) ? SC_DISAGREE : 0;
        const i64 hyper = (i64)SC_FN_MOD * frame;
        i64 t = ((i64)o.fn_first * frame - ((i64)p_first - 1)) % hyper; if (t < 0) t += hyper;
        o.frame_clock_start = (double)t;
    }
    if (lane == 0) out[stream] = o;
}

// ===================================================================================================
// Carrier fit of gsmcal_calibrate_carrier_fit_batch (definition: include/gsmcal.h): the tone of every FCCH row of pos_info from the
// periodogram maximum of the burst interior on r_correct, and the per-stream line through the tones over capture time.  The FCCH row
// list and its fcch_ok (FCCH_demod's 148*osr-sample window inside r_correct, which holds the 116*osr-sample interior) are
// demod_compact_kernel's.  osr 8 only.
// ===================================================================================================
struct CarrierFitDev {               // mirrors gsmcal_carrier_fit_result (include/gsmcal.h)
    int n_fcch, n_fit, flags, reserved;
    double t_mean, freq_hz, drift_hz_per_s, rms_hz, residual_ppm, carrier_fit_ppm, drift_ppm_per_s;
};
#define CF_NO_POS_INFO  1
#define CF_NO_R_CORRECT 2
#define CF_RANGE        4
#define CF_EDGE         8
#define CF_NOCONV      16
#define CF_FEW         32
#define CF_OFF    128                  // 16 symbols into the burst
#define CF_W      928                  // 116 symbols: the interior without the edges and the first differential symbol
#define CF_HALF   463.5                // m = n - (W-1)/2
#define CF_K      14                   // grid delta_k = k*fs/(4W), k = -14..14: 583.7 Hz steps over +-8172 Hz
#define CF_NGRID  (2 * CF_K + 1)
#define CF_NEWTON 5
#define CF_TOL_HZ 1e-4
#define CF_THREADS 256
#define CF_SMEM   ((size_t)(CF_W + GSMCAL_XCAP(CF_W) + CF_W + 8) * sizeof(double2))      // window | the loader's X, Y

// One block per (FCCH row, stream).  The window comes through the fine search's filtered-window cache where it covers it (as in
// fcch_demod_batch_kernel), then the dphi2 derotation and the nominal tone's removal.  Grid: warp w takes grid points w, w+8, ...; lane l
// samples l, l+32, ... with a rotation recurrence seeded by an exact sincospi at its first sample.  Newton: thread t takes samples
// t, t+256, ... seeded the same way; every thread gets the block sums and takes the same step.
__global__ void __launch_bounds__(CF_THREADS) carrier_fit_row_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                    const double *__restrict__ fcch_pos, const unsigned char *__restrict__ fcch_ok, int cap,
                                                                    double *__restrict__ f_out, double *__restrict__ t_out,
                                                                    unsigned char *__restrict__ row_flag) {
    extern __shared__ double2 sm[];
    __shared__ double2 ph0, tw32[32], gstep[CF_NGRID];
    __shared__ double pgrid[CF_NGRID], red[8 * 6];
    const int row = blockIdx.x, stream = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (row >= rec[stream].n_fcch) return;                     // also n_fcch = -1: the step does not run for this stream
    const i64 o = (i64)stream * cap + row;
    if (!fcch_ok[o]) {
        if (tid == 0) { f_out[o] = NAN; t_out[o] = NAN; row_flag[o] = CF_RANGE; }
        return;
    }
    const StreamCtl c = ctl[stream];
    const double p = fcch_pos[o];
    const i64 j0 = (i64)p - 1 + CF_OFF;                        // 0-based first sample of r_correct(p + 128 : p + 128 + 927)
    double2 *y = sm, *X = y + CF_W, *Y = X + GSMCAL_XCAP(CF_W);
    if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); ph0 = make_double2(cs, sn); }
    if (tid >= 32 && tid < 64) { double sn, cs; sincospi(-(double)(tid - 32) / 16.0, &sn, &cs); tw32[tid - 32] = make_double2(cs, sn); }
    if (tid >= 64 && tid < 64 + CF_NGRID) {                    // exp(-i*omega_k*32), omega_k = pi*k/(2W)
        double sn, cs; sincospi(-32.0 * (double)(tid - 64 - CF_K) / (2.0 * CF_W), &sn, &cs); gstep[tid - 64] = make_double2(cs, sn);
    }
    load_window(src, c, stream, j0, CF_W, y, X, Y, row);       // level 3; ends with a barrier
    derotate_post(y, CF_W, c.dphi2, ph0);                      // r_correct (carrier_correct_post_SCH.m:83)
    for (int i = tid; i < CF_W; i += CF_THREADS) y[i] = cmul(y[i], tw32[i & 31]);     // the same samples derotate_post gave this thread
    __syncthreads();
    // coarse grid
    for (int g = warp; g < CF_NGRID; g += CF_THREADS / 32) {
        double sn, cs; sincospi(-(double)(g - CF_K) * ((double)lane - CF_HALF) / (2.0 * CF_W), &sn, &cs);
        double2 z = make_double2(cs, sn);
        const double2 st = gstep[g];
        double ar = 0.0, ai = 0.0;
#pragma unroll 4
        for (int n = lane; n < CF_W; n += 32) {
            const double2 v = y[n];
            ar = fma(v.x, z.x, fma(-v.y, z.y, ar));
            ai = fma(v.x, z.y, fma(v.y, z.x, ai));
            z = cmul(z, st);
        }
        ar = warp_sum(ar); ai = warp_sum(ai);
        if (lane == 0) pgrid[g] = __dadd_rn(__dmul_rn(ar, ar), __dmul_rn(ai, ai));
    }
    __syncthreads();
    int kb = 0;
    for (int g = 1; g < CF_NGRID; ++g) if (pgrid[g] > pgrid[kb]) kb = g;                // first maximum
    if (kb == 0 || kb == CF_NGRID - 1) {
        if (tid == 0) { f_out[o] = NAN; t_out[o] = NAN; row_flag[o] = CF_EDGE; }
        return;
    }
    // Newton on P'(omega) = 0: P' = 2 Im(conj(S0) S1), P'' = 2 (|S1|^2 - Re(conj(S0) S2)), S_j = sum m^j y exp(-i omega m)
    double omega = GSMCAL_PI * (double)(kb - CF_K) / (2.0 * CF_W), step = 0.0;
    for (int it = 0; it < CF_NEWTON; ++it) {
        double sn, cs;
        sincos(-omega * ((double)tid - CF_HALF), &sn, &cs);
        double2 z = make_double2(cs, sn);
        sincos(-omega * (double)CF_THREADS, &sn, &cs);
        const double2 st = make_double2(cs, sn);
        double s[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};          // S0, S1, S2 (re, im)
        for (int n = tid; n < CF_W; n += CF_THREADS) {
            const double m = (double)n - CF_HALF;
            const double2 v = cmul(y[n], z);
            s[0] += v.x; s[1] += v.y;
            s[2] = fma(m, v.x, s[2]); s[3] = fma(m, v.y, s[3]);
            s[4] = fma(m * m, v.x, s[4]); s[5] = fma(m * m, v.y, s[5]);
            z = cmul(z, st);
        }
        block_sum_n<6, true>(s, red);
        const double num = s[0] * s[3] - s[1] * s[2];
        const double den = (s[2] * s[2] + s[3] * s[3]) - (s[0] * s[4] + s[1] * s[5]);
        step = -num / den;
        omega += step;
    }
    if (tid != 0) return;
    const double hz_per_rad = (((1625.0 / 6.0) * 1e3) * 8.0) / (2.0 * GSMCAL_PI);
    if (!(fabs(step) * hz_per_rad <= CF_TOL_HZ)) { f_out[o] = NAN; t_out[o] = NAN; row_flag[o] = CF_NOCONV; return; }
    f_out[o] = __dadd_rn(((1625.0 / 6.0) * 1e3) / 4.0, __dmul_rn(omega, hz_per_rad));
    const double s1 = __dadd_rn(1.0, __dmul_rn(c.sppm1, 1e-6)), s2 = __dadd_rn(1.0, __dmul_rn(c.sppm2, 1e-6));   // sampling_ppm[0], [1] of the record
    const double tau_c = p + (double)CF_OFF + CF_HALF;                                  // exact
    t_out[o] = __ddiv_rn(__dmul_rn(__dmul_rn(tau_c - 1.0, s2), s1), ((1625.0 / 6.0) * 1e3) * 8.0);
    row_flag[o] = 0;
}

// One warp per stream: the lanes gather the row flags and count the fitted rows, lane 0 fits f = a + b (t - t_mean) in row order
// (the sums as include/gsmcal.h states them, every product and sum rounded on its own) and composes the ppm figures.
__global__ void __launch_bounds__(32) carrier_fit_stream_kernel(const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                const unsigned char *__restrict__ row_flag, const double *__restrict__ f,
                                                                const double *__restrict__ t, int cap, double carrier_freq,
                                                                CarrierFitDev *__restrict__ out) {
    const int stream = blockIdx.x, lane = threadIdx.x;
    const DemodResultDev r = rec[stream];
    CarrierFitDev q;
    q.n_fcch = -1; q.n_fit = 0; q.flags = 0; q.reserved = 0;
    q.t_mean = q.freq_hz = q.drift_hz_per_s = q.rms_hz = q.residual_ppm = q.carrier_fit_ppm = q.drift_ppm_per_s = NAN;
    if (r.flags & (DM_NO_POS_INFO | DM_NO_R_CORRECT)) {
        q.flags = (r.flags & DM_NO_POS_INFO) ? CF_NO_POS_INFO : CF_NO_R_CORRECT;
        if (lane == 0) out[stream] = q;
        return;
    }
    const i64 base = (i64)stream * cap;
    const int n = r.n_fcch;
    unsigned fl = 0, nf = 0;
    for (int i = lane; i < n; i += 32) {
        fl |= row_flag[base + i];
        nf += isfinite(f[base + i]) ? 1u : 0u;
    }
    fl = __reduce_or_sync(0xffffffffu, fl);
    nf = __reduce_add_sync(0xffffffffu, nf);
    if (lane != 0) return;
    q.n_fcch = n; q.n_fit = (int)nf; q.flags = (int)fl;
    if (nf < 3) {
        q.flags |= CF_FEW;
        out[stream] = q;
        return;
    }
    double st = 0.0, sf = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!isfinite(f[base + i])) continue;
        st = __dadd_rn(st, t[base + i]);
        sf = __dadd_rn(sf, f[base + i]);
    }
    const double t_bar = st / (double)nf, a = sf / (double)nf;
    double stt = 0.0, stf = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!isfinite(f[base + i])) continue;
        const double dt = __dsub_rn(t[base + i], t_bar);
        stt = __dadd_rn(stt, __dmul_rn(dt, dt));
        stf = __dadd_rn(stf, __dmul_rn(dt, __dsub_rn(f[base + i], a)));
    }
    const double b = stf / stt;
    double ss = 0.0;
    for (int i = 0; i < n; ++i) {
        if (!isfinite(f[base + i])) continue;
        const double e = __dsub_rn(__dsub_rn(f[base + i], a), __dmul_rn(b, __dsub_rn(t[base + i], t_bar)));
        ss = __dadd_rn(ss, __dmul_rn(e, e));
    }
    const StreamCtl c = ctl[stream];
    q.t_mean = t_bar; q.freq_hz = a; q.drift_hz_per_s = b; q.rms_hz = sqrt(ss / (double)nf);
    q.residual_ppm = __dmul_rn(1e6, __dsub_rn(a, ((1625.0 / 6.0) * 1e3) / 4.0)) / carrier_freq;
    q.carrier_fit_ppm = total_ppm2(total_ppm2(c.cppm1, c.cppm2), q.residual_ppm);         // total_carrier_ppm of the record, then the residual
    q.drift_ppm_per_s = __dmul_rn(1e6, b) / carrier_freq;
    out[stream] = q;
}

// ===================================================================================================
// SCH_demod of gsmcal_calibrate_cell_batch (definition: include/gsmcal.h): every SCH row of pos_info on r_correct with the stream's
// carrier-fit line removed from its equaliser window, on what carrier_fit_stream_kernel wrote.  osr 8 only.
// ===================================================================================================
// df_i (Hz, r_correct's frame) of the SCH row at p: the fitted line at the capture time of the training centre r(p + 74*osr), mapped as
// carrier_fit_row_kernel maps its window centre; every operation rounded on its own.  NaN without a fit.
__device__ __forceinline__ double sch_resid_hz(const CarrierFitDev &q, const StreamCtl &c, double p) {
    if (q.flags & CF_FEW) return NAN;
    const double s1 = __dadd_rn(1.0, __dmul_rn(c.sppm1, 1e-6)), s2 = __dadd_rn(1.0, __dmul_rn(c.sppm2, 1e-6));
    const double t = __ddiv_rn(__dmul_rn(__dmul_rn(p + (double)(74 * 8 - 1), s2), s1), ((1625.0 / 6.0) * 1e3) * 8.0);   // p + 591: exact
    return __dadd_rn(__dsub_rn(q.freq_hz, ((1625.0 / 6.0) * 1e3) / 4.0), __dmul_rn(q.drift_hz_per_s, __dsub_rn(t, q.t_mean)));
}

// sch_demod_batch_kernel's body with the residual folded into the derotation it already does: no extra pass over the window.  df_out
// [stream][cap]: df_i, NaN without a fit and for rows beyond n_sch.
__global__ void __launch_bounds__(SDB_THREADS, 2) sch_demod_resid_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const DemodResultDev *__restrict__ rec,
                                                                        const double *__restrict__ sch_pos, const unsigned char *__restrict__ sch_ok, int cap,
                                                                        const double2 *__restrict__ tw, const double2 *__restrict__ Ft,
                                                                        const double2 *__restrict__ Wtab, const signed char *__restrict__ data_pm,
                                                                        const CarrierFitDev *__restrict__ carrier, unsigned char *__restrict__ demod_bits,
                                                                        unsigned char *__restrict__ dec_bits, double *__restrict__ corr_val,
                                                                        double *__restrict__ df_out) {
    const int row = blockIdx.x, stream = blockIdx.y;
    const i64 o = (i64)stream * cap + row;
    if (row >= rec[stream].n_sch) {
        if (threadIdx.x == 0) df_out[o] = NAN;
        return;
    }
    const double df = sch_resid_hz(carrier[stream], ctl[stream], sch_pos[o]);
    if (threadIdx.x == 0) df_out[o] = df;
    const double resid = isnan(df) ? 0.0 : __ddiv_rn(__dmul_rn(2.0 * GSMCAL_PI, df), ((1625.0 / 6.0) * 1e3) * 8.0);      // rad per sample
    sch_demod_body<true>(src, ctl, rec, sch_pos, sch_ok, cap, 8, tw, Ft, Wtab, data_pm, demod_bits, dec_bits, corr_val, resid);
}

// ===================================================================================================
// BCCH decoding of gsmcal_calibrate_sysinfo_batch (definition: include/gsmcal.h), behind sch_decode_batch_kernel on what the cell
// call wrote: the block list, every BCCH burst (one-tap equaliser on the normal training sequence of the cell's BCC, MLSE) and the
// block decoding (deinterleaver, Viterbi, Fire code, payload), the per-stream SI mask and the SI3 vote.  osr 8 only.
// ===================================================================================================
struct SysinfoDev {                  // mirrors gsmcal_sysinfo_result (include/gsmcal.h)
    int n_blocks, n_fire_ok, n_si3, n_si3_agree, flags, si_mask, mcc, mnc, mnc_digits, lac, ci, reserved;
};
#define SI_NO_POS_INFO   1
#define SI_NO_R_CORRECT  2
#define SI_NO_CELL       4
#define SI_UNCORRECTED   8
#define SI_NO_SI3       16
#define SI_SI3_DISAGREE 32
#define SI_ROW_RANGE     1
#define SI_ROW_EDGE      2
#define SI_BLK_FN        1
#define SI_BLK_ROW       2
#define SI_BLK_FIRE      4
#define SI_BLK_SHORT     8
#define SI_NO_LAG     (-128)
#define BB_N      1552                 // 194*osr: the equaliser window of SCH_demod
#define BB_L      208                  // 26*osr template samples
#define BB_LAG0   64                   // lags -64..+95
#define BB_NLAG   160
#define BB_NY     (BB_N + BB_NLAG - 1) // 1711 samples of y
#define BB_TR     552                  // 69*osr: the training start in x
#define BB_THREADS 384                 // the loader's unrolled FIR path covers ceil(1714 / 5) level-0 groups
#define BB_S ((GSMCAL_XCAP(BB_NY) + BB_NY + 8) > (BB_N + SD_NSYM * 16) ? (GSMCAL_XCAP(BB_NY) + BB_NY + 8) : (BB_N + SD_NSYM * 16))
#define BB_SMEM ((size_t)(BB_NY + 1 + BB_S) * sizeof(double2))      // y | the loader's X, Y, later x | branch correlations
#define SI_FIRE_G 0x10004820009ull       // D^40 + D^26 + D^23 + D^17 + D^3 + 1
__constant__ unsigned c_nts_bits[8] = {0x970897u, 0xb778b7u, 0x10ee90eu, 0x11ed11eu, 0x6b906bu, 0x13ac13au, 0x29f629fu, 0x3bc4bbcu};  // bit j at 25 - j

// One thread per stream: the blocks of pos_info (type-2 rows directly behind a type-1 row, pos_info order), at most cap; blk_n = -1 when
// the cell call's SCH stage did not run.
__global__ void bcch_block_kernel(const StreamCtl *__restrict__ ctl, const double *__restrict__ pos_info, const DemodResultDev *__restrict__ rec,
                                  int n_streams, int cap, int *__restrict__ blk_n, double *__restrict__ blk_pos, unsigned char *__restrict__ blk_nrow) {
    const int stream = blockIdx.x * blockDim.x + threadIdx.x;
    if (stream >= n_streams) return;
    if (rec[stream].n_sch < 0) { blk_n[stream] = -1; return; }
    const double *pi = pos_info + (i64)stream * 6 * cap * 2;
    const int rows = ctl[stream].n_pos_info;
    const i64 base = (i64)stream * cap;
    int n = 0, k = -1;                                             // k: rows of the open block, -1 = none open
    bool after_sch = false;
    for (int i = 0; i < rows; ++i) {
        const double t = pi[2 * i + 1];
        if (t == 2.0 && after_sch) {
            if (k < 0) { if (n >= cap) break; k = 0; ++n; }
            if (k < 4) { blk_pos[(base + n - 1) * 4 + k] = pi[2 * i]; ++k; blk_nrow[base + n - 1] = (unsigned char)k; }
            continue;
        }
        after_sch = (t == 1.0);
        k = -1;
    }
    blk_n[stream] = n;
}

// One block per (BCCH row, stream), row 4b + k = row k of block b: the 1711-sample window through the level-3 loader with
// dphi2 - 2*pi*df/fs folded into the derotation step (as sch_demod_resid_kernel), the 160-lag x 208-tap training correlation in fp64,
// the one-tap division, gmsk_viterbi_warp, and the 114 coded bits (two 57-bit words) and stealing bits of the burst.
__global__ void __launch_bounds__(BB_THREADS, 2) bcch_burst_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const int *__restrict__ blk_n,
                                                                   const double *__restrict__ blk_pos, const unsigned char *__restrict__ blk_nrow,
                                                                   const SchDecodeResultDev *__restrict__ sdec, const CarrierFitDev *__restrict__ carrier,
                                                                   const double2 *__restrict__ nts, const double2 *__restrict__ Wtab, int cap,
                                                                   signed char *__restrict__ lag_out, unsigned char *__restrict__ rflag_out,
                                                                   unsigned char *__restrict__ steal_out, unsigned long long *__restrict__ ibits) {
    extern __shared__ double2 sm[];
    __shared__ double2 tpl[BB_L], cr[BB_NLAG], wsh, ph0;
    __shared__ double pw[BB_NLAG], energy;
    __shared__ int lstar;
    __shared__ unsigned char bits[SD_NSYM + 2];
    const int j = blockIdx.x, stream = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = j >> 2, k = j & 3;
    if (b >= blk_n[stream]) return;
    const i64 o = (i64)stream * cap * 4 + j;
    const int bsic = sdec[stream].bsic;
    const double p = blk_pos[o];
    const StreamCtl c = ctl[stream];
    const double s0 = p - 128.0;                                   // g - 64 - 69*osr, g = p + 61*osr
    const bool run = bsic >= 0 && k < blk_nrow[(i64)stream * cap + b];
    const bool in_range = p == floor(p) && s0 >= 1.0 && s0 + (double)(BB_NY - 1) <= (double)c.len3;
    if (!run || !in_range) {
        if (tid == 0) {
            lag_out[o] = SI_NO_LAG; rflag_out[o] = run ? SI_ROW_RANGE : 0; steal_out[o] = 0;
            ibits[2 * o] = 0ull; ibits[2 * o + 1] = 0ull;
        }
        return;
    }
    double2 *y = sm, *S = y + BB_NY + 1, *x = S, *cb = S + BB_N;
    const i64 j0 = (i64)s0 - 1;
    const double df = sch_resid_hz(carrier[stream], c, p);
    const double resid = isnan(df) ? 0.0 : __ddiv_rn(__dmul_rn(2.0 * GSMCAL_PI, df), ((1625.0 / 6.0) * 1e3) * 8.0);     // rad per sample
    const double2 *t_col = nts + (i64)(bsic & 7) * BB_L;
    for (int n = tid; n < BB_L; n += BB_THREADS) tpl[n] = t_col[n];
    if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); ph0 = make_double2(cs, sn); }
    load_window(src, c, stream, j0, BB_NY, y, S, S + GSMCAL_XCAP(BB_NY));  // ends with a barrier
    derotate_post(y, BB_NY, c.dphi2 - resid, ph0);
    __syncthreads();
    if (tid == 0) {                                                // sum |t_n|^2 in n order
        double e = 0.0;
        for (int n = 0; n < BB_L; ++n) e += tpl[n].x * tpl[n].x + tpl[n].y * tpl[n].y;
        energy = e;
    }
    for (int li = warp; li < BB_NLAG; li += BB_THREADS / 32) {     // c(l), l = li - 64, over y(li + 552 + n)
        double ar = 0.0, ai = 0.0;
        for (int n = lane; n < BB_L; n += 32) {
            const double2 t = tpl[n], v = y[li + BB_TR + n];
            ar += t.x * v.x + t.y * v.y;                           // conj(t) * v
            ai += t.x * v.y - t.y * v.x;
        }
        ar = warp_sum(ar); ai = warp_sum(ai);
        if (lane == 0) { cr[li] = make_double2(ar, ai); pw[li] = ar * ar + ai * ai; }
    }
    __syncthreads();
    if (warp == 0) {                                               // first maximum
        double bv = -1.0; int bi = BB_NLAG;
        for (int li = lane; li < BB_NLAG; li += 32) if (pw[li] > bv) { bv = pw[li]; bi = li; }
        for (int s = 16; s > 0; s >>= 1) {
            const double v2 = __shfl_xor_sync(0xffffffffu, bv, s);
            const int i2 = __shfl_xor_sync(0xffffffffu, bi, s);
            if (v2 > bv || (v2 == bv && i2 < bi)) { bv = v2; bi = i2; }
        }
        if (lane == 0) {
            lstar = bi;
            const double2 h = make_double2(cr[bi].x / energy, cr[bi].y / energy);
            const double q = h.x * h.x + h.y * h.y;
            wsh = make_double2(h.x / q, -h.y / q);                 // 1/h = conj(h) / |h|^2
        }
    }
    __syncthreads();
    const int ls = lstar;
    const double2 w = wsh;
    for (int n = tid; n < BB_N; n += BB_THREADS) x[n] = cmul(y[ls + n], w);     // x(n) = y(l* + 64 + n) / h
    __syncthreads();
    for (int i = tid; i < SD_NSYM * 16; i += BB_THREADS) {         // sch_bits_body's branch correlations
        const int m = i >> 4, combo = i & 15;
        double ar = 0.0, ai = 0.0;
        for (int q = 0; q < 8; ++q) {
            const double2 v = x[m * 8 + q], wt = Wtab[combo * 8 + q];
            ar += v.x * wt.x + v.y * wt.y;                         // v * conj(w)
            ai += v.y * wt.x - v.x * wt.y;
        }
        cb[i] = make_double2(ar, ai);
    }
    __syncthreads();
    if (tid < 32) gmsk_viterbi_warp(cb, SD_NSYM, bits);
    __syncthreads();
    if (tid == 0) {
        const unsigned char *m = bits + SD_TB + SD_EX;             // burst symbols 0..147
        const unsigned tsc = c_nts_bits[bsic & 7];
        unsigned long long w0 = 0ull, w1 = 0ull;
        int bb = (int)(tsc >> 25) & 1;                             // b(61) = TSC bit 0, then backwards
        int steal = 0;
        for (int i = 60; i >= 0; --i) {
            bb ^= 1 - m[i + 1];
            if (i == 60) steal |= bb;
            else if (i >= 3) w0 |= (unsigned long long)bb << (i - 3);      // i(0..56) = b(3..59)
        }
        bb = (int)tsc & 1;                                         // b(86) = TSC bit 25, then forwards
        for (int i = 87; i <= 147; ++i) {
            bb ^= 1 - m[i];
            if (i == 87) steal |= bb << 1;
            else if (i <= 144) w1 |= (unsigned long long)bb << (i - 88);   // i(57..113) = b(88..144)
        }
        const int l = ls - BB_LAG0;
        lag_out[o] = (signed char)l;
        rflag_out[o] = (l == -BB_LAG0 || l == BB_NLAG - 1 - BB_LAG0) ? SI_ROW_EDGE : 0;
        steal_out[o] = (unsigned char)steal;
        ibits[2 * o] = w0; ibits[2 * o + 1] = w1;
    }
}

// One warp per stream, one lane per block (b = lane, lane + 32, ...): FN and TC, the deinterleaver, the 16-state hard-decision Viterbi
// over 228 steps with one 16-bit decision word per step in shared memory, the Fire check on 64-bit shift registers during the traceback,
// the payload; then the warp's SI mask and SI3 vote (keys: octets 3..9 of the SI3 blocks, ~0 for blocks that do not vote).
#define BD_STEPS 228
__global__ void __launch_bounds__(32) bcch_decode_kernel(const DemodResultDev *__restrict__ rec, const SchDecodeResultDev *__restrict__ sdec,
                                                         const CarrierFitDev *__restrict__ carrier, const double *__restrict__ sch_pos,
                                                         const int *__restrict__ blk_n, const double *__restrict__ blk_pos,
                                                         const unsigned char *__restrict__ blk_nrow, const unsigned char *__restrict__ rflag,
                                                         const unsigned long long *__restrict__ ibits, int cap, unsigned long long *__restrict__ key,
                                                         int *__restrict__ fn_out, unsigned char *__restrict__ tc_out, unsigned char *__restrict__ flag_out,
                                                         unsigned short *__restrict__ ham_out, unsigned char *__restrict__ payload,
                                                         SysinfoDev *__restrict__ out) {
    __shared__ unsigned short dec[32][BD_STEPS];
    __shared__ unsigned long long ib[32][8];
    const int stream = blockIdx.x, lane = threadIdx.x;
    const i64 base = (i64)stream * cap;
    const int n = blk_n[stream];
    const SchDecodeResultDev sd = sdec[stream];
    const bool cell = sd.bsic >= 0;
    const double p_first = (rec[stream].n_sch > 0) ? sch_pos[base] : 0.0;
    int n_fire = 0, n_si3 = 0, mask = 0;
    for (int b = lane; b < n; b += 32) {
        const i64 ob = base + b;
        int fn = -1, tc = 255, fl = 0, ham = 0;
        unsigned long long kv = ~0ull;
        unsigned char pay[23];
        for (int m = 0; m < 23; ++m) pay[m] = 0;
        if (cell) {
            const i64 f = (i64)(blk_pos[ob * 4] - p_first) / 10000;
            fn = (int)(((i64)sd.fn_first + f) % SC_FN_MOD);
            tc = (fn / 51) % 8;
            const int nr = blk_nrow[ob];
            if (nr < 4) fl |= SI_BLK_SHORT;
            if (fn % 51 != 2) fl |= SI_BLK_FN;
            for (int r = 0; r < nr; ++r) if (rflag[ob * 4 + r]) fl |= SI_BLK_ROW;
        }
        if (cell && !fl) {
            for (int q = 0; q < 8; ++q) ib[lane][q] = ibits[ob * 8 + q];     // row r's words at 2r, 2r + 1
            int metric[16];
#pragma unroll
            for (int s = 0; s < 16; ++s) metric[s] = (s == 0) ? 0 : 1 << 20;
            for (int t = 0; t < BD_STEPS; ++t) {
                int cc[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {                      // c(k) = i_(k mod 4)(2*((49k) mod 57) + ((k mod 8) div 4))
                    const int kk = 2 * t + h, jj = 2 * ((49 * kk) % 57) + ((kk & 7) >> 2);
                    const unsigned long long wd = ib[lane][2 * (kk & 3) + (jj >= 57)];
                    cc[h] = (int)(wd >> (jj >= 57 ? jj - 57 : jj)) & 1;
                }
                int nm[16];
                unsigned dw = 0u;
#pragma unroll
                for (int s = 0; s < 16; ++s) {                     // sch_decode_row's step
                    const int u = s & 1, p0 = s >> 1, p1 = p0 | 8;
                    const int a0 = u ^ ((p0 >> 2) & 1), a1 = u ^ (p0 & 1) ^ ((p0 >> 2) & 1);
                    const int m0 = metric[p0] + (a0 ^ cc[0]) + (a1 ^ cc[1]);
                    const int m1 = metric[p1] + (a0 ^ 1 ^ cc[0]) + (a1 ^ 1 ^ cc[1]);
                    const bool take1 = m1 < m0;                    // a tie keeps dropped bit 0
                    nm[s] = take1 ? m1 : m0;
                    dw |= (unsigned)take1 << s;
                }
#pragma unroll
                for (int s = 0; s < 16; ++s) metric[s] = nm[s];
                dec[lane][t] = (unsigned short)dw;
            }
            ham = metric[0];
            // traceback from state 0: u(t) = s & 1.  Fire: rem = sum u(t) D^(223-t) mod g, built from the low powers up.
            unsigned long long rem = 0ull, pwr = 1ull;
            int s = 0, acc = 0;
            for (int t = BD_STEPS - 1; t >= 0; --t) {
                const int u = s & 1;
                s = (s >> 1) | ((((int)dec[lane][t] >> s) & 1) << 3);
                if (t < 224) {
                    if (u) rem ^= pwr;
                    pwr <<= 1;
                    if (pwr >> 40) pwr ^= SI_FIRE_G;
                }
                if (t < 184) {
                    acc |= u << (t & 7);
                    if ((t & 7) == 0) { pay[t >> 3] = (unsigned char)acc; acc = 0; }
                }
            }
            if (rem != 0xFFFFFFFFFFull) fl |= SI_BLK_FIRE;
            else {
                ++n_fire;
                const int mt = pay[2];
                int bit = 256;
                if (pay[1] == 0x06) {
                    switch (mt) {
                        case 0x19: bit = 1; break;   case 0x1A: bit = 2; break;   case 0x02: bit = 4; break;
                        case 0x03: bit = 8; break;   case 0x07: bit = 16; break;  case 0x1B: bit = 32; break;
                        case 0x1C: bit = 64; break;  case 0x00: bit = 128; break; default: break;
                    }
                }
                mask |= bit;
                if (bit == 32) {
                    ++n_si3;
                    kv = 0ull;
                    for (int m = 0; m < 7; ++m) kv |= (unsigned long long)pay[3 + m] << (8 * m);
                }
            }
        }
        fn_out[ob] = fn; tc_out[ob] = (unsigned char)tc; flag_out[ob] = (unsigned char)fl; ham_out[ob] = (unsigned short)ham;
        for (int m = 0; m < 23; ++m) payload[ob * 23 + m] = pay[m];
        key[ob] = kv;
    }
    n_fire = __reduce_add_sync(0xffffffffu, n_fire);
    n_si3 = __reduce_add_sync(0xffffffffu, n_si3);
    mask = (int)__reduce_or_sync(0xffffffffu, (unsigned)mask);
    __syncwarp();                                                  // every lane's keys are visible to the warp
    SysinfoDev o;
    o.n_blocks = n; o.n_fire_ok = n_fire; o.n_si3 = n_si3; o.n_si3_agree = 0; o.flags = 0; o.si_mask = mask;
    o.mcc = o.mnc = o.mnc_digits = o.lac = o.ci = -1; o.reserved = 0;
    const int rf = rec[stream].flags;
    if (n < 0) o.flags = (rf & DM_NO_POS_INFO) ? SI_NO_POS_INFO : SI_NO_R_CORRECT;
    else {
        if (!cell) o.flags |= SI_NO_CELL;
        if (carrier[stream].flags & CF_FEW) o.flags |= SI_UNCORRECTED;
        if (n_si3 == 0) o.flags |= SI_NO_SI3;
        else {
            int best_cnt = 0, best_first = 0x7fffffff;
            unsigned long long best_key = ~0ull;
            for (int i = lane; i < n; i += 32) {
                const unsigned long long ki = key[base + i];
                if (ki == ~0ull) continue;
                int cnt = 0, first = i;
                for (int j = 0; j < n; ++j) {
                    if (key[base + j] != ki) continue;
                    ++cnt;
                    if (j < first) first = j;
                }
                if (cnt > best_cnt || (cnt == best_cnt && first < best_first)) { best_cnt = cnt; best_first = first; best_key = ki; }
            }
            for (int s = 16; s > 0; s >>= 1) {
                const int c2 = __shfl_xor_sync(0xffffffffu, best_cnt, s), f2 = __shfl_xor_sync(0xffffffffu, best_first, s);
                const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, best_key, s);
                if (c2 > best_cnt || (c2 == best_cnt && f2 < best_first)) { best_cnt = c2; best_first = f2; best_key = k2; }
            }
            auto oct = [&](int m) { return (int)(best_key >> (8 * (m - 3))) & 0xFF; };     // octets 3..9
            o.n_si3_agree = best_cnt;
            if (best_cnt < n_si3) o.flags |= SI_SI3_DISAGREE;
            o.ci = (oct(3) << 8) | oct(4);
            o.mcc = 100 * (oct(5) & 15) + 10 * (oct(5) >> 4) + (oct(6) & 15);
            const int d3 = oct(6) >> 4, m1 = oct(7) & 15, m2 = oct(7) >> 4;
            o.mnc_digits = (d3 == 15) ? 2 : 3;
            o.mnc = (d3 == 15) ? 10 * m1 + m2 : 100 * m1 + 10 * m2 + d3;
            o.lac = (oct(8) << 8) | oct(9);
        }
    }
    if (lane == 0) out[stream] = o;
}
