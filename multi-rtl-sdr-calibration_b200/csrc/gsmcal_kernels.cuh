// gsmcal_kernels.cuh - hand-written sm_100a kernels of the GSM sync/calibration hot path.
//
// Every kernel is new (the reference is MATLAB, SURVEY.md section 2); comments cite the reference
// arithmetic each one reproduces as file:line into JiaoXianjun/multi-rtl-sdr-calibration.
// All decision paths are IEEE fp64.  No cuFFT, no tensor cores (nothing here is a dense contraction).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

typedef long long i64;
typedef unsigned long long u64;

#define GSMCAL_MAX_TAPS 128
#define GSMCAL_PI 3.14159265358979323846

// FIR numerator of the current call (the analogue of `persistent coef`), zero-padded on both sides so that the unrolled
// kernels can index taps -4 .. MAX_TAPS+3 without a range check
__constant__ double c_tapsp[GSMCAL_MAX_TAPS + 8];
#define c_taps (c_tapsp + 4)

// ---------------------------------------------------------------------------------------------------
// per-stream control block: everything the tiny sequential stages decide, kept on the device so the
// batched pipeline never synchronises with the host between stages.
// ---------------------------------------------------------------------------------------------------
struct StreamCtl {
    u64    sum_i, sum_q;          // exact integer column sums of raw2iq.m:8
    double mu_re, mu_im;          // sum / N, written once per stream by mean_kernel (saves two fp64 divisions per thread per window load)
    // coarse
    int    n_coarse;              // -1: no FCCH found (FCCH_coarse_position.m:27-30)
    int    first_hit;             // 1-based window index of the first hit, -1 none
    double hit_avg_snr, hit_snr;
    // FCCH fine
    int    n_fine;                // first-round positions kept (last_idx, FCCH_fine_correction.m:65)
    int    n_fcch;                // returned FCCH_pos count, -1 = scalar -1
    int    interp1_on;            // r was resampled by (1+e1)
    int    tone1_enable;          // carrier estimate runs (num_fcch >= 5)
    int    derot1_on;
    double e1, dphi1, sppm1, cppm1;
    i64    len1;                  // length of r after FCCH_fine_correction, -1 = scalar -1
    // SCH
    int    sch_enable, n_sch, n_pos_info, interp2_on;
    double e2, sppm2;
    i64    len2;
    // post-SCH
    int    post_enable, n_post_fcch;
    double cppm2, dphi2;
    i64    len3;
    int    flags;
    int    pad_;
};

struct WinSrc {
    int            lazy;        // 0: read a materialised complex128 stream, 1: evaluate from the uint8 capture
    int            level;       // lazy: 0 filtered, 1 resampled(e1), 2 resampled+derotated, 3 resampled again (e2)
    const double2 *base;        // materialised stream(s)
    i64            base_len;    // samples per stream
    i64            base_stride; // distance between streams
    int            mat_interp;  // materialised: evaluate interp1(base, j*(1+e1)) on the fly
    const uint8_t *raw;         // lazy: [n_streams][2*n_iq]
    i64            n_iq;
    int            n_taps;
    int            dec;         // decimation applied on top (coarse stage: osr*dr), else 1
    // filtered-window cache (osr 8 fast path): the fine search stores every burst's filtered (level-0) search window
    // [ (p-65)*8, +2208 ) so that the two tone stages re-use it instead of re-filtering the capture (see gsmcal_burst8.cuh)
    const double2 *wcache;      // [n_streams][wc_cap][B8_WLEN] padded layout, nullptr = no cache
    const double  *wc_pos;      // [n_streams][wc_cap] coarse positions the windows were cut at
    int            wc_cap;
};
#define B8_NSMP 2208                        // samples of a fine-search window at osr 8 (1025 window starts + 1184 - 1)
#define B8_NCH  69                          // 32-sample chunks per window
#define B8_WPAD(i) ((i) + ((i) >> 5))       // one pad slot per chunk: chunk starts fall into different shared-memory banks
#define B8_WLEN (B8_NSMP + B8_NCH)          // padded entries per cached window (36,432 bytes)

// capacity (double2) of load_window's scratch X for a window of `count` samples
#define GSMCAL_XCAP(count) ((count) + GSMCAL_MAX_TAPS + 8)
__host__ __device__ __forceinline__ int xpad(int i) { return i; }   // 3 outputs per thread: 48-byte lane stride is conflict free as is

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cmulc(double2 a, double2 b) {   // a * conj(b)
    return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
// upper bound of sqrt(e) for the certificates (they only need |s| <= bound): both roundings go up, a handful of fp32 instructions
// instead of the ~20-instruction fp64 sqrt; at most 2.4e-7 above the true value, far inside the certificates' 1e-6 margin
__device__ __forceinline__ double sqrt_ub(double e) { return (double)__fsqrt_ru(__double2float_ru(e)); }
__device__ __forceinline__ double abs2_ref(double2 a) {            // abs(z).^2: sqrt first, then square
    double h = hypot(a.x, a.y);
    return h * h;
}
__device__ __forceinline__ double2 lerp_ref(double2 v0, double2 v1, double frac) {
    // interp1 'linear': v0 + frac*(v1-v0), product and sum rounded separately (matches the oracle bit for bit)
    return make_double2(__dadd_rn(v0.x, __dmul_rn(frac, __dsub_rn(v1.x, v0.x))),
                        __dadd_rn(v0.y, __dmul_rn(frac, __dsub_rn(v1.y, v0.y))));
}
__device__ __forceinline__ double stream_mean(u64 sum, i64 n) { return (double)sum / (double)n; }

// filtered sample L0[i] of one stream straight from the uint8 capture (zero initial state, DC removed):
//   filter(coef,1,raw2iq(a))(i)  - gsm_sync_demod.m:107,110; oldest tap first as direct-form-II-transposed nests them
__device__ __forceinline__ double2 fir_from_raw(const uint8_t *__restrict__ raw, i64 i, int n_taps, double mur, double mui) {
    double ar = 0.0, ai = 0.0;
    int kmax = (i < (i64)(n_taps - 1)) ? (int)i : n_taps - 1;
    const uchar2 *p = reinterpret_cast<const uchar2 *>(raw + 2 * (i - kmax));
#pragma unroll 8
    for (int k = kmax; k >= 0; --k, ++p) {
        const double h = c_taps[k];
        const uchar2 u = *p;
        ar = fma(h, (double)u.x - mur, ar);
        ai = fma(h, (double)u.y - mui, ai);
    }
    return make_double2(ar, ai);
}

// R consecutive FIR outputs from a register sliding window, fully unrolled for a compile-time tap count: every tap is a
// constant-bank operand of its DFMA and every staged sample is loaded once per R outputs (1 LDS.128 per 2R DFMA; a 128-bit
// shared load costs 4 cycles of the 128 B/clk crossbar, so R >= 4 keeps the loop FP64-bound).  Odd R: the R*16-byte lane
// stride is bank-conflict free.  Oldest input first, as direct-form-II-transposed nests the sum.
template <int NT, int R, int FENCE = 0>
__device__ __forceinline__ void fir_taps_const(const double2 *__restrict__ xb, double (&ar)[R], double (&ai)[R]) {
#pragma unroll
    for (int r = 0; r < R; ++r) { ar[r] = 0.0; ai[r] = 0.0; }
#pragma unroll
    for (int k = 0; k < NT - 1 + R; ++k) {
        if (FENCE > 0 && k > 0 && (k % FENCE) == 0) asm volatile("" ::: "memory");   // keeps the compiler from hoisting every load (register pressure)
        const double2 x = xb[k];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int tap = (NT - 1) + r - k;
            if (tap >= 0 && tap < NT) { ar[r] = fma(c_taps[tap], x.x, ar[r]); ai[r] = fma(c_taps[tap], x.y, ai[r]); }
        }
    }
}
#define LW_R 5
template <int NT>
__device__ __forceinline__ void fir_group_one(const double2 *__restrict__ X, double2 *__restrict__ l0, int n_l0, int gi) {
    double ar[LW_R], ai[LW_R];
    fir_taps_const<NT, LW_R, 6>(X + LW_R * gi, ar, ai);
    const int base = LW_R * gi;
#pragma unroll
    for (int r = 0; r < LW_R; ++r) if (base + r < n_l0) l0[base + r] = make_double2(ar[r], ai[r]);
}
template <int NT>
__device__ __forceinline__ void fir_groups_c(const double2 *__restrict__ X, double2 *__restrict__ l0, int n_l0, int tid) {
    // one group per thread, straight-line code (the caller guarantees ceil(n_l0 / LW_R) <= blockDim.x): inside a loop over groups the
    // compiler hoists all 2*NT tap registers out of it and spills uniform registers
    if (LW_R * tid < n_l0) fir_group_one<NT>(X, l0, n_l0, tid);
}
// exact uint8 -> double without the quarter-rate I2F: the integer sits in the low mantissa bits of 2^52
__device__ __forceinline__ double u8_to_f64(unsigned v) { return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0; }

// ---------------------------------------------------------------------------------------------------
// block-cooperative window loader: dst[0..count) = samples [start, start+count) (0-based) of the stream
// the stage works on.  X, Y: scratch of GSMCAL_XCAP(count) and (count + 8) double2.
// Lazy levels restate, per sample, FCCH_fine_correction.m:123-125 (interp1), :165 (derotation) and
// SCH_corr_rate_correction.m:126-127 (second interp1) on top of raw2iq + filter.
// ---------------------------------------------------------------------------------------------------
__device__ void load_window(const WinSrc &src, const StreamCtl &c, int stream, i64 start, int count,
                            double2 *dst, double2 *X, double2 *Y, int burst = -1) {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (!src.lazy) {
        const double2 *b = src.base + (i64)stream * src.base_stride;
        if (src.mat_interp && c.interp1_on) {
            const double scale = 1.0 + c.e1;
            for (int i = tid; i < count; i += nt) {
                double xq = (double)(start + i) * scale;
                i64 i0 = (i64)floor(xq);
                if (i0 > src.base_len - 1) i0 = src.base_len - 1;
                if (i0 < 0) i0 = 0;
                i64 i1 = (i0 + 1 > src.base_len - 1) ? src.base_len - 1 : i0 + 1;
                dst[i] = lerp_ref(b[i0], b[i1], xq - (double)i0);
            }
        } else {
            for (int i = tid; i < count; i += nt) {
                i64 j = start + i;
                dst[i] = (j >= 0 && j < src.base_len) ? b[j] : make_double2(0.0, 0.0);
            }
        }
        __syncthreads();
        return;
    }
    const uint8_t *raw = src.raw + (i64)stream * 2 * src.n_iq;
    const i64 n0 = src.n_iq;
    const double mur = c.mu_re, mui = c.mu_im;
    const bool use2 = (src.level == 3) && c.interp2_on;
    const bool use1 = (src.level >= 1) && c.interp1_on;
    const bool derot = (src.level >= 2) && c.derot1_on;
    const double s1 = 1.0 + c.e1, s2 = 1.0 + c.e2;
    const i64 len1 = use1 ? c.len1 : n0;
    i64 a2 = start, b2 = start + count - 1, a1 = a2, b1 = b2, a0, b0;
    if (use2) {
        a1 = (i64)floor((double)a2 * s2);
        b1 = (i64)floor((double)b2 * s2) + 1;
        if (b1 > len1 - 1) b1 = len1 - 1;
        if (a1 > b1) a1 = b1;
    }
    a0 = a1; b0 = b1;
    if (use1) {
        a0 = (i64)floor((double)a1 * s1);
        b0 = (i64)floor((double)b1 * s1) + 1;
        if (b0 > n0 - 1) b0 = n0 - 1;
        if (a0 > b0) a0 = b0;
    }
    if (a0 < 0) a0 = 0;
    if (b0 > n0 - 1) b0 = n0 - 1;
    // derotation base phasor exp(1i*a1*dphi1): the argument reaches 1e5..1e6 rad (Payne-Hanek path of sincos, ~150 instructions), so ONE
    // thread evaluates it while the others stage and filter; it is read after the barriers below
    __shared__ double2 lw_base, lw_step;                         // exp(1i*a1*dphi1); exp(1i*nt*dphi1), the per-iteration step of every thread
    if (derot && use1 && tid == 0) { double sn, cs; sincos((double)a1 * c.dphi1, &sn, &cs); lw_base = make_double2(cs, sn); }
    if (derot && use1 && tid == 32 % nt) { double sn, cs; sincos((double)nt * c.dphi1, &sn, &cs); lw_step = make_double2(cs, sn); }
    const int n_l0 = (int)(b0 - a0 + 1);
    // unrolled FIR variants (taps zero-padded on the old side), one group of LW_R outputs per thread; longer windows or filters take the rolled loop
    const int nt_sel = ((n_l0 + LW_R - 1) / LW_R > nt) ? 0 : ((src.n_taps == 47) ? 47 : ((src.n_taps <= 48) ? 48 : (src.n_taps <= 64 ? 64 : 0)));
    const int nt1 = (nt_sel ? nt_sel : src.n_taps) - 1;
    const int n_raw = n_l0 + nt1;
    double2 *l0 = (use1 || use2) ? Y : dst;
    // the fine search left this burst's filtered window in the cache: level 0 is a copy, no staging, no FIR
    bool from_cache = false;
    if (src.wcache && burst >= 0) {
        const i64 wbase = ((i64)src.wc_pos[(i64)stream * src.wc_cap + burst] - 65) * 8;
        if (a0 >= wbase && b0 < wbase + B8_NSMP) {
            const double2 *wc = src.wcache + ((i64)stream * src.wc_cap + burst) * B8_WLEN;
            const int o = (int)(a0 - wbase);
            for (int i = tid; i < n_l0; i += nt) l0[i] = wc[B8_WPAD(o + i)];
            from_cache = true;
        }
    }
    if (!from_cache) {
    // stage the DC-removed capture once (zero before the first sample: zero initial filter state).  One 2-byte IQ pair per
    // thread and load, four loads in flight; consecutive threads write consecutive 16-byte slots (conflict free).
    {
        const i64 j00 = a0 - nt1;                                // sample staged at X[0]
        const unsigned short *rp = reinterpret_cast<const unsigned short *>(raw);
        constexpr int MAXQ = 4;
        for (int i0 = 0; i0 < n_raw; i0 += MAXQ * nt) {
            unsigned wv[MAXQ];
#pragma unroll
            for (int q = 0; q < MAXQ; ++q) {
                const int i = i0 + tid + q * nt;
                const i64 j = j00 + i;
                wv[q] = (i < n_raw && j >= 0 && j < n0) ? (unsigned)__ldg(rp + j) : 0x10000u;      // bit 16: no sample here
            }
#pragma unroll
            for (int q = 0; q < MAXQ; ++q) {
                const int i = i0 + tid + q * nt;
                if (i < n_raw)
                    X[xpad(i)] = (wv[q] & 0x10000u) ? make_double2(0.0, 0.0)
                                                    : make_double2(u8_to_f64(wv[q] & 0xffu) - mur, u8_to_f64((wv[q] >> 8) & 0xffu) - mui);
            }
        }
    }
    if (tid < 8) X[n_raw + tid] = make_double2(0.0, 0.0);        // the last output group reads up to LW_R-1 samples past the window
    __syncthreads();
    if (nt_sel == 47) fir_groups_c<47>(X, l0, n_l0, tid);
    else if (nt_sel == 48) fir_groups_c<48>(X, l0, n_l0, tid);
    else if (nt_sel == 64) fir_groups_c<64>(X, l0, n_l0, tid);
    else {
        // generic tap count: 3 consecutive outputs per thread from a sliding register window of taps
        const int n_grp = (n_l0 + 2) / 3;
        for (int gi = tid; gi < n_grp; gi += nt) {
            double ar[3] = {0.0, 0.0, 0.0}, ai[3] = {0.0, 0.0, 0.0};
            double hw[3] = {c_taps[nt1], 0.0, 0.0};
            const int base = 3 * gi;
            for (int kk = 0; kk <= nt1 + 2; ++kk) {
                const int ii = base + kk;
                const double2 x = (ii < n_raw) ? X[xpad(ii)] : make_double2(0.0, 0.0);
#pragma unroll
                for (int r = 0; r < 3; ++r) { ar[r] = fma(hw[r], x.x, ar[r]); ai[r] = fma(hw[r], x.y, ai[r]); }
                hw[2] = hw[1]; hw[1] = hw[0];
                hw[0] = (nt1 - kk - 1 >= 0) ? c_taps[nt1 - kk - 1] : 0.0;
            }
#pragma unroll
            for (int r = 0; r < 3; ++r) if (base + r < n_l0) l0[base + r] = make_double2(ar[r], ai[r]);
        }
    }
    }
    __syncthreads();
    if (!use1 && !use2) {
        if (derot) {   // not reachable in the reference flow (derotation implies resampling) but keep it total
            for (int i = tid; i < count; i += nt) {
                double sn, cs; sincos((double)(start + i) * c.dphi1, &sn, &cs);
                dst[i] = cmul(dst[i], make_double2(cs, sn));
            }
            __syncthreads();
        }
        return;
    }
    if (use1) {
        double2 *l1 = use2 ? X : dst;
        const int n_l1 = (int)(b1 - a1 + 1);
        // derotation phasor exp(1i*j*dphi1) = base * exp(1i*tid*dphi1) for the thread's first sample (small arguments: the short
        // sincos path), then a fixed complex step of nt samples
        double2 ph = make_double2(1.0, 0.0), st = make_double2(1.0, 0.0);
        if (derot) {
            double sn, cs;
            sincos((double)tid * c.dphi1, &sn, &cs); ph = cmul(lw_base, make_double2(cs, sn));
            st = lw_step;
        }
        for (int i = tid; i < n_l1; i += nt) {
            i64 j = a1 + i;
            double xq = (double)j * s1;
            i64 i0 = (i64)floor(xq);
            if (i0 > n0 - 1) i0 = n0 - 1;
            i64 i1 = (i0 + 1 > n0 - 1) ? n0 - 1 : i0 + 1;
            double2 v = lerp_ref(Y[i0 - a0], Y[i1 - a0], xq - (double)i0);
            if (derot) { v = cmul(v, ph); ph = cmul(ph, st); }
            l1[i] = v;
        }
        __syncthreads();
    } else {   // level 3 with interp2 only (e1 path off): L1 == L0 (+derot)
        for (int i = tid; i < n_l0; i += nt) {
            double2 v = Y[i];
            if (derot) {
                double sn, cs; sincos((double)(a0 + i) * c.dphi1, &sn, &cs);
                v = cmul(v, make_double2(cs, sn));
            }
            X[i] = v;
        }
        __syncthreads();
    }
    if (use2) {
        for (int i = tid; i < count; i += nt) {
            double xq = (double)(a2 + i) * s2;
            i64 i0 = (i64)floor(xq);
            if (i0 > len1 - 1) i0 = len1 - 1;
            i64 i1 = (i0 + 1 > len1 - 1) ? len1 - 1 : i0 + 1;
            dst[i] = lerp_ref(X[i0 - a1], X[i1 - a1], xq - (double)i0);
        }
        __syncthreads();
    }
}

// one decimated sample of the stream the coarse stage sees: s(1:dec:end) - gsm_sync_demod.m:117
__device__ __forceinline__ double2 coarse_sample(const WinSrc &src, const StreamCtl &c, int stream, i64 idx0) {
    if (!src.lazy) return src.base[(i64)stream * src.base_stride + idx0];
    const uint8_t *raw = src.raw + (i64)stream * 2 * src.n_iq;
    return fir_from_raw(raw, idx0 * src.dec, src.n_taps, c.mu_re, c.mu_im);
}

// ---------------------------------------------------------------------------------------------------
// block reductions
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
// first-maximum argmax: larger value wins, equal values -> smaller index (MATLAB max returns the first)
__device__ __forceinline__ void argmax_combine(double &v, int &i, double v2, int i2) {
    if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}
__device__ void block_argmax(double &v, int &i, double *sv, int *si) {
    for (int o = 16; o > 0; o >>= 1) {
        double v2 = __shfl_down_sync(0xffffffffu, v, o);
        int i2 = __shfl_down_sync(0xffffffffu, i, o);
        argmax_combine(v, i, v2, i2);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (lane == 0) { sv[w] = v; si[w] = i; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double bv = sv[0]; int bi = si[0];
        for (int k = 1; k < nw; ++k) argmax_combine(bv, bi, sv[k], si[k]);
        sv[0] = bv; si[0] = bi;
    }
    __syncthreads();
    v = sv[0]; i = si[0];
    __syncthreads();
}
__device__ double block_sum(double v, double *sv) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (lane == 0) sv[w] = v;
    __syncthreads();
    if (w == 0) {
        double t = (lane < nw) ? sv[lane] : 0.0;
        t = warp_sum(t);
        if (lane == 0) sv[0] = t;
    }
    __syncthreads();
    double r = sv[0];
    __syncthreads();
    return r;
}

// several block sums at once.  ALL = true: every thread receives the totals (thread k adds the per-warp partials of value k, a third
// barrier publishes them - the earlier "every thread adds all 8*K partials" form cost more instructions than the FIR in the tone
// estimator).  ALL = false: only thread 0 receives them (K <= 4): warp 0 adds the partials with a segmented shuffle tree.
template <int K, bool ALL = true>
__device__ void block_sum_n(double (&v)[K], double *sv /* >= 8*K */) {
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = warp_sum(v[k]);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) sv[k * 8 + w] = v[k];
    }
    __syncthreads();
    if (ALL) {
        if (threadIdx.x < K) {
            double t = 0.0;
            for (int i = 0; i < nw; ++i) t += sv[threadIdx.x * 8 + i];
            sv[threadIdx.x * 8] = t;                             // row k is only touched by thread k
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < K; ++k) v[k] = sv[k * 8];
    } else {
        static_assert(ALL || K <= 4, "thread-0 variant handles up to 4 values (32 partials)");
        if (w == 0) {
            double t = (lane < 8 * K && (lane & 7) < nw) ? sv[lane] : 0.0;
            t += __shfl_down_sync(0xffffffffu, t, 4);
            t += __shfl_down_sync(0xffffffffu, t, 2);
            t += __shfl_down_sync(0xffffffffu, t, 1);
#pragma unroll
            for (int k = 0; k < K; ++k) v[k] = __shfl_sync(0xffffffffu, t, 8 * k);
        }
    }
    __syncthreads();
}
// inclusive prefix sum of a[0..n) in shared memory, executed by ONE full warp
__device__ void warp_scan_smem(double *a, int n, int lane) {
    const int per = (n + 31) >> 5, b = lane * per;
    double loc = 0.0;
    for (int i = 0; i < per; ++i) if (b + i < n) loc += a[b + i];
    double inc = loc;
    for (int d = 1; d < 32; d <<= 1) { const double t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    double run = inc - loc;
    for (int i = 0; i < per; ++i) if (b + i < n) { run += a[b + i]; a[b + i] = run; }
}

// ===================================================================================================
// K1  raw2iq.m:5-8
// ===================================================================================================
// exact integer column sums: 16-byte loads, dp4a byte sums, one 64-bit atomic per warp.
// grid (chunks, streams); each block owns `chunk_bytes` (multiple of 16) of one stream.
__device__ __forceinline__ void colsum_u8_chunk(const uint8_t *__restrict__ raw, i64 n_iq, i64 chunk_bytes, StreamCtl *ctl, int stream, i64 chunk_id) {
    const uint8_t *p = raw + (i64)stream * 2 * n_iq;
    const i64 total = 2 * n_iq;
    const i64 head = (16 - ((uintptr_t)p & 15)) & 15;            // even, since every stream starts on an even byte
    const i64 body = ((total - (head < total ? head : total)) / 16) * 16;
    unsigned si = 0, sq = 0;
    u64 li = 0, lq = 0;
    {
        const i64 c0 = chunk_id * chunk_bytes;
        i64 c1 = c0 + chunk_bytes; if (c1 > body) c1 = body;
        const uint4 *v = reinterpret_cast<const uint4 *>(p + head);
        const i64 i0 = c0 / 16, i1 = c1 / 16;
        const int nt = blockDim.x;                               // 256
        i64 i = i0 + threadIdx.x;
        for (; i + 3 * nt < i1; i += 4 * nt) {
            uint4 a = __ldg(v + i), b = __ldg(v + i + nt), c = __ldg(v + i + 2 * nt), d = __ldg(v + i + 3 * nt);
#define GSMCAL_ACC(w) si = __dp4a((w), 0x00010001u, si); sq = __dp4a((w), 0x01000100u, sq);
            GSMCAL_ACC(a.x) GSMCAL_ACC(a.y) GSMCAL_ACC(a.z) GSMCAL_ACC(a.w)
            GSMCAL_ACC(b.x) GSMCAL_ACC(b.y) GSMCAL_ACC(b.z) GSMCAL_ACC(b.w)
            GSMCAL_ACC(c.x) GSMCAL_ACC(c.y) GSMCAL_ACC(c.z) GSMCAL_ACC(c.w)
            GSMCAL_ACC(d.x) GSMCAL_ACC(d.y) GSMCAL_ACC(d.z) GSMCAL_ACC(d.w)
        }
        for (; i < i1; i += nt) {
            uint4 a = __ldg(v + i);
            GSMCAL_ACC(a.x) GSMCAL_ACC(a.y) GSMCAL_ACC(a.z) GSMCAL_ACC(a.w)
        }
#undef GSMCAL_ACC
    }
    li = si; lq = sq;
    if (chunk_id == 0) {                                          // ragged head / tail bytes, scalar
        const i64 hb = (head < total) ? head : total;
        for (i64 j = threadIdx.x; j < hb; j += blockDim.x) { if (j & 1) lq += p[j]; else li += p[j]; }
        for (i64 j = hb + body + threadIdx.x; j < total; j += blockDim.x) { if (j & 1) lq += p[j]; else li += p[j]; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        li += __shfl_down_sync(0xffffffffu, li, o);
        lq += __shfl_down_sync(0xffffffffu, lq, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (li) atomicAdd(&ctl[stream].sum_i, li);
        if (lq) atomicAdd(&ctl[stream].sum_q, lq);
    }
}

__global__ void __launch_bounds__(256) colsum_u8_kernel(const uint8_t *__restrict__ raw, i64 n_iq, i64 chunk_bytes, StreamCtl *ctl) {
    colsum_u8_chunk(raw, n_iq, chunk_bytes, ctl, blockIdx.y, blockIdx.x);
}

// "trickle" form for the staggered submit/collect pipeline (debug key 17): ONE warp per block, one block per SM, the bytes brought in by
// TMA bulk copies (cp.async.bulk -> UBLKCP) into a ring of 4 KB stages that complete on mbarriers.  What is in flight lives in shared
// memory, not in registers, so the footprint is 1 K registers + the ring (it fits beside four blocks of every FP64 kernel of the previous
// batch), and the ring size bounds the HBM rate (ring bytes / memory latency per SM): the sums of batch k+1 trickle in under the FP64
// stages of batch k instead of saturating HBM in front of them.  Same exact integer sums as colsum_u8_chunk, same (stream, chunk) units.
#define TRK_STAGE 4096
__global__ void __launch_bounds__(32) colsum_u8_trickle_kernel(const uint8_t *__restrict__ raw, i64 n_iq, i64 chunk_bytes, i64 n_chunks, i64 n_streams,
                                                               StreamCtl *ctl, int n_stage) {
    extern __shared__ __align__(128) unsigned char trk_sm[];     // [n_stage][TRK_STAGE] bytes, then n_stage mbarriers
    const int lane = threadIdx.x;
    const unsigned sm0 = (unsigned)__cvta_generic_to_shared(trk_sm), bar0 = sm0 + (unsigned)n_stage * TRK_STAGE;
    if (lane == 0) {
        for (int s = 0; s < n_stage; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8 * s));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    __syncwarp();
    const i64 total_units = n_chunks * n_streams, total = 2 * n_iq;
    struct Cur { i64 w, off, len; const uint8_t *base; };        // unit, byte offset inside it, its length, its first byte (16-byte aligned)
    auto open_unit = [&](Cur &c) {                               // skips empty units; len = 0 when the block has no more work
        for (; c.w < total_units; c.w += gridDim.x) {
            const int stream = (int)(c.w / n_chunks);
            const i64 chunk_id = c.w % n_chunks;
            const uint8_t *p = raw + (i64)stream * total;
            const i64 head = (16 - ((uintptr_t)p & 15)) & 15;
            const i64 body = ((total - (head < total ? head : total)) / 16) * 16;
            const i64 c0 = chunk_id * chunk_bytes;
            i64 c1 = c0 + chunk_bytes; if (c1 > body) c1 = body;
            if (c1 > c0 || chunk_id == 0) { c.off = 0; c.len = c1 > c0 ? c1 - c0 : 0; c.base = p + head + c0; return; }
        }
        c.off = 0; c.len = 0; c.base = nullptr;
    };
    // the producer cursor only visits units that have bytes; the consumer also visits empty chunk-0 units (ragged head / tail)
    auto prod_next = [&](Cur &c) {
        c.off += TRK_STAGE;
        if (c.off >= c.len) { do { c.w += gridDim.x; open_unit(c); } while (c.w < total_units && c.len == 0); }
    };
    auto issue = [&](const Cur &c, int stage) {                  // lane 0 only
        const i64 left = c.len - c.off;
        const unsigned bytes = (unsigned)(left < TRK_STAGE ? left : TRK_STAGE);
        const unsigned bar = bar0 + 8 * stage;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes));
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(sm0 + (unsigned)stage * TRK_STAGE), "l"(c.base + c.off), "r"(bytes), "r"(bar) : "memory");
    };
    Cur prod; prod.w = blockIdx.x; open_unit(prod);
    while (prod.w < total_units && prod.len == 0) { prod.w += gridDim.x; open_unit(prod); }
    Cur cons; cons.w = blockIdx.x; open_unit(cons);
    for (int s = 0; s < n_stage; ++s)
        if (prod.w < total_units) { if (lane == 0) issue(prod, s); prod_next(prod); }
    int stage = 0; unsigned phase = 0;
    unsigned si = 0, sq = 0;
    while (cons.w < total_units) {
        if (cons.len > 0) {
            const i64 left = cons.len - cons.off;
            const int bytes = (int)(left < TRK_STAGE ? left : TRK_STAGE);
            {
                unsigned done = 0;
                const unsigned bar = bar0 + 8 * stage;
                while (!done)
                    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                 : "=r"(done) : "r"(bar), "r"(phase) : "memory");
            }
            const uint4 *v = reinterpret_cast<const uint4 *>(trk_sm + (size_t)stage * TRK_STAGE);
            unsigned ti = 0, tq = 0, ui = 0, uq = 0, wi = 0, wq = 0;     // four independent dp4a chains per column
#define GSMCAL_ACC2(w, a, b) a = __dp4a((w), 0x00010001u, a); b = __dp4a((w), 0x01000100u, b);
            if (bytes == TRK_STAGE) {                            // all eight 16-byte loads in flight before the first use (one warp: latency is exposed)
                uint4 a[TRK_STAGE / 512];
#pragma unroll
                for (int k = 0; k < TRK_STAGE / 512; ++k) a[k] = v[lane + 32 * k];
#pragma unroll
                for (int k = 0; k < TRK_STAGE / 512; ++k) {
                    GSMCAL_ACC2(a[k].x, si, sq) GSMCAL_ACC2(a[k].y, ti, tq) GSMCAL_ACC2(a[k].z, ui, uq) GSMCAL_ACC2(a[k].w, wi, wq)
                }
            } else {
                for (int i = lane; 16 * i < bytes; i += 32) {
                    const uint4 a = v[i];
                    GSMCAL_ACC2(a.x, si, sq) GSMCAL_ACC2(a.y, ti, tq) GSMCAL_ACC2(a.z, ui, uq) GSMCAL_ACC2(a.w, wi, wq)
                }
            }
#undef GSMCAL_ACC2
            ti += ui; tq += uq; si += wi; sq += wq;
            si += ti; sq += tq;
            __syncwarp();                                        // every lane has read the stage before it is refilled
            if (prod.w < total_units) { if (lane == 0) issue(prod, stage); prod_next(prod); }
            if (++stage == n_stage) { stage = 0; phase ^= 1u; }
            cons.off += TRK_STAGE;
        }
        if (cons.off >= cons.len) {                              // unit done (at most 512 KB: the 32-bit lane sums cannot overflow)
            const int stream = (int)(cons.w / n_chunks);
            u64 li = si, lq = sq; si = 0; sq = 0;
            if (cons.w % n_chunks == 0) {                        // ragged head / tail bytes, scalar
                const uint8_t *p = raw + (i64)stream * total;
                const i64 head = (16 - ((uintptr_t)p & 15)) & 15;
                const i64 body = ((total - (head < total ? head : total)) / 16) * 16;
                const i64 hb = (head < total) ? head : total;
                for (i64 j = lane; j < hb; j += 32) { if (j & 1) lq += p[j]; else li += p[j]; }
                for (i64 j = hb + body + lane; j < total; j += 32) { if (j & 1) lq += p[j]; else li += p[j]; }
            }
            for (int o = 16; o > 0; o >>= 1) {
                li += __shfl_down_sync(0xffffffffu, li, o);
                lq += __shfl_down_sync(0xffffffffu, lq, o);
            }
            if (lane == 0) {
                if (li) atomicAdd(&ctl[stream].sum_i, li);
                if (lq) atomicAdd(&ctl[stream].sum_q, lq);
            }
            cons.w += gridDim.x; open_unit(cons);
        }
    }
}

// b = c - mean: one thread per IQ pair, 2-byte load, 16-byte store (warp stores 512 contiguous bytes)
__global__ void __launch_bounds__(256) raw2iq_store_kernel(const uint8_t *__restrict__ raw, i64 n_iq, const StreamCtl *__restrict__ ctl, double2 *__restrict__ out) {
    const int stream = blockIdx.y;
    const uchar2 *p = reinterpret_cast<const uchar2 *>(raw + (i64)stream * 2 * n_iq);
    double2 *o = out + (i64)stream * n_iq;
    const double mur = stream_mean(ctl[stream].sum_i, n_iq), mui = stream_mean(ctl[stream].sum_q, n_iq);
    const i64 stride = (i64)gridDim.x * 256;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < n_iq; i += stride) {
        uchar2 u = p[i];
        __stcs(o + i, make_double2((double)u.x - mur, (double)u.y - mui));
    }
}

// double-typed input (fread returns double, gsm_sync_demod.m:96): exact sums as long as values are 0..255 integers;
// done in fp64 with a fixed tree so the result is order-independent only for integer data (documented).
__global__ void __launch_bounds__(256) colsum_f64_kernel(const double *__restrict__ a, i64 n_iq, StreamCtl *ctl) {
    const int stream = blockIdx.y;
    const double2 *p = reinterpret_cast<const double2 *>(a + (i64)stream * 2 * n_iq);
    u64 li = 0, lq = 0;
    const i64 stride = (i64)gridDim.x * 256;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < n_iq; i += stride) {
        double2 v = p[i];
        li += (u64)(i64)v.x; lq += (u64)(i64)v.y;
    }
    for (int o = 16; o > 0; o >>= 1) {
        li += __shfl_down_sync(0xffffffffu, li, o);
        lq += __shfl_down_sync(0xffffffffu, lq, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&ctl[stream].sum_i, li); atomicAdd(&ctl[stream].sum_q, lq); }
}
__global__ void __launch_bounds__(256) raw2iq_store_f64_kernel(const double *__restrict__ a, i64 n_iq, const StreamCtl *__restrict__ ctl, double2 *__restrict__ out) {
    const int stream = blockIdx.y;
    const double2 *p = reinterpret_cast<const double2 *>(a + (i64)stream * 2 * n_iq);
    double2 *o = out + (i64)stream * n_iq;
    const double mur = stream_mean(ctl[stream].sum_i, n_iq), mui = stream_mean(ctl[stream].sum_q, n_iq);
    const i64 stride = (i64)gridDim.x * 256;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < n_iq; i += stride) {
        double2 v = p[i];
        o[i] = make_double2(v.x - mur, v.y - mui);
    }
}

// ===================================================================================================
// K2  filter(coef,1,s) [+ s(1:decim:end)]   gsm_sync_demod.m:110, chn_filter_8x_4x.m:13-15
// ===================================================================================================
// Full-rate FIR, complex128 in/out (or uint8 in with DC removal fused).  Each thread produces R=8
// consecutive outputs from a register-blocked sliding window, so every staged input is read from shared
// memory once per 8 outputs.  Shared rows are padded (one slot per 8) to keep the 128-byte-strided
// per-thread reads bank-conflict free.  NT = taps rounded up (zero-padded on the old side: adds exact 0).
#define FIR_R 8
#define FIR_THREADS 128
#define FIR_TILE (FIR_R * FIR_THREADS)
__device__ __forceinline__ int fir_pad(int i) { return i + (i >> 3); }

template <int NT, bool FROM_U8>
__global__ void __launch_bounds__(FIR_THREADS) fir_full_kernel(const void *__restrict__ in_, i64 n, i64 in_stride, const StreamCtl *__restrict__ ctl,
                                                              double2 *__restrict__ out, i64 out_stride) {
    extern __shared__ double2 sm[];
    const int stream = blockIdx.y;
    const i64 t0 = (i64)blockIdx.x * FIR_TILE;                    // first output of the tile
    const int n_in = FIR_TILE + NT - 1;
    double mur = 0.0, mui = 0.0;
    if (FROM_U8) { mur = stream_mean(ctl[stream].sum_i, n); mui = stream_mean(ctl[stream].sum_q, n); }
    {   // all of a thread's loads are issued before the first is consumed (one memory latency per tile, not per element)
        constexpr int NLD = (FIR_TILE + NT - 1 + FIR_THREADS - 1) / FIR_THREADS;
        double2 v[NLD];
        uchar2 u[NLD];
#pragma unroll
        for (int q = 0; q < NLD; ++q) {
            const int i = threadIdx.x + q * FIR_THREADS;
            const i64 j = t0 - (NT - 1) + i;
            v[q] = make_double2(0.0, 0.0); u[q] = make_uchar2(0, 0);
            if (i < n_in && j >= 0 && j < n) {
                if (FROM_U8) u[q] = reinterpret_cast<const uchar2 *>(static_cast<const uint8_t *>(in_) + (i64)stream * in_stride)[j];
                else v[q] = __ldcs(static_cast<const double2 *>(in_) + (i64)stream * in_stride + j);
            }
        }
#pragma unroll
        for (int q = 0; q < NLD; ++q) {
            const int i = threadIdx.x + q * FIR_THREADS;
            const i64 j = t0 - (NT - 1) + i;
            if (i < n_in) {
                if (FROM_U8) v[q] = (j >= 0 && j < n) ? make_double2((double)u[q].x - mur, (double)u[q].y - mui) : make_double2(0.0, 0.0);
                sm[fir_pad(i)] = v[q];
            }
        }
    }
    __syncthreads();
    double ar[FIR_R], ai[FIR_R];
#pragma unroll
    for (int r = 0; r < FIR_R; ++r) { ar[r] = 0.0; ai[r] = 0.0; }
    const int base = threadIdx.x * FIR_R;                         // staged index of the oldest input of output 0
#pragma unroll
    for (int k = 0; k < NT - 1 + FIR_R; ++k) {
        double2 x = sm[fir_pad(base + k)];
#pragma unroll
        for (int r = 0; r < FIR_R; ++r) {
            const int tap = (NT - 1) + r - k;                     // oldest input first: h[NT-1] ... h[0]
            if (tap >= 0 && tap < NT) {
                ar[r] = fma(c_taps[tap], x.x, ar[r]);
                ai[r] = fma(c_taps[tap], x.y, ai[r]);
            }
        }
    }
    double2 *o = out + (i64)stream * out_stride;
#pragma unroll
    for (int r = 0; r < FIR_R; ++r) {
        i64 j = t0 + base + r;
        if (j < n) __stcs(o + j, make_double2(ar[r], ai[r]));
    }
}

// Full-rate complex128 FIR, persistent + TMA double buffering.  Each block loops over tiles of FT_TILE outputs; the
// (FT_TILE + NT - 1)-sample input tile (18.7 KB, contiguous, 16-byte aligned) is fetched by ONE cp.async.bulk (UBLKCP)
// per tile that completes on an mbarrier, two tiles in flight, so the FP64 pipe never waits for global memory.  Each
// thread produces 9 consecutive outputs from a register sliding window; 9*16 B = 144 B lane stride is bank-conflict
// free on the dense layout the bulk copy writes, so no re-layout pass is needed.
#define FT_R 9
#define FT_THREADS 128
#define FT_TILE (FT_R * FT_THREADS)
template <int NT>
__global__ void __launch_bounds__(FT_THREADS) fir_full_tma_kernel(const double2 *__restrict__ in, i64 n, i64 n_col, double2 *__restrict__ out) {
    extern __shared__ __align__(16) double2 sm[];                // [2][FT_TILE + NT - 1]
    __shared__ __align__(8) unsigned long long full_bar[2];
    constexpr int TILE_IN = FT_TILE + NT - 1;
    const i64 tiles_per_col = (n + FT_TILE - 1) / FT_TILE, n_tiles = tiles_per_col * n_col;
    const unsigned bar0 = (unsigned)__cvta_generic_to_shared(&full_bar[0]);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8));
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    __syncthreads();
    auto issue = [&](i64 tile, int stage) {                      // thread 0 only
        const i64 col = tile / tiles_per_col, t0 = (tile % tiles_per_col) * FT_TILE;
        const i64 j0 = (t0 - (NT - 1) > 0) ? t0 - (NT - 1) : 0;                       // first valid input sample
        i64 j1 = t0 + FT_TILE; if (j1 > n) j1 = n;
        const unsigned bytes = (unsigned)((j1 - j0) * sizeof(double2));
        const unsigned dst = (unsigned)__cvta_generic_to_shared(sm + (size_t)stage * TILE_IN + (j0 - (t0 - (NT - 1))));
        const unsigned bar = bar0 + 8 * stage;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes));
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst), "l"(in + col * n + j0), "r"(bytes), "r"(bar) : "memory");
    };
    i64 tile = blockIdx.x;
    if (threadIdx.x == 0) {
        if (tile < n_tiles) issue(tile, 0);
        if (tile + gridDim.x < n_tiles) issue(tile + gridDim.x, 1);
    }
    unsigned phase[2] = {0u, 0u};
    for (int it = 0; tile < n_tiles; tile += gridDim.x, ++it) {
        const int stage = it & 1;
        const i64 col = tile / tiles_per_col, t0 = (tile % tiles_per_col) * FT_TILE;
        double2 *buf = sm + (size_t)stage * TILE_IN;
        {
            unsigned done = 0;
            const unsigned bar = bar0 + 8 * stage;
            while (!done)
                asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                             : "=r"(done) : "r"(bar), "r"(phase[stage]) : "memory");
            phase[stage] ^= 1u;
        }
        if (t0 == 0) {                                           // zero initial filter state: the halo before the first sample
            for (int i = threadIdx.x; i < NT - 1; i += FT_THREADS) buf[i] = make_double2(0.0, 0.0);
            __syncthreads();
        }
        double ar[FT_R], ai[FT_R];
#pragma unroll
        for (int r = 0; r < FT_R; ++r) { ar[r] = 0.0; ai[r] = 0.0; }
        const double2 *xb = buf + threadIdx.x * FT_R;
#pragma unroll
        for (int k = 0; k < NT - 1 + FT_R; ++k) {
            const double2 x = xb[k];
#pragma unroll
            for (int r = 0; r < FT_R; ++r) {
                const int tap = (NT - 1) + r - k;                // oldest input first: h[NT-1] ... h[0]
                if (tap >= 0 && tap < NT) { ar[r] = fma(c_taps[tap], x.x, ar[r]); ai[r] = fma(c_taps[tap], x.y, ai[r]); }
            }
        }
        double2 *o = out + col * n + t0 + threadIdx.x * FT_R;
#pragma unroll
        for (int r = 0; r < FT_R; ++r)
            if (t0 + threadIdx.x * FT_R + r < n) __stcs(o + r, make_double2(ar[r], ai[r]));
        __syncthreads();                                         // every thread is done reading this stage
        if (threadIdx.x == 0 && tile + 2 * (i64)gridDim.x < n_tiles) issue(tile + 2 * (i64)gridDim.x, stage);
    }
}

// Decimating FIR: one thread per kept output r(1+m*decim); input tile staged contiguously (coalesced) in
// shared memory.  Used for decim > 1 (2: chn_filter_8x_4x, 20: split scanner, 64: coarse stream).
#define FIRD_THREADS 128
template <bool FROM_U8>
__global__ void __launch_bounds__(FIRD_THREADS) fir_decim_kernel(const void *__restrict__ in_, i64 n, i64 in_stride, const StreamCtl *__restrict__ ctl, int n_taps,
                                                                int decim, int outs_per_block, double2 *__restrict__ out, i64 n_out, i64 out_stride,
                                                                double *__restrict__ power_acc) {
    extern __shared__ double2 sm[];
    const int stream = blockIdx.y;
    const i64 m0 = (i64)blockIdx.x * outs_per_block;
    i64 m1 = m0 + outs_per_block; if (m1 > n_out) m1 = n_out;
    const int n_o = (int)(m1 - m0);
    const i64 j0 = m0 * decim - (n_taps - 1);
    const int n_in = (n_o - 1) * decim + n_taps;
    double mur = 0.0, mui = 0.0;
    if (FROM_U8) { mur = stream_mean(ctl[stream].sum_i, n); mui = stream_mean(ctl[stream].sum_q, n); }
    const bool sparse = decim >= n_taps;          // windows do not overlap: skip the unused inputs between them
    for (int i = threadIdx.x; i < n_in; i += FIRD_THREADS) {
        if (sparse && ((i % decim) >= n_taps)) continue;
        i64 j = j0 + i;
        double2 v = make_double2(0.0, 0.0);
        if (j >= 0 && j < n) {
            if (FROM_U8) {
                uchar2 u = reinterpret_cast<const uchar2 *>(static_cast<const uint8_t *>(in_) + (i64)stream * in_stride)[j];
                v = make_double2((double)u.x - mur, (double)u.y - mui);
            } else {
                v = static_cast<const double2 *>(in_)[(i64)stream * in_stride + j];
            }
        }
        sm[i + i / 8] = v;
    }
    __syncthreads();
    double pw = 0.0;
    for (int o = threadIdx.x; o < n_o; o += FIRD_THREADS) {
        const int b = o * decim;
        double ar = 0.0, ai = 0.0;
        for (int k = n_taps - 1; k >= 0; --k) {
            int idx = b + (n_taps - 1 - k);
            double2 x = sm[idx + idx / 8];
            ar = fma(c_taps[k], x.x, ar);
            ai = fma(c_taps[k], x.y, ai);
        }
        if (out) out[(i64)stream * out_stride + m0 + o] = make_double2(ar, ai);
        if (power_acc) { double h = hypot(ar, ai); pw += h * h; }
    }
    if (power_acc) {
        __shared__ double red[8];
        double t = block_sum(pw, red);
        if (threadIdx.x == 0) atomicAdd(&power_acc[stream], t);
    }
}

// Decimating FIR straight from the uint8 capture when the windows do not overlap (decim >= n_taps: the /64 coarse
// stream, multi_rtl_sdr_gsm_FCCH_scanner.m:133-135).  One thread per kept output; its 2*n_taps bytes are fetched as
// 8-byte aligned words that are ALL in flight before the first use (the per-sample loop of the staged kernel paid a
// memory latency per iteration), then unpacked and filtered in registers.  The byte phase of a row is the same for
// every output of a stream (2*decim*m is a multiple of 8 for decim % 4 == 0), so tap indices stay warp-uniform.
#define FDD_THREADS 128
template <int MAXW>
__global__ void __launch_bounds__(FDD_THREADS) fir_decim_direct_u8_kernel(const uint8_t *__restrict__ in, i64 n, const StreamCtl *__restrict__ ctl, int n_taps, int decim,
                                                                         double2 *__restrict__ out, i64 n_out, double *__restrict__ power_acc) {
    const int stream = blockIdx.y;
    const uint8_t *raw = in + (i64)stream * 2 * n;
    const double mur = stream_mean(ctl[stream].sum_i, n), mui = stream_mean(ctl[stream].sum_q, n);
    const i64 m = (i64)blockIdx.x * FDD_THREADS + threadIdx.x;
    const int nt1 = n_taps - 1;
    double ar = 0.0, ai = 0.0;
    bool valid = m < n_out;
    if (valid) {
        const i64 j0 = m * decim - nt1;                           // oldest sample of this output's window
        const uintptr_t a = (uintptr_t)(raw + 2 * j0);
        const int off = (int)((a & 7) >> 1);                      // samples between the aligned word and j0 (warp-uniform)
        const int nw = (n_taps + off + 3) >> 2;
        const i64 jw0 = j0 - off;                                 // sample index of the first aligned word
        if (jw0 >= 0 && jw0 + 4 * (i64)nw <= n) {
            const uint2 *wp = reinterpret_cast<const uint2 *>(a & ~(uintptr_t)7);
            uint2 w[MAXW];
#pragma unroll
            for (int q = 0; q < MAXW; ++q) w[q] = (q < nw) ? __ldg(wp + q) : make_uint2(0u, 0u);
#pragma unroll
            for (int q = 0; q < MAXW; ++q) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int t = 4 * q + e - off;                // 0 = oldest sample -> tap nt1 - t
                    if (q < nw && t >= 0 && t <= nt1) {
                        const unsigned pr2 = ((e < 2) ? w[q].x : w[q].y) >> (16 * (e & 1));
                        const double h = c_taps[nt1 - t];
                        ar = fma(h, (double)(pr2 & 0xffu) - mur, ar);
                        ai = fma(h, (double)((pr2 >> 8) & 0xffu) - mui, ai);
                    }
                }
            }
        } else {                                                  // first / last outputs of a row: scalar, zero initial state
            const double2 v = fir_from_raw(raw, m * decim, n_taps, mur, mui);
            ar = v.x; ai = v.y;
        }
        if (out) out[(i64)stream * n_out + m] = make_double2(ar, ai);
    }
    if (power_acc) {
        __shared__ double red[8];
        double pw = 0.0;
        if (valid) { const double h = hypot(ar, ai); pw = h * h; }
        const double t = block_sum(pw, red);
        if (threadIdx.x == 0) atomicAdd(&power_acc[stream], t);
    }
}

// mean(abs(raw2iq(a)).^2) without a filter: scan_band_power_spectrum.m:80-85
__global__ void __launch_bounds__(256) power_u8_kernel(const uint8_t *__restrict__ raw, i64 n_iq, const StreamCtl *__restrict__ ctl, int decim, double *__restrict__ power_acc) {
    __shared__ double red[8];
    const int stream = blockIdx.y;
    const uchar2 *p = reinterpret_cast<const uchar2 *>(raw + (i64)stream * 2 * n_iq);
    const double mur = stream_mean(ctl[stream].sum_i, n_iq), mui = stream_mean(ctl[stream].sum_q, n_iq);
    const i64 n_out = (n_iq + decim - 1) / decim;
    double pw = 0.0;
    for (i64 m = (i64)blockIdx.x * 256 + threadIdx.x; m < n_out; m += (i64)gridDim.x * 256) {
        uchar2 u = p[m * decim];
        double h = hypot((double)u.x - mur, (double)u.y - mui);
        pw += h * h;
    }
    double t = block_sum(pw, red);
    if (threadIdx.x == 0) atomicAdd(&power_acc[stream], t);
}

// ===================================================================================================
// K6 / K7  whole-stream resample (interp1 'linear') and derotation
//          FCCH_fine_correction.m:118-125,163-165; SCH_corr_rate_correction.m:120-128; carrier_correct_post_SCH.m:81-83
// ===================================================================================================
// out[j] = lerp(in, j*(1+e)) * exp(1i*j*dphi).  The phasor is evaluated exactly (fp64 sincos of the rounded
// product, as the reference does) for the first of each thread's DEROT_K samples and advanced by a fixed
// complex step for the others; the error is < 1e-15 per step and the samples stay coalesced.
#define DEROT_K 8
__global__ void __launch_bounds__(256) resample_derotate_kernel(const double2 *__restrict__ in, i64 len_in, double e, int do_interp,
                                                               double dphi, int do_derot, double2 *__restrict__ out, i64 len_out) {
    const i64 blk0 = (i64)blockIdx.x * (256 * DEROT_K);
    const double scale = 1.0 + e;
    double2 ph = make_double2(1.0, 0.0), step = make_double2(1.0, 0.0);
    if (do_derot) {
        double sn, cs;
        sincos((double)(blk0 + threadIdx.x) * dphi, &sn, &cs); ph = make_double2(cs, sn);
        sincos(256.0 * dphi, &sn, &cs); step = make_double2(cs, sn);
    }
#pragma unroll
    for (int k = 0; k < DEROT_K; ++k) {
        i64 j = blk0 + (i64)k * 256 + threadIdx.x;
        if (j < len_out) {
            double2 v;
            if (do_interp) {
                double xq = (double)j * scale;
                i64 i0 = (i64)floor(xq);
                if (i0 > len_in - 1) i0 = len_in - 1;
                i64 i1 = (i0 + 1 > len_in - 1) ? len_in - 1 : i0 + 1;
                v = lerp_ref(in[i0], in[i1], xq - (double)i0);
            } else {
                v = in[j];
            }
            if (do_derot) v = cmul(v, ph);
            __stcs(out + j, v);
        }
        if (do_derot) ph = cmul(ph, step);
    }
}

// ===================================================================================================
// K3  moving-FFT SNR statistic   move_fft_snr_runtime_avg.m:17-28, specific_fft_snr_fix_avg.m:10-20
// ===================================================================================================
// SNR of one fft_len-point window held in w[] (fft_len <= 128): direct DFT with an exact twiddle table.
// FL > 0: compile-time length, powers stay in registers; FL == 0: runtime length.
template <int FL>
__device__ double window_snr_t(const double2 *w, int fft_len_rt, const double2 *tw /* exp(-2*pi*i*j/fft_len) */) {
    const int fft_len = FL > 0 ? FL : fft_len_rt;
    double p[FL > 0 ? FL : 128];
    double2 x[FL > 0 ? FL : 1];
    if (FL > 0) {
#pragma unroll
        for (int n = 0; n < FL; ++n) x[n] = w[n];
    }
    double tot = 0.0, best = -1.0;
    int kbest = 0;
#pragma unroll
    for (int k = 0; k < fft_len; ++k) {
        double xr = 0.0, xi = 0.0;
#pragma unroll
        for (int n = 0; n < fft_len; ++n) {
            const double2 t = tw[(k * n) % fft_len];
            const double2 v = FL > 0 ? x[n] : w[n];
            xr += v.x * t.x - v.y * t.y;
            xi += v.x * t.y + v.y * t.x;
        }
        double h = hypot(xr, xi);
        p[k] = h * h;
        tot += p[k];
        if (p[k] > best) { best = p[k]; kbest = k; }             // first maximum
    }
    double sig;
    if (FL > 0) {
        double pm = 0.0, pp = 0.0;
#pragma unroll
        for (int k = 0; k < fft_len; ++k) {
            if (k == (kbest + fft_len - 1) % fft_len) pm = p[k];
            if (k == (kbest + 1) % fft_len) pp = p[k];
        }
        sig = pm + best + pp;
    } else {
        sig = p[(kbest + fft_len - 1) % fft_len] + p[kbest] + p[(kbest + 1) % fft_len];
    }
    double noise = tot - sig;
    return 10.0 * log10(sig / noise);
}
// 16-point window (the reference's case: fft_len = 2^floor(log2(148/8)), FCCH_coarse_position.m:17): radix-4 x radix-4
// FFT in registers, X[k1+4*k2] = sum_{n2} W16^{n2*k1} W4^{n2*k2} sum_{n1} x[4*n1+n2] W4^{n1*k1}.
__device__ __forceinline__ void radix4(double2 a0, double2 a1, double2 a2, double2 a3, double2 &y0, double2 &y1, double2 &y2, double2 &y3) {
    const double2 s02 = make_double2(a0.x + a2.x, a0.y + a2.y), d02 = make_double2(a0.x - a2.x, a0.y - a2.y);
    const double2 s13 = make_double2(a1.x + a3.x, a1.y + a3.y), d13 = make_double2(a1.x - a3.x, a1.y - a3.y);
    y0 = make_double2(s02.x + s13.x, s02.y + s13.y);
    y2 = make_double2(s02.x - s13.x, s02.y - s13.y);
    y1 = make_double2(d02.x + d13.y, d02.y - d13.x);            // d02 - i*d13
    y3 = make_double2(d02.x - d13.y, d02.y + d13.x);            // d02 + i*d13
}
__device__ double window_snr16(const double2 *w) {
    const double C1 = 0.92387953251128673848, S1 = 0.38268343236508978178, R2 = 0.70710678118654752440;
    double2 A[4][4];
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) radix4(w[n2], w[4 + n2], w[8 + n2], w[12 + n2], A[n2][0], A[n2][1], A[n2][2], A[n2][3]);
    // twiddles W16^{n2*k1} = (cos, -sin)(2*pi*n2*k1/16)
    A[1][1] = cmul(A[1][1], make_double2(C1, -S1)); A[1][2] = cmul(A[1][2], make_double2(R2, -R2)); A[1][3] = cmul(A[1][3], make_double2(S1, -C1));
    A[2][1] = cmul(A[2][1], make_double2(R2, -R2)); A[2][2] = make_double2(A[2][2].y, -A[2][2].x); A[2][3] = cmul(A[2][3], make_double2(-R2, -R2));
    A[3][1] = cmul(A[3][1], make_double2(S1, -C1)); A[3][2] = cmul(A[3][2], make_double2(-R2, -R2)); A[3][3] = cmul(A[3][3], make_double2(-C1, S1));
    double p[16];
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) {
        double2 y0, y1, y2, y3;
        radix4(A[0][k1], A[1][k1], A[2][k1], A[3][k1], y0, y1, y2, y3);
        p[k1] = fma(y0.x, y0.x, y0.y * y0.y); p[k1 + 4] = fma(y1.x, y1.x, y1.y * y1.y);
        p[k1 + 8] = fma(y2.x, y2.x, y2.y * y2.y); p[k1 + 12] = fma(y3.x, y3.x, y3.y * y3.y);
    }
    double tot = 0.0, best = -1.0; int kbest = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) { tot += p[k]; if (p[k] > best) { best = p[k]; kbest = k; } }   // first maximum
    double pm = 0.0, pp = 0.0;
#pragma unroll
    for (int k = 0; k < 16; ++k) { if (k == ((kbest + 15) & 15)) pm = p[k]; if (k == ((kbest + 1) & 15)) pp = p[k]; }
    const double sig = pm + best + pp;
    return 10.0 * log10(sig / (tot - sig));
}
__device__ __forceinline__ double window_snr(const double2 *w, int fft_len, const double2 *tw) {
    return (fft_len == 16) ? window_snr16(w) : window_snr_t<0>(w, fft_len, tw);
}

// SNR of windows [w0, w0+n_win) (0-based window starts) of each stream -> snr[stream][0..n_win)
#define SNR_THREADS 128
__global__ void __launch_bounds__(SNR_THREADS) snr_map_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, i64 w0, i64 n_win, int fft_len,
                                                             double *__restrict__ snr, i64 snr_stride) {
    extern __shared__ double2 sm[];
    double2 *tw = sm;                       // fft_len
    double2 *buf = sm + fft_len;            // SNR_THREADS + fft_len - 1 samples
    const int stream = blockIdx.y;
    const i64 b0 = (i64)blockIdx.x * SNR_THREADS;
    if (b0 >= n_win) return;
    for (int j = threadIdx.x; j < fft_len; j += SNR_THREADS) {
        double sn, cs; sincospi(-2.0 * (double)j / (double)fft_len, &sn, &cs);
        tw[j] = make_double2(cs, sn);
    }
    i64 rem = n_win - b0;
    const int nw = rem < SNR_THREADS ? (int)rem : SNR_THREADS;
    const int ns = nw + fft_len - 1;
    StreamCtl c = ctl[stream];
    for (int i = threadIdx.x; i < ns; i += SNR_THREADS) buf[i] = coarse_sample(src, c, stream, w0 + b0 + i);
    __syncthreads();
    if (threadIdx.x < nw) snr[(i64)stream * snr_stride + b0 + threadIdx.x] = window_snr(buf + threadIdx.x, fft_len, tw);
}

// sequential first-hit scan, one warp per stream
//   move_fft_snr_runtime_avg.m:11-12,30-41 (sum_snr updated as "subtract oldest, add newest", FIFO seeded with 999).
// Until the first hit every window is pushed, so the running sum S_i seen by window i does not depend on any decision:
// all lanes replay the two-add recurrence for 32 windows (same order of operations as the reference), lane k keeps
// S_k, and the 32 threshold tests (with their divisions) are then evaluated in parallel; the first set lane wins.
__global__ void first_hit_scan_kernel(const double *__restrict__ snr, i64 snr_stride, i64 n_win, int mv_len, double th, StreamCtl *ctl, int n_streams) {
    const int stream = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (stream >= n_streams) return;
    const double *s = snr + (i64)stream * snr_stride;
    double sum_snr = 999.0 * (double)mv_len;
    int hit = -1; double hit_snr = 0.0, hit_avg = 0.0;
    for (i64 c0 = 0; c0 < n_win && hit < 0; c0 += 32) {
        const i64 i = c0 + lane;
        const double cur = (i < n_win) ? s[i] : 0.0;
        const double old = (i < n_win) ? ((i >= mv_len) ? s[i - mv_len] : 999.0) : 0.0;
        double mine = 0.0;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            const double v = __shfl_sync(0xffffffffu, cur, k);
            const double o = __shfl_sync(0xffffffffu, old, k);
            if (lane == k) mine = sum_snr;
            sum_snr = sum_snr - o;
            sum_snr = sum_snr + v;
        }
        const double peak_to_avg = cur - (mine / (double)mv_len);
        const unsigned mask = __ballot_sync(0xffffffffu, (i < n_win) && (peak_to_avg > th));
        if (mask) {
            const int l = __ffs(mask) - 1;
            hit = (int)(c0 + l) + 1;
            hit_snr = __shfl_sync(0xffffffffu, cur, l);
            hit_avg = hit_snr - __shfl_sync(0xffffffffu, peak_to_avg, l);
        }
    }
    if (lane == 0) {
        ctl[stream].first_hit = hit;
        ctl[stream].hit_snr = hit_snr;
        ctl[stream].hit_avg_snr = hit_avg;
    }
}

// specific_fft_snr_fix_avg.m:10-29 for one stream (drop-in entry point): first window in [t0,t1] over threshold
__global__ void specific_hit_kernel(const double *__restrict__ snr, i64 n, double th, double avg, int *hit_off, double *hit_snr) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        *hit_off = -1;
        for (i64 i = 0; i < n; ++i)
            if (snr[i] - avg > th) { *hit_off = (int)i; *hit_snr = snr[i]; break; }
    }
}

// ===================================================================================================
// K4  burst chain  FCCH_coarse_position.m:32-91 - one warp per stream, 11 candidate windows per step
// ===================================================================================================
#define CHAIN_THREADS 64
#define PF_BYTES 5120              // raw bytes one prefetched candidate range may hold ((2*5+2*5+16+3)*64+46 samples at dec 64 = 5084 B + alignment)
#define PF_STRIDE (PF_BYTES + PF_BYTES / 8 + 32)   // with one 16-byte pad per 128 bytes (bank spreading for the 128-byte window stride)
#define PF_RANGES 2                // candidate ranges per step: after a 10-frame step, after an 11-frame step
// 112 registers and 24 KB: three chains fit into the registers and shared memory one retiring FP64 block (56 x 256 registers, 40-50 KB)
// frees, so the high-priority chains of batch k+1 displace a third fewer blocks of batch k's burst kernels
__global__ void __maxnreg__(112) coarse_chain_kernel(WinSrc src, StreamCtl *ctl, i64 len, int fft_len, double th, int step10, int step11,
                                                                    int dr, int cap, double *__restrict__ position, double *__restrict__ snr_out,
                                                                    unsigned long long *__restrict__ prof) {
    // debug key 13: thread 0 adds the cycles between the marks of a step to prof[phase], prof[7] counts steps, prof[6] blocks
    long long t_prev = prof ? clock64() : 0;
#define CH_MARK(ph) do { if (prof && threadIdx.x == 0) { const long long t_now = clock64(); atomicAdd(prof + (ph), (unsigned long long)(t_now - t_prev)); t_prev = t_now; } } while (0)
    // Each step evaluates the 11 windows around the 10-frame prediction (:47-58) AND the 11 around the 11-frame
    // prediction (:65-76) at once; the second set is only consulted when the first has no hit, as in the reference.
    // Lazy source: the raw bytes a step can touch are prefetched one step ahead into a double-buffered shared-memory ring with
    // cp.async, then every decimated sample is a FIR over shared memory.  The footprint (26 KB, 64 threads) lets 7 blocks share an
    // SM, so the dependent chains of 1024 streams run side by side instead of in waves.
    extern __shared__ double2 chain_sm[];                        // tw[fft_len] | buf[2][2*5 + fft_len]
    __shared__ int sh_hit; __shared__ double sh_snr;
    __shared__ __align__(16) unsigned char pf_buf[2 * PF_RANGES * PF_STRIDE];
    __shared__ i64 pf_lo[2][PF_RANGES], pf_hi[2][PF_RANGES];
    const int stream = blockIdx.x, tid = threadIdx.x;
    const int max_offset = 5;
    const int n_cand = 2 * max_offset + 1;
    const int ns = 2 * max_offset + fft_len;
    double2 *tw = chain_sm, *buf0 = chain_sm + fft_len, *buf1 = buf0 + ns;
    if (tid < 2 * PF_RANGES) { pf_lo[tid / PF_RANGES][tid % PF_RANGES] = 0; pf_hi[tid / PF_RANGES][tid % PF_RANGES] = 0; }
    int step_no = 0;
    StreamCtl c = ctl[stream];
    double *pos_o = position + (i64)stream * cap;
    double *snr_o = snr_out + (i64)stream * cap;
    if (c.first_hit < 0) {
        if (tid == 0) ctl[stream].n_coarse = -1;
        return;
    }
    for (int j = tid; j < fft_len; j += CHAIN_THREADS) {
        double sn, cs; sincospi(-2.0 * (double)j / (double)fft_len, &sn, &cs);
        tw[j] = make_double2(cs, sn);
    }
    const i64 limit = (len - (fft_len - 1)) - max_offset;
    const int dec = src.dec, nt1 = src.n_taps - 1;
    const uint8_t *raw = src.raw + (i64)stream * 2 * src.n_iq;
    const double mur = c.mu_re, mui = c.mu_im;
    // prefetch of the raw bytes around two window centres (decimated indices) into ring slot `slot`
    auto prefetch = [&](int slot, i64 cen0, i64 cen1) {
        const i64 centers[PF_RANGES] = {cen0, cen1};
#pragma unroll
        for (int q = 0; q < PF_RANGES; ++q) {
            const i64 lo = (centers[q] - 2 * max_offset - 2) * (i64)dec - nt1, hi = (centers[q] + 2 * max_offset + fft_len + 1) * (i64)dec;
            const bool okr = lo >= 8 && hi + 8 < src.n_iq && (hi - lo) * 2 + 32 <= PF_BYTES;
            const uintptr_t a0 = ((uintptr_t)(raw + 2 * lo)) & ~(uintptr_t)15;
            const int nchunk = okr ? (int)(((uintptr_t)(raw + 2 * hi) - a0 + 15) >> 4) : 0;
            unsigned char *dstb = pf_buf + (slot * PF_RANGES + q) * PF_STRIDE;
            for (int ch = tid; ch < nchunk; ch += CHAIN_THREADS) {
                const unsigned sa = (unsigned)__cvta_generic_to_shared(dstb + 16 * ch + 16 * (ch >> 3));
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(a0 + 16 * (uintptr_t)ch));
            }
            if (tid == 0) {
                pf_lo[slot][q] = okr ? (i64)(((const uint8_t *)a0 - raw) / 2) : 0;      // sample index of byte 0 (a0 >= raw, even offset)
                pf_hi[slot][q] = okr ? pf_lo[slot][q] + 8 * (i64)nchunk : 0;            // exclusive
            }
        }
        asm volatile("cp.async.commit_group;");
    };
    i64 pos = c.first_hit;
    int count = 1;
    if (tid == 0) { pos_o[0] = (double)((pos - 1) * dr + 1); snr_o[0] = c.hit_snr; }
    __syncthreads();
    if (src.lazy) prefetch(0, pos + step10, pos + step11);       // what the first step reads
    while (count < cap) {
        const i64 nextA = pos + step10, nextB = pos + step11;
        if (nextA > limit) break;                                // run out of sampled signal (:49-51)
        const bool b_ok = nextB <= limit;                        // (:67-69)
        __syncthreads();
        // ---- what the FOLLOWING step can touch: its windows sit within +-5 of the 10-frame successor of a group-A hit, or of
        //      pos + 10 + 11 frames (an A hit followed by an 11-frame step, or a B hit followed by a 10-frame step). ----
        const int cur = step_no & 1, nxt = cur ^ 1;
        if (src.lazy) {
            prefetch(nxt, nextA + step10, nextA + step11);
            asm volatile("cp.async.wait_group 1;");              // everything except the group just committed has landed
        }
        __syncthreads();
        // which prefetched range serves this step's groups?
        int srcA = -1, srcB = -1;
        if (src.lazy) {
            const i64 needA0 = (nextA - max_offset - 1) * (i64)dec - nt1, needA1 = (nextA + max_offset + fft_len - 1) * (i64)dec;
            const i64 needB0 = (nextB - max_offset - 1) * (i64)dec - nt1, needB1 = (nextB + max_offset + fft_len - 1) * (i64)dec;
            for (int q = 0; q < PF_RANGES; ++q) {
                if (srcA < 0 && pf_hi[cur][q] > 0 && needA0 >= pf_lo[cur][q] && needA1 <= pf_hi[cur][q]) srcA = q;
                if (srcB < 0 && pf_hi[cur][q] > 0 && needB0 >= pf_lo[cur][q] && needB1 <= pf_hi[cur][q]) srcB = q;
            }
        }
        const bool fast = src.lazy && srcA >= 0 && (srcB >= 0 || !b_ok);
        ++step_no;
        CH_MARK(0);                                              // prefetch issue, wait for the previous one, range lookup
        if (fast) {
            for (int i = tid; i < 2 * ns; i += CHAIN_THREADS) {
                const int g = i / ns, r = i % ns;
                if (g == 1 && !b_ok) continue;
                const int q = g == 0 ? srcA : srcB;
                const unsigned char *pb = pf_buf + (cur * PF_RANGES + q) * PF_STRIDE;
                const i64 s0 = ((g == 0 ? nextA : nextB) - max_offset - 1 + r) * (i64)dec - nt1;   // oldest raw sample of this decimated sample
                int bo = (int)(2 * (s0 - pf_lo[cur][q]));                                            // byte offset (unpadded)
                double ar = 0.0, ai = 0.0;
                for (int k = nt1; k >= 0; --k, bo += 2) {        // oldest tap first
                    const unsigned u = *reinterpret_cast<const unsigned short *>(pb + bo + 16 * (bo >> 7));
                    ar = fma(c_taps[k], u8_to_f64(u & 0xffu) - mur, ar);
                    ai = fma(c_taps[k], u8_to_f64(u >> 8) - mui, ai);
                }
                (g == 0 ? buf0 : buf1)[r] = make_double2(ar, ai);
            }
        } else {                                                 // first samples / last samples of a capture, materialised source
            for (int i = tid; i < 2 * ns; i += CHAIN_THREADS) {
                const int g = i / ns, r = i % ns;
                if (g == 0 || b_ok) (g == 0 ? buf0 : buf1)[r] = coarse_sample(src, c, stream, (g == 0 ? nextA : nextB) - max_offset - 1 + r);
            }
        }
        __syncthreads();
        CH_MARK(fast ? 1 : 2);                                   // the 2 x 26 decimated samples (FIR over the prefetched bytes / slow path)
        if (tid < 32) {
            double v = 0.0; bool h = false;
            const int g = tid / n_cand, r = tid % n_cand;
            if (tid < 2 * n_cand && (g == 0 || b_ok)) { v = window_snr((g == 0 ? buf0 : buf1) + r, fft_len, tw); h = (v - c.hit_avg_snr) > th; }
            CH_MARK(4);                                          // (inside phase 3) the window SNRs alone
            const unsigned mask = __ballot_sync(0xffffffffu, h);
            const unsigned mA = mask & ((1u << n_cand) - 1), mB = (mask >> n_cand) & ((1u << n_cand) - 1);
            int l = -1;
            if (mA) l = __ffs(mA) - 1; else if (mB) l = n_cand + __ffs(mB) - 1;
            const double hv = __shfl_sync(0xffffffffu, v, l < 0 ? 0 : l);
            if (tid == 0) { sh_hit = l; sh_snr = hv; }
        }
        __syncthreads();
        CH_MARK(3);                                              // 22 window SNRs, first hit
        if (prof && tid == 0) atomicAdd(prof + 7, 1ull);
        const int l = sh_hit;
        if (l < 0) break;
        pos = (l < n_cand) ? nextA - max_offset + l : nextB - max_offset + (l - n_cand);
        if (tid == 0) { pos_o[count] = (double)((pos - 1) * dr + 1); snr_o[count] = sh_snr; }
        ++count;
    }
    asm volatile("cp.async.wait_group 0;");                      // no copy may still be in flight when the block retires
    if (prof && tid == 0) atomicAdd(prof + 6, 1ull);
    if (tid == 0) ctl[stream].n_coarse = count;
}

// ===================================================================================================
// K5  fine FCCH position  FCCH_fine_correction.m:32-64
// ===================================================================================================
// One block per (burst, stream).  All n_win sliding windows' max-bin power by a sliding DFT:
//   X_{m+1}[k] = (X_m[k] - s[m] + s[m+N]) * exp(+2*pi*i*k/N)
// each thread owns FP_BPT bins in registers and remembers the first window where its bins peak; the block
// then takes the first-maximum over bins.  (max_m max_k == max_k max_m, and the first window attaining the
// global maximum is the same either way, so no per-window reduction is needed.)
#define FP_BPT 4
#define FALL_GRID 256     // bursts tier 3 (multi-block band search) handles per launch; beyond that this single-block kernel takes over
__device__ void fine_peak_full_body(const WinSrc &src, StreamCtl *__restrict__ ctl, const double *__restrict__ base_pos, int cap,
                                    int osr, i64 len_s_ov, const double2 *__restrict__ tw /* exp(-2*pi*i*j/N) */,
                                    double *__restrict__ fine_raw, bool listed, int burst, int stream, double2 *sm, double *red_v, int *red_i) {
    const StreamCtl c = ctl[stream];
    if (c.n_coarse < 5 || burst >= c.n_coarse) return;
    const int N = 148 * osr;
    const int max_offset = 64;
    const int n_win = 2 * max_offset * osr + 1;
    const int n_smp = n_win + N - 1;
    const i64 len_s = len_s_ov / osr;
    const i64 position = (i64)base_pos[(i64)stream * cap + burst];
    double *o = fine_raw + (i64)stream * cap + burst;
    if (position + max_offset > len_s - 148 + 1) {            // run out of sampled signal (:35-38)
        if (threadIdx.x == 0) *o = INFINITY;
        return;
    }
    if (listed && threadIdx.x == 0) atomicOr(&ctl[stream].flags, 32);
    const i64 sp = (position - max_offset - 1) * osr + 1;     // 1-based
    double2 *win = sm;
    double2 *X = win + n_smp;
    double2 *Y = X + GSMCAL_XCAP(n_smp);
    load_window(src, c, stream, sp - 1, n_smp, win, X, Y);

    double xr[FP_BPT], xi[FP_BPT], wr[FP_BPT], wi[FP_BPT], best[FP_BPT];
    int bestm[FP_BPT];
    const int T = blockDim.x;
#pragma unroll
    for (int b = 0; b < FP_BPT; ++b) {
        const int k = threadIdx.x + b * T;
        xr[b] = 0.0; xi[b] = 0.0; best[b] = -1.0; bestm[b] = 0;
        double2 w = (k < N) ? tw[k] : make_double2(1.0, 0.0);
        wr[b] = w.x; wi[b] = -w.y;                               // exp(+2*pi*i*k/N)
    }
    // X_0[k] by direct DFT
    {
        int idx[FP_BPT];
#pragma unroll
        for (int b = 0; b < FP_BPT; ++b) idx[b] = 0;
        for (int n = 0; n < N; ++n) {
            const double2 s = win[n];
#pragma unroll
            for (int b = 0; b < FP_BPT; ++b) {
                const int k = threadIdx.x + b * T;
                if (k < N) {
                    const double2 t = tw[idx[b]];
                    xr[b] = fma(s.x, t.x, fma(-s.y, t.y, xr[b]));
                    xi[b] = fma(s.x, t.y, fma(s.y, t.x, xi[b]));
                    idx[b] += k; if (idx[b] >= N) idx[b] -= N;
                }
            }
        }
    }
    for (int m = 0; m < n_win; ++m) {
#pragma unroll
        for (int b = 0; b < FP_BPT; ++b) {
            const double p = fma(xr[b], xr[b], xi[b] * xi[b]);
            if (p > best[b]) { best[b] = p; bestm[b] = m; }
        }
        if (m + 1 < n_win) {
            const double2 s_old = win[m], s_new = win[m + N];
            const double dr_ = s_new.x - s_old.x, di_ = s_new.y - s_old.y;
#pragma unroll
            for (int b = 0; b < FP_BPT; ++b) {
                const double tr = xr[b] + dr_, ti = xi[b] + di_;
                xr[b] = fma(tr, wr[b], -(ti * wi[b]));
                xi[b] = fma(tr, wi[b], ti * wr[b]);
            }
        }
    }
    double v = -1.0; int mi = 0x7fffffff;
#pragma unroll
    for (int b = 0; b < FP_BPT; ++b) {
        const int k = threadIdx.x + b * T;
        if (k < N) argmax_combine(v, mi, best[b], bestm[b]);
    }
    block_argmax(v, mi, red_v, red_i);
    if (threadIdx.x == 0) *o = (double)(sp + mi);              // sp + max_idx - 1, max_idx = mi + 1
}

// direct mode (fall_list == nullptr): grid (cap, streams), every burst - the drop-in / forced path and the tiers' test oracle.
// list mode: a small grid walks the tier-3 work list, and only when it is longer than the multi-block tier handles.
__global__ void __launch_bounds__(320) fine_peak_full_kernel(WinSrc src, StreamCtl *__restrict__ ctl, const double *__restrict__ base_pos, int cap,
                                                             int osr, i64 len_s_ov, const double2 *__restrict__ tw,
                                                             double *__restrict__ fine_raw, const int *__restrict__ fall_list,
                                                             const int *__restrict__ fall_count, int fall_limit) {
    extern __shared__ double2 sm[];
    __shared__ double red_v[16];
    __shared__ int red_i[16];
    if (!fall_list) {
        fine_peak_full_body(src, ctl, base_pos, cap, osr, len_s_ov, tw, fine_raw, false, blockIdx.x, blockIdx.y, sm, red_v, red_i);
        return;
    }
    const int cnt = *fall_count;
    if (cnt <= fall_limit) return;
    for (int wi = blockIdx.x; wi < cnt; wi += gridDim.x) {
        const int id = fall_list[wi];
        __syncthreads();
        fine_peak_full_body(src, ctl, base_pos, cap, osr, len_s_ov, tw, fine_raw, true, id % cap, id / cap, sm, red_v, red_i);
    }
}

// ---------------------------------------------------------------------------------------------------
// K5, fast path: the same argmax from a 64-bin band around the FCCH tone, with a proof that no other bin
// can matter.  For every window m the reference takes max_k |X_m[k]|^2 over ALL N bins; here
//   * the band S = [k0-48, k0+16) (k0 from a phase-slope estimate of the centre window; the GMSK data
//     energy sits ~37 bins below the tone, hence the asymmetry) is tracked exactly by the sliding DFT,
//   * every 16th window c is "certified": by Parseval sum_{k not in S} |X_c[k]|^2 = N*E_c - sum_{k in S} |X_c[k]|^2
//     =: R_c bounds every out-of-band bin, and since |X_{m+1}[k]| <= |X_m[k]| + |s[m]| + |s[m+N]| the bound
//     sqrt(R_c) + sum_{i=c}^{c+14} (|s[i]|+|s[i+N]|) holds for windows c..c+15.
// If that bound squared stays below the best in-band power G for all windows, no out-of-band bin reaches G,
// so the first window attaining the maximum - the reference's answer - is the in-band one.  Otherwise the
// burst is flagged and fine_peak_full_kernel recomputes it over all bins.  Work drops ~18x.
#define FB_BINS 64
#define FB_SEGS 4
#define FB_THREADS (FB_BINS * FB_SEGS)
#define FB_LO 48
#define FB_CERT 16
// Fallback kernels behind a `need` mask (the bursts an earlier tier could not certify - few or none): a block owns `gsz` consecutive
// bursts of a stream and runs the body for the flagged ones: 1/gsz of the blocks to dispatch, an unflagged group costs one 4-byte load per thread.
__device__ __forceinline__ unsigned group_mask(const int *__restrict__ need, i64 row0, int first, int gsz, int cap) {
    const int lane = threadIdx.x & 31;
    const bool f = lane < gsz && first + lane < cap && (need == nullptr || need[row0 + first + lane] != 0);
    return __ballot_sync(0xffffffffu, f);                        // every warp evaluates the same mask: block-uniform without a barrier
}
__device__ __forceinline__ void fine_peak_band_body(const WinSrc &src, const StreamCtl *__restrict__ ctl, const double *__restrict__ base_pos, int cap,
                                                    int osr, i64 len_s_ov, const double2 *__restrict__ tw, double *__restrict__ fine_raw,
                                                    int *__restrict__ need_full,
                                                    int mode, int *__restrict__ fall_list, int *__restrict__ fall_count,
                                                    double *__restrict__ fall_best, int *__restrict__ fall_m, int force_fail, int burst, int stream) {
    // mode 0 (tier 2): grid (cap, streams); the band sits around the tone and must pass the certificate, otherwise the
    //                  burst is appended to fall_list.
    // mode 1 (tier 3): grid (ceil(N/64), FALL_GRID); block (z, y) searches bins [64z, 64z+64) of the y-th listed burst, no
    //                  certificate needed because the blocks of a burst cover every bin; fine_fall_combine_kernel merges them.
    extern __shared__ double2 sm[];
    __shared__ double red_v[8];
    __shared__ int red_i[8];
    __shared__ double part[2 * (8 * 128 / FB_CERT + 2)];
    __shared__ double scan_sv[16];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const StreamCtl c = ctl[stream];
    if (c.n_coarse < 5 || burst >= c.n_coarse) return;
    const int N = 148 * osr;
    const int max_offset = 64;
    const int n_win = 2 * max_offset * osr + 1;
    const int n_smp = n_win + N - 1;
    const i64 len_s = len_s_ov / osr;
    const i64 position = (i64)base_pos[(i64)stream * cap + burst];
    double *o = fine_raw + (i64)stream * cap + burst;
    if (position + max_offset > len_s - 148 + 1) {            // run out of sampled signal (:35-38)
        if (tid == 0) *o = INFINITY;
        return;
    }
    const i64 sp = (position - max_offset - 1) * osr + 1;
    double2 *win = sm;
    double2 *X = win + n_smp;
    if (src.wcache && osr == 8) {   // tier 1 (fine_core8_kernel) left the filtered window in the cache: no staging, no FIR
        const double2 *wc = src.wcache + ((i64)stream * src.wc_cap + burst) * B8_WLEN;
        for (int i = tid; i < n_smp; i += FB_THREADS) win[i] = wc[B8_WPAD(i)];
        __syncthreads();
    } else {   // level 0: only the staging scratch X is used; three passes keep it small (4 blocks per SM)
        const int part_n = (n_smp + 2) / 3;
        for (int off = 0; off < n_smp; off += part_n)
            load_window(src, c, stream, sp - 1 + off, (n_smp - off < part_n) ? n_smp - off : part_n, win + off, X, X);
    }
    // ---- energy / magnitude sums per 16-sample chunk, prefix over chunks (N and the certified windows are multiples of 16) ----
    const int n_chunk = n_smp / FB_CERT;                        // 138 at osr 8 (n_smp = 16*138)
    double *pe16 = reinterpret_cast<double *>(X + 8 * FB_BINS), *pa16 = pe16 + n_chunk + 2, *pa15 = pa16 + n_chunk + 2;   // behind the piece sums
    if (tid < n_chunk) {
        double se = 0.0, sa = 0.0, sa15 = 0.0;
        for (int i = 0; i < FB_CERT; ++i) {
            const double2 v = win[tid * FB_CERT + i];
            const double e = v.x * v.x + v.y * v.y;
            se += e;
            const double a = sqrt_ub(e);
            sa += a; if (i < FB_CERT - 1) sa15 += a;
        }
        pe16[tid + 1] = se; pa16[tid + 1] = sa; pa15[tid] = sa15;
    }
    if (tid == 0) { pe16[0] = 0.0; pa16[0] = 0.0; }
    __syncthreads();
    // pe16[i] = sum_{n<16i}|s|^2, pa16 likewise (two warps scan in parallel), pa15[i] = sum_{n<16i+15}|s|
    if (warp == 0) warp_scan_smem(pe16, n_chunk + 1, lane);
    if (warp == 1) { warp_scan_smem(pa16, n_chunk + 1, lane); __syncwarp(); for (int i = lane; i < n_chunk; i += 32) pa15[i] += pa16[i]; }
    // ---- band centre from the phase slope of the centre window ----
    const int mc = (n_win - 1) / 2;
    double pq[2] = {0.0, 0.0};
    for (int n = mc + tid; n < mc + N - 1; n += FB_THREADS) {
        const double2 q2 = cmulc(win[n + 1], win[n]);
        pq[0] += q2.x; pq[1] += q2.y;
    }
    block_sum_n<2, false>(pq, scan_sv);
    if (tid == 0) red_i[0] = (int)floor(atan2(pq[1], pq[0]) * (double)N / (2.0 * GSMCAL_PI) + 0.5);     // one atan2 per block
    __syncthreads();
    const int k0 = red_i[0];
    __syncthreads();
    // ---- thread = (segment g of windows, bin j).  Segment-start spectra from shared piece sums (absolute phase):
    //      pieces [0,q) [q,2q) [2q,3q) [3q,4q) [4q,N) [N,N+q) [N+q,N+2q) [N+2q,N+3q); window g*q = pieces g..g+4 ----
    const int g = tid / FB_BINS, j = tid % FB_BINS;
    int k = ((mode == 1 ? FB_BINS * (int)blockIdx.x : k0 - FB_LO) + j) % N; if (k < 0) k += N;
    const int q = (n_win - 1) / FB_SEGS;
    const double2 wk = tw[k];                                    // exp(-2*pi*i*k/N)
    double2 *PS = X;                                             // [8][FB_BINS]
    const double2 wk2 = tw[(2 * k) % N], wk3 = tw[(3 * k) % N], wk4 = tw[(4 * k) % N];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int pc = g + 4 * half;
        const int a = (pc <= 4) ? pc * q : N + (pc - 5) * q;
        const int b = (pc < 4) ? a + q : (pc == 4 ? N : a + q);
        // sample n+r (r<4) carries W^{(n+r)k} = t * W^{rk}: four accumulators share one twiddle, advanced by W^{4k};
        // t is re-seeded exactly from the table every 32 samples
        double a0r = 0.0, a0i = 0.0, a1r = 0.0, a1i = 0.0, a2r = 0.0, a2i = 0.0, a3r = 0.0, a3i = 0.0;
        for (int n0 = a; n0 < b; n0 += 32) {
            double2 t = tw[(int)(((i64)n0 * k) % N)];
            const int n1 = (n0 + 32 < b) ? n0 + 32 : b;
            int n = n0;
            for (; n + 3 < n1; n += 4) {
                const double2 s0 = win[n], s1 = win[n + 1], s2 = win[n + 2], s3 = win[n + 3];
                a0r = fma(s0.x, t.x, fma(-s0.y, t.y, a0r)); a0i = fma(s0.x, t.y, fma(s0.y, t.x, a0i));
                a1r = fma(s1.x, t.x, fma(-s1.y, t.y, a1r)); a1i = fma(s1.x, t.y, fma(s1.y, t.x, a1i));
                a2r = fma(s2.x, t.x, fma(-s2.y, t.y, a2r)); a2i = fma(s2.x, t.y, fma(s2.y, t.x, a2i));
                a3r = fma(s3.x, t.x, fma(-s3.y, t.y, a3r)); a3i = fma(s3.x, t.y, fma(s3.y, t.x, a3i));
                t = cmul(t, wk4);
            }
            if (n < n1)     { const double2 s0 = win[n];     a0r = fma(s0.x, t.x, fma(-s0.y, t.y, a0r)); a0i = fma(s0.x, t.y, fma(s0.y, t.x, a0i)); }
            if (n + 1 < n1) { const double2 s1 = win[n + 1]; a1r = fma(s1.x, t.x, fma(-s1.y, t.y, a1r)); a1i = fma(s1.x, t.y, fma(s1.y, t.x, a1i)); }
            if (n + 2 < n1) { const double2 s2 = win[n + 2]; a2r = fma(s2.x, t.x, fma(-s2.y, t.y, a2r)); a2i = fma(s2.x, t.y, fma(s2.y, t.x, a2i)); }
        }
        const double2 c1 = cmul(make_double2(a1r, a1i), wk), c2 = cmul(make_double2(a2r, a2i), wk2), c3 = cmul(make_double2(a3r, a3i), wk3);
        PS[pc * FB_BINS + j] = make_double2((a0r + c1.x) + (c2.x + c3.x), (a0i + c1.y) + (c2.y + c3.y));
    }
    __syncthreads();
    const int m0 = g * q, m_end = (g == FB_SEGS - 1) ? n_win : m0 + q;
    double xr, xi;
    {
        double yr = 0.0, yi = 0.0;
#pragma unroll
        for (int pc = 0; pc < 5; ++pc) { const double2 v = PS[(g + pc) * FB_BINS + j]; yr += v.x; yi += v.y; }
        const double2 t = tw[(int)(((i64)m0 * k) % N)];          // X_{m0}[k] = Y_{m0}[k] * exp(+2*pi*i*m0*k/N)
        xr = yr * t.x + yi * t.y;
        xi = yi * t.x - yr * t.y;
    }
    // ---- d[m] = s[m+N] - s[m] in place (m < 4q <= N, so the sources s[m+N] are never overwritten) ----
    for (int m = tid; m < n_win - 1; m += FB_THREADS) {
        const double2 s_old = win[m], s_new = win[m + N];
        win[m] = make_double2(s_new.x - s_old.x, s_new.y - s_old.y);
    }
    __syncthreads();
    const double wr = wk.x, wi = -wk.y;                          // exp(+2*pi*i*k/N)
    double best = -1.0; int bestm = 0;
    for (int m = m0; m < m_end; ++m) {
        const double p = fma(xr, xr, xi * xi);
        if (p > best) { best = p; bestm = m; }
        if ((m % FB_CERT) == 0) {
            double s2 = p;
            for (int d = 16; d > 0; d >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, d);
            if (lane == 0) part[2 * (m / FB_CERT) + (warp & 1)] = s2;
        }
        if (m + 1 < m_end) {
            const double2 d = win[m];
            const double tr = xr + d.x, ti = xi + d.y;
            xr = fma(tr, wr, -(ti * wi));
            xi = fma(tr, wi, ti * wr);
        }
    }
    block_argmax(best, bestm, red_v, red_i);                     // also orders the part[] writes before the reads below
    const int n_cert = (n_win - 1) / FB_CERT + 1;
    int ok = 1;
    if (tid < n_cert) {
        const int ci = tid, nc = N / FB_CERT;                    // window c = 16*ci covers samples [16*ci, 16*(ci+nc))
        const double sum_s = part[2 * ci] + part[2 * ci + 1];
        const double R = (double)N * (pe16[ci + nc] - pe16[ci]) - sum_s;
        // windows c..c+15 (only c itself for the last one): slack = sum_{i=c}^{c+14} (|s[i]| + |s[i+N]|)
        const double A = (ci == n_cert - 1) ? 0.0 : (pa15[ci] - pa16[ci]) + (pa15[ci + nc] - pa16[ci + nc]);
        const double bound = sqrt_ub(R > 0.0 ? R : 0.0) + A;
        ok = (bound * bound < best * (1.0 - 1e-6)) ? 1 : 0;
    }
    ok = __syncthreads_and(ok);
    if (tid == 0) {
        if (mode == 1) {
            const int nb3 = (N + FB_BINS - 1) / FB_BINS;
            fall_best[(i64)blockIdx.y * nb3 + blockIdx.x] = best;
            fall_m[(i64)blockIdx.y * nb3 + blockIdx.x] = bestm;
        } else {
            *o = (double)(sp + bestm);
            if (force_fail) ok = 0;                               // test hook: exercise tier 3 on every burst that reaches tier 2
            need_full[(i64)stream * cap + burst] = ok ? 0 : 1;
            if (!ok) fall_list[atomicAdd(fall_count, 1)] = stream * cap + burst;
        }
    }
}
__global__ void __launch_bounds__(FB_THREADS, 4) fine_peak_band_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const double *__restrict__ base_pos, int cap,
                                                                   int osr, i64 len_s_ov, const double2 *__restrict__ tw, double *__restrict__ fine_raw,
                                                                   const int *__restrict__ need_band, int *__restrict__ need_full,
                                                                   int mode, int *__restrict__ fall_list, int *__restrict__ fall_count,
                                                                   double *__restrict__ fall_best, int *__restrict__ fall_m, int force_fail, int gsz /* mode 0: 1..32 */) {
    if (mode == 1) {
        const int cnt = *fall_count;
        if ((int)blockIdx.y >= cnt || cnt > force_fail) return;    // in mode 1 `force_fail` carries the list-length limit of this tier
        const int id = fall_list[blockIdx.y];
        fine_peak_band_body(src, ctl, base_pos, cap, osr, len_s_ov, tw, fine_raw, need_full, mode, fall_list, fall_count, fall_best, fall_m, force_fail, id % cap, id / cap);
        return;
    }
    // mode 0: a block owns gsz consecutive bursts of a stream and searches the ones tier 1 left open (see tone_est_kernel)
    const int stream = blockIdx.y, first = blockIdx.x * gsz;
    unsigned m = group_mask(need_band, (i64)stream * cap, first, gsz, cap);
    while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        fine_peak_band_body(src, ctl, base_pos, cap, osr, len_s_ov, tw, fine_raw, need_full, mode, fall_list, fall_count, fall_best, fall_m, force_fail, first + b, stream);
        if (m) __syncthreads();
    }
}

// merges the per-band results of tier 3: first maximum over all bins = larger power, then earlier window
__global__ void fine_fall_combine_kernel(const int *__restrict__ fall_list, const int *__restrict__ fall_count, const double *__restrict__ fall_best,
                                         const int *__restrict__ fall_m, int nb3, const double *__restrict__ base_pos, int cap, int osr,
                                         double *__restrict__ fine_raw, StreamCtl *ctl, int fall_limit) {
    const int wi = blockIdx.x * blockDim.x + threadIdx.x;
    const int cnt = *fall_count;
    if (wi >= cnt || cnt > fall_limit) return;
    const int id = fall_list[wi];
    double v = -1.0; int m = 0x7fffffff;
    for (int z = 0; z < nb3; ++z) argmax_combine(v, m, fall_best[(i64)wi * nb3 + z], fall_m[(i64)wi * nb3 + z]);
    const i64 position = (i64)base_pos[id];
    const i64 sp = (position - 64 - 1) * osr + 1;
    fine_raw[id] = (double)(sp + m);
    atomicOr(&ctl[id / cap].flags, 32);
}

// ---------------------------------------------------------------------------------------------------
// K5, tier 1: the same search tracking only FC_BINS = 8 bins around the tone, 32 window segments per burst.
// Chunk sums (absolute phase) over 69 chunks of 4*osr samples + a prefix over chunks give every segment-start
// spectrum as a difference of two prefix entries; each thread then slides 4*osr windows.  The Parseval/triangle
// certificate (see fine_peak_band_kernel) is evaluated against these 8 bins; it holds for ~85-90 % of bursts
// (it fails when the tone sits between two bins and the +-64-symbol edge windows hold 43 % GMSK data), the rest
// go to the 64-bin band kernel and, if that cannot prove it either, to the all-bin kernel.
#define FC_BINS 8
#define FC_LO 3
#define FC_THREADS 256
__global__ void __launch_bounds__(FC_THREADS, 4) fine_peak_core_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const double *__restrict__ base_pos, int cap,
                                                                      int osr, i64 len_s_ov, const double2 *__restrict__ tw, double *__restrict__ fine_raw,
                                                                      int *__restrict__ need_band, int force_fail) {
    extern __shared__ double2 sm[];
    __shared__ double red_v[8];
    __shared__ int red_i[8];
    __shared__ double scan_sv[16];
    const int burst = blockIdx.x, stream = blockIdx.y, tid = threadIdx.x;
    const StreamCtl c = ctl[stream];
    if (c.n_coarse < 5 || burst >= c.n_coarse) return;
    const int N = 148 * osr;
    const int max_offset = 64;
    const int n_win = 2 * max_offset * osr + 1;
    const int n_smp = n_win + N - 1;
    const i64 len_s = len_s_ov / osr;
    const i64 position = (i64)base_pos[(i64)stream * cap + burst];
    double *o = fine_raw + (i64)stream * cap + burst;
    if (position + max_offset > len_s - 148 + 1) {            // run out of sampled signal (:35-38)
        if (tid == 0) *o = INFINITY;
        return;
    }
    const i64 sp = (position - max_offset - 1) * osr + 1;
    double2 *win = sm;
    double2 *X = win + n_smp;
    {
        const int part_n = (n_smp + 2) / 3;
        for (int off = 0; off < n_smp; off += part_n)
            load_window(src, c, stream, sp - 1 + off, (n_smp - off < part_n) ? n_smp - off : part_n, win + off, X, X);
    }
    const int CH = 4 * osr;                                     // chunk = segment length; n_smp = 69*CH, N = 37*CH, n_win-1 = 32*CH
    const int n_ch = n_smp / CH, n_seg = (n_win - 1) / CH, wch = N / CH;
    double2 *CS = X;                                             // [FC_BINS][n_ch + 1] prefix of chunk sums (bin-major: the scans read contiguously)
    const int csl = n_ch + 1;
#define CSI(cc, jj) ((jj) * csl + (cc))
    const int n_chunk = n_smp / FB_CERT;
    double *pe16 = reinterpret_cast<double *>(X + (n_ch + 1) * FC_BINS), *pa16 = pe16 + n_chunk + 2, *pa15 = pa16 + n_chunk + 2;
    if (tid < n_chunk) {
        double se = 0.0, sa = 0.0, sa15 = 0.0;
        for (int i = 0; i < FB_CERT; ++i) {
            const double2 v = win[tid * FB_CERT + i];
            const double e = v.x * v.x + v.y * v.y;
            se += e;
            const double a = sqrt_ub(e);
            sa += a; if (i < FB_CERT - 1) sa15 += a;
        }
        pe16[tid + 1] = se; pa16[tid + 1] = sa; pa15[tid] = sa15;
    }
    if (tid == 0) { pe16[0] = 0.0; pa16[0] = 0.0; }
    // band centre from the phase slope of the centre window
    const int mc = (n_win - 1) / 2;
    double pq[2] = {0.0, 0.0};
    for (int n = mc + tid; n < mc + N - 1; n += FC_THREADS) {
        const double2 q2 = cmulc(win[n + 1], win[n]);
        pq[0] += q2.x; pq[1] += q2.y;
    }
    block_sum_n<2, false>(pq, scan_sv);
    if (tid == 0) red_i[0] = (int)floor(atan2(pq[1], pq[0]) * (double)N / (2.0 * GSMCAL_PI) + 0.5);     // one atan2 per block
    __syncthreads();
    const int k0 = red_i[0];
    __syncthreads();
    {
        const int lane = tid & 31, warp = tid >> 5;
        if (warp == 0) warp_scan_smem(pe16, n_chunk + 1, lane);
        if (warp == 1) { warp_scan_smem(pa16, n_chunk + 1, lane); __syncwarp(); for (int i = lane; i < n_chunk; i += 32) pa15[i] += pa16[i]; }
    }
    // Two passes at most.  Pass 0 tracks the 8 bins k0-3 .. k0+4.  If its certificate fails, pass 1 adds k0-7 .. k0-4 and
    // k0+5 .. k0+8 (16 tracked bins in total: their tracked power only tightens every bound) and re-checks; the samples
    // are restored from the in-place differences first.  Whatever still cannot be proven goes to the 64-bin band kernel.
    double *T2 = pa15 + n_chunk + 2 + ((n_chunk & 1) ? 1 : 0);                      // [n_seg+1][8] tracked power of pass 0 per (window, split), behind the prefix arrays
    double g_best = -1.0; int g_bestm = 0x7fffffff;
    int ok = 0;
    for (int pass = 0; pass < 2 && !ok; ++pass) {
        if (pass == 1) {                                         // s[m] = s[m+N] - d[m] for m < n_win-1 (d was stored in place)
            for (int m = tid; m < n_win - 1; m += FC_THREADS) {
                const double2 dd = win[m], s_new = win[m + N];
                win[m] = make_double2(s_new.x - dd.x, s_new.y - dd.y);
            }
            __syncthreads();
        }
        // chunk sums sum_{n in chunk} s[n] W^{n*k}: (chunk, bin) pairs over the block, 4 accumulators per twiddle
        for (int p = tid; p < n_ch * FC_BINS; p += FC_THREADS) {
            const int cidx = p / FC_BINS, j = p % FC_BINS;
            int k = (k0 + ((pass == 0) ? j - FC_LO : (j < 4 ? j - 7 : j + 1))) % N; if (k < 0) k += N;
            const double2 wk = tw[k], wk2 = tw[(2 * k) % N], wk3 = tw[(3 * k) % N], wk4 = tw[(4 * k) % N];
            const int a = cidx * CH;
            double2 t = tw[(int)(((i64)a * k) % N)];
            double a0r = 0.0, a0i = 0.0, a1r = 0.0, a1i = 0.0, a2r = 0.0, a2i = 0.0, a3r = 0.0, a3i = 0.0;
            for (int n = a; n < a + CH; n += 4) {
                const double2 s0 = win[n], s1 = win[n + 1], s2 = win[n + 2], s3 = win[n + 3];
                a0r = fma(s0.x, t.x, fma(-s0.y, t.y, a0r)); a0i = fma(s0.x, t.y, fma(s0.y, t.x, a0i));
                a1r = fma(s1.x, t.x, fma(-s1.y, t.y, a1r)); a1i = fma(s1.x, t.y, fma(s1.y, t.x, a1i));
                a2r = fma(s2.x, t.x, fma(-s2.y, t.y, a2r)); a2i = fma(s2.x, t.y, fma(s2.y, t.x, a2i));
                a3r = fma(s3.x, t.x, fma(-s3.y, t.y, a3r)); a3i = fma(s3.x, t.y, fma(s3.y, t.x, a3i));
                t = cmul(t, wk4);
            }
            const double2 c1 = cmul(make_double2(a1r, a1i), wk), c2 = cmul(make_double2(a2r, a2i), wk2), c3 = cmul(make_double2(a3r, a3i), wk3);
            CS[CSI(cidx + 1, j)] = make_double2((a0r + c1.x) + (c2.x + c3.x), (a0i + c1.y) + (c2.y + c3.y));
        }
        __syncthreads();
        {   // prefix over chunks: warp b scans bin b (lanes own ceil(n_ch/32) consecutive chunks)
            const int lane = tid & 31, bin = tid >> 5;
            if (bin < FC_BINS) {
                const int per = (n_ch + 31) >> 5, b0 = 1 + lane * per;
                double lr = 0.0, li = 0.0;
                for (int i = 0; i < per; ++i) if (b0 + i <= n_ch) { const double2 v = CS[CSI(b0 + i, bin)]; lr += v.x; li += v.y; }
                double ir = lr, ii = li;
                for (int d = 1; d < 32; d <<= 1) {
                    const double tr = __shfl_up_sync(0xffffffffu, ir, d), ti = __shfl_up_sync(0xffffffffu, ii, d);
                    if (lane >= d) { ir += tr; ii += ti; }
                }
                double rr = ir - lr, ri = ii - li;
                for (int i = 0; i < per; ++i) if (b0 + i <= n_ch) { const double2 v = CS[CSI(b0 + i, bin)]; rr += v.x; ri += v.y; CS[CSI(b0 + i, bin)] = make_double2(rr, ri); }
                if (lane == 0) CS[CSI(0, bin)] = make_double2(0.0, 0.0);
            }
        }
        __syncthreads();
        const int g = tid / FC_BINS, j = tid % FC_BINS;
        const bool active = g < n_seg;
        int k = (k0 + ((pass == 0) ? j - FC_LO : (j < 4 ? j - 7 : j + 1))) % N; if (k < 0) k += N;
        const double2 wk = tw[k];
        const int m0 = g * CH, m_end = (g == n_seg - 1) ? n_win : m0 + CH;
        double xr = 0.0, xi = 0.0;
        if (active) {
            const double2 hi = CS[CSI(g + wch, j)], lo = CS[CSI(g, j)];
            const double yr = hi.x - lo.x, yi = hi.y - lo.y;
            const double2 t = tw[(int)(((i64)m0 * k) % N)];      // X_{m0}[k] = Y_{m0}[k] * exp(+2*pi*i*m0*k/N)
            xr = yr * t.x + yi * t.y;
            xi = yi * t.x - yr * t.y;
        }
        for (int m = tid; m < n_win - 1; m += FC_THREADS) {      // d[m] = s[m+N] - s[m] in place
            const double2 s_old = win[m], s_new = win[m + N];
            win[m] = make_double2(s_new.x - s_old.x, s_new.y - s_old.y);
        }
        __syncthreads();
        const double wr = wk.x, wi = -wk.y;
        double best = -1.0; int bestm = 0x7fffffff;
        if (active) {
            for (int m = m0; m < m_end; ++m) {
                const double p = fma(xr, xr, xi * xi);
                if (p > best) { best = p; bestm = m; }
                if (m + 1 < m_end) {
                    const double2 d = win[m];
                    const double tr = xr + d.x, ti = xi + d.y;
                    xr = fma(tr, wr, -(ti * wi));
                    xi = fma(tr, wi, ti * wr);
                }
            }
        }
        block_argmax(best, bestm, red_v, red_i);
        if (pass == 0) { g_best = best; g_bestm = bestm; }
        else if (best > g_best || (best == g_best && bestm < g_bestm)) break;   // the extra bins would move the argmax: leave it to tier 2
        // ---- certificate at every segment-start window c = CH*g (g = 0..n_seg), straight from the chunk prefix table.
        // For any split of the window into a part P1 of d samples and the rest P2, every untracked bin obeys
        //   |X_c[k]| <= |P1[k]| + |P2[k]| <= sqrt(d*E_P1) + sqrt(N*E_P2 - sum_tracked |P2[k']|^2)
        // (Cauchy-Schwarz on P1, Parseval on the zero-padded P2).  Putting the non-FCCH samples of an edge window into P1
        // (d ~ |m* - c|, a few chunk-aligned candidates) is much tighter than Parseval on the whole window, whose bound
        // charges all of the GMSK data energy to a single bin.  d = 0 is the plain Parseval bound. ----
        // threads = (window, candidate split): 8 lanes per window, candidate 0 = plain Parseval, 1..6 = d0-2 .. d0+3 chunks
        ok = 1;
        for (int w0 = 0; w0 <= n_seg; w0 += FC_THREADS / 8) {
            const int gq = w0 + (tid >> 3), cand = tid & 7;
            double bnd = INFINITY;
            if (gq <= n_seg && cand < 7) {
                const int cw = gq * CH, per16 = CH / FB_CERT;
                const bool lead = cw < g_bestm;
                const int dist = lead ? g_bestm - cw : cw - g_bestm;
                const int dch = (cand == 0) ? 0 : (dist + CH - 1) / CH - 3 + cand;
                if (dch == 0 || (cw != g_bestm && dch >= 1 && dch < wch)) {
                    // P1 = first dch chunks (window starts before the burst) or last dch chunks (window runs past it)
                    const int p1a = lead ? gq : gq + wch - dch, p1b = p1a + dch;
                    const int p2a = lead ? gq + dch : gq, p2b = lead ? gq + wch : gq + wch - dch;
                    const double e1 = pe16[p1b * per16] - pe16[p1a * per16], e2 = pe16[p2b * per16] - pe16[p2a * per16];
                    double t2 = (pass == 0) ? 0.0 : T2[gq * 8 + cand];
#pragma unroll
                    for (int jj = 0; jj < FC_BINS; ++jj) {
                        const double2 hi = CS[CSI(p2b, jj)], lo = CS[CSI(p2a, jj)];
                        const double yr = hi.x - lo.x, yi = hi.y - lo.y;
                        t2 += yr * yr + yi * yi;
                    }
                    if (pass == 0) T2[gq * 8 + cand] = t2;
                    const double r2 = (double)N * e2 - t2;
                    bnd = sqrt_ub((double)(dch * CH) * (e1 > 0.0 ? e1 : 0.0)) + sqrt_ub(r2 > 0.0 ? r2 : 0.0);
                }
            }
            bnd = fmin(bnd, __shfl_xor_sync(0xffffffffu, bnd, 1));
            bnd = fmin(bnd, __shfl_xor_sync(0xffffffffu, bnd, 2));
            bnd = fmin(bnd, __shfl_xor_sync(0xffffffffu, bnd, 4));
            if (gq <= n_seg && cand == 0) {
                const int per16 = CH / FB_CERT;
                // windows cw .. cw+CH-1 (only cw itself for the last one): slack = sum_{i=cw}^{cw+CH-2} (|s[i]| + |s[i+N]|)
                const int i16 = gq * per16 + per16 - 1, j16 = (gq + wch) * per16 + per16 - 1;     // pa15[i16] = sum_{n < cw+CH-1} |s|
                const double A = (gq == n_seg) ? 0.0 : (pa15[i16] - pa16[gq * per16]) + (pa15[j16] - pa16[(gq + wch) * per16]);
                const double bound = bnd + A;
                if (!(bound * bound < g_best * (1.0 - 1e-6))) ok = 0;
            }
        }
        ok = __syncthreads_and(ok);
    }
    const int bestm = g_bestm;
    if (tid == 0) {
        *o = (double)(sp + bestm);
        need_band[(i64)stream * cap + burst] = (ok && !force_fail) ? 0 : 1;       // force_fail: test hook, sends every burst to tier 2
    }
#undef CSI
}

// ===================================================================================================
// N = M * 37 point DFT, second factorisation (n = 37*n1 + n2, k = k1 + M*k2):
//   X[k1 + M*k2] = sum_{n2<37} W_37^{n2*k2} * T[n2][k1],   T[n2][k1] = W_N^{n2*k1} * FFT_M(x[37*n1+n2])[k1]
// fft_rows computes T (37 M-point FFTs, Stockham radix-2 when M is a power of two); dft_col then yields any
// single bin in 37 MACs, so a stage that needs few bins (band around the tone, the SNR-gate bins) never pays
// for all N.
// ===================================================================================================
__device__ double2 *fft_rows(const double2 *in, double2 *a, double2 *b, int N, const double2 *__restrict__ tw) {
    const int M = N / 37, T = blockDim.x, tid = threadIdx.x;
    double2 *src = a, *dst = b;
    if ((M & (M - 1)) == 0) {
        const int lm = 31 - __clz(M), half = M / 2;
        __shared__ double2 twm[64];                              // exp(-2*pi*i*j/M), j < M/2 (M <= 128)
        for (int i = tid; i < half; i += T) twm[i] = tw[i * 37];
        for (int i = tid; i < N; i += T) { const int n2 = i >> lm, n1 = i & (M - 1); src[i] = in[37 * n1 + n2]; }
        __syncthreads();
        int tsh = lm - 1;                                        // twiddle index k * (M / (2*Ns)) = k << tsh
        for (int Ns = 1; Ns < M; Ns <<= 1, --tsh) {
            for (int i = tid; i < 37 * half; i += T) {
                const int row = i >> (lm - 1), j = i & (half - 1), k = j & (Ns - 1);
                const double2 x0 = src[row * M + j];
                const double2 x1 = cmul(src[row * M + j + half], twm[k << tsh]);
                const int o = row * M + ((j - k) << 1) + k;
                dst[o] = make_double2(x0.x + x1.x, x0.y + x1.y);
                dst[o + Ns] = make_double2(x0.x - x1.x, x0.y - x1.y);
            }
            __syncthreads();
            double2 *t = src; src = dst; dst = t;
        }
    } else {                                                  // generic M: direct row DFTs
        for (int i = tid; i < N; i += T) {
            const int n2 = i / M, k1 = i % M;
            double ar = 0.0, ai = 0.0;
            int t = 0; const int stp = (37 * k1) % N;
            for (int n1 = 0; n1 < M; ++n1) {
                const double2 x = in[37 * n1 + n2], w = tw[t];
                ar = fma(x.x, w.x, fma(-x.y, w.y, ar));
                ai = fma(x.x, w.y, fma(x.y, w.x, ai));
                t += stp; if (t >= N) t -= N;
            }
            dst[i] = make_double2(ar, ai);
        }
        __syncthreads();
        double2 *t = src; src = dst; dst = t;
    }
    for (int i = tid; i < N; i += T) { const int n2 = i / M, k1 = i - n2 * M; src[i] = cmul(src[i], tw[n2 * k1]); }   // n2*k1 < 37*M = N
    __syncthreads();
    return src;
}
__device__ __forceinline__ double2 dft_col(const double2 *Tm, int k, int N, const double2 *__restrict__ tw) {
    const int M = N / 37, k1 = k % M, k2 = k / M;
    double ar = 0.0, ai = 0.0;
    int t = 0; const int stp = M * k2;                         // < N
#pragma unroll 4
    for (int n2 = 0; n2 < 37; ++n2) {
        const double2 x = Tm[n2 * M + k1], w = tw[t];
        ar = fma(x.x, w.x, fma(-x.y, w.y, ar));
        ai = fma(x.x, w.y, fma(x.y, w.x, ai));
        t += stp; if (t >= N) t -= N;
    }
    return make_double2(ar, ai);
}

// ===================================================================================================
// K8  per-burst tone frequency (+ SNR gate)   FCCH_fine_correction.m:143-155,185-189; carrier_correct_post_SCH.m:58-72
// ===================================================================================================
// The integer bin is the first maximum of the fftshift-ed power spectrum (:148-150).  It is found from a 16-bin
// band around a phase-slope estimate and accepted only if Parseval proves every other bin smaller
// (N*sum|u|^2 - sum_band P < max_band P); otherwise all N bins are evaluated.
#define TONE_THREADS 256
#define TONE_BAND 16
__device__ __forceinline__ void tone_est_body(const WinSrc &src, const StreamCtl *__restrict__ ctl, int which /* 1: fine stage, 2: post-SCH */,
                                              const double *__restrict__ pos, int cap, int osr, const double2 *__restrict__ tw,
                                              double *__restrict__ fo_out, double *__restrict__ gate_out, const int burst, const int stream) {
    extern __shared__ double2 sm[];
    __shared__ double red_v[8];
    __shared__ int red_i[8];
    __shared__ double2 step_sh;
    __shared__ double red_n[80];
    __shared__ int sh_k0;
    __shared__ double sh_pr;
    const int tid = threadIdx.x;
    const StreamCtl c = ctl[stream];
    const int nb = (which == 1) ? (c.tone1_enable ? c.n_fcch : 0) : (c.post_enable ? c.n_post_fcch : 0);
    if (burst >= nb) return;
    const int N = 148 * osr;
    const double sampling_rate = ((1625.0 / 6.0) * 1e3) * (double)osr;
    double2 *u = sm, *A = u + N, *F = A + N;
    double2 *X = A, *Y = X + GSMCAL_XCAP(N);                  // the loader's scratch aliases the FFT work buffers
    const i64 sp = (i64)pos[(i64)stream * cap + burst];
    load_window(src, c, stream, sp - 1, N, u, X, Y, burst);       // burst: level 0 comes from the fine search's window cache when it covers the range
    // energy and phase slope -> band centre
    double epq[3] = {0.0, 0.0, 0.0};
    for (int n = tid; n < N; n += TONE_THREADS) {
        const double2 v = u[n];
        epq[0] = fma(v.x, v.x, fma(v.y, v.y, epq[0]));
        if (n + 1 < N) { const double2 q = cmulc(u[n + 1], v); epq[1] += q.x; epq[2] += q.y; }
    }
    block_sum_n<3>(epq, red_n);
    const double e = epq[0];
    if (tid == 0) sh_k0 = (int)floor(atan2(epq[2], epq[1]) * (double)N / (2.0 * GSMCAL_PI) + 0.5);     // one atan2 per block, not per thread
    __syncthreads();
    const int k0 = sh_k0;
    // band search without an FFT: 16 bins x 16 sample segments, absolute-phase partial DFTs (4 accumulators per twiddle,
    // as in the fine search), summed over the segments through shared memory.
    // shifted index j <-> bin (j + N/2) mod N; first maximum in j order (:149-150)
    double v = -1.0; int j_best = 0x7fffffff; double band_sum = 0.0;
    {
        const int bin = tid & (TONE_BAND - 1), seg = tid / TONE_BAND, n_segs = TONE_THREADS / TONE_BAND;
        int k = (k0 - TONE_BAND / 2 + bin) % N; if (k < 0) k += N;
        const int per = (N + n_segs - 1) / n_segs, na = seg * per, nb2 = (na + per < N) ? na + per : N;
        const double2 wk = tw[k], wk2 = tw[(2 * k) % N], wk3 = tw[(3 * k) % N], wk4 = tw[(4 * k) % N];
        double2 t = tw[(int)(((i64)na * k) % N)];
        double a0r = 0.0, a0i = 0.0, a1r = 0.0, a1i = 0.0, a2r = 0.0, a2i = 0.0, a3r = 0.0, a3i = 0.0;
        int n = na;
        for (; n + 3 < nb2; n += 4) {
            const double2 s0 = u[n], s1 = u[n + 1], s2 = u[n + 2], s3 = u[n + 3];
            a0r = fma(s0.x, t.x, fma(-s0.y, t.y, a0r)); a0i = fma(s0.x, t.y, fma(s0.y, t.x, a0i));
            a1r = fma(s1.x, t.x, fma(-s1.y, t.y, a1r)); a1i = fma(s1.x, t.y, fma(s1.y, t.x, a1i));
            a2r = fma(s2.x, t.x, fma(-s2.y, t.y, a2r)); a2i = fma(s2.x, t.y, fma(s2.y, t.x, a2i));
            a3r = fma(s3.x, t.x, fma(-s3.y, t.y, a3r)); a3i = fma(s3.x, t.y, fma(s3.y, t.x, a3i));
            t = cmul(t, wk4);
        }
        if (n < nb2)     { const double2 s0 = u[n];     a0r = fma(s0.x, t.x, fma(-s0.y, t.y, a0r)); a0i = fma(s0.x, t.y, fma(s0.y, t.x, a0i)); }
        if (n + 1 < nb2) { const double2 s1 = u[n + 1]; a1r = fma(s1.x, t.x, fma(-s1.y, t.y, a1r)); a1i = fma(s1.x, t.y, fma(s1.y, t.x, a1i)); }
        if (n + 2 < nb2) { const double2 s2 = u[n + 2]; a2r = fma(s2.x, t.x, fma(-s2.y, t.y, a2r)); a2i = fma(s2.x, t.y, fma(s2.y, t.x, a2i)); }
        const double2 c1 = cmul(make_double2(a1r, a1i), wk), c2 = cmul(make_double2(a2r, a2i), wk2), c3 = cmul(make_double2(a3r, a3i), wk3);
        A[seg * TONE_BAND + bin] = make_double2((a0r + c1.x) + (c2.x + c3.x), (a0i + c1.y) + (c2.y + c3.y));
        __syncthreads();
        if (tid < TONE_BAND) {
            double xr = 0.0, xi = 0.0;
            for (int sgi = 0; sgi < n_segs; ++sgi) { const double2 q = A[sgi * TONE_BAND + tid]; xr += q.x; xi += q.y; }
            int j = k - N / 2; if (j < 0) j += N;                // here k is the bin of thread (seg 0, bin tid)
            v = abs2_ref(make_double2(xr, xi)); j_best = j; band_sum = v;
        }
    }
    band_sum = block_sum(band_sum, red_v);
    block_argmax(v, j_best, red_v, red_i);
    if (!((double)N * e - band_sum < v * (1.0 - 1e-9))) {     // not certified: every bin through the row FFT (uniform branch)
        const double2 *Tm = fft_rows(u, A, F, N, tw);
        v = -1.0; j_best = 0x7fffffff;
        for (int j = tid; j < N; j += TONE_THREADS) {
            int k = j + N / 2; if (k >= N) k -= N;
            argmax_combine(v, j_best, abs2_ref(dft_col(Tm, k, N, tw)), j);
        }
        block_argmax(v, j_best, red_v, red_i);
    }
    const int jr = j_best + 1 - ((N / 2) + 1);                 // max_idx - (fft_len/2 + 1)
    const double int_phase_rotate = 2.0 * GSMCAL_PI * (double)jr / (double)N;
    // integer-bin derotation exp(-1i*n*int_phase_rotate) == twiddle table entry (n*jr mod N); unit phasors (:152-153)
    int jm = jr % N; if (jm < 0) jm += N;
    int tidx = (int)(((i64)tid * jm) % N);
    const int tinc = (int)(((i64)TONE_THREADS * jm) % N);
    for (int n = tid; n < N; n += TONE_THREADS, tidx = (tidx + tinc >= N) ? tidx + tinc - N : tidx + tinc) {
        const double2 w = cmul(u[n], tw[tidx]);
        u[n] = w;
        const double h2 = fma(w.x, w.x, w.y * w.y);
        const double inv = rsqrt(h2);                            // exp(1i*angle(w)) = w/|w| (samples are O(1..100): no over/underflow)
        A[n] = (h2 > 0.0) ? make_double2(w.x * inv, w.y * inv) : make_double2(1.0, 0.0);
    }
    __syncthreads();
    double rri[2] = {0.0, 0.0};
    for (int n = tid; n < N - 1; n += TONE_THREADS) {
        const double2 a = A[n + 1], b = A[n];                      // a / b with |b| = 1 to 1 ulp: a * conj(b) (the division by |b|^2 changes
        rri[0] += a.x * b.x + a.y * b.y;                           // the mean by < 2e-16 relative and cost a reciprocal per sample)
        rri[1] += a.y * b.x - a.x * b.y;
    }
    block_sum_n<2, false>(rri, red_n);
    if (tid == 0) sh_pr = atan2(rri[1] / (double)(N - 1), rri[0] / (double)(N - 1));
    __syncthreads();
    const double phase_rotate = sh_pr;
    const double fo = sampling_rate * (int_phase_rotate + phase_rotate) / (2 * GSMCAL_PI);
    if (tid == 0) fo_out[(i64)stream * cap + burst] = fo;
    if (which != 1) return;
    // SNR gate (:185-189): fine derotation, then only the bins the gate reads: [1:3,end-1:end] vs [4:hnl, end-hnl+1:end-2]
    if (tid == 0) { double sn, cs; sincos((double)TONE_THREADS * phase_rotate, &sn, &cs); step_sh = make_double2(cs, -sn); }
    __syncthreads();
    double sg[10] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};   // bins 0, +1, -1, +2, -2 of the derotated burst (re, im)
    {
        double sn, cs; sincos((double)tid * phase_rotate, &sn, &cs);
        double2 ph = make_double2(cs, -sn);
        const double2 st = step_sh;
        for (int n = tid; n < N; n += TONE_THREADS) {
            const double2 w = cmul(u[n], ph);
            u[n] = w;
            ph = cmul(ph, st);
            const double2 t1 = tw[n], t2 = tw[(2 * n) % N];
            sg[0] += w.x; sg[1] += w.y;
            sg[2] += w.x * t1.x - w.y * t1.y; sg[3] += w.x * t1.y + w.y * t1.x;      // * W^{n}
            sg[4] += w.x * t1.x + w.y * t1.y; sg[5] += w.y * t1.x - w.x * t1.y;      // * conj(W^{n})
            sg[6] += w.x * t2.x - w.y * t2.y; sg[7] += w.x * t2.y + w.y * t2.x;
            sg[8] += w.x * t2.x + w.y * t2.y; sg[9] += w.y * t2.x - w.x * t2.y;
        }
    }
    block_sum_n<10>(sg, red_n);                                  // also orders the u[] writes before the FFT below
    // Only the DECISION "SNR >= 5 dB" leaves this stage (:192-196).  The five signal bins [1:3, end-1:end] are computed
    // directly; every noise bin is among the other N-5, whose total power is N*E - sig by Parseval (derotation keeps the
    // energy E).  So sig >= 10^0.5 * (N*E - sig) proves the burst passes the gate without any FFT; bursts that cannot be
    // proven this way evaluate the 110 bins exactly.
    {
        double sig5 = 0.0;
#pragma unroll
        for (int q = 0; q < 5; ++q) sig5 += sg[2 * q] * sg[2 * q] + sg[2 * q + 1] * sg[2 * q + 1];
        if (sig5 >= 3.16227766016838 * (1.0 + 1e-9) * ((double)N * e - sig5)) {
            if (tid == 0) gate_out[(i64)stream * cap + burst] = 99.0;      // "certified above the 5 dB gate"
            return;
        }
    }
    const double2 *Tm = fft_rows(u, A, F, N, tw);
    const int hnl = (int)ceil(((double)N * 200e3 / sampling_rate) / 2.0);
    double sn2[2] = {0.0, 0.0};
    for (int i = tid; i < 2 * hnl; i += TONE_THREADS) {
        const int k = (i < hnl) ? i : N - 2 * hnl + i;           // 0..hnl-1 and N-hnl..N-1
        const double p = abs2_ref(dft_col(Tm, k, N, tw));
        if (k < 3 || k >= N - 2) sn2[0] += p; else sn2[1] += p;
    }
    block_sum_n<2, false>(sn2, red_n);
    if (tid == 0) gate_out[(i64)stream * cap + burst] = 10.0 * log10(sn2[0] / sn2[1]);
}
// (group_mask: see fine_peak_band_kernel)
__global__ void __launch_bounds__(TONE_THREADS, 3) tone_est_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, int which, const double *__restrict__ pos, int cap,
                                                               int osr, const double2 *__restrict__ tw, double *__restrict__ fo_out,
                                                               double *__restrict__ gate_out, const int *__restrict__ need, int gsz /* 1..32 */) {
    const int stream = blockIdx.y, first = blockIdx.x * gsz;
    unsigned m = group_mask(need, (i64)stream * cap, first, gsz, cap);
    while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        tone_est_body(src, ctl, which, pos, cap, osr, tw, fo_out, gate_out, first + b, stream);
        if (m) __syncthreads();                                  // the next burst reuses the shared buffers
    }
}

// ===================================================================================================
// K9  SCH training-sequence correlation   SCH_corr_rate_correction.m:37-63
// ===================================================================================================
#define SCH_THREADS 256
#define SCH_LPG 6       // lags per warp and pass of the fp64 correlation
#define SCH_PASSES 2
#define SCH_NSL 16      // template samples per lane
#define SCH_SLPW 12     // lags per warp of the fp32 screen: one pass, 8 x 12 = 96 >= 89
#define SCH_MAXC 8      // candidate lags the screen may leave (one warp each); more -> the full fp64 correlation
#define SCH_NSTAT 9     // counters: [0] bursts that ran the full fp64 correlation, [c] bursts the screen decided with c candidates
// screen bound eps = SCH_EPS_K * 2^-24 * sqrt(E_win * E_tpl) + SCH_EPS_ABS * (1 + sqrt(L * E_tpl) + sqrt(L * E_win)), valid while both
// energies are <= SCH_E_MAX (no fp32 overflow); derivation in DESIGN.md section 4
#define SCH_EPS_K   64.0
#define SCH_EPS_ABS 7.888609052210118e-31       // 2^-100
#define SCH_E_MAX   1.329227995784916e36        // 2^120
__host__ __device__ constexpr int sch_tplf_len(int L) { return L + (L >> 4); }   // float2 entries of the padded fp32 template

// fp64 register-tiled correlation of all n_lag lags into corr / corr_i: per pass warp w owns lags [6(8p+w), +6), lane owns template
// samples [16*lane, 16*lane+16); a 6-deep sliding register window of the burst is advanced one sample per step (2 shared loads per 6
// complex MACs).  wp / tp hold window and template with one pad slot per 16 samples so the 256-byte lane stride is conflict free.  Two
// passes of 6 lags (instead of one of 12) keep the kernel at 64 registers, and the lane partials are folded to 8 lanes by shuffles
// before they go through shared memory (7 KB instead of 50 KB): 4 blocks per SM instead of 2.  Not inlined: next to the screen, the
// 56-register build spilled inside this loop.
__device__ __noinline__ void sch_corr_tiled_fp64(const double2 *wp, const double2 *tp, double *part, double *corr, double *corr_i,
                                                    int n_lag, int n_smp) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = SCH_THREADS >> 5;
    const int nb = SCH_NSL * lane;
#pragma unroll 1
    for (int pass = 0; pass < SCH_PASSES; ++pass) {
        double ar[SCH_LPG], ai[SCH_LPG];
        double2 wr_[SCH_LPG];
#pragma unroll
        for (int l = 0; l < SCH_LPG; ++l) { ar[l] = 0.0; ai[l] = 0.0; }
        const int l0 = SCH_LPG * (pass * nw + w);
#pragma unroll
        for (int l = 0; l < SCH_LPG - 1; ++l) { const int i = l0 + nb + l; wr_[l] = (i < n_smp) ? wp[i + (i >> 4)] : make_double2(0.0, 0.0); }
#pragma unroll
        for (int n = 0; n < SCH_NSL; ++n) {
            const int iw = l0 + nb + n + SCH_LPG - 1, it = nb + n;
            wr_[SCH_LPG - 1] = (iw < n_smp) ? wp[iw + (iw >> 4)] : make_double2(0.0, 0.0);
            const double2 tt = tp[it + (it >> 4)];
#pragma unroll
            for (int l = 0; l < SCH_LPG; ++l) {              // conj(ts) .* window
                ar[l] = fma(wr_[l].x, tt.x, fma(wr_[l].y, tt.y, ar[l]));
                ai[l] = fma(wr_[l].y, tt.x, fma(-wr_[l].x, tt.y, ai[l]));
            }
#pragma unroll
            for (int l = 0; l < SCH_LPG - 1; ++l) wr_[l] = wr_[l + 1];
        }
        // fold 32 lanes to 8 (lanes 0..7 hold the sums of lanes {i, i+8, i+16, i+24}), then rows (lag, re|im) of 9 doubles
#pragma unroll
        for (int l = 0; l < SCH_LPG; ++l) {
            ar[l] += __shfl_down_sync(0xffffffffu, ar[l], 16); ai[l] += __shfl_down_sync(0xffffffffu, ai[l], 16);
            ar[l] += __shfl_down_sync(0xffffffffu, ar[l], 8);  ai[l] += __shfl_down_sync(0xffffffffu, ai[l], 8);
        }
        if (pass > 0) __syncthreads();                       // the rows of the previous pass have been consumed
        if (lane < 8) {
#pragma unroll
            for (int l = 0; l < SCH_LPG; ++l) {
                part[(2 * (SCH_LPG * w + l)) * 9 + lane] = ar[l];
                part[(2 * (SCH_LPG * w + l) + 1) * 9 + lane] = ai[l];
            }
        }
        __syncthreads();
        if (threadIdx.x < 2 * nw * SCH_LPG) {
            const double *row = part + threadIdx.x * 9;
            const double s0 = (row[0] + row[1]) + (row[2] + row[3]), s1 = (row[4] + row[5]) + (row[6] + row[7]);
            const int lag = SCH_LPG * pass * nw + (threadIdx.x >> 1);
            if (lag < n_lag) { if (threadIdx.x & 1) corr_i[lag] = s0 + s1; else corr[lag] = s0 + s1; }
        }
    }
}

// |corr|^2 of ONE lag, evaluated by one warp in sch_corr_tiled_fp64's exact operation order (the same lane chains, the fold by 16 and 8,
// the same row sums, then abs2_ref): the value is bit-identical to the tiled correlation's.  The template comes from global memory (8 KB,
// L2/L1 resident); lane j reads 16 consecutive samples of it.
__device__ __forceinline__ double sch_lag_fp64(const double2 *wp, const double2 *__restrict__ tpl, int lag, int lane) {
    const int nb = SCH_NSL * lane;
    double ar = 0.0, ai = 0.0;
#pragma unroll
    for (int n = 0; n < SCH_NSL; ++n) {
        const int iw = lag + nb + n;
        const double2 x = wp[iw + (iw >> 4)], tt = __ldg(tpl + nb + n);
        ar = fma(x.x, tt.x, fma(x.y, tt.y, ar));
        ai = fma(x.y, tt.x, fma(-x.x, tt.y, ai));
    }
    ar += __shfl_down_sync(0xffffffffu, ar, 16); ai += __shfl_down_sync(0xffffffffu, ai, 16);
    ar += __shfl_down_sync(0xffffffffu, ar, 8);  ai += __shfl_down_sync(0xffffffffu, ai, 8);
    // the row sum ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)) by three more halvings: lane 0 ends with the same value
#pragma unroll
    for (int k = 1; k < 8; k <<= 1) { ar += __shfl_down_sync(0xffffffffu, ar, k); ai += __shfl_down_sync(0xffffffffu, ai, k); }
    return abs2_ref(make_double2(ar, ai));                   // (lane 0's)
}

// tplf: the template in fp32, padded like tp (sch_tplf_len(L) entries); tpl_e: its energy in fp64, rounded up.  mode: 0 = fp32 screen,
// 1 = always the fp64 correlation, 2 = screen, then take the fallback as if it had failed.  stats: SCH_NSTAT counters (see SCH_NSTAT).
// 64 registers: four blocks fill the register file
__global__ void __maxnreg__(64) sch_corr_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, const double *__restrict__ fcch_pos, int cap,
                                                              int osr, const double2 *__restrict__ tpl, const float2 *__restrict__ tplf,
                                                              const double *__restrict__ tpl_e, int mode, unsigned *__restrict__ stats,
                                                              double *__restrict__ sch_raw, int *__restrict__ sch_edge) {
    extern __shared__ double2 sm[];
    __shared__ double red_v[8];
    __shared__ int red_i[8];
    __shared__ double corr[160], corr_i[160];
    __shared__ unsigned cmask[3];
    const int burst = blockIdx.x, stream = blockIdx.y;
    const StreamCtl c = ctl[stream];
    if (!c.sch_enable || burst >= c.n_fcch) return;
    const int L = 64 * osr;
    const int max_offset = 8 * osr;
    const i64 len_s = c.len1;
    const int slot_ov = (625 * osr) / 4;
    const int fix_off = slot_ov * 8 + 42 * osr;
    const i64 training_sp = (i64)fcch_pos[(i64)stream * cap + burst] + fix_off;
    double *o = sch_raw + (i64)stream * cap + burst;
    if (training_sp + max_offset > len_s - L + 1) {            // run out (:40-43)
        if (threadIdx.x == 0) { *o = INFINITY; sch_edge[(i64)stream * cap + burst] = 0; }
        return;
    }
    const i64 sp = training_sp - max_offset;
    const int n_lag = 2 * max_offset - 5 * osr + 1;            // 89 at osr 8
    const int n_smp = n_lag + L - 1;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = SCH_THREADS >> 5;
    // the tiled paths are written for osr 8: L = 32 * SCH_NSL and n_lag = 89 <= SCH_PASSES * nw * SCH_LPG = nw * SCH_SLPW
    const bool tiled = (osr == 8);
    const bool screen = tiled && mode != 1;
    double2 *win = sm, *t = win + n_smp, *X = t + L, *Y = X + GSMCAL_XCAP(n_smp);
    // the template (the fp64 one, 8 KB at osr 8, or the padded fp32 one of the screen, 4.25 KB) is staged by ONE TMA bulk copy
    // (cp.async.bulk -> UBLKCP) that completes on an mbarrier while all threads evaluate the burst window; it is consumed only after the
    // wait below
    __shared__ __align__(8) unsigned long long tpl_bar;
    const unsigned bar_a = (unsigned)__cvta_generic_to_shared(&tpl_bar);
    const void *tsrc = screen ? (const void *)tplf : (const void *)tpl;
    const unsigned tbytes = screen ? (unsigned)(sch_tplf_len(L) * sizeof(float2)) : (unsigned)(L * sizeof(double2));
    const bool tma_ok = (((uintptr_t)tsrc & 15) == 0) && (((uintptr_t)t & 15) == 0) && ((tbytes & 15) == 0);
    if (tma_ok) {
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
            asm volatile("fence.mbarrier_init.release.cluster;");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(tbytes));
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"((unsigned)__cvta_generic_to_shared(t)), "l"(tsrc), "r"(tbytes), "r"(bar_a) : "memory");
        }
    } else if (screen) {
        for (int i = threadIdx.x; i < sch_tplf_len(L); i += SCH_THREADS) reinterpret_cast<float2 *>(t)[i] = tplf[i];
    } else {
        for (int i = threadIdx.x; i < L; i += SCH_THREADS) t[i] = tpl[i];
    }
    load_window(src, c, stream, sp - 1, n_smp, win, X, Y);
    if (tma_ok) {                                                // phase 0 of the barrier: spin until the bulk copy has landed
        unsigned done = 0;
        while (!done) {
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(bar_a), "r"(0u) : "memory");
        }
    }
    if (tiled) {
        double2 *wp = X, *tp = X + (n_smp + (n_smp >> 4) + 2);      // X and Y are contiguous: 924 + 608 slots >= 640 + 544
        double *part = reinterpret_cast<double *>(tp + (L + (L >> 4) + 2));      // [2 * nw * SCH_LPG][9]
        if (screen) {
            // fp32 screen.  Only the index of the first maximum of |corr|^2 leaves the kernel, so every lag is correlated in fp32 and
            // the bound eps >= |screened corr - fp64 corr| (DESIGN.md section 4) rules out the lags that cannot hold the maximum; the
            // few that can are evaluated in fp64 exactly as the tiled correlation does, so the index is the one it would give.
            float2 *wf = reinterpret_cast<float2 *>(tp);            // the fp64 template is not staged: its slots hold the fp32 window
            float *part_f = reinterpret_cast<float *>(wf + (n_smp + (n_smp >> 4) + 2));  // [2 * nw * SCH_SLPW][9]
            const float2 *tf = reinterpret_cast<const float2 *>(t);
            double e = 0.0;
            for (int i = threadIdx.x; i < n_smp; i += SCH_THREADS) {
                const double2 v = win[i];
                wp[i + (i >> 4)] = v;
                wf[i + (i >> 4)] = make_float2((float)v.x, (float)v.y);
                e = fma(v.x, v.x, fma(v.y, v.y, e));
            }
            const double e_win = block_sum(e, red_v) * (1.0 + 1e-12);   // its barriers also publish wp / wf; rounded up
            const double e_tpl = *tpl_e;
            const bool bounded = e_win <= SCH_E_MAX && e_tpl <= SCH_E_MAX;         // false for inf / NaN too
            const double eps = SCH_EPS_K * 5.9604644775390625e-8 * sqrt(e_win * e_tpl) * (1.0 + 1e-12)
                             + SCH_EPS_ABS * (1.0 + sqrt((double)L * e_tpl) + sqrt((double)L * e_win));
            if (bounded) {
                // warp w owns lags [SLPW*w, +SLPW), lane owns template samples [16*lane, +16); an SLPW-deep sliding register
                // window of the burst advances one sample per step: 2 LDS.64 (2 wavefronts each, conflict free with the pad) per 4*SLPW
                // FFMA.  One pass of 12 lags at 64 registers
                constexpr int SLPW = SCH_SLPW;
                const int nb = SCH_NSL * lane;
                const int l0 = SLPW * w;
                float ar[SLPW], ai[SLPW];
                float2 wr_[SLPW];
#pragma unroll
                for (int l = 0; l < SLPW; ++l) { ar[l] = 0.0f; ai[l] = 0.0f; }
#pragma unroll
                for (int l = 0; l < SLPW - 1; ++l) { const int i = l0 + nb + l; wr_[l] = (i < n_smp) ? wf[i + (i >> 4)] : make_float2(0.0f, 0.0f); }
#pragma unroll
                for (int n = 0; n < SCH_NSL; ++n) {
                    const int iw = l0 + nb + n + SLPW - 1, it = nb + n;
                    wr_[SLPW - 1] = (iw < n_smp) ? wf[iw + (iw >> 4)] : make_float2(0.0f, 0.0f);
                    const float2 tt = tf[it + (it >> 4)];
#pragma unroll
                    for (int l = 0; l < SLPW; ++l) {
                        ar[l] = fmaf(wr_[l].x, tt.x, fmaf(wr_[l].y, tt.y, ar[l]));
                        ai[l] = fmaf(wr_[l].y, tt.x, fmaf(-wr_[l].x, tt.y, ai[l]));
                    }
#pragma unroll
                    for (int l = 0; l < SLPW - 1; ++l) wr_[l] = wr_[l + 1];
                }
#pragma unroll
                for (int l = 0; l < SLPW; ++l) {
                    ar[l] += __shfl_down_sync(0xffffffffu, ar[l], 16); ai[l] += __shfl_down_sync(0xffffffffu, ai[l], 16);
                    ar[l] += __shfl_down_sync(0xffffffffu, ar[l], 8);  ai[l] += __shfl_down_sync(0xffffffffu, ai[l], 8);
                }
                if (lane < 8) {                                 // rows (lag, re|im) of 9 floats, every lag of the burst
#pragma unroll
                    for (int l = 0; l < SLPW; ++l) {
                        part_f[(2 * (l0 + l)) * 9 + lane] = ar[l];
                        part_f[(2 * (l0 + l) + 1) * 9 + lane] = ai[l];
                    }
                }
            }
            __syncthreads();
            if (bounded && threadIdx.x < 2 * nw * SCH_SLPW) {
                const float *row = part_f + threadIdx.x * 9;
                const float s0 = (row[0] + row[1]) + (row[2] + row[3]), s1 = (row[4] + row[5]) + (row[6] + row[7]);
                const int lag = threadIdx.x >> 1;
                if (lag < n_lag) { if (threadIdx.x & 1) corr_i[lag] = (double)(s0 + s1); else corr[lag] = (double)(s0 + s1); }
            }
            __syncthreads();
            // candidates: M = max (|c^| - eps); a lag whose |c^| + eps stays below M (with the certificates' relative margin) is below
            // the lag that attains M, whatever the exact values are
            double a = 0.0, lo = -INFINITY;
            if (bounded && threadIdx.x < n_lag) {
                const double cr = corr[threadIdx.x], ci = corr_i[threadIdx.x];
                a = sqrt(cr * cr + ci * ci);
                lo = a - eps;
            }
#pragma unroll
            for (int k = 16; k > 0; k >>= 1) lo = fmax(lo, __shfl_xor_sync(0xffffffffu, lo, k));
            if (lane == 0) red_v[w] = lo;
            __syncthreads();
            double M = red_v[0];
#pragma unroll
            for (int k = 1; k < nw; ++k) M = fmax(M, red_v[k]);
            const bool cand = bounded && threadIdx.x < n_lag && (a + eps) * (1.0 + 1e-9) >= M * (1.0 - 1e-9);
            const unsigned bal = __ballot_sync(0xffffffffu, cand);
            if (lane == 0 && w < 3) cmask[w] = bal;                 // n_lag <= 96
            const int n_c = __syncthreads_count(cand);              // also orders the red_v reads before any later write
            if (bounded && mode == 0 && n_c >= 1 && n_c <= SCH_MAXC) {
                if (w < n_c) {                                      // warp w: the w-th candidate in lag order
                    int k = w, lag = 0;
#pragma unroll 1
                    for (int q = 0; q < 3; ++q) {
                        unsigned m = cmask[q];
                        const int pc = __popc(m);
                        if (k < pc) {
                            for (; k > 0; --k) m &= m - 1;
                            lag = 32 * q + __ffs(m) - 1;
                            break;
                        }
                        k -= pc;
                    }
                    const double v = sch_lag_fp64(wp, tpl, lag, lane);
                    if (lane == 0) { corr_i[w] = v; red_i[w] = lag; }
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    double v = -1.0; int bi = 0x7fffffff;
                    for (int k = 0; k < n_c; ++k) argmax_combine(v, bi, corr_i[k], red_i[k]);
                    *o = (double)(sp + bi);
                    sch_edge[(i64)stream * cap + burst] = (bi == 0 || bi == n_lag - 1) ? 1 : 0;
                    atomicAdd(stats + n_c, 1u);
                }
                return;
            }
            // fallback: the full fp64 correlation; the fp64 template goes over the fp32 window (read before the barriers above)
            for (int i = threadIdx.x; i < L; i += SCH_THREADS) tp[i + (i >> 4)] = __ldg(tpl + i);
        } else {
            for (int i = threadIdx.x; i < n_smp; i += SCH_THREADS) wp[i + (i >> 4)] = win[i];
            for (int i = threadIdx.x; i < L; i += SCH_THREADS) tp[i + (i >> 4)] = t[i];
        }
        if (threadIdx.x == 0) atomicAdd(stats, 1u);
        __syncthreads();
        // corr / corr_i reach the helper as opaque shared addresses: as its only caller this kernel would otherwise have them folded into
        // the helper, and then ptxas spills 8 bytes here at 64 registers
        unsigned a_c = (unsigned)__cvta_generic_to_shared(corr), a_ci = (unsigned)__cvta_generic_to_shared(corr_i);
        asm("" : "+r"(a_c), "+r"(a_ci));
        sch_corr_tiled_fp64(wp, tp, part, (double *)__cvta_shared_to_generic(a_c), (double *)__cvta_shared_to_generic(a_ci), n_lag, n_smp);
    } else {
        for (int lag = w; lag < n_lag; lag += nw) {              // generic shapes: one warp per lag
            double ar = 0.0, ai = 0.0;
            for (int n = lane; n < L; n += 32) {
                const double2 p = cmulc(win[lag + n], t[n]);      // conj(ts) .* window
                ar += p.x; ai += p.y;
            }
            ar = warp_sum(ar); ai = warp_sum(ai);
            if (lane == 0) { corr[lag] = ar; corr_i[lag] = ai; }
        }
    }
    __syncthreads();
    if (threadIdx.x < n_lag) corr[threadIdx.x] = abs2_ref(make_double2(corr[threadIdx.x], corr_i[threadIdx.x]));   // abs(.)^2, one lag per thread
    __syncthreads();
    double v = -1.0; int bi = 0x7fffffff;
    for (int lag = threadIdx.x; lag < n_lag; lag += SCH_THREADS) argmax_combine(v, bi, corr[lag], lag);
    block_argmax(v, bi, red_v, red_i);
    if (threadIdx.x == 0) {
        *o = (double)(sp + bi);
        sch_edge[(i64)stream * cap + burst] = (bi == 0 || bi == n_lag - 1) ? 1 : 0;
    }
}

// ===================================================================================================
// sequential per-stream stages (one thread per stream): ppm solves, regridding, pos_info
// ===================================================================================================
__device__ __forceinline__ double mround(double x) { return (x >= 0.0) ? floor(x + 0.5) : -floor(-x + 0.5); }   // MATLAB round

// 10-frame / 11-frame spacing classification - FCCH_fine_correction.m:74-113 == SCH_corr_rate_correction.m:89-116.
// kind[i] = 0 (10 frames) / 1 (11 frames) / 2 (both windows, cannot happen with these thresholds).
__device__ bool classify_spacing(const double *pos, int n, int osr, double max_ppm, double *expected, double *d10o, double *d11o, unsigned char *kind) {
    const double num_sym_per_frame = (625.0 / 4.0) * 8.0;
    const double d10 = 10.0 * num_sym_per_frame * osr, d11 = 11.0 * num_sym_per_frame * osr;
    const double th10 = floor(d10 * max_ppm * 1e-6), th11 = floor(d11 * max_ppm * 1e-6);
    int na = 0, nb = 0;
    for (int i = 0; i + 1 < n; ++i) {
        const double d = pos[i + 1] - pos[i];
        const bool a = fabs(d - d10) < th10, b = fabs(d - d11) < th11;
        na += a; nb += b;
        kind[i] = b ? 1 : 0;
        if (a && b) kind[i] = 2;
    }
    *expected = (double)na * d10 + (double)nb * d11;
    *d10o = d10; *d11o = d11;
    return (na + nb) == n - 1;
}

// The per-stream stages below run as ONE WARP per stream: the lanes stage the stream's small arrays in shared memory
// with coalesced loads, lane 0 replays the reference's sequential logic on shared memory (global-memory latency was
// the whole cost of the one-thread-per-stream version), and the lanes write the results back together.
#define PS_THREADS 32
__global__ void __launch_bounds__(PS_THREADS) fine_ppm_kernel(StreamCtl *ctl, int n_streams, int cap, int osr, i64 n_iq, const double *__restrict__ fine_raw,
                                                             double *__restrict__ fcch_pos, unsigned char *__restrict__ kind_scratch) {
    extern __shared__ double ps_sm[];
    double *fr = ps_sm, *fp = fr + cap;
    unsigned char *kind = reinterpret_cast<unsigned char *>(fp + cap);
    __shared__ StreamCtl cs;
    const int stream = blockIdx.x, lane = threadIdx.x;
    if (stream >= n_streams) return;
    if (lane == 0) cs = ctl[stream];
    __syncwarp();
    const int nc = cs.n_coarse;
    for (int i = lane; i < nc; i += PS_THREADS) fr[i] = fine_raw[(i64)stream * cap + i];
    __syncwarp();
    if (lane == 0) {
        StreamCtl c = cs;
        c.n_fcch = -1; c.len1 = -1; c.sppm1 = INFINITY; c.cppm1 = INFINITY; c.interp1_on = 0; c.tone1_enable = 0; c.derot1_on = 0;
        c.e1 = 0.0; c.dphi1 = 0.0; c.n_fine = 0;
        const int fft_len = 148 * osr;
        if (c.n_coarse >= 5) {
            int last_idx = c.n_coarse;
            for (int i = 0; i < c.n_coarse; ++i) if (isinf(fr[i])) { last_idx = i; break; }
            c.n_fine = last_idx;
            c.n_fcch = last_idx;
            for (int i = 0; i < last_idx; ++i) fp[i] = fr[i];
            if (last_idx >= 5) {
                c.len1 = n_iq;                                        // r = s (:72)
                double expected, d10, d11;
                if (!classify_spacing(fr, last_idx, osr, 4000.0, &expected, &d10, &d11, kind)) {
                    c.n_fcch = -1; c.flags |= 1;                      // :95-102
                } else {
                    const double actual = fr[last_idx - 1] - fr[0];
                    const double e = (actual - expected) / expected;
                    c.e1 = e; c.sppm1 = e * 1e6; c.interp1_on = 1;
                    c.len1 = (e >= 0.0) ? (i64)floor((double)n_iq / (1.0 + e)) : n_iq;
                    const double first = mround((fr[0] - 1.0) / (1.0 + e)) + 1.0;
                    double acc = 1.0;
                    fp[0] = acc + first - 1.0;
                    for (int i = 0; i + 1 < last_idx; ++i) { acc += (kind[i] == 1) ? d11 : d10; fp[i + 1] = acc + first - 1.0; }
                    int n = last_idx;
                    if (fp[n - 1] + fft_len - 1 > (double)c.len1) n -= 1;     // :135-137
                    c.n_fcch = n;
                    c.tone1_enable = (n >= 5);
                }
            }
        }
        cs = c;
        ctl[stream] = c;
    }
    __syncwarp();
    const int n_out = cs.n_fine > cs.n_fcch ? cs.n_fine : cs.n_fcch;
    for (int i = lane; i < n_out; i += PS_THREADS) fcch_pos[(i64)stream * cap + i] = fp[i];
    (void)kind_scratch;
}

__global__ void __launch_bounds__(PS_THREADS) fine_carrier_kernel(StreamCtl *ctl, int n_streams, int cap, int osr, double carrier_freq, const double *__restrict__ fo,
                                                                 const double *__restrict__ gate) {
    extern __shared__ double ps_sm[];
    double *f = ps_sm, *g = f + cap;
    const int stream = blockIdx.x, lane = threadIdx.x;
    if (stream >= n_streams) return;
    StreamCtl c = ctl[stream];
    if (c.tone1_enable) {
        for (int i = lane; i < c.n_fcch; i += PS_THREADS) { f[i] = fo[(i64)stream * cap + i]; g[i] = gate[(i64)stream * cap + i]; }
        __syncwarp();
    }
    if (lane != 0) return;
    if (c.tone1_enable) {
        const double symbol_rate = (1625.0 / 6.0) * 1e3, sampling_rate = symbol_rate * osr, target = symbol_rate / 4.0;
        double acc = 0.0;
        for (int i = 0; i < c.n_fcch; ++i) acc += f[i];
        const double fom = acc / (double)c.n_fcch;
        c.cppm1 = 1e6 * (fom - target) / carrier_freq;
        c.dphi1 = (target - fom) * 2 * GSMCAL_PI / sampling_rate;
        c.derot1_on = 1;
        int low = 0;
        for (int i = 0; i < c.n_fcch; ++i) low += (g[i] < 5.0);
        if (low > 0) { c.n_fcch = -1; c.flags |= 2; }             // :192-196
    }
    c.sch_enable = (c.n_fcch >= 5);
    ctl[stream] = c;
}

__global__ void __launch_bounds__(PS_THREADS) sch_ppm_kernel(StreamCtl *ctl, int n_streams, int cap, int osr, const double *__restrict__ sch_raw, const int *__restrict__ sch_edge,
                                                            double *__restrict__ sch_pos_scratch, unsigned char *__restrict__ kind_scratch, double *__restrict__ pos_info /* [stream][6*cap][2] */,
                                                            double *__restrict__ post_pos) {
    extern __shared__ double ps_sm[];
    double *sr = ps_sm, *sp_ = sr + cap;
    int *se = reinterpret_cast<int *>(sp_ + cap);
    unsigned char *kind = reinterpret_cast<unsigned char *>(se + cap);
    __shared__ StreamCtl cs;
    __shared__ int sh_fill;
    const int stream = blockIdx.x, lane = threadIdx.x;
    if (stream >= n_streams) return;
    if (lane == 0) { cs = ctl[stream]; sh_fill = 0; }
    __syncwarp();
    double *pi = pos_info + (i64)stream * 6 * cap * 2;
    double *pp = post_pos + (i64)stream * cap;
    const int H = cs.sch_enable ? cs.n_fcch : 0;
    for (int i = lane; i < H; i += PS_THREADS) { sr[i] = sch_raw[(i64)stream * cap + i]; se[i] = sch_edge[(i64)stream * cap + i]; }
    __syncwarp();
    if (lane == 0) {
        StreamCtl c = cs;
        c.n_pos_info = -1; c.len2 = -1; c.sppm2 = INFINITY; c.interp2_on = 0; c.e2 = 0.0; c.n_sch = 0; c.post_enable = 0; c.n_post_fcch = 0;
        c.cppm2 = INFINITY; c.dphi2 = 0.0; c.len3 = -1;
        if (c.sch_enable) {
            int num_sch = H; bool edge = false;
            for (int i = 0; i < H; ++i) {
                if (isinf(sr[i])) { num_sch = i; break; }
                if (se[i]) { edge = true; break; }
            }
            if (edge) {
                c.flags |= 4;                                         // pos_info = [-1,-1], r = -1 (:59-63)
            } else {
                c.n_sch = num_sch;
                c.n_pos_info = 3 * H;                                 // -1.*ones(3*num_fcch_hit,2) (:32)
                sh_fill = 3 * H;
                if (num_sch >= 5) {
                    c.len2 = c.len1;                                  // r = s (:87)
                    double expected, d10, d11;
                    if (!classify_spacing(sr, num_sch, osr, 400.0, &expected, &d10, &d11, kind)) {
                        c.flags |= 8;                                 // :106-112
                    } else {
                        const double actual = sr[num_sch - 1] - sr[0];
                        const double e = (actual - expected) / expected;
                        c.e2 = e; c.sppm2 = e * 1e6;
                        if (e != 0.0) {
                            c.interp2_on = 1;
                            c.len2 = (e > 0.0) ? (i64)floor((double)c.len1 / (1.0 + e)) : c.len1;
                        }
                        const double first = mround((sr[0] - 1.0) / (1.0 + e)) + 1.0;
                        double acc = 1.0;
                        sp_[0] = acc + first - 1.0;
                        for (int i = 0; i + 1 < num_sch; ++i) { acc += (kind[i] == 1) ? d11 : d10; sp_[i + 1] = acc + first - 1.0; }
                        // BCCH_flag (:138-141), 1-based: flag(b_idx+1) and flag(b_idx-4) for b_idx>=5, b_idx = 11-frame gaps
                        const int slot_ov = (625 * osr) / 4, frame_ov = slot_ov * 8;
                        const double fix_off = (double)(frame_ov + 42 * osr), pre_ov = (double)(42 * osr);
                        const double len_r = (double)c.len2;
                        int row = 0, n_f = 0, n_b = 0;
                        sh_fill = 0;                                  // rows are written explicitly below
                        for (int i = 0; i < num_sch; ++i) {
                            const bool flag = (i >= 1 && kind[i - 1] == 1) || (i + 4 < num_sch - 1 && kind[i + 4] == 1);
                            pi[2 * row] = sp_[i] - fix_off; pi[2 * row + 1] = 0.0; pp[n_f++] = sp_[i] - fix_off; ++row;
                            const double s0 = sp_[i] - pre_ov;
                            if (s0 + slot_ov - 1 <= len_r) { pi[2 * row] = s0; pi[2 * row + 1] = 1.0; ++row; } else break;
                            if (flag) {
                                bool runout = false;
                                for (int k = 1; k <= 4; ++k) {
                                    const double b0 = s0 + (double)k * frame_ov;
                                    if (b0 + slot_ov - 1 <= len_r) { pi[2 * row] = b0; pi[2 * row + 1] = 2.0; ++row; ++n_b; }
                                    else { runout = true; break; }
                                }
                                if (runout) break;
                            }
                        }
                        c.n_pos_info = row;
                        c.n_post_fcch = n_f;
                        // carrier_correct_post_SCH.m:10-19: all -1 cannot happen here; needs >= 4 BCCH rows
                        if (n_b >= 4) { c.post_enable = 1; c.len3 = c.len2; } else c.flags |= 16;
                    }
                }
            }
        }
        ctl[stream] = c;
    }
    __syncwarp();
    const int fill = sh_fill;                                         // the -1 sentinel matrix (:32), written by all lanes
    for (int i = lane; i < 2 * fill; i += PS_THREADS) pi[i] = -1.0;
    (void)sch_pos_scratch; (void)kind_scratch;
}

__device__ __forceinline__ double total_ppm2(double a, double b) {     // total_ppm_calculation.m:5-21
    if (isinf(a) && a > 0 && isinf(b) && b > 0) return INFINITY;
    double acc = 1.0;
    acc = acc * (1.0 + a * 1e-6);
    acc = acc * (1.0 + b * 1e-6);
    return (acc - 1.0) * 1e6;
}

struct StreamResultDev {            // mirrors gsmcal_stream_result (include/gsmcal.h)
    int n_coarse, n_fcch, n_pos_info, flags;
    i64 r_len[3];
    double sampling_ppm[2], carrier_ppm[2], total_sampling_ppm, total_carrier_ppm;
};

__global__ void __launch_bounds__(PS_THREADS) post_carrier_kernel(StreamCtl *ctl, int n_streams, int cap, int osr, double carrier_freq, const double *__restrict__ fo, StreamResultDev *res) {
    extern __shared__ double ps_sm[];
    const int stream = blockIdx.x, lane = threadIdx.x;
    if (stream >= n_streams) return;
    StreamCtl c = ctl[stream];
    if (c.post_enable) {
        for (int i = lane; i < c.n_post_fcch; i += PS_THREADS) ps_sm[i] = fo[(i64)stream * cap + i];
        __syncwarp();
    }
    if (lane != 0) return;
    if (c.post_enable) {
        const double symbol_rate = (1625.0 / 6.0) * 1e3, sampling_rate = symbol_rate * osr, target = symbol_rate / 4.0;
        double acc = 0.0;
        for (int i = 0; i < c.n_post_fcch; ++i) acc += ps_sm[i];
        const double fom = acc / (double)c.n_post_fcch;
        c.cppm2 = 1e6 * (fom - target) / carrier_freq;
        c.dphi2 = (target - fom) * 2 * GSMCAL_PI / sampling_rate;
    }
    ctl[stream] = c;
    if (res) {
        StreamResultDev r;
        r.n_coarse = c.n_coarse; r.n_fcch = c.n_fcch; r.n_pos_info = c.n_pos_info; r.flags = c.flags;
        r.r_len[0] = c.len1; r.r_len[1] = c.len2; r.r_len[2] = c.len3;
        r.sampling_ppm[0] = c.sppm1; r.sampling_ppm[1] = c.sppm2;
        r.carrier_ppm[0] = c.cppm1; r.carrier_ppm[1] = c.cppm2;
        r.total_sampling_ppm = total_ppm2(c.sppm1, c.sppm2);
        r.total_carrier_ppm = total_ppm2(c.cppm1, c.cppm2);
        res[stream] = r;
    }
}

// ===================================================================================================
// r_correct of the batched pipeline: the stream gsm_sync_demod.m:120 hands to SCH_demod (:145), straight from the uint8 capture:
//   filter(coef,1,raw2iq(a)) -> interp1 by (1+e1) (FCCH_fine_correction.m:125) -> .*exp(1i*n*dphi1) (:165)
//   -> interp1 by (1+e2) (SCH_corr_rate_correction.m:127) -> .*exp(1i*n*dphi2) (carrier_correct_post_SCH.m:83)
// One pass, 2 bytes in and 16 bytes out per sample (the function-by-function chain moves 178).  Persistent blocks walk tiles of MAT_T
// outputs; the levels are load_window's, the last derotation uses one slow-path sincos per tile.  FP64-bound by the 47-tap FIR.
// ===================================================================================================
#define MAT_T 1200
#define MAT_THREADS 256
__global__ void __launch_bounds__(MAT_THREADS, 3) materialise_r_kernel(WinSrc src, const StreamCtl *__restrict__ ctl, double2 *__restrict__ r_out, i64 r_stride,
                                                                   i64 tiles_per_stream) {
    extern __shared__ double2 sm[];
    __shared__ double2 base2;
    double2 *dst = sm, *X = dst + MAT_T, *Y = X + GSMCAL_XCAP(MAT_T + 8);
    const int stream = blockIdx.y, tid = threadIdx.x;
    const StreamCtl c = ctl[stream];
    if (c.len3 < 0) return;                                      // r = -1 on this stream's path: nothing to materialise
    double2 *o = r_out + (i64)stream * r_stride;
    double2 st2 = make_double2(1.0, 0.0), ph_t = make_double2(1.0, 0.0);
    {
        double sn, cs;
        sincos((double)tid * c.dphi2, &sn, &cs); ph_t = make_double2(cs, sn);
        sincos((double)MAT_THREADS * c.dphi2, &sn, &cs); st2 = make_double2(cs, sn);
    }
    for (i64 tile = blockIdx.x; tile < tiles_per_stream; tile += gridDim.x) {
        const i64 j0 = tile * MAT_T;
        if (j0 >= c.len3) break;
        const int count = (c.len3 - j0 < MAT_T) ? (int)(c.len3 - j0) : MAT_T;
        __syncthreads();                                         // the previous tile's reads of dst are done
        if (tid == 0) { double sn, cs; sincos((double)j0 * c.dphi2, &sn, &cs); base2 = make_double2(cs, sn); }
        load_window(src, c, stream, j0, count, dst, X, Y);       // level 3; ends with a barrier
        double2 ph = cmul(base2, ph_t);
        for (int i = tid; i < count; i += MAT_THREADS) {
            __stcs(o + j0 + i, cmul(dst[i], ph));
            ph = cmul(ph, st2);
        }
    }
}

// FCCH scanner acceptance: multi_rtl_sdr_gsm_FCCH_scanner.m:165-186
__global__ void scan_accept_kernel(const StreamCtl *ctl, int n_chan, int cap, const double *__restrict__ position, const double *__restrict__ snr,
                                   double *__restrict__ snr_out, double *__restrict__ num_hit) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_chan) return;
    const int n = ctl[ch].n_coarse;
    double s = 0.0, h = 0.0;
    if (n >= 3) {
        const double *p = position + (i64)ch * cap;
        bool all_a = true, all_b = true;
        for (int i = 0; i + 1 < n; ++i) {
            const double d = p[i + 1] - p[i];
            const bool a = fabs(d - 12500.0) > 50.0;
            if (a) { all_a = false; if (fabs(d - 13750.0) > 50.0) all_b = false; }
        }
        if (all_a || all_b) {
            double acc = 0.0;
            for (int i = 0; i < n; ++i) acc += snr[(i64)ch * cap + i];
            s = acc / (double)n; h = (double)n;
        }
    }
    snr_out[ch] = s; num_hit[ch] = h;
}

// multi_rtl_sdr_diversity_scanner.m:150-176: per-dongle mean power (:155) and the incoherent combination over dongles
// (mean(power_spectrum, 1), :172), both on the device: power_acc[i * n_freq + f] holds sum(abs(r_flt(1:decim:end, f)).^2) of dongle i.
__global__ void diversity_combine_kernel(const double *__restrict__ power_acc, i64 n_out, int n_freq, int n_dongle,
                                         double *__restrict__ power_spectrum /* n_dongle x n_freq, column-major */, double *__restrict__ combine) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_freq) return;
    double acc = 0.0;
    for (int i = 0; i < n_dongle; ++i) {                         // MATLAB sums a column top to bottom
        const double p = power_acc[(i64)i * n_freq + f] / (double)n_out;
        power_spectrum[(i64)f * n_dongle + i] = p;
        acc += p;
    }
    combine[f] = acc / (double)n_dongle;
}

__global__ void mean_kernel(StreamCtl *ctl, int n_streams, i64 n_iq) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < n_streams) { ctl[d].mu_re = stream_mean(ctl[d].sum_i, n_iq); ctl[d].mu_im = stream_mean(ctl[d].sum_q, n_iq); }
}

// tw[0..N): exp(-2*pi*i*j/N).  Behind it, three compact copies for the Horner segment / chunk rotations of tone8_kernel and
// fine_core8_kernel: tw[N + s] = W^(10 s), tw[N + TW_SEG + s] = W^(20 s), tw[N + 2 TW_SEG + s] = W^(32 s), s < TW_SEG - the same values as
// tw[(10 s) % N] ..., but a warp reads 16 consecutive entries (2 cache lines) instead of 16 lines
#define TW_SEG 128
#define TW_EXTRA (3 * TW_SEG)
__global__ void twiddle_init_kernel(double2 *tw, int N) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < N + TW_EXTRA) {
        const int t = (j - N) / TW_SEG, sidx = (j - N) % TW_SEG;
        const int e = (j < N) ? j : (int)(((t == 0 ? 10ll : (t == 1 ? 20ll : 32ll)) * sidx) % N);
        double sn, cs; sincospi(-2.0 * (double)e / (double)N, &sn, &cs);
        tw[j] = make_double2(cs, sn);
    }
}

// FP64 pipe microbenchmark (8 independent DFMA chains per thread): the denominator for the FP64-bound burst stages,
// which MEASURED_PEAKS.json (HBM copy + bf16 GEMM) does not provide.
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    if (a == 123.456) out[blockIdx.x * 256 + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}
