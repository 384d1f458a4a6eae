// gsmcal_api.cu - the C ABI declared in include/gsmcal.h: host-side sequencing of the sm_100a kernels.
// No torch types, no CPU fallback: every compute entry point fails with GSMCAL_ERR_CUDA without a device.
#include "../../include/gsmcal.h"
#include "gsmcal_kernels.cuh"
#include "gsmcal_burst8.cuh"
#include "gsmcal_demod.cuh"

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "chn_filter_taps.inc"

static_assert(sizeof(gsmcal_stream_result) == sizeof(StreamResultDev), "result record layout");
static_assert(sizeof(gsmcal_demod_result) == sizeof(DemodResultDev) && sizeof(gsmcal_demod_result) == 32, "demod record layout");
static_assert(GSMCAL_DEMOD_NO_POS_INFO == DM_NO_POS_INFO && GSMCAL_DEMOD_NO_R_CORRECT == DM_NO_R_CORRECT && GSMCAL_DEMOD_SCH_RANGE == DM_SCH_RANGE &&
              GSMCAL_DEMOD_FCCH_RANGE == DM_FCCH_RANGE, "demod flags");
static_assert(sizeof(gsmcal_bcch_result) == sizeof(BcchResultDev) && sizeof(gsmcal_bcch_result) == 272 && offsetof(gsmcal_bcch_result, nts_idx) == 8 &&
              offsetof(gsmcal_bcch_result, flags) == 12 && offsetof(gsmcal_bcch_result, corr_abs) == 16, "BCCH record layout");
static_assert(GSMCAL_BCCH_NO_POS_INFO == BC_NO_POS_INFO && GSMCAL_BCCH_FEW_BCCH == BC_FEW_BCCH && GSMCAL_BCCH_FCCH_RANGE == BC_FCCH_RANGE &&
              GSMCAL_BCCH_TRAIN_RANGE == BC_TRAIN_RANGE, "BCCH flags");
static_assert(sizeof(gsmcal_sch_timing_result) == sizeof(TimingResultDev) && sizeof(gsmcal_sch_timing_result) == 40 &&
              offsetof(gsmcal_sch_timing_result, t0) == 16 && offsetof(gsmcal_sch_timing_result, rms) == 32, "SCH timing record layout");
static_assert(GSMCAL_TIMING_NO_POS_INFO == TM_NO_POS_INFO && GSMCAL_TIMING_NO_R_CORRECT == TM_NO_R_CORRECT && GSMCAL_TIMING_RANGE == TM_RANGE &&
              GSMCAL_TIMING_EDGE == TM_EDGE && GSMCAL_TIMING_FEW == TM_FEW, "SCH timing flags");
static_assert(sizeof(gsmcal_sch_decode_result) == sizeof(SchDecodeResultDev) && sizeof(gsmcal_sch_decode_result) == 32 &&
              offsetof(gsmcal_sch_decode_result, fn_first) == 20 && offsetof(gsmcal_sch_decode_result, frame_clock_start) == 24, "SCH decode record layout");
static_assert(GSMCAL_SCHDEC_NO_POS_INFO == SC_NO_POS_INFO && GSMCAL_SCHDEC_NO_R_CORRECT == SC_NO_R_CORRECT && GSMCAL_SCHDEC_NONE == SC_NONE &&
              GSMCAL_SCHDEC_DISAGREE == SC_DISAGREE && GSMCAL_SCHDEC_ROW_WINDOW == SC_ROW_WINDOW && GSMCAL_SCHDEC_ROW_ALIGN == SC_ROW_ALIGN &&
              GSMCAL_SCHDEC_ROW_CRC == SC_ROW_CRC && GSMCAL_SCHDEC_ROW_FIELD == SC_ROW_FIELD, "SCH decode flags");
static_assert(sizeof(gsmcal_carrier_fit_result) == sizeof(CarrierFitDev) && sizeof(gsmcal_carrier_fit_result) == 72 &&
              offsetof(gsmcal_carrier_fit_result, t_mean) == 16 && offsetof(gsmcal_carrier_fit_result, drift_ppm_per_s) == 64, "carrier fit record layout");
static_assert(GSMCAL_CARRIER_NO_POS_INFO == CF_NO_POS_INFO && GSMCAL_CARRIER_NO_R_CORRECT == CF_NO_R_CORRECT && GSMCAL_CARRIER_RANGE == CF_RANGE &&
              GSMCAL_CARRIER_EDGE == CF_EDGE && GSMCAL_CARRIER_NOCONV == CF_NOCONV && GSMCAL_CARRIER_FEW == CF_FEW, "carrier fit flags");

namespace {

std::mutex g_mu;
thread_local std::string g_err;
thread_local int g_device = 0;
std::atomic<long long> g_launches{0};
int *g_last_need_full = nullptr, *g_last_need_band = nullptr; long long g_last_need_full_n = 0;
int g_debug_groups = 4;           // stream groups per batch (1 = strictly sequential stages, enables per-stage timing)
int g_debug_fall_limit = FALL_GRID;  // tier 3 handles work lists up to this length (tests set 0 to exercise the single-block list mode)
int g_debug_fail_tier2 = 0;       // tests: pretend the 64-bin certificate failed
int g_debug_force_full = 0;       // tests: run the all-bin fine search for every burst
int g_debug_submit_groups = 2;    // stream groups inside a submitted batch (debug key 8)
int g_debug_hi_prio = 1;          // burst chain of each stream group on a high-priority CUDA stream
int g_debug_core8_passes = B8_NPASS; // passes of 8 tracked bins in fine_core8_kernel (1..8)
unsigned *g_last_pass_hist = nullptr, *g_prev_pass_hist = nullptr;   // counters of the last / the one-before-last batch (debug_get 50.., 150..)
int g_debug_sch_mode = 0;          // debug key 24: sch_corr_kernel at osr 8: 0 = fp32 screen, 1 = always fp64, 2 = screen + forced fallback
unsigned *g_last_sch_stats = nullptr;   // SCH_NSTAT counters of the last call that ran the SCH stage (debug_get 120..)
int g_debug_trickle = 2;           // debug key 17: ring stages (x 4 KB, 1..24) of colsum_u8_trickle_kernel in submit/collect
int g_debug_trickle_blocks = 3;    // debug key 18: its blocks per SM (3 x 2 stages: 22 GB in 7 ms under the FP64 stages, profiles/r2q)
int g_debug_timeline = 0;          // submit/collect print the device timeline of every batch to stderr (A/B of overlap)
cudaEvent_t g_tl_base = nullptr;
int g_debug_prof = 0;              // fine_core8_kernel accumulates per-phase cycle counts (debug_get 50..65)
int g_debug_no_tone8 = 0;          // tests / A-B: 1 = generic tone estimator for every burst
int g_debug_no_core8 = 0;         // tests / A-B: 1 = round-1 tier-1 kernel and no filtered-window cache

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
    return code;
}

#define CU(expr)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (expr);                                                                          \
        if (e_ != cudaSuccess) return fail(GSMCAL_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define TRY(expr) do { int rc_ = (expr); if (rc_ != GSMCAL_OK) return rc_; } while (0)
#define LAUNCH(kern, grid, block, smem, st, ...)                                                          \
    do { kern<<<(grid), (block), (smem), (st)>>>(__VA_ARGS__); ++g_launches; CU(cudaGetLastError()); } while (0)

struct DevBuf {
    void *p = nullptr; size_t cap = 0;
    int get(size_t bytes, void **out) {
        if (bytes > cap) {
            if (p) cudaFree(p);
            p = nullptr; cap = 0;
            size_t want = bytes + bytes / 8 + 256;
            cudaError_t e = cudaMalloc(&p, want);
            if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
            if (e != cudaSuccess) return fail(GSMCAL_ERR_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
            cap = want;
        }
        *out = p;
        return GSMCAL_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// one in-flight batch of the submit/collect API: its own workspace, streams and pinned result staging, so that consecutive batches
// overlap on the device (the ~1 ms latency-bound front of batch k+1 - column sums, burst chain - runs under the FP64 kernels of batch k)
constexpr int kSlots = 4;
struct Slot {
    DevBuf work, wc;                                            // wc: filtered-window cache of the osr-8 fast path
    cudaStream_t front_hi = nullptr;
    std::vector<cudaStream_t> grp, hi;
    cudaEvent_t done = nullptr;
    cudaEvent_t tl[8] = {};                                     // debug key 14: front start, column sums done, burst chain done, FP64 stages done,
                                                                // FP64 stages start, fine search done, fine tone done, SCH done
    bool tl_on = false;
    bool busy = false;
    char *stage = nullptr; size_t stage_cap = 0;               // pinned host staging of the results
    gsmcal_stream_result *results = nullptr; double *coarse_pos = nullptr, *coarse_snr = nullptr, *fcch_pos = nullptr, *pos_info = nullptr;
    size_t n_res = 0, n_per = 0;                                // bytes of the result records / of one D*cap double array
};
#include "gsmcal_hostcopy.inc"

constexpr int kNumStageEvents = 8;
struct Ctx {
    StageRing ring;                  // pinned staging for pageable host buffers
    int last_slot = -1;              // slot of the most recently submitted batch (submit/collect pipeline)
    bool attrs = false;
    cudaEvent_t stage_ev[kNumStageEvents];
    bool stage_ev_ok = false;
    Slot slots[kSlots];
    DevBuf in, out, work, tplbuf, wc, dem;     // dem: outputs and row lists of gsmcal_calibrate_demod_batch
    std::map<int, double2 *> tw;     // N -> exp(-2*pi*i*j/N)
    std::vector<cudaStream_t> side;  // extra streams: stream groups of a batch overlap their latency-bound stages
    std::vector<cudaStream_t> side_hi; // one high-priority stream per group for the latency-bound burst chain (see gsmcal_calibrate_batch)
};
std::map<int, Ctx> g_ctx;

// per-stage CUDA-event timing of the last gsmcal_calibrate_batch call (events are recorded on the call's stream; they belong to the
// device's Ctx - an event of another device cannot be recorded on this one's streams)
int g_stage_n = 0;
float g_stage_ms[kNumStageEvents];
int stage_mark(Ctx &c, cudaStream_t st) {
    if (!c.stage_ev_ok) {
        for (int i = 0; i < kNumStageEvents; ++i) CU(cudaEventCreate(&c.stage_ev[i]));
        c.stage_ev_ok = true;
    }
    if (g_stage_n < kNumStageEvents) CU(cudaEventRecord(c.stage_ev[g_stage_n++], st));
    return GSMCAL_OK;
}

int ensure_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) { cudaGetLastError(); return fail(GSMCAL_ERR_CUDA, "no CUDA device (the sm_100a kernels are the only implementation; there is no CPU fallback)"); }
    CU(cudaSetDevice(g_device));
    return GSMCAL_OK;
}

constexpr int kFineThreads = 320;
size_t fine_smem(int osr) { int N = 148 * osr, ns = 2 * 64 * osr + 1 + N - 1; return (size_t)(2 * ns + 8 + GSMCAL_XCAP(ns)) * sizeof(double2); }
size_t fine_band_smem(int osr) {
    // window + scratch; the scratch holds the loader's staging for one third of the window, later the piece / chunk sums
    // and the three 16-sample prefix arrays of the certificate
    const int N = 148 * osr, ns = 2 * 64 * osr + 1 + N - 1, n_chunk = ns / 16, pre = (3 * (n_chunk + 2) + 1) / 2 + 2;
    int x = GSMCAL_XCAP((ns + 2) / 3);
    const int need_band = 8 * FB_BINS + pre, need_core = (ns / (4 * osr) + 1) * FC_BINS + pre + 4 + (2 * 64 * osr / (4 * osr) + 2) * 4;   // + pass-0 tracked powers [n_seg+1][8] doubles
    if (x < need_band) x = need_band;
    if (x < need_core) x = need_core;
    return (size_t)(ns + x) * sizeof(double2);
}
size_t tone_smem(int osr) {
    int N = 148 * osr, work = GSMCAL_XCAP(N) + N + 8;
    if (work < 2 * N) work = 2 * N;
    return (size_t)(N + work) * sizeof(double2);
}
size_t sch_smem(int osr) {
    int L = 64 * osr, ns = 16 * osr - 5 * osr + 1 + L - 1;
    size_t slots = (size_t)(2 * ns + L + 8 + GSMCAL_XCAP(ns));
    if (osr == 8) {     // register-tiled path: padded window + padded template + 96 partial-sum rows of 9 doubles behind X
        size_t need = (size_t)(ns + L + 8) + (size_t)(ns + (ns >> 4) + 2) + (size_t)(L + (L >> 4) + 2) + (96 * 9 + 1) / 2 + 2;
        if (slots < need) slots = need;
    }
    return slots * sizeof(double2);
}

int get_ctx(Ctx **out) {
    TRY(ensure_device());
    Ctx &c = g_ctx[g_device];
    if (!c.attrs) {
        CU(cudaFuncSetAttribute(fine_peak_full_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CU(cudaFuncSetAttribute(fine_peak_band_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CU(cudaFuncSetAttribute(fine_peak_core_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CU(cudaFuncSetAttribute(fine_core8_kernel<47, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B8_SMEM));
        CU(cudaFuncSetAttribute(fine_core8_kernel<47, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B8_SMEM));
        CU(cudaFuncSetAttribute(fine_core8_kernel<48, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B8_SMEM));
        CU(cudaFuncSetAttribute(fine_core8_kernel<64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B8_SMEM));
        CU(cudaFuncSetAttribute(tone8_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T8_SMEM));
        CU(cudaFuncSetAttribute(tone8_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T8_SMEM));
        CU(cudaFuncSetAttribute(tone_est_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CU(cudaFuncSetAttribute(sch_corr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(colsum_u8_trickle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 24 * (TRK_STAGE + 8)));
        CU(cudaFuncSetAttribute(colsum_u8_trickle_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CU(cudaFuncSetAttribute(materialise_r_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fir_full_tma_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fir_full_tma_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(coarse_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fine_ppm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fine_carrier_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(sch_ppm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(post_carrier_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fir_decim_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fir_decim_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(fcch_demod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));      // (attributes are per device:
        CU(cudaFuncSetAttribute(fde_template_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));    //  all of them live here, keyed by
        CU(cudaFuncSetAttribute(sch_demod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));       //  the device's Ctx)
        CU(cudaFuncSetAttribute(sch_demod_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(sch_demod_resid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        CU(cudaFuncSetAttribute(bcch_burst_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BB_SMEM));
        CU(cudaFuncSetAttribute(fcch_demod_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        c.attrs = true;
    }
    *out = &c;
    return GSMCAL_OK;
}

int get_twiddle(Ctx &c, int N, cudaStream_t st, const double2 **out) {
    auto it = c.tw.find(N);
    if (it == c.tw.end()) {
        double2 *p = nullptr;
        CU(cudaMalloc(&p, sizeof(double2) * (N + TW_EXTRA)));
        LAUNCH(twiddle_init_kernel, (N + TW_EXTRA + 127) / 128, 128, 0, st, p, N);
        c.tw[N] = p;
        *out = p;
    } else *out = it->second;
    return GSMCAL_OK;
}

double g_taps_host[GSMCAL_MAX_TAPS + 8]; int g_taps_n = -1; int g_taps_dev = -1;
bool any_slot_busy() {
    for (auto &kv : g_ctx) for (Slot &sl : kv.second.slots) if (sl.busy) return true;
    return false;
}
int set_taps(const double *coef, int n_taps, cudaStream_t st) {
    if (n_taps < 1 || n_taps > GSMCAL_MAX_TAPS) return fail(GSMCAL_ERR_ARG, "n_taps must be 1..%d", GSMCAL_MAX_TAPS);
    double tmp[GSMCAL_MAX_TAPS + 8];
    memset(tmp, 0, sizeof tmp);                          // zero padding (4 before, the rest after) adds exact zeros
    memcpy(tmp + 4, coef, sizeof(double) * n_taps);
    if (g_taps_n == n_taps && g_taps_dev == g_device && memcmp(tmp, g_taps_host, sizeof tmp) == 0) return GSMCAL_OK;   // the constant table already holds them
    if (any_slot_busy()) CU(cudaDeviceSynchronize());    // submitted batches still read the old table
    CU(cudaMemcpyToSymbolAsync(c_tapsp, tmp, sizeof tmp, 0, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));                       // tmp lives on this stack frame
    memcpy(g_taps_host, tmp, sizeof tmp); g_taps_n = n_taps; g_taps_dev = g_device;
    return GSMCAL_OK;
}

// ---- workspace carve-up ----------------------------------------------------------------------------
struct Work {
    StreamCtl *ctl; StreamResultDev *res;
    double *coarse_pos, *coarse_snr, *fine_raw, *fcch_pos, *fo, *gate, *sch_raw, *sch_pos, *post_pos, *pos_info, *snr_map, *power;
    int *sch_edge, *need_full, *need_band, *tone_need, *fall_list, *fall_count, *fall_m; double *fall_best; unsigned char *kind; double2 *tpl;
    const float2 *tplf; const double *tpl_e;   // behind tpl: the screen's padded fp32 template and the template energy (tpl_pack)
    unsigned *sch_stats;          // [SCH_NSTAT] sch_corr_kernel counters
    i64 snr_stride;
    unsigned *pass_hist;          // [16] fine_core8_kernel: bursts proven after p passes ([0] = left to the band kernel)
    double2 *wcache;              // [D][cap][B8_WLEN] or nullptr (set by attach_wcache)
    bool wc_valid;                // the fine search of this call filled the cache
};
size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }
// the SCH template as the device reads it: fp64 [L] | fp32 with one pad slot per 16 samples [sch_tplf_len(L)], 16-byte aligned for the
// TMA copy | the fp64 energy sum |t|^2, rounded up (the screen's bound needs an upper bound)
size_t tplf_off(int L) { return sizeof(double2) * (size_t)L; }
size_t tpl_e_off(int L) { return tplf_off(L) + ((sizeof(float2) * (size_t)sch_tplf_len(L) + 15) & ~(size_t)15); }
size_t tpl_pack_bytes(int L) { return tpl_e_off(L) + 16; }
void tpl_pack(const double *tpl, int L, unsigned char *dst) {
    memset(dst, 0, tpl_pack_bytes(L));
    memcpy(dst, tpl, sizeof(double2) * (size_t)L);
    float2 *f = reinterpret_cast<float2 *>(dst + tplf_off(L));
    double e = 0.0;
    for (int i = 0; i < L; ++i) {
        const double x = tpl[2 * i], y = tpl[2 * i + 1];
        f[i + (i >> 4)] = make_float2((float)x, (float)y);
        e += x * x + y * y;
    }
    e *= 1.0 + 1e-12;                                    // L <= 512: the sum's relative error is below 1e-13
    memcpy(dst + tpl_e_off(L), &e, sizeof e);
}
constexpr int kMaxGroups = 32;     // stream groups per batch (tier-3 scratch is per group); ceil(148*8/64) = 19 <= 24 bands

int make_work(DevBuf &wb, i64 D, int cap, i64 snr_len, int tpl_len, Work *w) {
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
    size_t o_ctl = take(sizeof(StreamCtl) * D), o_res = take(sizeof(StreamResultDev) * D);
    size_t per = sizeof(double) * D * cap;
    size_t o_cp = take(per), o_cs = take(per), o_fr = take(per), o_fp = take(per), o_fo = take(per), o_g = take(per), o_sr = take(per), o_sp = take(per), o_pp = take(per);
    size_t o_pi = take(per * 12), o_snr = take(sizeof(double) * D * snr_len), o_pw = take(sizeof(double) * D);
    size_t o_se = take(sizeof(int) * D * cap), o_nf = take(sizeof(int) * D * cap), o_nb = take(sizeof(int) * D * cap), o_tn = take(sizeof(int) * D * cap), o_fl = take(sizeof(int) * D * cap), o_fc = take(sizeof(int) * D), o_fm = take(sizeof(int) * (size_t)FALL_GRID * 24 * kMaxGroups), o_fb = take(sizeof(double) * (size_t)FALL_GRID * 24 * kMaxGroups), o_k = take(D * cap), o_tpl = take(tpl_pack_bytes(tpl_len > 0 ? tpl_len : 1)), o_ph = take(sizeof(unsigned) * 16 + sizeof(unsigned long long) * 64), o_ss = take(sizeof(unsigned) * SCH_NSTAT);
    void *base;
    TRY(wb.get(off, &base));
    char *b = static_cast<char *>(base);
    w->ctl = (StreamCtl *)(b + o_ctl); w->res = (StreamResultDev *)(b + o_res);
    w->coarse_pos = (double *)(b + o_cp); w->coarse_snr = (double *)(b + o_cs); w->fine_raw = (double *)(b + o_fr); w->fcch_pos = (double *)(b + o_fp);
    w->fo = (double *)(b + o_fo); w->gate = (double *)(b + o_g); w->sch_raw = (double *)(b + o_sr); w->sch_pos = (double *)(b + o_sp); w->post_pos = (double *)(b + o_pp);
    w->pos_info = (double *)(b + o_pi); w->snr_map = (double *)(b + o_snr); w->power = (double *)(b + o_pw);
    w->sch_edge = (int *)(b + o_se); w->need_full = (int *)(b + o_nf); w->need_band = (int *)(b + o_nb); w->tone_need = (int *)(b + o_tn); w->fall_list = (int *)(b + o_fl); w->fall_count = (int *)(b + o_fc); w->fall_m = (int *)(b + o_fm); w->fall_best = (double *)(b + o_fb); w->kind = (unsigned char *)(b + o_k); w->tpl = (double2 *)(b + o_tpl);
    w->tplf = (const float2 *)(b + o_tpl + tplf_off(tpl_len)); w->tpl_e = (const double *)(b + o_tpl + tpl_e_off(tpl_len)); w->sch_stats = (unsigned *)(b + o_ss);
    w->snr_stride = snr_len;
    w->pass_hist = (unsigned *)(b + o_ph);
    w->wcache = nullptr; w->wc_valid = false;
    return GSMCAL_OK;
}

// filtered-window cache of the osr-8 fast path: 36,432 bytes per (stream, burst); skipped (the stages re-filter) when it would not fit
constexpr size_t kMaxWcacheBytes = (size_t)24 << 30;
int attach_wcache(DevBuf &buf, i64 D, int cap, int osr, Work *w) {
    w->wcache = nullptr;
    if (osr != 8) return GSMCAL_OK;
    const size_t bytes = (size_t)D * cap * B8_WLEN * sizeof(double2);
    if (bytes > kMaxWcacheBytes) return GSMCAL_OK;
    void *p;
    if (buf.get(bytes, &p) != GSMCAL_OK) { cudaGetLastError(); return GSMCAL_OK; }   // no memory for it: run without
    w->wcache = (double2 *)p;
    return GSMCAL_OK;
}

Work sub_work(const Work &w, i64 d0, int cap, int group) {
    Work s = w;
    s.ctl += d0; s.res += d0; s.power += d0;
    s.coarse_pos += d0 * cap; s.coarse_snr += d0 * cap; s.fine_raw += d0 * cap; s.fcch_pos += d0 * cap; s.fo += d0 * cap; s.gate += d0 * cap;
    s.sch_raw += d0 * cap; s.sch_pos += d0 * cap; s.post_pos += d0 * cap; s.pos_info += d0 * cap * 12; s.snr_map += d0 * w.snr_stride;
    s.sch_edge += d0 * cap; s.need_full += d0 * cap; s.need_band += d0 * cap; s.tone_need += d0 * cap; s.kind += d0 * cap;
    s.fall_list += d0 * cap; s.fall_count += d0;
    s.fall_m += (size_t)group * FALL_GRID * 24; s.fall_best += (size_t)group * FALL_GRID * 24;
    if (s.wcache) s.wcache += (size_t)d0 * cap * B8_WLEN;
    return s;
}

WinSrc mat_src(const double2 *base, i64 len, i64 stride, int interp) {
    WinSrc s; memset(&s, 0, sizeof s);
    s.lazy = 0; s.base = base; s.base_len = len; s.base_stride = stride; s.mat_interp = interp; s.dec = 1;
    return s;
}
WinSrc lazy_src(const uint8_t *raw, i64 n_iq, int n_taps, int level, int dec) {
    WinSrc s; memset(&s, 0, sizeof s);
    s.lazy = 1; s.raw = raw; s.n_iq = n_iq; s.n_taps = n_taps; s.level = level; s.dec = dec;
    return s;
}
WinSrc with_cache(WinSrc s, const Work &w, int cap) {            // level-0 samples of cached bursts come from the fine search's window cache
    if (w.wcache && w.wc_valid) { s.wcache = w.wcache; s.wc_pos = w.coarse_pos; s.wc_cap = cap; }
    return s;
}

// ---- stage launchers (device buffers) -------------------------------------------------------------
int run_colsum_u8(const uint8_t *raw, i64 n_iq, i64 D, StreamCtl *ctl, cudaStream_t st) {
    if (((uintptr_t)raw & 1) != 0) return fail(GSMCAL_ERR_ARG, "uint8 capture must start on an even address");
    const i64 chunk = 512 * 1024;
    i64 chunks = (2 * n_iq + chunk - 1) / chunk; if (chunks < 1) chunks = 1;
    if (D > 65535) return fail(GSMCAL_ERR_ARG, "more than 65535 streams per call");
    LAUNCH(colsum_u8_kernel, dim3((unsigned)chunks, (unsigned)D), 256, 0, st, raw, n_iq, chunk, ctl);
    return GSMCAL_OK;
}

int run_colsum_u8_trickle(const uint8_t *raw, i64 n_iq, i64 D, StreamCtl *ctl, int blocks, int n_stage, cudaStream_t st) {
    if (((uintptr_t)raw & 1) != 0) return fail(GSMCAL_ERR_ARG, "uint8 capture must start on an even address");
    const i64 chunk = 512 * 1024;
    i64 chunks = (2 * n_iq + chunk - 1) / chunk; if (chunks < 1) chunks = 1;
    LAUNCH(colsum_u8_trickle_kernel, (unsigned)blocks, 32, (size_t)n_stage * (TRK_STAGE + 8), st, raw, n_iq, chunk, chunks, D, ctl, n_stage);
    return GSMCAL_OK;
}

struct CoarseParams { int fft_len, mv_len, step10, step11, dr; i64 n_first; double th; };
double host_mround(double x) { return x >= 0 ? floor(x + 0.5) : -floor(-x + 0.5); }
int coarse_params(int dr, CoarseParams *p) {
    if (dr < 1 || dr > 148) return fail(GSMCAL_ERR_ARG, "decimation_ratio out of range");
    const double num_sym_per_frame = (625.0 / 4.0) * 8.0;
    p->fft_len = 1 << (int)floor(log2(148.0 / dr));            // FCCH_coarse_position.m:17
    p->mv_len = 10 * p->fft_len;                                // :22
    p->th = 10.0;                                               // :21
    p->n_first = (i64)ceil(23.0 * num_sym_per_frame / dr);      // :25
    p->step10 = (int)host_mround(10.0 * num_sym_per_frame / dr);   // :35
    p->step11 = (int)host_mround(11.0 * num_sym_per_frame / dr);   // :36
    p->dr = dr;
    return GSMCAL_OK;
}

int run_coarse(WinSrc src, i64 len, const CoarseParams &p, i64 D, int cap, Work &w, cudaStream_t st) {
    const i64 n_win = p.n_first - (p.fft_len - 1);
    size_t smem = sizeof(double2) * (p.fft_len + SNR_THREADS + p.fft_len);
    LAUNCH(snr_map_kernel, dim3((unsigned)((n_win + SNR_THREADS - 1) / SNR_THREADS), (unsigned)D), SNR_THREADS, smem, st,
           src, w.ctl, (i64)0, n_win, p.fft_len, w.snr_map, w.snr_stride);
    LAUNCH(first_hit_scan_kernel, (unsigned)((D + 3) / 4), 128, 0, st, w.snr_map, w.snr_stride, n_win, p.mv_len, p.th, w.ctl, (int)D);
    const size_t chain_smem = sizeof(double2) * (size_t)(p.fft_len + 2 * (2 * 5 + p.fft_len));    // twiddles + the two candidate groups
    LAUNCH(coarse_chain_kernel, (unsigned)D, CHAIN_THREADS, chain_smem, st, src, w.ctl, len, p.fft_len, p.th, p.step10, p.step11, p.dr, cap, w.coarse_pos, w.coarse_snr,
           g_debug_prof ? (unsigned long long *)(w.pass_hist + 16) + 48 : nullptr);
    return GSMCAL_OK;
}

constexpr int kNeedGroup = 8;      // bursts per block of the fallback kernels that run behind a need-mask (tone_est_kernel, tier 2)
int run_fine_peak(Ctx &c, WinSrc src_peak, i64 n_iq, int osr, i64 D, int cap, Work &w, cudaStream_t st) {
    const double2 *tw; TRY(get_twiddle(c, 148 * osr, st, &tw));
    if (g_debug_force_full || (osr % 4) != 0) {      // the band kernel's 16-sample certificate grid needs osr % 4 == 0
        LAUNCH(fine_peak_full_kernel, dim3((unsigned)cap, (unsigned)D), kFineThreads, fine_smem(osr), st, src_peak, w.ctl, w.coarse_pos, cap, osr, n_iq, tw, w.fine_raw, (const int *)nullptr, (const int *)nullptr, 0);
        return GSMCAL_OK;
    }
    CU(cudaMemsetAsync(w.need_full, 0, sizeof(int) * D * cap, st));
    CU(cudaMemsetAsync(w.need_band, 0, sizeof(int) * D * cap, st));
    w.wc_valid = false;
    if (src_peak.lazy && osr == 8 && src_peak.n_taps <= 64 && !g_debug_no_core8) {
        // osr-8 fast path: FIR once per burst, filtered window cached for tier 2 and the tone stages
        const dim3 grid((unsigned)cap, (unsigned)D);
#define CORE8_ARGS src_peak.raw, n_iq, w.ctl, w.coarse_pos, cap, tw, w.fine_raw, w.need_band, g_debug_fail_tier2, w.wcache, g_debug_core8_passes, w.pass_hist, \
                   (unsigned long long *)(w.pass_hist + 16)
        if (src_peak.n_taps == 47 && g_debug_prof) LAUNCH((fine_core8_kernel<47, true>), grid, B8_THREADS, B8_SMEM, st, CORE8_ARGS);
        else if (src_peak.n_taps == 47) LAUNCH((fine_core8_kernel<47, false>), grid, B8_THREADS, B8_SMEM, st, CORE8_ARGS);
        else if (src_peak.n_taps <= 48) LAUNCH((fine_core8_kernel<48, false>), grid, B8_THREADS, B8_SMEM, st, CORE8_ARGS);
        else                            LAUNCH((fine_core8_kernel<64, false>), grid, B8_THREADS, B8_SMEM, st, CORE8_ARGS);
#undef CORE8_ARGS
        w.wc_valid = (w.wcache != nullptr);
        src_peak = with_cache(src_peak, w, cap);
    } else
    LAUNCH(fine_peak_core_kernel, dim3((unsigned)cap, (unsigned)D), FC_THREADS, fine_band_smem(osr), st, src_peak, w.ctl, w.coarse_pos, cap, osr, n_iq, tw, w.fine_raw, w.need_band, g_debug_fail_tier2);
    CU(cudaMemsetAsync(w.fall_count, 0, sizeof(int), st));
    LAUNCH(fine_peak_band_kernel, dim3((unsigned)((cap + kNeedGroup - 1) / kNeedGroup), (unsigned)D), FB_THREADS, fine_band_smem(osr), st, src_peak, w.ctl, w.coarse_pos, cap, osr, n_iq, tw, w.fine_raw,
           (const int *)w.need_band, w.need_full, 0, w.fall_list, w.fall_count, w.fall_best, w.fall_m, g_debug_fail_tier2, kNeedGroup);
    const int nb3 = (148 * osr + FB_BINS - 1) / FB_BINS;
    LAUNCH(fine_peak_band_kernel, dim3((unsigned)nb3, (unsigned)FALL_GRID), FB_THREADS, fine_band_smem(osr), st, src_peak, w.ctl, w.coarse_pos, cap, osr, n_iq, tw, w.fine_raw,
           (const int *)nullptr, (int *)nullptr, 1, w.fall_list, w.fall_count, w.fall_best, w.fall_m, g_debug_fall_limit, 1);
    LAUNCH(fine_fall_combine_kernel, FALL_GRID / 128, 128, 0, st, w.fall_list, w.fall_count, w.fall_best, w.fall_m, nb3, w.coarse_pos, cap, osr, w.fine_raw, w.ctl, g_debug_fall_limit);
    LAUNCH(fine_peak_full_kernel, 296, kFineThreads, fine_smem(osr), st, src_peak, w.ctl, w.coarse_pos, cap, osr, n_iq, tw, w.fine_raw,
           (const int *)w.fall_list, (const int *)w.fall_count, g_debug_fall_limit);
    return GSMCAL_OK;
}
// per-burst tone estimate: with the filtered-window cache (osr 8) tone8_kernel does every burst it can certify and flags the others
// for the generic row-FFT kernel; without a cache the generic kernel does them all
int run_tone(WinSrc src, int which, const double *pos, int osr, i64 D, int cap, const double2 *tw, Work &w, cudaStream_t st) {
    const int *need = nullptr;
    if (src.lazy && src.wcache && osr == 8 && !g_debug_no_tone8) {
        CU(cudaMemsetAsync(w.tone_need, 0, sizeof(int) * D * cap, st));
        unsigned long long *prof = (unsigned long long *)(w.pass_hist + 16) + 16 * which;      // [1]: fine stage, [2]: post stage (debug key 13)
        if (g_debug_prof) LAUNCH(tone8_kernel<true>, dim3((unsigned)cap, (unsigned)D), T8_THREADS, T8_SMEM, st, src, w.ctl, which, pos, cap, tw, w.fo, w.gate, w.tone_need, prof);
        else              LAUNCH(tone8_kernel<false>, dim3((unsigned)cap, (unsigned)D), T8_THREADS, T8_SMEM, st, src, w.ctl, which, pos, cap, tw, w.fo, w.gate, w.tone_need, prof);
        need = w.tone_need;
    }
    const int gsz = need ? kNeedGroup : 1;                       // behind tone8_kernel's mask: groups of bursts per block (few or none are flagged)
    LAUNCH(tone_est_kernel, dim3((unsigned)((cap + gsz - 1) / gsz), (unsigned)D), TONE_THREADS, tone_smem(osr), st, src, w.ctl, which, pos, cap, osr, tw, w.fo, w.gate, need, gsz);
    return GSMCAL_OK;
}

int run_fine_rest(Ctx &c, WinSrc src_tone, i64 n_iq, int osr, double carrier_freq, i64 D, int cap, Work &w, cudaStream_t st) {
    const double2 *tw; TRY(get_twiddle(c, 148 * osr, st, &tw));
    LAUNCH(fine_ppm_kernel, (unsigned)D, PS_THREADS, (size_t)cap * 17 + 16, st, w.ctl, (int)D, cap, osr, n_iq, w.fine_raw, w.fcch_pos, w.kind);
    TRY(run_tone(src_tone, 1, w.fcch_pos, osr, D, cap, tw, w, st));
    LAUNCH(fine_carrier_kernel, (unsigned)D, PS_THREADS, (size_t)cap * 16, st, w.ctl, (int)D, cap, osr, carrier_freq, w.fo, w.gate);
    return GSMCAL_OK;
}

int run_fine(Ctx &c, WinSrc src_peak, WinSrc src_tone, i64 n_iq, int osr, double carrier_freq, i64 D, int cap, Work &w, cudaStream_t st) {
    TRY(run_fine_peak(c, src_peak, n_iq, osr, D, cap, w, st));
    return run_fine_rest(c, src_tone, n_iq, osr, carrier_freq, D, cap, w, st);
}

int run_sch(WinSrc src, int osr, i64 D, int cap, Work &w, cudaStream_t st) {
    LAUNCH(sch_corr_kernel, dim3((unsigned)cap, (unsigned)D), SCH_THREADS, sch_smem(osr), st,
           src, w.ctl, w.fcch_pos, cap, osr, w.tpl, w.tplf, w.tpl_e, g_debug_sch_mode, w.sch_stats, w.sch_raw, w.sch_edge);
    LAUNCH(sch_ppm_kernel, (unsigned)D, PS_THREADS, (size_t)cap * 21 + 16, st, w.ctl, (int)D, cap, osr, w.sch_raw, w.sch_edge, w.sch_pos, w.kind, w.pos_info, w.post_pos);
    return GSMCAL_OK;
}

int run_post(Ctx &c, WinSrc src, int osr, double carrier_freq, i64 D, int cap, Work &w, bool want_res, cudaStream_t st) {
    const double2 *tw; TRY(get_twiddle(c, 148 * osr, st, &tw));
    TRY(run_tone(src, 2, w.post_pos, osr, D, cap, tw, w, st));
    LAUNCH(post_carrier_kernel, (unsigned)D, PS_THREADS, (size_t)cap * 8, st, w.ctl, (int)D, cap, osr, carrier_freq, w.fo, want_res ? w.res : nullptr);
    return GSMCAL_OK;
}

template <bool U8>
int run_fir(const void *in, i64 n, i64 in_stride, const StreamCtl *ctl, int n_taps, int decim, i64 D, double2 *out, i64 n_out, double *power, cudaStream_t st) {
    if (decim < 1) return fail(GSMCAL_ERR_ARG, "decim must be >= 1");
    if (n <= 0) return GSMCAL_OK;
    if (decim == 1 && !power && !U8 && n_taps <= 64 && in_stride == n && n_out == n && (((uintptr_t)in & 15) == 0)) {
        // complex128 in/out: persistent TMA-pipelined kernel
        const i64 n_tiles = ((n + FT_TILE - 1) / FT_TILE) * D;
        i64 gx = 148 * 4; if (gx > n_tiles) gx = n_tiles;        // 4 resident blocks per SM (122 registers, 38 KB)
        if (n_taps <= 48) LAUNCH((fir_full_tma_kernel<48>), (unsigned)gx, FT_THREADS, sizeof(double2) * 2 * (FT_TILE + 47), st, (const double2 *)in, n, D, out);
        else              LAUNCH((fir_full_tma_kernel<64>), (unsigned)gx, FT_THREADS, sizeof(double2) * 2 * (FT_TILE + 63), st, (const double2 *)in, n, D, out);
        return GSMCAL_OK;
    }
    if (decim == 1 && !power) {
        unsigned gx = (unsigned)((n + FIR_TILE - 1) / FIR_TILE);
        auto smem = [](int NT) { int n_in = FIR_TILE + NT - 1; return sizeof(double2) * (size_t)(n_in + n_in / 8 + 2); };
        if (n_taps <= 32)      LAUNCH((fir_full_kernel<32, U8>), dim3(gx, (unsigned)D), FIR_THREADS, smem(32), st, in, n, in_stride, ctl, out, n_out);
        else if (n_taps <= 48) LAUNCH((fir_full_kernel<48, U8>), dim3(gx, (unsigned)D), FIR_THREADS, smem(48), st, in, n, in_stride, ctl, out, n_out);
        else if (n_taps <= 64) LAUNCH((fir_full_kernel<64, U8>), dim3(gx, (unsigned)D), FIR_THREADS, smem(64), st, in, n, in_stride, ctl, out, n_out);
        else                   LAUNCH((fir_full_kernel<128, U8>), dim3(gx, (unsigned)D), FIR_THREADS, smem(128), st, in, n, in_stride, ctl, out, n_out);
        return GSMCAL_OK;
    }
    if (U8 && decim >= n_taps && (decim % 4) == 0 && n_taps <= 64) {
        unsigned gx = (unsigned)((n_out + FDD_THREADS - 1) / FDD_THREADS);
        LAUNCH(fir_decim_direct_u8_kernel<17>, dim3(gx, (unsigned)D), FDD_THREADS, 0, st, (const uint8_t *)in, n, ctl, n_taps, decim, out, n_out, power);
        return GSMCAL_OK;
    }
    int opb = 2048 / decim; if (opb < 1) opb = 1; if (opb > 1024) opb = 1024;
    int n_in = (opb - 1) * decim + n_taps;
    size_t smem = sizeof(double2) * (size_t)(n_in + n_in / 8 + 2);
    unsigned gx = (unsigned)((n_out + opb - 1) / opb);
    LAUNCH(fir_decim_kernel<U8>, dim3(gx, (unsigned)D), FIRD_THREADS, smem, st, in, n, in_stride, ctl, n_taps, decim, opb, out, n_out, n_out, power);
    return GSMCAL_OK;
}

int run_resample_derotate(const double2 *in, i64 len_in, double e, int do_interp, double dphi, int do_derot, double2 *out, i64 len_out, cudaStream_t st) {
    if (len_out <= 0) return GSMCAL_OK;
    unsigned g = (unsigned)((len_out + 256 * DEROT_K - 1) / (256 * DEROT_K));
    LAUNCH(resample_derotate_kernel, g, 256, 0, st, in, len_in, e, do_interp, dphi, do_derot, out, len_out);
    return GSMCAL_OK;
}

int check_fir_args(const double *coef, int n_taps, const void *s, i64 n, i64 n_col, const void *r) {
    if (!coef || !s || !r || n < 0 || n_col < 1) return fail(GSMCAL_ERR_ARG, "null pointer or negative size");
    if (n_taps < 1 || n_taps > GSMCAL_MAX_TAPS) return fail(GSMCAL_ERR_ARG, "n_taps must be 1..%d", GSMCAL_MAX_TAPS);
    return GSMCAL_OK;
}

// ---- what the drop-in entry points share (they run on stream 0; fcch_scan passes the caller's stream) ---------------------------
// They touch the device, so every entry point calls them after its host-decided sentinels and argument errors.
// one complex128 stream: the device's context, s (n samples) on the device and a one-stream workspace of cap bursts
int upload_s(const double *s, i64 n, int cap, i64 snr_len, int tpl_len, cudaStream_t st, Ctx **c, const double2 **din, Work *w) {
    TRY(get_ctx(c));
    void *p; TRY((*c)->in.get(sizeof(double2) * (size_t)n, &p));
    TRY(make_work((*c)->work, 1, cap, snr_len, tpl_len, w));
    TRY(copy_h2d((*c)->ring, g_device, p, s, sizeof(double2) * (size_t)n, st));
    *din = (const double2 *)p;
    return GSMCAL_OK;
}
// n_col columns of n_iq uint8 I/Q pairs as the kernels read them: a workspace of n_col streams x cap bursts, the FIR taps when coef is
// given, a device copy of a host capture, and the column sums behind zeroed control blocks
int u8_input(Ctx &c, const uint8_t *a, int mem, i64 n_iq, i64 n_col, int cap, i64 snr_len, const double *coef, int n_taps, cudaStream_t st,
             const uint8_t **draw, Work *w) {
    const size_t bytes = (size_t)2 * n_iq * n_col;
    void *p = (void *)a;
    if (mem == GSMCAL_MEM_HOST) TRY(c.in.get(bytes, &p));
    TRY(make_work(c.work, n_col, cap, snr_len, 0, w));
    if (coef) TRY(set_taps(coef, n_taps, st));
    if (mem == GSMCAL_MEM_HOST) TRY(copy_h2d(c.ring, g_device, p, a, bytes, st));
    CU(cudaMemsetAsync(w->ctl, 0, sizeof(StreamCtl) * n_col, st));
    *draw = (const uint8_t *)p;
    return run_colsum_u8(*draw, n_iq, n_col, w->ctl, st);
}
unsigned raw2iq_grid(i64 n_iq) { i64 gx = (n_iq + 256 * 8 - 1) / (256 * 8); if (gx > 148 * 16) gx = 148 * 16; return (unsigned)gx; }
// one stream's control block to / from the host, complete on return
int put_ctl(StreamCtl *dev, const StreamCtl &h, cudaStream_t st) {
    CU(cudaMemcpyAsync(dev, &h, sizeof h, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return GSMCAL_OK;
}
int get_ctl(const StreamCtl *dev, StreamCtl *h, cudaStream_t st) {
    CU(cudaMemcpyAsync(h, dev, sizeof *h, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GSMCAL_OK;
}
// r (len samples) of a correction drop-in: s (n samples, din on the device) resampled by (1+e) and / or derotated by dphi, or s itself
int return_r(Ctx &c, const double *s, const double2 *din, i64 n, i64 len, double e, int do_interp, double dphi, int do_derot, double *r,
             cudaStream_t st) {
    if (!do_interp && !do_derot) { memcpy(r, s, sizeof(double2) * (size_t)len); return GSMCAL_OK; }
    void *dout; TRY(c.out.get(sizeof(double2) * (size_t)len, &dout));
    TRY(run_resample_derotate(din, n, e, do_interp, dphi, do_derot, (double2 *)dout, len, st));
    return copy_d2h(c.ring, g_device, r, dout, sizeof(double2) * (size_t)len, st);
}

void gmsk_template(int osr, double *out);
size_t fcch_demod_smem(int osr);
size_t sch_demod_smem(int osr);
void gmsk_branch_table(int osr, double *W);
void sch_training_pm(signed char *data_pm);

// ---- the stage behind post-SCH ("tail") of gsmcal_calibrate_demod_batch, _demod_bcch_batch, _sch_decode_batch, _sch_timing_batch,
// _carrier_fit_batch, _cell_batch and _sysinfo_batch --
// It is the SCH timing block when `timing` is set, the carrier fit block when `carrier` is set (with `sdec`: then the residual-corrected
// SCH_demod and the SCH decoding block, and with `si` as well the BCCH decoding block), else the demod block (batched SCH_demod / FCCH_demod) with the BCCH block when `nts` is set and
// the SCH decoding block when `sdec` is set.
struct TailOut {                     // the caller's host outputs; an array left NULL is not read back
    gsmcal_demod_result *demod; uint8_t *sch_ok, *bits, *dec; double *corr, *freq, *snr, *idx;
    const double *nts; gsmcal_bcch_result *bcch;
    gsmcal_sch_decode_result *sdec; int32_t *fn, *bsic; uint8_t *ham, *rflag;
    gsmcal_sch_timing_result *timing; double *tau, *x;
    gsmcal_carrier_fit_result *carrier; double *cf_f, *cf_t; uint8_t *cf_flag;
    double *sch_df;
    gsmcal_sysinfo_result *si; int8_t *lag; uint8_t *bflag, *steal; int32_t *bfn; uint8_t *btc, *bblk; uint16_t *bham; uint8_t *pay;
};
struct TailDev {                     // device buffers of the same blocks
    DemodResultDev *rec; double *sch_pos, *fcch_pos; unsigned char *sch_ok, *fcch_ok;                       // the row lists
    double *corr, *freq, *snr, *idx; unsigned char *bits, *dec; double2 *Ft /* N */, *Wtab /* 16*osr */; signed char *dpm /* 64 */;
    double2 *nts /* (26*osr) x 8 */; BcchResultDev *bcch;
    SchDecodeResultDev *sdec; int *key, *fn, *bsic; unsigned char *ham, *rflag;
    TimingResultDev *timing; double *tau, *x; unsigned char *row_flag;
    CarrierFitDev *carrier; double *cf_f, *cf_t; unsigned char *cf_flag;
    double *sch_df;
    SysinfoDev *si; int *blk_n; double *blk_pos; unsigned char *blk_nrow; signed char *lag; unsigned char *bflag, *steal;
    unsigned long long *ibits, *skey; int *bfn; unsigned char *btc, *bblk; unsigned short *bham; unsigned char *pay;
};
// every per-stream array ([D] records, [D][cap] rows) of the blocks `o` asks for: f(device pointer, bytes per stream, the caller's host
// array or NULL).  Set-up, the slice of a stream group and the read-back all walk this one list.  The per-call constants (Ft, Wtab, dpm,
// nts) are not in it.
template <class F> void tail_arrays(TailDev &t, const TailOut &o, int cap, F &&f) {
    const size_t r = (size_t)cap;
    f(t.rec, sizeof(DemodResultDev), o.demod); f(t.sch_pos, 8 * r, nullptr); f(t.fcch_pos, 8 * r, nullptr);
    f(t.sch_ok, r, o.sch_ok); f(t.fcch_ok, r, nullptr);
    if (o.timing) {
        f(t.timing, sizeof(TimingResultDev), o.timing); f(t.tau, 8 * r, o.tau); f(t.x, 8 * r, o.x); f(t.row_flag, r, nullptr);
        return;
    }
    if (o.carrier) {
        f(t.carrier, sizeof(CarrierFitDev), o.carrier); f(t.cf_f, 8 * r, o.cf_f); f(t.cf_t, 8 * r, o.cf_t); f(t.cf_flag, r, o.cf_flag);
        if (o.sdec) {                // the corrected SCH rows (bits_to_decoder is written, not returned) and their decoding
            f(t.bits, 148 * r, o.bits); f(t.dec, 148 * r, nullptr); f(t.corr, 8 * 85 * r, o.corr); f(t.sch_df, 8 * r, o.sch_df);
            f(t.sdec, sizeof(SchDecodeResultDev), o.sdec); f(t.key, 4 * r, nullptr); f(t.fn, 4 * r, o.fn); f(t.bsic, 4 * r, o.bsic);
            f(t.ham, r, o.ham); f(t.rflag, r, o.rflag);
        }
        if (o.si) {                  // the block list, the BCCH rows ([cap][4] per stream) and the blocks
            f(t.si, sizeof(SysinfoDev), o.si); f(t.blk_n, 4, nullptr); f(t.blk_pos, 8 * 4 * r, nullptr); f(t.blk_nrow, r, nullptr);
            f(t.lag, 4 * r, o.lag); f(t.bflag, 4 * r, o.bflag); f(t.steal, 4 * r, o.steal); f(t.ibits, 8 * 8 * r, nullptr);
            f(t.skey, 8 * r, nullptr); f(t.bfn, 4 * r, o.bfn); f(t.btc, r, o.btc); f(t.bblk, r, o.bblk); f(t.bham, 2 * r, o.bham);
            f(t.pay, 23 * r, o.pay);
        }
        return;
    }
    f(t.bits, 148 * r, o.bits); f(t.dec, 148 * r, o.dec); f(t.corr, 8 * 85 * r, o.corr); f(t.freq, 8 * r, o.freq); f(t.snr, 8 * r, o.snr);
    f(t.idx, 8 * r, o.idx);
    if (o.nts) f(t.bcch, sizeof(BcchResultDev), o.bcch);
    if (o.sdec) {
        f(t.sdec, sizeof(SchDecodeResultDev), o.sdec); f(t.key, 4 * r, nullptr); f(t.fn, 4 * r, o.fn); f(t.bsic, 4 * r, o.bsic);
        f(t.ham, r, o.ham); f(t.rflag, r, o.rflag);
    }
}
template <class T> void place(T *&p, uintptr_t a) { p = (T *)a; }
// the buffers of D streams in c.dem, and for the demod block the branch table, training bits and fft(template) (SCH_demod.m:47-59) and
// with nts (host, (26*osr) x 8 complex) the normal training sequences; once per call on `st` before the stream groups fork
// (gsmcal_SCH_demod: the demod block alone, one stream of its H bursts)
int tail_setup(Ctx &c, i64 D, int cap, int osr, const double2 *tpl_dev, const TailOut &o, std::vector<double> &W, signed char *data_pm,
               cudaStream_t st, TailDev *t) {
    const int N = SD_NSYM * osr;
    const bool sch = !o.timing && (!o.carrier || o.sdec);        // SCH rows are demodulated
    *t = TailDev{};
    auto layout = [&](uintptr_t base) {          // points every buffer into [base, base + the size it returns)
        size_t off = 0;
        auto take = [&](auto *&p, size_t bytes) { place(p, base + off); off = align_up(off + bytes); };
        tail_arrays(*t, o, cap, [&](auto *&p, size_t per, const void *) { take(p, per * D); });
        if (sch) { take(t->Ft, sizeof(double2) * N); take(t->Wtab, sizeof(double2) * 16 * osr); take(t->dpm, 64); }
        if (o.nts) take(t->nts, sizeof(double2) * 8 * 26 * osr);
        return off;
    };
    void *base; TRY(c.dem.get(layout(0), &base));
    layout((uintptr_t)base);
    if (!sch) return GSMCAL_OK;
    if (o.nts) CU(cudaMemcpyAsync(t->nts, o.nts, sizeof(double2) * 8 * 26 * (size_t)osr, cudaMemcpyHostToDevice, st));
    W.assign(2 * 16 * (size_t)osr, 0.0);
    gmsk_branch_table(osr, W.data());
    sch_training_pm(data_pm);
    CU(cudaMemcpyAsync(t->Wtab, W.data(), sizeof(double) * W.size(), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(t->dpm, data_pm, 64, cudaMemcpyHostToDevice, st));
    const double2 *tw; TRY(get_twiddle(c, N, st, &tw));
    LAUNCH(fde_template_kernel, 1, SD_THREADS, 3 * (size_t)N * sizeof(double2), st, tpl_dev, osr, tw, t->Ft);
    return GSMCAL_OK;
}
// one stream group: row lists + sentinels, then either the timing of every SCH row and the per-stream fit (osr 8), or the tone of every
// FCCH row and the per-stream carrier fit (osr 8) with, for _cell_batch, the SCH bursts less the fitted residual and their decoding (and
// for _sysinfo_batch the BCCH blocks behind them), or
// SCH bursts, SCH decoding and BCCH_demod when their outputs were asked for, FCCH
// bursts, FCCH means
int run_tail(Ctx &c, WinSrc src, const Work &ws, const TailDev &t, int osr, double carrier_freq, i64 nd, int cap, cudaStream_t st) {
    LAUNCH(demod_compact_kernel, (unsigned)nd, 32, 0, st, ws.ctl, ws.pos_info, cap, osr, t.rec, t.sch_pos, t.sch_ok, t.fcch_pos, t.fcch_ok);
    if (t.timing) {
        LAUNCH(sch_timing_batch_kernel, dim3((unsigned)cap, (unsigned)nd), SCH_THREADS, TM_SMEM, st, src, ws.ctl, t.rec, t.sch_pos, cap, ws.tpl,
               t.tau, t.row_flag);
        LAUNCH(sch_timing_fit_kernel, (unsigned)nd, 32, 0, st, ws.ctl, t.rec, t.sch_pos, t.row_flag, t.tau, cap, t.x, t.timing);
        return GSMCAL_OK;
    }
    if (t.carrier) {
        LAUNCH(carrier_fit_row_kernel, dim3((unsigned)cap, (unsigned)nd), CF_THREADS, CF_SMEM, st, with_cache(src, ws, cap), ws.ctl, t.rec, t.fcch_pos,
               t.fcch_ok, cap, t.cf_f, t.cf_t, t.cf_flag);
        LAUNCH(carrier_fit_stream_kernel, (unsigned)nd, 32, 0, st, ws.ctl, t.rec, t.cf_flag, t.cf_f, t.cf_t, cap, carrier_freq, t.carrier);
        if (!t.sdec) return GSMCAL_OK;
        const double2 *tw_s; TRY(get_twiddle(c, SD_NSYM * osr, st, &tw_s));        // built by the set-up: no launch here
        LAUNCH(sch_demod_resid_kernel, dim3((unsigned)cap, (unsigned)nd), SDB_THREADS, sch_demod_smem(osr), st, src, ws.ctl, t.rec, t.sch_pos, t.sch_ok,
               cap, tw_s, t.Ft, t.Wtab, t.dpm, t.carrier, t.bits, t.dec, t.corr, t.sch_df);
        LAUNCH(sch_decode_batch_kernel, (unsigned)nd, 32, 0, st, t.rec, t.sch_pos, t.sch_ok, t.bits, t.corr, cap, osr, t.key, t.fn, t.bsic,
               t.ham, t.rflag, t.sdec);
        if (!t.si) return GSMCAL_OK;
        LAUNCH(bcch_block_kernel, (unsigned)((nd + 127) / 128), 128, 0, st, ws.ctl, ws.pos_info, t.rec, (int)nd, cap, t.blk_n, t.blk_pos, t.blk_nrow);
        LAUNCH(bcch_burst_kernel, dim3(4 * (unsigned)cap, (unsigned)nd), BB_THREADS, BB_SMEM, st, src, ws.ctl, t.blk_n, t.blk_pos, t.blk_nrow, t.sdec,
               t.carrier, t.nts, t.Wtab, cap, t.lag, t.bflag, t.steal, t.ibits);
        LAUNCH(bcch_decode_kernel, (unsigned)nd, 32, 0, st, t.rec, t.sdec, t.carrier, t.sch_pos, t.blk_n, t.blk_pos, t.blk_nrow, t.bflag, t.ibits, cap,
               t.skey, t.bfn, t.btc, t.bblk, t.bham, t.pay, t.si);
        return GSMCAL_OK;
    }
    const double2 *tw_s, *tw_f;                  // both built by the set-up: no launch here
    TRY(get_twiddle(c, SD_NSYM * osr, st, &tw_s));
    TRY(get_twiddle(c, 148 * osr, st, &tw_f));
    LAUNCH(sch_demod_batch_kernel, dim3((unsigned)cap, (unsigned)nd), SDB_THREADS, sch_demod_smem(osr), st, src, ws.ctl, t.rec, t.sch_pos, t.sch_ok,
           cap, osr, tw_s, t.Ft, t.Wtab, t.dpm, t.bits, t.dec, t.corr);
    if (t.sdec)
        LAUNCH(sch_decode_batch_kernel, (unsigned)nd, 32, 0, st, t.rec, t.sch_pos, t.sch_ok, t.bits, t.corr, cap, osr, t.key, t.fn, t.bsic,
               t.ham, t.rflag, t.sdec);
    const size_t fs = fcch_demod_smem(osr), fs_load = sizeof(double2) * (3 * 148 * (size_t)osr + 144);      // + the loader's scratch behind u
    LAUNCH(fcch_demod_batch_kernel, dim3((unsigned)cap, (unsigned)nd), FD_THREADS, fs > fs_load ? fs : fs_load, st, with_cache(src, ws, cap), ws.ctl, t.rec,
           t.fcch_pos, t.fcch_ok, cap, osr, tw_f, t.freq, t.snr, t.idx);
    LAUNCH(demod_fcch_mean_kernel, (unsigned)((nd + 127) / 128), 128, 0, st, t.rec, (int)nd, t.freq, cap, carrier_freq);
    if (t.bcch) {
        const int L = 26 * osr;
        LAUNCH(bcch_demod_batch_kernel, (unsigned)nd, BC_THREADS, sizeof(double2) * (size_t)(L + GSMCAL_XCAP(L) + L + 8), st, src, ws.ctl, t.rec, ws.pos_info,
               cap, osr, t.nts, t.bcch);
    }
    return GSMCAL_OK;
}

// ---- what gsmcal_calibrate_batch* and gsmcal_calibrate_batch_submit share ---------------------------------------------------------
// `to` waits for what has been enqueued on `from` so far
int hand_off(cudaStream_t from, cudaStream_t to) {
    cudaEvent_t ev; CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(cudaEventRecord(ev, from)); CU(cudaStreamWaitEvent(to, ev, 0)); CU(cudaEventDestroy(ev));
    return GSMCAL_OK;
}

struct Batch { CoarseParams p; int dec; i64 len_dec; int cap; Work w; };
// argument checks and sizes; no device is touched, so a malformed call fails the same way on every machine
int batch_args(const char *name, const void *raw, const double *tpl, const double *coef, const void *results, i64 n_iq, i64 D, int osr,
               int coarse_dr, Batch *b) {
    if (!raw || !tpl || !coef || !results || n_iq < 1 || D < 1 || osr < 1 || osr > 8) return fail(GSMCAL_ERR_ARG, "%s: bad arguments (osr 1..8)", name);
    TRY(coarse_params(coarse_dr, &b->p));
    b->dec = osr * coarse_dr;
    b->len_dec = (n_iq + b->dec - 1) / b->dec;
    if (b->p.n_first > b->len_dec) return fail(GSMCAL_ERR_RANGE, "%s: capture shorter than 23 frames", name);
    b->cap = (int)gsmcal_max_bursts(b->len_dec, coarse_dr);
    return GSMCAL_OK;
}
// the per-call set-up on st: workspace and window cache, FIR taps, zeroed control blocks and counters, the packed SCH template (through
// h_tpl, tpl_pack_bytes(64 * osr) bytes that stay valid until the copy has run) and the twiddles, built before the stream groups fork
int batch_setup(Ctx &c, DevBuf &work, DevBuf &wc, const double *tpl, const double *coef, int n_taps, int osr, i64 D, unsigned char *h_tpl,
                cudaStream_t st, Batch *b) {
    Work &w = b->w;
    const int cap = b->cap;
    TRY(make_work(work, D, cap, b->p.n_first, 64 * osr, &w));
    TRY(attach_wcache(wc, D, cap, osr, &w));
    TRY(set_taps(coef, n_taps, st));
    CU(cudaMemsetAsync(w.ctl, 0, sizeof(StreamCtl) * D, st));
    CU(cudaMemsetAsync(w.need_full, 0, sizeof(int) * D * cap, st));
    CU(cudaMemsetAsync(w.need_band, 0, sizeof(int) * D * cap, st));
    tpl_pack(tpl, 64 * osr, h_tpl);
    CU(cudaMemcpyAsync((void *)w.tpl, h_tpl, tpl_pack_bytes(64 * osr), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(w.sch_stats, 0, sizeof(unsigned) * SCH_NSTAT, st));
    { const double2 *twp; TRY(get_twiddle(c, 148 * osr, st, &twp)); }
    CU(cudaMemsetAsync(w.pass_hist, 0, sizeof(unsigned) * 16 + sizeof(unsigned long long) * 64, st));
    g_last_sch_stats = w.sch_stats;
    g_last_need_full = w.need_full; g_last_need_band = w.need_band; g_last_need_full_n = (long long)D * cap;
    g_last_pass_hist = w.pass_hist;
    return GSMCAL_OK;
}

// the burst stages of one stream group, in order on sg: fine peak, fine rest (ppm, tone, carrier), SCH, post-SCH and, with tail, the tail
// stage.  With marks, marks[i] is recorded on sg behind stage i (null entries are skipped)
int run_burst_stages(Ctx &c, const uint8_t *graw, i64 n_iq, int n_taps, int osr, double carrier_freq, i64 nd, int cap, Work &ws,
                     const TailDev *tail, cudaStream_t sg, const cudaEvent_t *marks) {
    auto mark = [&](int i) { if (marks && marks[i]) CU(cudaEventRecord(marks[i], sg)); return GSMCAL_OK; };
    TRY(run_fine_peak(c, lazy_src(graw, n_iq, n_taps, 0, 1), n_iq, osr, nd, cap, ws, sg));
    TRY(mark(0));
    TRY(run_fine_rest(c, with_cache(lazy_src(graw, n_iq, n_taps, 1, 1), ws, cap), n_iq, osr, carrier_freq, nd, cap, ws, sg));
    TRY(mark(1));
    TRY(run_sch(lazy_src(graw, n_iq, n_taps, 2, 1), osr, nd, cap, ws, sg));
    TRY(mark(2));
    TRY(run_post(c, with_cache(lazy_src(graw, n_iq, n_taps, 3, 1), ws, cap), osr, carrier_freq, nd, cap, ws, true, sg));
    TRY(mark(3));
    if (tail) {
        TRY(run_tail(c, lazy_src(graw, n_iq, n_taps, 3, 1), ws, *tail, osr, carrier_freq, nd, cap, sg));
        TRY(mark(4));
    }
    return GSMCAL_OK;
}

}  // namespace

// ====================================================================================================
extern "C" {

int gsmcal_abi_version(void) { return GSMCAL_ABI_VERSION; }
const char *gsmcal_last_error(void) { return g_err.c_str(); }
int gsmcal_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int gsmcal_set_device(int device) {
    int n = gsmcal_device_count();
    if (device < 0 || device >= n) return fail(GSMCAL_ERR_CUDA, "device %d not available (%d devices)", device, n);
    g_device = device;
    return GSMCAL_OK;
}
void gsmcal_release(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    g_last_need_full = nullptr; g_last_need_band = nullptr; g_last_need_full_n = 0; g_last_pass_hist = nullptr; g_prev_pass_hist = nullptr; g_last_sch_stats = nullptr;   // they point into the workspaces freed below
    for (auto &kv : g_ctx) {
        cudaSetDevice(kv.first);
        kv.second.ring.release(); kv.second.in.release(); kv.second.out.release(); kv.second.work.release(); kv.second.tplbuf.release(); kv.second.wc.release(); kv.second.dem.release();
        for (auto &t : kv.second.tw) cudaFree(t.second);
        kv.second.tw.clear();
        if (kv.second.stage_ev_ok) { for (cudaEvent_t e : kv.second.stage_ev) cudaEventDestroy(e); kv.second.stage_ev_ok = false; }
        for (cudaStream_t s2 : kv.second.side) cudaStreamDestroy(s2);
        kv.second.side.clear();
        for (cudaStream_t s2 : kv.second.side_hi) cudaStreamDestroy(s2);
        kv.second.side_hi.clear();
        for (Slot &sl : kv.second.slots) {
            if (sl.done) { cudaEventSynchronize(sl.done); cudaEventDestroy(sl.done); sl.done = nullptr; }
            for (cudaStream_t s2 : sl.grp) cudaStreamDestroy(s2);
            for (cudaStream_t s2 : sl.hi) cudaStreamDestroy(s2);
            if (sl.front_hi) cudaStreamDestroy(sl.front_hi);
            sl.front_hi = nullptr;
            sl.grp.clear(); sl.hi.clear();
            if (sl.stage) cudaFreeHost(sl.stage);
            sl.stage = nullptr; sl.stage_cap = 0; sl.busy = false;
            sl.work.release(); sl.wc.release();
        }
    }
}
int64_t gsmcal_debug_get(int key) {
    // key 1: bursts of the last fine search (this device) that needed the all-bin fallback
    std::lock_guard<std::mutex> lk(g_mu);
    if (key == 40) return (int64_t)g_debug_core8_passes;
    if (key >= 150 && key < 214) {                               // the same counters of the batch submitted before the last one (other slot)
        if (!g_prev_pass_hist) return 0;
        unsigned long long v = 0;
        if (cudaMemcpy(&v, (unsigned long long *)(g_prev_pass_hist + 16) + (key - 150), sizeof v, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return (int64_t)v;
    }
    if (key >= 50 && key < 114) {                                 // per-phase cycle sums (debug key 13), [15] = blocks: 50.. fine_core8, 66.. tone8 (fine), 82.. tone8 (post)
        if (!g_last_pass_hist) return 0;
        unsigned long long v = 0;
        if (cudaMemcpy(&v, (unsigned long long *)(g_last_pass_hist + 16) + (key - 50), sizeof v, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return (int64_t)v;
    }
    if (key >= 120 && key < 121 + SCH_NSTAT) {                  // sch_corr_kernel counters of the last call (SCH_NSTAT)
        if (!g_last_sch_stats) return 0;
        unsigned h[SCH_NSTAT];
        if (cudaMemcpy(h, g_last_sch_stats, sizeof h, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        if (key == 120) { int64_t n = 0; for (int k = 1; k < SCH_NSTAT; ++k) n += h[k]; return n; }
        return (int64_t)h[key - 121];
    }
    if (key == 30) return (int64_t)g_staged_bytes.load();           // bytes that went through the pinned staging ring (pageable host buffers)
    if (key >= 10 && key < 26) {                                 // 10 + p: bursts the osr-8 tier-1 kernel proved after p passes (p = 0: left open)
        if (!g_last_pass_hist) return 0;
        unsigned v = 0;
        if (cudaMemcpy(&v, g_last_pass_hist + (key - 10), sizeof v, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return (int64_t)v;
    }
    if (key == 1 || key == 2) {
        const int *src = (key == 1) ? g_last_need_full : g_last_need_band;
        if (!src || g_last_need_full_n <= 0) return 0;
        std::vector<int> h((size_t)g_last_need_full_n);
        if (cudaMemcpy(h.data(), src, sizeof(int) * h.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        int64_t n = 0;
        for (int v : h) n += (v != 0);
        return n;
    }
    return -1;
}
int gsmcal_debug_set(int key, int value) {
    if (key == 0) { g_debug_force_full = value; return GSMCAL_OK; }
    if (key == 4) { g_debug_fail_tier2 = value; return GSMCAL_OK; }
    if (key == 5) { g_debug_fall_limit = value < 0 ? 0 : (value > FALL_GRID ? FALL_GRID : value); return GSMCAL_OK; }
    if (key == 6) { g_debug_hi_prio = value ? 1 : 0; return GSMCAL_OK; }
    if (key == 9) { g_debug_no_core8 = value ? 1 : 0; return GSMCAL_OK; }
    if (key == 11) { g_debug_no_tone8 = value ? 1 : 0; return GSMCAL_OK; }
    if (key == 12) { g_debug_no_staging = value ? 1 : 0; return GSMCAL_OK; }
    if (key == 13) { g_debug_prof = value ? 1 : 0; return GSMCAL_OK; }
    if (key == 14) { g_debug_timeline = value ? 1 : 0; return GSMCAL_OK; }
    if (key == 24) { if (value < 0 || value > 2) return fail(GSMCAL_ERR_ARG, "debug_set 24: 0, 1 or 2"); g_debug_sch_mode = value; return GSMCAL_OK; }
    if (key == 17) { g_debug_trickle = value < 1 ? 1 : (value > 24 ? 24 : value); return GSMCAL_OK; }
    if (key == 18) { g_debug_trickle_blocks = value < 1 ? 1 : (value > 4 ? 4 : value); return GSMCAL_OK; }
    if (key == 10) { g_debug_core8_passes = value < 1 ? 1 : (value > 8 ? 8 : value); return GSMCAL_OK; }
    if (key == 8) { g_debug_submit_groups = value < 1 ? 1 : (value > kMaxGroups / 2 ? kMaxGroups / 2 : value); return GSMCAL_OK; }
    if (key == 3) { g_debug_groups = value < 1 ? 1 : (value > kMaxGroups / 2 ? kMaxGroups / 2 : value); return GSMCAL_OK; }
    return fail(GSMCAL_ERR_ARG, "debug_set: unknown key");
}
int64_t gsmcal_launch_count(int reset) { long long v = g_launches.load(); if (reset) g_launches = 0; return v; }

int64_t gsmcal_max_bursts(int64_t len_decimated, int decimation_ratio) {
    const double num_sym_per_frame = (625.0 / 4.0) * 8.0;
    return (int64_t)ceil((double)len_decimated / (10.0 * num_sym_per_frame / decimation_ratio)) + 2;
}

// ---------------------------------------------------------------------------------------------------
int gsmcal_raw2iq_u8(const uint8_t *a, int64_t n_iq, int64_t n_col, double *b) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!a || !b || n_iq < 0 || n_col < 1) return fail(GSMCAL_ERR_ARG, "raw2iq: bad arguments");
    if (n_iq == 0) return GSMCAL_OK;
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = 0;
    const uint8_t *din; void *dout; Work w;
    TRY(c->out.get(sizeof(double2) * (size_t)n_iq * n_col, &dout));
    TRY(u8_input(*c, a, GSMCAL_MEM_HOST, n_iq, n_col, 1, 1, nullptr, 0, st, &din, &w));
    LAUNCH(raw2iq_store_kernel, dim3(raw2iq_grid(n_iq), (unsigned)n_col), 256, 0, st, din, n_iq, w.ctl, (double2 *)dout);
    TRY(copy_d2h(c->ring, g_device, b, dout, sizeof(double2) * (size_t)n_iq * n_col, st));
    return GSMCAL_OK;
}

int gsmcal_raw2iq_f64(const double *a, int64_t n_iq, int64_t n_col, double *b) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!a || !b || n_iq < 0 || n_col < 1) return fail(GSMCAL_ERR_ARG, "raw2iq: bad arguments");
    if (n_iq == 0) return GSMCAL_OK;
    for (int64_t i = 0; i < 2 * n_iq * n_col; ++i)
        if (!(a[i] >= 0.0 && a[i] <= 255.0 && a[i] == floor(a[i])))
            return fail(GSMCAL_ERR_ARG, "raw2iq: double input must hold integers 0..255 (what fread(...,'uint8') returns)");
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = 0;
    void *din, *dout; Work w;
    TRY(c->in.get(sizeof(double) * (size_t)2 * n_iq * n_col, &din));
    TRY(c->out.get(sizeof(double2) * (size_t)n_iq * n_col, &dout));
    TRY(make_work(c->work, n_col, 1, 1, 0, &w));
    TRY(copy_h2d(c->ring, g_device, din, a, sizeof(double) * (size_t)2 * n_iq * n_col, st));
    CU(cudaMemsetAsync(w.ctl, 0, sizeof(StreamCtl) * n_col, st));
    const dim3 grid(raw2iq_grid(n_iq), (unsigned)n_col);
    LAUNCH(colsum_f64_kernel, grid, 256, 0, st, (const double *)din, n_iq, w.ctl);
    LAUNCH(raw2iq_store_f64_kernel, grid, 256, 0, st, (const double *)din, n_iq, w.ctl, (double2 *)dout);
    TRY(copy_d2h(c->ring, g_device, b, dout, sizeof(double2) * (size_t)n_iq * n_col, st));
    return GSMCAL_OK;
}

// ---------------------------------------------------------------------------------------------------
int gsmcal_fir1(int order, double wn, double *coef) {
    // MATLAB fir1(n, Wn): low-pass, Hamming window, scaled so the DC gain is exactly 1 (gsm_sync_demod.m:34)
    if (order < 1 || order + 1 > GSMCAL_MAX_TAPS || !(wn > 0.0 && wn < 1.0) || !coef) return fail(GSMCAL_ERR_ARG, "fir1: bad arguments");
    const int n = order + 1;
    const double alpha = 0.5 * order;
    double sum = 0.0;
    for (int i = 0; i < n; ++i) {
        const double m = i - alpha;
        const double x = wn * m;
        const double sinc = (x == 0.0) ? 1.0 : sin(M_PI * x) / (M_PI * x);
        const double win = 0.54 - 0.46 * cos(2.0 * M_PI * i / order);
        coef[i] = wn * sinc * win;
        sum += coef[i];
    }
    for (int i = 0; i < n; ++i) coef[i] /= sum;
    return GSMCAL_OK;
}

int gsmcal_fir_filter(const double *coef, int n_taps, const double *s, int64_t n, int64_t n_col, int decim, double *r) {
    std::lock_guard<std::mutex> lk(g_mu);
    TRY(check_fir_args(coef, n_taps, s, n, n_col, r));
    if (n == 0) return GSMCAL_OK;
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = 0;
    const i64 n_out = (n + decim - 1) / decim;
    void *din, *dout;
    TRY(c->in.get(sizeof(double2) * (size_t)n * n_col, &din));
    TRY(c->out.get(sizeof(double2) * (size_t)n_out * n_col, &dout));
    TRY(set_taps(coef, n_taps, st));
    TRY(copy_h2d(c->ring, g_device, din, s, sizeof(double2) * (size_t)n * n_col, st));
    TRY(run_fir<false>(din, n, n, nullptr, n_taps, decim, n_col, (double2 *)dout, n_out, nullptr, st));
    TRY(copy_d2h(c->ring, g_device, r, dout, sizeof(double2) * (size_t)n_out * n_col, st));
    return GSMCAL_OK;
}

int gsmcal_raw2iq_fir_u8(const uint8_t *a, int64_t n_iq, int64_t n_col, const double *coef, int n_taps, int decim, double *r) {
    std::lock_guard<std::mutex> lk(g_mu);
    TRY(check_fir_args(coef, n_taps, a, n_iq, n_col, r));
    if (n_iq == 0) return GSMCAL_OK;
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = 0;
    const i64 n_out = (n_iq + decim - 1) / decim;
    const uint8_t *din; void *dout; Work w;
    TRY(c->out.get(sizeof(double2) * (size_t)n_out * n_col, &dout));
    TRY(u8_input(*c, a, GSMCAL_MEM_HOST, n_iq, n_col, 1, 1, coef, n_taps, st, &din, &w));
    TRY(run_fir<true>(din, n_iq, 2 * n_iq, w.ctl, n_taps, decim, n_col, (double2 *)dout, n_out, nullptr, st));
    TRY(copy_d2h(c->ring, g_device, r, dout, sizeof(double2) * (size_t)n_out * n_col, st));
    return GSMCAL_OK;
}

int gsmcal_chn_filter_taps(int which, double *coef, int *n_taps) {
    if (!coef || !n_taps) return fail(GSMCAL_ERR_ARG, "chn_filter_taps: null");
    if (which == 8) { memcpy(coef, kNum8x, sizeof kNum8x); *n_taps = 60; return GSMCAL_OK; }
    if (which == 4) { memcpy(coef, kNum4x, sizeof kNum4x); *n_taps = 30; return GSMCAL_OK; }
    return fail(GSMCAL_ERR_ARG, "chn_filter_taps: which must be 8 or 4");
}
int gsmcal_chn_filter_8x_4x(const double *s, int64_t n, int64_t n_col, double *r) { return gsmcal_fir_filter(kNum8x, 60, s, n, n_col, 2, r); }
int gsmcal_chn_filter_4x(const double *s, int64_t n, int64_t n_col, double *r) { return gsmcal_fir_filter(kNum4x, 30, s, n, n_col, 1, r); }

int gsmcal_band_power_u8(const uint8_t *a, int64_t n_iq, int64_t n_col, const double *coef, int n_taps, int decim, double *power) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!a || !power || n_iq < 1 || n_col < 1 || decim < 1) return fail(GSMCAL_ERR_ARG, "band_power: bad arguments");
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = 0;
    const uint8_t *din; Work w;
    TRY(u8_input(*c, a, GSMCAL_MEM_HOST, n_iq, n_col, 1, 1, coef, n_taps, st, &din, &w));
    CU(cudaMemsetAsync(w.power, 0, sizeof(double) * n_col, st));
    const i64 n_out = (n_iq + decim - 1) / decim;
    if (coef) {
        TRY(run_fir<true>(din, n_iq, 2 * n_iq, w.ctl, n_taps, decim, n_col, nullptr, n_out, w.power, st));
    } else {
        i64 gx = (n_out + 2047) / 2048; if (gx > 1024) gx = 1024;
        LAUNCH(power_u8_kernel, dim3((unsigned)gx, (unsigned)n_col), 256, 0, st, din, n_iq, w.ctl, decim, w.power);
    }
    CU(cudaMemcpyAsync(power, w.power, sizeof(double) * n_col, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < n_col; ++i) power[i] /= (double)n_out;
    return GSMCAL_OK;
}

int gsmcal_diversity_power_u8(const uint8_t *s_all, int64_t n_iq, int64_t n_freq, int64_t n_dongle, const double *coef, int n_taps, int decim,
                              double *power_spectrum, double *power_spectrum_combine) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!s_all || !coef || !power_spectrum || !power_spectrum_combine || n_iq < 1 || n_freq < 1 || n_dongle < 1 || decim < 1)
        return fail(GSMCAL_ERR_ARG, "diversity_power: bad arguments");
    const i64 n_col = n_freq * n_dongle;
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = 0;
    const uint8_t *din; Work w;
    TRY(u8_input(*c, s_all, GSMCAL_MEM_HOST, n_iq, n_col, 3, 1, coef, n_taps, st, &din, &w));   // cap 3: room for power | per-dongle spectrum | combination in the [D][cap] arrays
    CU(cudaMemsetAsync(w.power, 0, sizeof(double) * n_col, st));
    const i64 n_out = (n_iq + decim - 1) / decim;
    TRY(run_fir<true>(din, n_iq, 2 * n_iq, w.ctl, n_taps, decim, n_col, nullptr, n_out, w.power, st));
    LAUNCH(diversity_combine_kernel, (unsigned)((n_freq + 127) / 128), 128, 0, st, w.power, n_out, (int)n_freq, (int)n_dongle, w.fo, w.gate);
    CU(cudaMemcpyAsync(power_spectrum, w.fo, sizeof(double) * n_col, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(power_spectrum_combine, w.gate, sizeof(double) * n_freq, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GSMCAL_OK;
}

// ---------------------------------------------------------------------------------------------------
static int snr_windows(const double *s, int64_t len, int fft_len, i64 w0, i64 n_win, Ctx **cout, Work *w, cudaStream_t st) {
    if (!s || len < 1 || fft_len < 1 || fft_len > 128) return fail(GSMCAL_ERR_ARG, "moving fft: bad arguments (fft_len <= 128)");
    const double2 *din;
    TRY(upload_s(s, len, 1, n_win > 0 ? n_win : 1, 0, st, cout, &din, w));
    CU(cudaMemsetAsync(w->ctl, 0, sizeof(StreamCtl), st));
    if (n_win > 0) {
        size_t smem = sizeof(double2) * (fft_len + SNR_THREADS + fft_len);
        LAUNCH(snr_map_kernel, dim3((unsigned)((n_win + SNR_THREADS - 1) / SNR_THREADS), 1), SNR_THREADS, smem, st, mat_src(din, len, len, 0), w->ctl, w0, n_win, fft_len,
               w->snr_map, w->snr_stride);
    }
    return GSMCAL_OK;
}

int gsmcal_move_fft_snr_runtime_avg(const double *s, int64_t len, int mv_len, int fft_len, double th,
                                    int *hit_flag, double *hit_idx, double *hit_avg_snr, double *hit_snr) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!hit_flag || !hit_idx || !hit_avg_snr || !hit_snr || mv_len < 1) return fail(GSMCAL_ERR_ARG, "move_fft_snr_runtime_avg: bad arguments");
    cudaStream_t st = 0; Ctx *c; Work w;
    const i64 n_win = len - (fft_len - 1);
    TRY(snr_windows(s, len, fft_len, 0, n_win, &c, &w, st));
    StreamCtl h; memset(&h, 0, sizeof h); h.first_hit = -1;
    if (n_win > 0) {
        LAUNCH(first_hit_scan_kernel, 1, 32, 0, st, w.snr_map, w.snr_stride, n_win, mv_len, th, w.ctl, 1);
        TRY(get_ctl(w.ctl, &h, st));
    }
    if (h.first_hit > 0) { *hit_flag = 1; *hit_idx = h.first_hit; *hit_avg_snr = h.hit_avg_snr; *hit_snr = h.hit_snr; }
    else { *hit_flag = 0; *hit_idx = -1; *hit_avg_snr = INFINITY; *hit_snr = INFINITY; }
    return GSMCAL_OK;
}

int gsmcal_move_fft_snr_trace(const double *s, int64_t len, int fft_len, double *snr) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!snr) return fail(GSMCAL_ERR_ARG, "snr trace: null output");
    cudaStream_t st = 0; Ctx *c; Work w;
    const i64 n_win = len - (fft_len - 1);
    if (n_win < 1) return fail(GSMCAL_ERR_ARG, "snr trace: stream shorter than fft_len");
    TRY(snr_windows(s, len, fft_len, 0, n_win, &c, &w, st));
    CU(cudaMemcpyAsync(snr, w.snr_map, sizeof(double) * n_win, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GSMCAL_OK;
}

int gsmcal_specific_fft_snr_fix_avg(const double *s, int64_t len, int64_t t0, int64_t t1, int fft_len, double th, double avg_snr,
                                    int *hit_flag, double *hit_idx, double *hit_snr) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!hit_flag || !hit_idx || !hit_snr) return fail(GSMCAL_ERR_ARG, "specific_fft_snr_fix_avg: null output");
    *hit_flag = 0; *hit_idx = -1; *hit_snr = INFINITY;
    if (t1 < t0) return GSMCAL_OK;
    if (t0 < 1 || t1 + fft_len - 1 > len) return fail(GSMCAL_ERR_RANGE, "specific_fft_snr_fix_avg: window outside the stream (MATLAB would raise an index error)");
    cudaStream_t st = 0; Ctx *c; Work w;
    const i64 n_win = t1 - t0 + 1;
    TRY(snr_windows(s, len, fft_len, t0 - 1, n_win, &c, &w, st));
    LAUNCH(specific_hit_kernel, 1, 32, 0, st, w.snr_map, n_win, th, avg_snr, w.sch_edge, w.power);
    int off; double v;
    CU(cudaMemcpyAsync(&off, w.sch_edge, sizeof off, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&v, w.power, sizeof v, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (off >= 0) { *hit_flag = 1; *hit_idx = (double)(t0 + off); *hit_snr = v; }
    return GSMCAL_OK;
}

int gsmcal_FCCH_coarse_position(const double *s, int64_t len, int decimation_ratio, double *position, double *snr, int64_t cap_out, int64_t *n_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!s || !position || !snr || !n_out || len < 1) return fail(GSMCAL_ERR_ARG, "FCCH_coarse_position: bad arguments");
    CoarseParams p; TRY(coarse_params(decimation_ratio, &p));
    if (p.n_first > len) return fail(GSMCAL_ERR_RANGE, "FCCH_coarse_position: stream shorter than 23 frames (s(1:%lld) would raise an index error)", (long long)p.n_first);
    const int cap = (int)gsmcal_max_bursts(len, decimation_ratio);
    cudaStream_t st = 0; Ctx *c; const double2 *din; Work w;
    TRY(upload_s(s, len, cap, p.n_first, 0, st, &c, &din, &w));
    CU(cudaMemsetAsync(w.ctl, 0, sizeof(StreamCtl), st));
    TRY(run_coarse(mat_src(din, len, len, 0), len, p, 1, cap, w, st));
    StreamCtl h; TRY(get_ctl(w.ctl, &h, st));
    if (h.n_coarse < 0) { *n_out = -1; return GSMCAL_OK; }
    if (h.n_coarse > cap_out) return fail(GSMCAL_ERR_CAPACITY, "FCCH_coarse_position: %d hits, capacity %lld", h.n_coarse, (long long)cap_out);
    CU(cudaMemcpy(position, w.coarse_pos, sizeof(double) * h.n_coarse, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(snr, w.coarse_snr, sizeof(double) * h.n_coarse, cudaMemcpyDeviceToHost));
    *n_out = h.n_coarse;
    return GSMCAL_OK;
}

// ---------------------------------------------------------------------------------------------------
int gsmcal_FCCH_fine_correction(const double *s, int64_t n, const double *base_position, int64_t n_base, int osr, double carrier_freq,
                                double *FCCH_pos, int64_t pos_cap, int64_t *n_pos, double *r, int64_t r_cap, int64_t *r_len,
                                double *sampling_ppm, double *carrier_ppm) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!s || !n_pos || !r_len || !sampling_ppm || !carrier_ppm || n < 1 || n_base < 0 || osr < 1 || osr > 8) return fail(GSMCAL_ERR_ARG, "FCCH_fine_correction: bad arguments (osr 1..8)");
    *n_pos = -1; *r_len = -1; *sampling_ppm = INFINITY; *carrier_ppm = INFINITY;
    if (n_base < 5) return GSMCAL_OK;                                   // FCCH_fine_correction.m:12-15
    if (!base_position || !FCCH_pos) return fail(GSMCAL_ERR_ARG, "FCCH_fine_correction: null positions");
    const i64 len_s = n / osr;
    for (int64_t i = 0; i < n_base; ++i) {
        const double p = base_position[i];
        if (p + 64 > (double)(len_s - 148 + 1)) break;
        if (p != floor(p) || p - 64 < 1) return fail(GSMCAL_ERR_RANGE, "FCCH_fine_correction: base_position(%lld)=%g puts the search window before the first sample", (long long)i + 1, p);
    }
    const int cap = (int)n_base;
    cudaStream_t st = 0; Ctx *c; const double2 *din; Work w;
    TRY(upload_s(s, n, cap, 1, 0, st, &c, &din, &w));
    CU(cudaMemcpyAsync(w.coarse_pos, base_position, sizeof(double) * cap, cudaMemcpyHostToDevice, st));
    StreamCtl h; memset(&h, 0, sizeof h); h.n_coarse = cap;
    TRY(put_ctl(w.ctl, h, st));
    TRY(run_fine(*c, mat_src(din, n, n, 0), mat_src(din, n, n, 1), n, osr, carrier_freq, 1, cap, w, st));
    TRY(get_ctl(w.ctl, &h, st));
    *sampling_ppm = h.sppm1; *carrier_ppm = h.cppm1; *n_pos = h.n_fcch;
    if (h.n_fcch > 0) {
        if (h.n_fcch > pos_cap) return fail(GSMCAL_ERR_CAPACITY, "FCCH_fine_correction: FCCH_pos capacity");
        CU(cudaMemcpy(FCCH_pos, w.fcch_pos, sizeof(double) * h.n_fcch, cudaMemcpyDeviceToHost));
    }
    *r_len = h.len1;
    if (h.len1 >= 0) {
        if (!r || h.len1 > r_cap) return fail(GSMCAL_ERR_CAPACITY, "FCCH_fine_correction: r capacity %lld < %lld", (long long)r_cap, (long long)h.len1);
        TRY(return_r(*c, s, din, n, h.len1, h.e1, h.interp1_on, h.dphi1, h.derot1_on, r, st));     // r = s when neither is on (:72)
    }
    return GSMCAL_OK;
}

int gsmcal_SCH_training_sequence_gen(int osr, double *s) {
    if (!s || osr < 1 || osr > 64) return fail(GSMCAL_ERR_ARG, "gsm_SCH_training_sequence_gen: bad arguments");
    gmsk_template(osr, s);
    return GSMCAL_OK;
}

int gsmcal_SCH_corr_rate_correction(const double *s, int64_t n, const double *FCCH_pos, int64_t n_fcch, const double *tpl, int osr,
                                    double *pos_info, int64_t rows_cap, int64_t *n_rows, double *r, int64_t r_cap, int64_t *r_len, double *sampling_ppm) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!n_rows || !r_len || !sampling_ppm || osr < 1 || osr > 8) return fail(GSMCAL_ERR_ARG, "SCH_corr_rate_correction: bad arguments (osr 1..8)");
    *n_rows = -1; *r_len = -1; *sampling_ppm = INFINITY;
    if (n_fcch < 5) return GSMCAL_OK;                                    // SCH_corr_rate_correction.m:11-14
    if (!s || !FCCH_pos || !tpl || !pos_info || n < 1) return fail(GSMCAL_ERR_ARG, "SCH_corr_rate_correction: null input");
    const int cap = (int)n_fcch;
    const int L = 64 * osr;
    for (int i = 0; i < cap; ++i) if (FCCH_pos[i] != floor(FCCH_pos[i]) || FCCH_pos[i] + (625 * osr / 4) * 8 + 42 * osr - 8 * osr < 1)
        return fail(GSMCAL_ERR_RANGE, "SCH_corr_rate_correction: FCCH_pos(%d) puts the search window before the first sample", i + 1);
    cudaStream_t st = 0; Ctx *c; const double2 *din; Work w;
    TRY(upload_s(s, n, cap, 1, L, st, &c, &din, &w));
    std::vector<unsigned char> tpk(tpl_pack_bytes(L));
    tpl_pack(tpl, L, tpk.data());
    CU(cudaMemcpyAsync((void *)w.tpl, tpk.data(), tpk.size(), cudaMemcpyHostToDevice, st));
    g_last_sch_stats = w.sch_stats;
    CU(cudaMemsetAsync(w.sch_stats, 0, sizeof(unsigned) * SCH_NSTAT, st));
    CU(cudaMemcpyAsync(w.fcch_pos, FCCH_pos, sizeof(double) * cap, cudaMemcpyHostToDevice, st));
    StreamCtl h; memset(&h, 0, sizeof h); h.n_fcch = cap; h.sch_enable = 1; h.len1 = n;
    TRY(put_ctl(w.ctl, h, st));
    TRY(run_sch(mat_src(din, n, n, 0), osr, 1, cap, w, st));
    TRY(get_ctl(w.ctl, &h, st));
    *sampling_ppm = h.sppm2; *n_rows = h.n_pos_info;
    if (h.n_pos_info > 0) {
        if (h.n_pos_info > rows_cap) return fail(GSMCAL_ERR_CAPACITY, "SCH_corr_rate_correction: pos_info capacity %lld < %d", (long long)rows_cap, h.n_pos_info);
        std::vector<double> tmp(2 * (size_t)h.n_pos_info);
        CU(cudaMemcpy(tmp.data(), w.pos_info, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost));
        for (int i = 0; i < h.n_pos_info; ++i) { pos_info[i] = tmp[2 * i]; pos_info[h.n_pos_info + i] = tmp[2 * i + 1]; }
    }
    *r_len = h.len2;
    if (h.len2 >= 0) {
        if (!r || h.len2 > r_cap) return fail(GSMCAL_ERR_CAPACITY, "SCH_corr_rate_correction: r capacity");
        TRY(return_r(*c, s, din, n, h.len2, h.e2, h.interp2_on, 0.0, 0, r, st));                // r = s without resampling (:87,:120)
    }
    return GSMCAL_OK;
}

int gsmcal_carrier_correct_post_SCH(const double *s, int64_t n, const double *pos_info, int64_t n_rows, int osr, double carrier_freq,
                                    double *r, int64_t r_cap, int64_t *r_len, double *carrier_ppm) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!r_len || !carrier_ppm || n_rows < 0 || osr < 1 || osr > 8) return fail(GSMCAL_ERR_ARG, "carrier_correct_post_SCH: bad arguments");
    *r_len = -1; *carrier_ppm = INFINITY;
    if (n_rows > 0 && !pos_info) return fail(GSMCAL_ERR_ARG, "carrier_correct_post_SCH: null pos_info");
    bool all_m1 = n_rows > 0;                                            // `if pos_info==-1` is true only when ALL elements are -1 (:10)
    for (int64_t i = 0; i < 2 * n_rows; ++i) if (pos_info[i] != -1.0) { all_m1 = false; break; }
    if (all_m1) return GSMCAL_OK;
    int n_b = 0; std::vector<double> fpos;
    for (int64_t i = 0; i < n_rows; ++i) {
        if (pos_info[n_rows + i] == 2.0) ++n_b;
        if (pos_info[n_rows + i] == 0.0) fpos.push_back(pos_info[i]);
    }
    if (n_b < 4) return GSMCAL_OK;                                       // :15-19
    if (!s || n < 1) return fail(GSMCAL_ERR_ARG, "carrier_correct_post_SCH: null stream");
    const int N = 148 * osr;
    for (double p : fpos) if (p != floor(p) || p < 1 || p + N - 1 > (double)n) return fail(GSMCAL_ERR_RANGE, "carrier_correct_post_SCH: FCCH window outside the stream");
    if (fpos.empty()) return fail(GSMCAL_ERR_RANGE, "carrier_correct_post_SCH: no FCCH rows (mean of empty is NaN in the reference)");
    if (!r || n > r_cap) return fail(GSMCAL_ERR_CAPACITY, "carrier_correct_post_SCH: r capacity");
    const int cap = (int)fpos.size();
    cudaStream_t st = 0; Ctx *c; const double2 *din; Work w;
    TRY(upload_s(s, n, cap, 1, 0, st, &c, &din, &w));
    CU(cudaMemcpyAsync(w.post_pos, fpos.data(), sizeof(double) * cap, cudaMemcpyHostToDevice, st));
    StreamCtl h; memset(&h, 0, sizeof h); h.post_enable = 1; h.n_post_fcch = cap; h.len2 = n;
    h.sppm1 = h.sppm2 = h.cppm1 = INFINITY;
    TRY(put_ctl(w.ctl, h, st));
    TRY(run_post(*c, mat_src(din, n, n, 0), osr, carrier_freq, 1, cap, w, false, st));
    TRY(get_ctl(w.ctl, &h, st));
    *carrier_ppm = h.cppm2;
    TRY(return_r(*c, s, din, n, n, 0.0, 0, h.dphi2, 1, r, st));
    *r_len = n;
    return GSMCAL_OK;
}

int gsmcal_total_ppm_calculation(const double *ppm_in, int64_t n, double *ppm_out) {
    // total_ppm_calculation.m:5-21 - pure scalar host arithmetic (there is nothing to put on a GPU)
    if (!ppm_out || n < 0 || (n > 0 && !ppm_in)) return fail(GSMCAL_ERR_ARG, "total_ppm_calculation: bad arguments");
    bool all_inf = n > 0;
    for (int64_t i = 0; i < n; ++i) if (!(std::isinf(ppm_in[i]) && ppm_in[i] > 0)) { all_inf = false; break; }
    if (all_inf) { *ppm_out = INFINITY; return GSMCAL_OK; }
    double acc = 1.0;
    for (int64_t i = 0; i < n; ++i) acc = acc * (1.0 + ppm_in[i] * 1e-6);
    *ppm_out = (acc - 1.0) * 1e6;
    return GSMCAL_OK;
}

// ---------------------------------------------------------------------------------------------------
static int calibrate_batch_impl(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                double *r_out, int r_mem, int64_t r_stride, const TailOut *tail = nullptr) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (r_out && r_stride < n_iq) return fail(GSMCAL_ERR_ARG, "calibrate_batch_r: r_stride must be >= n_iq");
    Batch b; TRY(batch_args("calibrate_batch", raw, tpl, coef, results, n_iq, D, osr, coarse_dr, &b));
    const int cap = b.cap;
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    std::vector<unsigned char> tpk(tpl_pack_bytes(64 * osr));       // pageable: cudaMemcpyAsync stages it before it returns
    TRY(batch_setup(*c, c->work, c->wc, tpl, coef, n_taps, osr, D, tpk.data(), st, &b));
    Work &w = b.w;
    const uint8_t *draw = raw;
    if (raw_mem == GSMCAL_MEM_HOST) {
        void *din; TRY(c->in.get((size_t)2 * n_iq * D, &din));
        draw = (const uint8_t *)din;
    }
    TailDev td;
    std::vector<double> tail_w; signed char tail_pm[64];             // host sources of the uploads, alive until the final synchronise
    if (tail) TRY(tail_setup(*c, D, cap, osr, w.tpl, *tail, tail_w, tail_pm, st, &td));
    g_stage_n = 0;
    // Streams are independent, so the batch is cut into groups that run the stage sequence on their own CUDA
    // streams: the latency-bound stages of one group (burst chain, per-stream solves) overlap the FP64-bound
    // stages of the others, and with host input the H2D copy of group g+1 overlaps the compute of group g.
    int n_groups = g_debug_groups;
    if (raw_mem == GSMCAL_MEM_HOST && n_groups > 1) n_groups *= 2;
    if (D < 2 * n_groups) n_groups = 1;
    const bool timing = (n_groups == 1);
    while ((int)c->side.size() < n_groups + 1) { cudaStream_t s2; CU(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking)); c->side.push_back(s2); }
    if (g_debug_hi_prio) {
        int lo_p = 0, hi_p = 0; CU(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
        while ((int)c->side_hi.size() < n_groups) { cudaStream_t s2; CU(cudaStreamCreateWithPriority(&s2, cudaStreamNonBlocking, hi_p)); c->side_hi.push_back(s2); }
    }
    cudaStream_t cp = c->side[n_groups];                                         // H2D copies
    cudaEvent_t ev_fork; CU(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    CU(cudaEventRecord(ev_fork, st));
    if (raw_mem == GSMCAL_MEM_HOST) CU(cudaStreamWaitEvent(cp, ev_fork, 0));
    std::vector<cudaEvent_t> ev_done;
    const size_t per = (size_t)2 * n_iq;
    if (timing) TRY(stage_mark(*c, st));
    for (int g = 0; g < n_groups; ++g) {
        const i64 d0 = D * g / n_groups, d1 = D * (g + 1) / n_groups, nd = d1 - d0;
        cudaStream_t sg = (n_groups == 1) ? st : c->side[g];
        if (sg != st) CU(cudaStreamWaitEvent(sg, ev_fork, 0));
        Work ws = sub_work(w, d0, cap, g);
        const uint8_t *graw = draw + d0 * per;
        if (raw_mem == GSMCAL_MEM_HOST) {
            TRY(copy_h2d(c->ring, g_device, (void *)graw, raw + d0 * per, per * nd, cp));
            TRY(hand_off(cp, sg));
            TRY(run_colsum_u8(graw, n_iq, nd, ws.ctl, sg));
        } else if (sg == st) {
            TRY(run_colsum_u8(graw, n_iq, nd, ws.ctl, sg));
        } else {
            // device input: the HBM-bound column sums run on the caller's stream (group 0 gets the whole bandwidth first)
            TRY(run_colsum_u8(graw, n_iq, nd, ws.ctl, st));
            TRY(hand_off(st, sg));
        }
        LAUNCH(mean_kernel, (unsigned)((nd + 127) / 128), 128, 0, sg, ws.ctl, (int)nd, n_iq);
        if (timing) TRY(stage_mark(*c, sg));
        if (sg != st && g_debug_hi_prio) {
            // the coarse stage is a handful of small latency-bound kernels (a 0.8 ms dependent burst chain): on the group's own stream
            // their blocks queue behind the thousands of pending blocks of the other groups' FP64 kernels.  A high-priority stream
            // lets the block scheduler place them as soon as a slot frees, so the chain runs underneath the heavy kernels.
            cudaStream_t sh = c->side_hi[g];
            TRY(hand_off(sg, sh));
            TRY(run_coarse(lazy_src(graw, n_iq, n_taps, 0, b.dec), b.len_dec, b.p, nd, cap, ws, sh));
            TRY(hand_off(sh, sg));
        } else
        TRY(run_coarse(lazy_src(graw, n_iq, n_taps, 0, b.dec), b.len_dec, b.p, nd, cap, ws, sg));
        if (timing) TRY(stage_mark(*c, sg));
        // stagger the groups (see gsmcal_calibrate_batch_submit): the FP64 stages of group g wait for group g-1, its front does not
        if (!ev_done.empty()) CU(cudaStreamWaitEvent(sg, ev_done.back(), 0));
        TailDev gtd = td;                                        // the group's rows of every per-stream array
        if (tail) tail_arrays(gtd, *tail, cap, [&](auto *&p, size_t per, const void *) { place(p, (uintptr_t)p + d0 * per); });
        TRY(run_burst_stages(*c, graw, n_iq, n_taps, osr, carrier_freq, nd, cap, ws, tail ? &gtd : nullptr, sg,
                             timing ? c->stage_ev + g_stage_n : nullptr));
        if (timing) g_stage_n += tail ? 5 : 4;                   // 3 + 5 <= kNumStageEvents
        if (sg != st) {
            cudaEvent_t ev; CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            CU(cudaEventRecord(ev, sg));
            ev_done.push_back(ev);
        }
    }
    for (cudaEvent_t ev : ev_done) { CU(cudaStreamWaitEvent(st, ev, 0)); CU(cudaEventDestroy(ev)); }   // join (after ALL groups are enqueued)
    CU(cudaEventDestroy(ev_fork));
    if (r_out) {
        // r_correct (gsm_sync_demod.m:120 -> :145) for every stream whose chain completed: one fused pass from the uint8 capture
        double2 *r_dev = (double2 *)r_out;
        if (r_mem == GSMCAL_MEM_HOST) { void *p; TRY(c->out.get(sizeof(double2) * (size_t)r_stride * D, &p)); r_dev = (double2 *)p; }
        const i64 tiles = (n_iq + MAT_T - 1) / MAT_T;
        i64 gx = (148 * 3 + D - 1) / D; if (gx < 1) gx = 1; if (gx > tiles) gx = tiles;
        const size_t smem = sizeof(double2) * (size_t)(MAT_T + GSMCAL_XCAP(MAT_T + 8) + MAT_T + 16);
        LAUNCH(materialise_r_kernel, dim3((unsigned)gx, (unsigned)D), MAT_THREADS, smem, st, lazy_src(draw, n_iq, n_taps, 3, 1), w.ctl, r_dev, (i64)r_stride, tiles);
        if (r_mem == GSMCAL_MEM_HOST) {                          // only the r_len[2] samples of every completed stream go back (nothing else is written)
            CU(cudaMemcpyAsync(results, w.res, sizeof(StreamResultDev) * D, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            for (i64 d = 0; d < D; ++d)
                if (results[d].r_len[2] > 0)
                    TRY(copy_d2h(c->ring, g_device, r_out + 2 * (size_t)r_stride * d, r_dev + (size_t)r_stride * d, sizeof(double2) * (size_t)results[d].r_len[2], st));
        }
    }
    CU(cudaMemcpyAsync(results, w.res, sizeof(StreamResultDev) * D, cudaMemcpyDeviceToHost, st));
    if (coarse_pos) CU(cudaMemcpyAsync(coarse_pos, w.coarse_pos, sizeof(double) * D * cap, cudaMemcpyDeviceToHost, st));
    if (coarse_snr) CU(cudaMemcpyAsync(coarse_snr, w.coarse_snr, sizeof(double) * D * cap, cudaMemcpyDeviceToHost, st));
    if (fcch_pos) CU(cudaMemcpyAsync(fcch_pos, w.fcch_pos, sizeof(double) * D * cap, cudaMemcpyDeviceToHost, st));
    if (pos_info) CU(cudaMemcpyAsync(pos_info, w.pos_info, sizeof(double) * D * cap * 12, cudaMemcpyDeviceToHost, st));
    if (tail) {
        int rc = GSMCAL_OK;
        tail_arrays(td, *tail, cap, [&](auto *p, size_t per, void *h) { if (h && rc == GSMCAL_OK) rc = copy_d2h(c->ring, g_device, h, p, per * D, st); });
        TRY(rc);
    }
    CU(cudaStreamSynchronize(st));
    if (timing) for (int i = 0; i + 1 < g_stage_n; ++i) CU(cudaEventElapsedTime(&g_stage_ms[i], c->stage_ev[i], c->stage_ev[i + 1]));
    if (!timing) g_stage_n = 0;
    return GSMCAL_OK;
}

int gsmcal_calibrate_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                           const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                           double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream) {
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0);
}

int gsmcal_calibrate_batch_r(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                             const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                             double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                             double *r_correct, int r_mem, int64_t r_stride) {
    if (!r_correct) return fail(GSMCAL_ERR_ARG, "calibrate_batch_r: null r_correct");
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, r_correct, r_mem, r_stride);
}

int gsmcal_calibrate_demod_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                 const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                 double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                 gsmcal_demod_result *demod, uint8_t *sch_ok, uint8_t *demod_bits, uint8_t *bits_to_decoder, double *corr_val,
                                 double *fcch_freq, double *fcch_snr, double *fcch_max_idx) {
    if (!demod) return fail(GSMCAL_ERR_ARG, "calibrate_demod_batch: null demod");
    TailOut o{};
    o.demod = demod; o.sch_ok = sch_ok; o.bits = demod_bits; o.dec = bits_to_decoder; o.corr = corr_val; o.freq = fcch_freq; o.snr = fcch_snr;
    o.idx = fcch_max_idx;
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o);
}

int gsmcal_calibrate_demod_bcch_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                      const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                      double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                      gsmcal_demod_result *demod, uint8_t *sch_ok, uint8_t *demod_bits, uint8_t *bits_to_decoder, double *corr_val,
                                      double *fcch_freq, double *fcch_snr, double *fcch_max_idx,
                                      const double *normal_training_sequence, gsmcal_bcch_result *bcch) {
    if (!demod || !normal_training_sequence || !bcch) return fail(GSMCAL_ERR_ARG, "calibrate_demod_bcch_batch: null demod, normal_training_sequence or bcch");
    TailOut o{};
    o.demod = demod; o.sch_ok = sch_ok; o.bits = demod_bits; o.dec = bits_to_decoder; o.corr = corr_val; o.freq = fcch_freq; o.snr = fcch_snr;
    o.idx = fcch_max_idx; o.nts = normal_training_sequence; o.bcch = bcch;
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o);
}

int gsmcal_calibrate_sch_decode_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                      const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                      double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                      gsmcal_demod_result *demod, uint8_t *sch_ok, uint8_t *demod_bits, uint8_t *bits_to_decoder, double *corr_val,
                                      double *fcch_freq, double *fcch_snr, double *fcch_max_idx,
                                      const double *normal_training_sequence, gsmcal_bcch_result *bcch,
                                      gsmcal_sch_decode_result *dec, int32_t *sch_fn, int32_t *sch_bsic, uint8_t *sch_hamming, uint8_t *sch_row_flags) {
    if (!demod || !dec) return fail(GSMCAL_ERR_ARG, "calibrate_sch_decode_batch: null demod or dec");
    if (!normal_training_sequence != !bcch) return fail(GSMCAL_ERR_ARG, "calibrate_sch_decode_batch: normal_training_sequence and bcch must both be set or both NULL");
    TailOut o{};
    o.demod = demod; o.sch_ok = sch_ok; o.bits = demod_bits; o.dec = bits_to_decoder; o.corr = corr_val; o.freq = fcch_freq; o.snr = fcch_snr;
    o.idx = fcch_max_idx; o.nts = normal_training_sequence; o.bcch = bcch;
    o.sdec = dec; o.fn = sch_fn; o.bsic = sch_bsic; o.ham = sch_hamming; o.rflag = sch_row_flags;
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o);
}

int gsmcal_calibrate_sch_timing_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                      const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                      double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                      gsmcal_sch_timing_result *timing, double *sch_tau, double *sch_x) {
    if (!timing) return fail(GSMCAL_ERR_ARG, "calibrate_sch_timing_batch: null timing");
    if (osr != 8) return fail(GSMCAL_ERR_ARG, "calibrate_sch_timing_batch: oversampling_ratio must be 8");
    TailOut o{};
    o.timing = timing; o.tau = sch_tau; o.x = sch_x;
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o);
}

int gsmcal_calibrate_carrier_fit_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                       const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                       double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                       gsmcal_carrier_fit_result *carrier, double *fcch_f, double *fcch_t, uint8_t *fcch_row_flags) {
    if (!carrier) return fail(GSMCAL_ERR_ARG, "calibrate_carrier_fit_batch: null carrier");
    if (osr != 8) return fail(GSMCAL_ERR_ARG, "calibrate_carrier_fit_batch: oversampling_ratio must be 8");
    TailOut o{};
    o.carrier = carrier; o.cf_f = fcch_f; o.cf_t = fcch_t; o.cf_flag = fcch_row_flags;
    return calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                                cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o);
}

int gsmcal_calibrate_cell_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                gsmcal_carrier_fit_result *carrier, double *fcch_f, double *fcch_t, uint8_t *fcch_row_flags,
                                gsmcal_sch_decode_result *dec, uint8_t *sch_ok, uint8_t *demod_bits, double *corr_val,
                                double *sch_df, int32_t *sch_fn, int32_t *sch_bsic, uint8_t *sch_hamming, uint8_t *sch_row_flags) {
    if (!carrier || !dec) return fail(GSMCAL_ERR_ARG, "calibrate_cell_batch: null carrier or dec");
    if (osr != 8) return fail(GSMCAL_ERR_ARG, "calibrate_cell_batch: oversampling_ratio must be 8");
    TailOut o{};
    o.carrier = carrier; o.cf_f = fcch_f; o.cf_t = fcch_t; o.cf_flag = fcch_row_flags;
    o.sdec = dec; o.sch_ok = sch_ok; o.bits = demod_bits; o.corr = corr_val; o.sch_df = sch_df;
    o.fn = sch_fn; o.bsic = sch_bsic; o.ham = sch_hamming; o.rflag = sch_row_flags;
    TRY(calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                             cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o));
    for (int64_t d = 0; d < D; ++d)                              // SCH_demod ran on r_correct as it is: the rows of _demod_batch
        if (dec[d].n_sch >= 0 && (carrier[d].flags & GSMCAL_CARRIER_FEW)) dec[d].flags |= GSMCAL_SCHDEC_UNCORRECTED;
    return GSMCAL_OK;
}

int gsmcal_calibrate_sysinfo_batch(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                   const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                   double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream,
                                   gsmcal_carrier_fit_result *carrier, double *fcch_f, double *fcch_t, uint8_t *fcch_row_flags,
                                   gsmcal_sch_decode_result *dec, uint8_t *sch_ok, uint8_t *demod_bits, double *corr_val,
                                   double *sch_df, int32_t *sch_fn, int32_t *sch_bsic, uint8_t *sch_hamming, uint8_t *sch_row_flags,
                                   const double *nts, gsmcal_sysinfo_result *sysinfo, int8_t *bcch_lag, uint8_t *bcch_row_flags,
                                   uint8_t *bcch_steal, int32_t *blk_fn, uint8_t *blk_tc, uint8_t *blk_flags, uint16_t *blk_hamming,
                                   uint8_t *blk_payload) {
    if (!carrier || !dec || !nts || !sysinfo) return fail(GSMCAL_ERR_ARG, "calibrate_sysinfo_batch: null carrier, dec, normal_training_sequence or sysinfo");
    if (osr != 8) return fail(GSMCAL_ERR_ARG, "calibrate_sysinfo_batch: oversampling_ratio must be 8");
    TailOut o{};
    o.carrier = carrier; o.cf_f = fcch_f; o.cf_t = fcch_t; o.cf_flag = fcch_row_flags;
    o.sdec = dec; o.sch_ok = sch_ok; o.bits = demod_bits; o.corr = corr_val; o.sch_df = sch_df;
    o.fn = sch_fn; o.bsic = sch_bsic; o.ham = sch_hamming; o.rflag = sch_row_flags;
    o.nts = nts; o.si = sysinfo; o.lag = bcch_lag; o.bflag = bcch_row_flags; o.steal = bcch_steal;
    o.bfn = blk_fn; o.btc = blk_tc; o.bblk = blk_flags; o.bham = blk_hamming; o.pay = blk_payload;
    TRY(calibrate_batch_impl(raw, raw_mem, n_iq, D, carrier_freq, tpl, coef, n_taps, osr, coarse_dr, results, coarse_pos, coarse_snr, fcch_pos, pos_info,
                             cuda_stream, nullptr, GSMCAL_MEM_DEVICE, 0, &o));
    for (int64_t d = 0; d < D; ++d)                              // as gsmcal_calibrate_cell_batch
        if (dec[d].n_sch >= 0 && (carrier[d].flags & GSMCAL_CARRIER_FEW)) dec[d].flags |= GSMCAL_SCHDEC_UNCORRECTED;
    return GSMCAL_OK;
}

// ---- submit / collect: the same pipeline, several batches in flight -----------------------------------------------------------
int gsmcal_calibrate_batch_submit(int slot, const uint8_t *raw_dev, int64_t n_iq, int64_t D, double carrier_freq, const double *tpl,
                                  const double *coef, int n_taps, int osr, int coarse_dr, gsmcal_stream_result *results,
                                  double *coarse_pos, double *coarse_snr, double *fcch_pos, double *pos_info, void *cuda_stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (slot < 0 || slot >= kSlots) return fail(GSMCAL_ERR_ARG, "calibrate_batch_submit: slot must be 0..%d", kSlots - 1);
    Batch b; TRY(batch_args("calibrate_batch_submit", raw_dev, tpl, coef, results, n_iq, D, osr, coarse_dr, &b));
    const int cap = b.cap;
    Ctx *c; TRY(get_ctx(&c));
    Slot &sl = c->slots[slot];
    if (sl.busy) return fail(GSMCAL_ERR_ARG, "calibrate_batch_submit: slot %d still holds an uncollected batch", slot);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int n_groups = g_debug_submit_groups;                       // 2: in the staggered pipeline a batch's stages run alone, so the per-stream kernels and
                                                                // the grid tails of one half overlap the burst kernels of the other (31.15 -> 30.85 ms, profiles/r2x)
    if (D < 2 * n_groups) n_groups = 1;
    if (!sl.done) CU(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    int lo_p = 0, hi_p = 0; CU(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
    if (!sl.front_hi) CU(cudaStreamCreateWithPriority(&sl.front_hi, cudaStreamNonBlocking, hi_p));
    while ((int)sl.grp.size() < n_groups) { cudaStream_t s2; CU(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking)); sl.grp.push_back(s2); }
    while ((int)sl.hi.size() < n_groups) { cudaStream_t s2; CU(cudaStreamCreateWithPriority(&s2, cudaStreamNonBlocking, hi_p)); sl.hi.push_back(s2); }
    // pinned staging: records | coarse_pos | coarse_snr | fcch_pos | pos_info (x12) | the packed SCH template (the caller's template may be
    // pageable and short-lived)
    sl.n_res = sizeof(StreamResultDev) * (size_t)D; sl.n_per = sizeof(double) * (size_t)D * cap;
    const size_t need = align_up(sl.n_res) + 15 * sl.n_per + tpl_pack_bytes(64 * osr);
    if (need > sl.stage_cap) {
        if (sl.stage) cudaFreeHost(sl.stage);
        sl.stage = nullptr; sl.stage_cap = 0;
        CU(cudaMallocHost((void **)&sl.stage, need));
        sl.stage_cap = need;
    }
    char *h_res = sl.stage, *h_arr = sl.stage + align_up(sl.n_res), *h_tpl = h_arr + 15 * sl.n_per;
    // normal-priority kernels of different streams are dispatched in arrival order: behind the 10^5 queued blocks of the previous batch's fine
    // search even a memset waits milliseconds (device timeline, debug key 14), so the whole front runs at high priority
    cudaStream_t fr = sl.front_hi;
    TRY(hand_off(st, fr));                                       // the capture is ready on the caller's stream
    unsigned *prev_pass_hist = g_last_pass_hist;
    TRY(batch_setup(*c, sl.work, sl.wc, tpl, coef, n_taps, osr, D, (unsigned char *)h_tpl, fr, &b));
    g_prev_pass_hist = prev_pass_hist;
    Work &w = b.w;
    const size_t per = (size_t)2 * n_iq;
    sl.tl_on = g_debug_timeline != 0;
    if (sl.tl_on) {
        if (!sl.tl[0]) for (auto &e : sl.tl) CU(cudaEventCreate(&e));
        if (!g_tl_base) { CU(cudaEventCreate(&g_tl_base)); CU(cudaEventRecord(g_tl_base, fr)); }
        CU(cudaEventRecord(sl.tl[0], fr));
    }
    // the column sums as launches of fixed footprint on the front stream (see colsum_u8_trickle_kernel), one per stream group, back to back:
    // the burst chain of group g starts under the sums of group g+1
    int n_sm = 148; CU(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, g_device));
    for (int g = 0; g < n_groups; ++g) {
        const i64 d0 = D * g / n_groups, d1 = D * (g + 1) / n_groups;
        TRY(run_colsum_u8_trickle(raw_dev + d0 * per, n_iq, d1 - d0, w.ctl + d0, n_sm * g_debug_trickle_blocks, g_debug_trickle, fr));
        TRY(hand_off(fr, sl.hi[g]));
    }
    if (sl.tl_on) CU(cudaEventRecord(sl.tl[1], fr));
    for (int g = 0; g < n_groups; ++g) {
        const i64 d0 = D * g / n_groups, d1 = D * (g + 1) / n_groups, nd = d1 - d0;
        cudaStream_t sg = sl.grp[g], sh = sl.hi[g];
        Work ws = sub_work(w, d0, cap, g);
        const uint8_t *graw = raw_dev + d0 * per;
        LAUNCH(mean_kernel, (unsigned)((nd + 127) / 128), 128, 0, sh, ws.ctl, (int)nd, n_iq);
        TRY(run_coarse(lazy_src(graw, n_iq, n_taps, 0, b.dec), b.len_dec, b.p, nd, cap, ws, sh));      // latency-bound chain: high priority
        TRY(hand_off(sh, sg));
        const bool tl_g = sl.tl_on && g == n_groups - 1;
        if (tl_g) CU(cudaEventRecord(sl.tl[2], sh));
        // Staggered batches: the FP64 stages of batch k+1 start when batch k is done, and the front of batch k+1 - on the high-priority
        // streams, with the column sums as the small-footprint TMA-ring kernel - runs UNDER the FP64 stages of batch k.  Without this wait
        // two batches in flight run in lockstep (normal-priority kernels are dispatched in arrival order, so their stages interleave and
        // both finish together) and both fronts execute while nothing else does.  Device timelines and the cost of the overlap (the ring's
        // shared-memory traffic, the burst chain): profiles/r2n, r2p, r2q, r2z, r2ak and DESIGN.md section 4.
        if (c->last_slot >= 0 && c->last_slot != slot && c->slots[c->last_slot].busy)
            CU(cudaStreamWaitEvent(sg, c->slots[c->last_slot].done, 0));
        if (tl_g) CU(cudaEventRecord(sl.tl[4], sg));
        const cudaEvent_t marks[4] = {sl.tl[5], sl.tl[6], sl.tl[7], sl.tl[3]};
        TRY(run_burst_stages(*c, graw, n_iq, n_taps, osr, carrier_freq, nd, cap, ws, nullptr, sg, tl_g ? marks : nullptr));
        TRY(hand_off(sg, fr));
    }
    CU(cudaMemcpyAsync(h_res, w.res, sl.n_res, cudaMemcpyDeviceToHost, fr));
    if (coarse_pos) CU(cudaMemcpyAsync(h_arr, w.coarse_pos, sl.n_per, cudaMemcpyDeviceToHost, fr));
    if (coarse_snr) CU(cudaMemcpyAsync(h_arr + sl.n_per, w.coarse_snr, sl.n_per, cudaMemcpyDeviceToHost, fr));
    if (fcch_pos) CU(cudaMemcpyAsync(h_arr + 2 * sl.n_per, w.fcch_pos, sl.n_per, cudaMemcpyDeviceToHost, fr));
    if (pos_info) CU(cudaMemcpyAsync(h_arr + 3 * sl.n_per, w.pos_info, 12 * sl.n_per, cudaMemcpyDeviceToHost, fr));
    CU(cudaEventRecord(sl.done, fr));
    sl.results = results; sl.coarse_pos = coarse_pos; sl.coarse_snr = coarse_snr; sl.fcch_pos = fcch_pos; sl.pos_info = pos_info;
    sl.busy = true;
    c->last_slot = slot;
    return GSMCAL_OK;
}

int gsmcal_calibrate_batch_collect(int slot) {
    cudaEvent_t done;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (slot < 0 || slot >= kSlots) return fail(GSMCAL_ERR_ARG, "calibrate_batch_collect: slot must be 0..%d", kSlots - 1);
        Ctx *c; TRY(get_ctx(&c));
        if (!c->slots[slot].busy) return fail(GSMCAL_ERR_ARG, "calibrate_batch_collect: nothing was submitted to slot %d", slot);
        done = c->slots[slot].done;
    }
    CU(cudaEventSynchronize(done));                              // outside the lock: other slots can be submitted meanwhile
    std::lock_guard<std::mutex> lk(g_mu);
    Ctx *c; TRY(get_ctx(&c));
    Slot &sl = c->slots[slot];
    if (sl.tl_on && g_tl_base) {
        float t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int i = 0; i < 8; ++i) cudaEventElapsedTime(&t[i], g_tl_base, sl.tl[i]);
        fprintf(stderr, "[gsmcal timeline] slot %d: front start %.3f ms, column sums done %.3f, burst chain done %.3f, FP64 stages start %.3f, "
                        "fine search +%.3f, fine tone +%.3f, SCH +%.3f, post +%.3f, done %.3f\n",
                slot, t[0], t[1], t[2], t[4], t[5] - t[4], t[6] - t[5], t[7] - t[6], t[3] - t[7], t[3]);
        cudaGetLastError();
    }
    const char *h_res = sl.stage, *h_arr = sl.stage + align_up(sl.n_res);
    memcpy(sl.results, h_res, sl.n_res);
    if (sl.coarse_pos) memcpy(sl.coarse_pos, h_arr, sl.n_per);
    if (sl.coarse_snr) memcpy(sl.coarse_snr, h_arr + sl.n_per, sl.n_per);
    if (sl.fcch_pos) memcpy(sl.fcch_pos, h_arr + 2 * sl.n_per, sl.n_per);
    if (sl.pos_info) memcpy(sl.pos_info, h_arr + 3 * sl.n_per, 12 * sl.n_per);
    sl.busy = false;
    return GSMCAL_OK;
}

int gsmcal_calibrate_batch_cancel(int slot) {
    // gives the slot back without delivering results: waits for the batch (its kernels read the capture and write the slot's own
    // staging, never the caller's result pointers, which are only touched by _collect) and forgets the pointers
    cudaEvent_t done;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (slot < 0 || slot >= kSlots) return fail(GSMCAL_ERR_ARG, "calibrate_batch_cancel: slot must be 0..%d", kSlots - 1);
        Ctx *c; TRY(get_ctx(&c));
        if (!c->slots[slot].busy) return GSMCAL_OK;
        done = c->slots[slot].done;
    }
    CU(cudaEventSynchronize(done));
    std::lock_guard<std::mutex> lk(g_mu);
    Ctx *c; TRY(get_ctx(&c));
    Slot &sl = c->slots[slot];
    sl.results = nullptr; sl.coarse_pos = sl.coarse_snr = sl.fcch_pos = sl.pos_info = nullptr;
    sl.busy = false;
    return GSMCAL_OK;
}

int gsmcal_last_batch_stage_ms(double *ms, int cap_n) {
    // colsum(+H2D), coarse, fine_peak, fine ppm+tone+carrier, SCH, post-SCH (+ demod) - of the last gsmcal_calibrate_batch* call
    int n = g_stage_n > 0 ? g_stage_n - 1 : 0;
    for (int i = 0; i < n && i < cap_n; ++i) ms[i] = g_stage_ms[i];
    return n;
}

int gsmcal_fcch_scan(const uint8_t *raw, int raw_mem, int64_t n_iq, int64_t n_chan, const double *coef, int n_taps, int osr, int coarse_dr,
                     double *snr, double *num_hit, double *position, int32_t *n_position, void *cuda_stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!raw || !coef || !snr || !num_hit || n_iq < 1 || n_chan < 1 || osr < 1) return fail(GSMCAL_ERR_ARG, "fcch_scan: bad arguments");
    CoarseParams p; TRY(coarse_params(coarse_dr, &p));
    const int dec = osr * coarse_dr;
    const i64 len_dec = (n_iq + dec - 1) / dec;
    if (p.n_first > len_dec) return fail(GSMCAL_ERR_RANGE, "fcch_scan: capture shorter than 23 frames");
    const int cap = (int)gsmcal_max_bursts(len_dec, coarse_dr);
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const uint8_t *draw; Work w;
    TRY(u8_input(*c, raw, raw_mem, n_iq, n_chan, cap, p.n_first, coef, n_taps, st, &draw, &w));
    LAUNCH(mean_kernel, (unsigned)((n_chan + 127) / 128), 128, 0, st, w.ctl, (int)n_chan, n_iq);
    TRY(run_coarse(lazy_src(draw, n_iq, n_taps, 0, dec), len_dec, p, n_chan, cap, w, st));
    LAUNCH(scan_accept_kernel, (unsigned)((n_chan + 63) / 64), 64, 0, st, w.ctl, (int)n_chan, cap, w.coarse_pos, w.coarse_snr, w.fo, w.gate);
    CU(cudaMemcpyAsync(snr, w.fo, sizeof(double) * n_chan, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(num_hit, w.gate, sizeof(double) * n_chan, cudaMemcpyDeviceToHost, st));
    if (position) CU(cudaMemcpyAsync(position, w.coarse_pos, sizeof(double) * n_chan * cap, cudaMemcpyDeviceToHost, st));
    std::vector<StreamCtl> h;
    if (n_position) { h.resize(n_chan); CU(cudaMemcpyAsync(h.data(), w.ctl, sizeof(StreamCtl) * n_chan, cudaMemcpyDeviceToHost, st)); }
    CU(cudaStreamSynchronize(st));
    if (n_position) for (int64_t i = 0; i < n_chan; ++i) n_position[i] = h[i].n_coarse;
    return GSMCAL_OK;
}

int gsmcal_fp64_peak(double *tflops, void *cuda_stream) {
    // measured DFMA throughput of this GPU (2 flop per DFMA), CUDA events around a register-only FMA kernel
    std::lock_guard<std::mutex> lk(g_mu);
    if (!tflops) return fail(GSMCAL_ERR_ARG, "fp64_peak: null output");
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    cudaDeviceProp prop; CU(cudaGetDeviceProperties(&prop, g_device));
    const int blocks = prop.multiProcessorCount * 8, iters = 1 << 14;
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CU(cudaEventRecord(e0, st));
        LAUNCH(fp64_peak_kernel, blocks, 256, 0, st, (double *)nullptr, iters, 0.999999, 1e-9);
        CU(cudaEventRecord(e1, st));
        CU(cudaEventSynchronize(e1));
        float ms; CU(cudaEventElapsedTime(&ms, e0, e1));
        const double tf = 2.0 * 8.0 * iters * 256.0 * blocks / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    CU(cudaEventDestroy(e0)); CU(cudaEventDestroy(e1));
    *tflops = best;
    return GSMCAL_OK;
}

int gsmcal_stage_launch(int stage, const void *in, void *out, int64_t n_iq, int64_t n_col, const double *coef, int n_taps, void *cuda_stream) {
    std::lock_guard<std::mutex> lk(g_mu);
    Ctx *c; TRY(get_ctx(&c));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    Work w; TRY(make_work(c->work, n_col, 1, 1, 0, &w));       // the control blocks of stage 0's column sums stay at offset 0
    if (coef) TRY(set_taps(coef, n_taps, st));
    switch (stage) {
    case 0:
        CU(cudaMemsetAsync(w.ctl, 0, sizeof(StreamCtl) * n_col, st));
        return run_colsum_u8((const uint8_t *)in, n_iq, n_col, w.ctl, st);
    case 1:
        LAUNCH(raw2iq_store_kernel, dim3(raw2iq_grid(n_iq), (unsigned)n_col), 256, 0, st, (const uint8_t *)in, n_iq, w.ctl, (double2 *)out);
        return GSMCAL_OK;
    case 2: return run_fir<false>(in, n_iq, n_iq, nullptr, n_taps, 1, n_col, (double2 *)out, n_iq, nullptr, st);
    case 3: return run_fir<true>(in, n_iq, 2 * n_iq, w.ctl, n_taps, 1, n_col, (double2 *)out, n_iq, nullptr, st);
    case 4: for (i64 d = 0; d < n_col; ++d) TRY(run_resample_derotate((const double2 *)in + d * n_iq, n_iq, -35e-6, 1, 0.0, 0, (double2 *)out + d * n_iq, n_iq, st)); return GSMCAL_OK;
    case 5: for (i64 d = 0; d < n_col; ++d) TRY(run_resample_derotate((const double2 *)in + d * n_iq, n_iq, 0.0, 0, 0.0123, 1, (double2 *)out + d * n_iq, n_iq, st)); return GSMCAL_OK;
    case 6: return run_fir<true>(in, n_iq, 2 * n_iq, w.ctl, n_taps, 64, n_col, (double2 *)out, (n_iq + 63) / 64, nullptr, st);
    default: return fail(GSMCAL_ERR_ARG, "stage_launch: unknown stage %d", stage);
    }
}

}  // extern "C"

// ====================================================================================================
// T1  gsm_SCH_training_sequence_gen.m:17-19,32,39 - GMSK per GSM 05.04 (host code: 512 samples, once per session)
// ====================================================================================================
namespace {
double gq_big_f(double u) { return u * 0.5 * erfc(-u / sqrt(2.0)) + exp(-0.5 * u * u) / sqrt(2.0 * M_PI); }
double gq_big_g(double t) {
    const double sigma = sqrt(log(2.0)) / (2.0 * M_PI * 0.3);
    return (sigma / 2.0) * (gq_big_f((t + 0.5) / sigma) - gq_big_f((t - 0.5) / sigma));
}
double gmsk_q(double tau) {
    if (tau < 0.0) tau = 0.0;
    if (tau > 4.0) tau = 4.0;
    const double g0 = gq_big_g(-2.0), g1 = gq_big_g(2.0);
    return (gq_big_g(tau - 2.0) - g0) / (g1 - g0);
}
void gmsk_bits(const int *bits, int nb, int osr, double *out) {      // differential encoding against a leading 0, bit 1 -> +1, then GMSK
    std::vector<double> a((size_t)nb);
    int prev = 0;
    for (int k = 0; k < nb; ++k) { a[k] = (bits[k] == prev) ? 1.0 : -1.0; prev = bits[k]; }   // ~abs(diff([0;data]))
    for (int n = 0; n < nb * osr; ++n) {
        double phase = 0.0;
        for (int k = 0; k < nb; ++k) phase += a[k] * gmsk_q(((double)n - (double)k * osr) / osr);
        out[2 * n] = cos((M_PI / 2.0) * phase);
        out[2 * n + 1] = sin((M_PI / 2.0) * phase);
    }
}
void gmsk_template(int osr, double *out) {
    static const int bits[64] = {1, 0, 1, 1, 1, 0, 0, 1, 0, 1, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0,
                                 0, 0, 0, 0, 0, 1, 1, 1, 1, 0, 0, 1, 0, 1, 1, 0, 1, 0, 1, 0, 0, 0,
                                 1, 0, 1, 0, 1, 1, 1, 0, 1, 1, 0, 0, 0, 0, 1, 1, 0, 1, 1};
    gmsk_bits(bits, 64, osr, out);
}
}  // namespace

#include "gsmcal_demod_api.inc"
