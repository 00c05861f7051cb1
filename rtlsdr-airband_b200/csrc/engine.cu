// Host side of the B200 demodulation engine: configuration -> device tables and per-channel state, raw-sample
// ingest, run scheduling (K1 then K2 per run), result queueing, and the C ABI declared in include/airband_b200.h.
//
// Config-time arithmetic restated here (host, double/float exactly as the reference does it):
//   window                      reference src/rtl_airband.cpp:335-351
//   sincos LUT                  reference src/util.cpp:103-111
//   Squelch constructor/setters reference src/squelch.cpp:36-116
//   Goertzel coefficients, bank reference src/ctcss.cpp:31-42,62-73,92-111
//   NotchFilter coefficients    reference src/filters.cpp:30-47
//   LowpassFilter design        reference src/filters.cpp:67-144
//   initial channel state       reference src/config.cpp:265-281,313-331
// There is no CPU execution path: every entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <complex>
#include <deque>
#include <memory>
#include <string>
#include <vector>

#include "../../include/airband_b200.h"
#include "abg_internal.h"

namespace {

// Small host->device parameter uploads go through a KERNEL (payload passed by value), not cudaMemcpyAsync: a copy would
// queue on the host->device copy engine behind whatever bulk ingest copies (abg_push of the NEXT run) are already
// enqueued, and the run that needs these few hundred bytes would wait for megabytes of unrelated input (measured: ~1 ms
// per step on the pipelined host path).  A launch is ordered only by its own stream.
struct UploadBlob {
    uint4 q[240];  // 3840 bytes: stays below the 4 KB kernel-parameter limit together with the other arguments
};
__global__ void upload_kernel(const UploadBlob b, uint4* dst, int n16) {
    const int i = threadIdx.x;
    if (i < n16) dst[i] = b.q[i];
}
// dst: 16-byte aligned device buffer with room for nbytes rounded up to 16; returns the number of launches (or -1)
int upload_small(void* dst, const void* src, size_t nbytes, cudaStream_t s) {
    int launches = 0;
    for (size_t off = 0; off < nbytes; off += sizeof(UploadBlob)) {
        const size_t chunk = std::min(sizeof(UploadBlob), nbytes - off);
        UploadBlob b;
        memcpy(b.q, static_cast<const char*>(src) + off, chunk);
        if (chunk % 16) memset(reinterpret_cast<char*>(b.q) + chunk, 0, 16 - chunk % 16);
        const int n16 = (int)((chunk + 15) / 16);
        upload_kernel<<<1, 256, 0, s>>>(b, reinterpret_cast<uint4*>(static_cast<char*>(dst) + off), n16);
        if (cudaGetLastError() != cudaSuccess) return -1;
        ++launches;
    }
    return launches;
}

thread_local std::string g_err;
int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t _e = (call);                                                                              \
        if (_e != cudaSuccess) return fail(ABG_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

const float kStandardTones[51] = {67.0,  69.3,  71.9,  74.4,  77.0,  79.7,  82.5,  85.4,  88.5,  91.5,  94.8,  97.4,  100.0,
                                  103.5, 107.2, 110.9, 114.8, 118.8, 123.0, 127.3, 131.8, 136.5, 141.3, 146.2, 150.0, 151.4,
                                  156.7, 159.8, 162.2, 165.5, 167.9, 171.3, 173.8, 177.3, 179.9, 183.5, 186.2, 189.9, 192.8,
                                  196.6, 199.5, 203.5, 206.5, 210.7, 218.1, 225.7, 229.1, 233.6, 241.8, 250.3, 254.1};  // ctcss.cpp:87-89

// Goertzel coefficient of one detector, ctcss.cpp:31-42 (same operand types: int*float/float, +0.5 in double, float omega)
float goertzel_coeff(float tone_freq, float sample_rate, int window_size) {
    int k = (0.5 + window_size * tone_freq / sample_rate);
    float omega = (2.0 * M_PI * k) / window_size;
    float coeff = 2.0 * cos(omega);
    return coeff;
}
// bank for one CTCSS object: wanted tone first, then standard tones not within 5 Hz, dropping coefficient collisions
std::vector<float> tone_bank(float ctcss_freq, float sample_rate, int window_size) {
    std::vector<float> coeffs;
    auto try_add = [&](float f) {
        float c = goertzel_coeff(f, sample_rate, window_size);
        for (float e : coeffs)
            if (e == c) return;
        coeffs.push_back(c);
    };
    try_add(ctcss_freq);
    for (float tone : kStandardTones) {
        if (std::abs(ctcss_freq - tone) < 5) continue;
        try_add(tone);
    }
    return coeffs;
}

// LowpassFilter::LowpassFilter, filters.cpp:67-96 (+ blt/expand/multin/eval :98-144)
typedef std::complex<double> cd;
cd lp_blt(cd pz) { return (2.0 + pz) / (2.0 - pz); }
void lp_multin(cd w, int npz, cd coeffs[]) {
    cd nw = -w;
    for (int i = npz; i >= 1; i--) coeffs[i] = (nw * coeffs[i]) + coeffs[i - 1];
    coeffs[0] = nw * coeffs[0];
}
bool lp_expand(cd pz[], int npz, cd coeffs[]) {
    coeffs[0] = 1.0;
    for (int i = 0; i < npz; i++) coeffs[i + 1] = 0.0;
    for (int i = 0; i < npz; i++) lp_multin(pz[i], npz, coeffs);
    for (int i = 0; i < npz + 1; i++)
        if (fabs(coeffs[i].imag()) > 1e-10) return false;
    return true;
}
cd lp_eval(cd coeffs[], int npz, cd z) {
    cd sum(0.0);
    for (int i = npz; i >= 0; i--) sum = (sum * z) + coeffs[i];
    return sum;
}
bool lowpass_design(float freq, float sample_freq, float* gain, float* yc0, float* yc1) {
    double raw_alpha = (double)freq / sample_freq;
    double warped_alpha = tan(M_PI * raw_alpha) / M_PI;
    cd zeros[2] = {-1.0, -1.0};
    cd poles[2];
    poles[0] = lp_blt(M_PI * 2 * warped_alpha * cd(-1.10160133059e+00, 6.36009824757e-01));
    poles[1] = lp_blt(M_PI * 2 * warped_alpha * conj(cd(-1.10160133059e+00, 6.36009824757e-01)));
    cd top[3], bot[3];
    if (!lp_expand(zeros, 2, top) || !lp_expand(poles, 2, bot)) return false;
    cd g = lp_eval(top, 2, 1.0) / lp_eval(bot, 2, 1.0);
    *gain = hypot(g.imag(), g.real());
    *yc0 = -(bot[0].real() / bot[2].real());
    *yc1 = -(bot[1].real() / bot[2].real());
    return true;
}

struct Plan {
    int r1, r2, r3;
};
bool plan_for(int n, Plan* p) {  // must match Plan<LOGN> in k1_fft.cu
    switch (n) {
        case 256: *p = {16, 16, 0}; return true;
        case 512: *p = {32, 16, 0}; return true;
        case 1024: *p = {32, 32, 0}; return true;
        case 2048: *p = {64, 32, 0}; return true;
        case 4096: *p = {64, 64, 0}; return true;
        case 8192: *p = {32, 16, 16}; return true;
    }
    return false;
}

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaError_t alloc(size_t count) {
        n = count;
        return cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
    }
    void free() {
        if (p) cudaFree(p);
        p = nullptr;
    }
};

struct Device {
    int sfmt = 0, bpc = 0, sample_rate = 0, hop = 0, hop_bytes = 0;
    float fullscale = 0;
    int g0 = 0, C = 0, group = 0;
    bool primed = false, has_afc = false;
    // raw sample stream (ping-pong linear buffers)
    unsigned char* raw[2] = {nullptr, nullptr};
    int cur = 0;
    size_t cap = 0, fill = 0, consumed = 0;
    int runs_since_compaction = 1;  // K1 launches that read raw[cur] since the last compaction
    // resident replay stream
    unsigned char* res = nullptr;
    size_t res_bytes = 0;
    bool res_primed = false;
    float2* spec = nullptr;  // [nbmax][N] when has_afc
    std::deque<std::pair<int, int>> ready;  // (slot, batch-in-run)
};

// ---- scan mode: per-frequency freq_t sets (rtl_airband.h:223-233,250-252) ------------------------------------------------
// A scan channel keeps one FreqSet per freqlist[] entry in device memory.  The live slot (params/state/sqbuf/tone banks
// of channel g, what K2 reads) holds the current entry; abg_scan_select() swaps entries with one small kernel on the
// K2 stream, i.e. between the batches of two runs, which is when demodulate() re-reads freq_idx (rtl_airband.cpp:498).
struct FreqSet {
    ChanParams p;  // freq-level fields only: modulation, ampfactor, notch, low-pass, CTCSS
    ChanState s;   // freq-level fields only: Squelch, CTCSS counters, filter delay elements, agcavgfast, active_counter
    float sqbuf[ABG_SQ_BUF];
    float tone_coeff[2][ABG_MAX_TONES], tone_q1[2][ABG_MAX_TONES], tone_q2[2][ABG_MAX_TONES], tone_mag[2][ABG_MAX_TONES];
};
struct ScanView {
    ChanParams* params;
    ChanState* state;
    float *sqbuf, *tone_coeff, *tone_q1, *tone_q2, *tone_mag;
    int Gp;
};
__device__ void freq_fields_copy(ChanParams& dp, ChanState& ds, const ChanParams& sp, const ChanState& ss) {
    // channel_t members stay with the channel: dev, needs_raw_iq, has_iq_outputs, dm_dphi, alpha, afc / dm_phi, pr, pj,
    // prev_waveout, axc_prev
    dp.modulation = sp.modulation; dp.ampfactor = sp.ampfactor;
    dp.notch_on = sp.notch_on; dp.nd0 = sp.nd0; dp.nd1 = sp.nd1; dp.nd2 = sp.nd2;
    dp.lp_on = sp.lp_on; dp.lp_gain = sp.lp_gain; dp.lp_yc0 = sp.lp_yc0; dp.lp_yc1 = sp.lp_yc1;
    dp.ctcss_on = sp.ctcss_on;
    for (int w = 0; w < 2; w++) { dp.n_tones[w] = sp.n_tones[w]; dp.window[w] = sp.window[w]; }
    const uint32_t dm_phi = ds.dm_phi;
    const float pr = ds.pr, pj = ds.pj, prev_waveout = ds.prev_waveout;
    const int32_t axc_prev = ds.axc_prev;
    ds = ss;
    ds.dm_phi = dm_phi; ds.pr = pr; ds.pj = pj; ds.prev_waveout = prev_waveout; ds.axc_prev = axc_prev;
}
__global__ void scan_swap_kernel(const ScanView v, int g, FreqSet* save_to, const FreqSet* load_from) {
    const int t = threadIdx.x, Gp = v.Gp;
    if (t == 0) {
        save_to->p = v.params[g];
        save_to->s = v.state[g];
        ChanParams p = v.params[g];
        ChanState s = v.state[g];
        freq_fields_copy(p, s, load_from->p, load_from->s);
        v.params[g] = p;
        v.state[g] = s;
    }
    for (int i = t; i < ABG_SQ_BUF; i += blockDim.x) {
        save_to->sqbuf[i] = v.sqbuf[(size_t)i * Gp + g];
        v.sqbuf[(size_t)i * Gp + g] = load_from->sqbuf[i];
    }
    for (int i = t; i < 2 * ABG_MAX_TONES; i += blockDim.x) {
        const int w = i / ABG_MAX_TONES, k = i % ABG_MAX_TONES;
        const size_t o = (size_t)i * Gp + g;
        save_to->tone_coeff[w][k] = v.tone_coeff[o]; v.tone_coeff[o] = load_from->tone_coeff[w][k];
        save_to->tone_q1[w][k] = v.tone_q1[o];       v.tone_q1[o] = load_from->tone_q1[w][k];
        save_to->tone_q2[w][k] = v.tone_q2[o];       v.tone_q2[o] = load_from->tone_q2[w][k];
        save_to->tone_mag[w][k] = v.tone_mag[o];     v.tone_mag[o] = load_from->tone_mag[w][k];
    }
}

struct Group {
    int sfmt, hop_bytes;
    float fullscale;
    std::vector<int> devs;
    int frames_per_tile = 0, tile_bytes_cap = 0;      // full-spectrum kernel (k1_fft.cu)
    int p_frames_per_tile = 0, p_tile_bytes_cap = 0;  // output-pruned kernel (k1_pruned.cu)
    int max_channels = 0;
    bool pruned = false;                               // which kernel this group runs
    DevBuf<float> wsc;
    std::vector<float> h_wsc;
    K1Dev* d_k1 = nullptr;  // device array [devs.size() + 1]: the extra (all-zero) entry is the tensor-core kernel's tile counter
    std::vector<K1Dev> h_k1;  // host copy, uploaded by value with every run (upload_small)
    // tensor-core K1 (k1_tc.cu)
    bool use_tc = false;
    K1TcPlan tc{};
    DevBuf<signed char> tc_btab;
    DevBuf<long long> tc_sq;
    DevBuf<int32_t> tc_tab_of_dev;
    double tc_cscale = 0.0;
    int tc_tables = 0;
};

// One run's results.  Page-locked host memory by default; HBM after abg_set_result_location(ABG_RESULTS_DEVICE).
struct Slot {
    float* wout = nullptr;    // [G][nbmax*B]
    float* iqout = nullptr;   // [G][nbmax*B][2] or null
    unsigned char* axc = nullptr;  // [nbmax][Gp]
    float* mix = nullptr;     // [nbmax][n_mixers][2][B]
    int32_t* mixflag = nullptr;  // [nbmax][n_mixers]
    int mix_pending = 0;
    cudaEvent_t done = nullptr;
    int pending = 0;          // unfetched device-batches referencing this slot
    // device mode: recorded on the caller's stream after the gather of a device fetch that read this slot; a later
    // run's mixer and export kernels wait for it before they overwrite the slot
    cudaEvent_t released = nullptr;
    bool release_pending = false;
};

}  // namespace

struct abg_engine {
    int N = 0, W = 0, B = 0, fm_demod = 0, nbmax = 4, P = 0, G = 0, Gp = 0, fft_mode = 0;
    int cuda_dev = 0, sm_count = 148, tc_digits = 4;
    bool tc_auto = true;               // fft_mode 0 picks the tensor-core K1 for eligible groups (ABG_K1_TC_AUTO=0: FP32 kernels only)
    int32_t* tc_status = nullptr;      // pinned + mapped: the tensor-core K1 reports a stalled pipeline here (never hangs)
    int32_t* tc_status_dev = nullptr;
    bool any_iq_out = false;
    std::vector<Device> dev;
    std::vector<Group> groups;
    std::vector<ChanParams> h_params;
    bool any_nfm = false;  // some channel or scan-list entry demodulates NFM
    struct ScanChan {
        int g = 0, n_freqs = 0, cur = 0;
        FreqSet* stash = nullptr;  // device array [n_freqs]; entry `cur` is stale while it is live
    };
    std::vector<ScanChan> scan;
    // device memory
    DevBuf<ChanParams> params;
    DevBuf<ChanState> state;
    DevBuf<int32_t> bins, base_bins;
    DevBuf<float> win[2], wout, sqbuf, tone_coeff, tone_q1, tone_q2, tone_mag, lut;  // win/iqin are double-buffered: K1 of run i+1
    DevBuf<float2> iqin[2], iqout, tw1, tw2, twn;                                           // fills one while K2 of run i reads the other
    DevBuf<unsigned char> axc;
    K2Dev* d_k2 = nullptr;
    std::vector<K2Dev> h_k2;  // host copy, uploaded by value with every run (upload_small)
    std::vector<Slot> slots;
    int next_slot = 0;
    cudaStream_t stream = nullptr;   // stream A: ingest copies + K1
    bool own_stream = false;
    cudaStream_t stream_b = nullptr; // stream B: K2, mixers, result copies, tail copy
    cudaStream_t stream_c = nullptr; // stream C: ingest (abg_push host->device copies, buffer compaction)
    cudaEvent_t ev_ingest = nullptr; // last ingest operation
    cudaEvent_t ev_caller = nullptr; // abg_push_device: the caller's stream up to the push
    int results_where = ABG_RESULTS_HOST;
    bool ingest_dirty = false;
    cudaEvent_t ev_k1[2] = {nullptr, nullptr}, ev_k2[2] = {nullptr, nullptr};
    uint64_t run_index = 0;
    bool any_afc = false;
    int k2_lpw = 32;
    uint64_t launches = 0;
    // timing events of the last TL_RUNS runs: [0] K1 start, [1] K1 end (stream A); [2] K2 start, [3] K2 end, [4] end of run (stream B)
    static constexpr int TL_RUNS = 8;
    cudaEvent_t tl[TL_RUNS][5] = {};
    bool tev_valid = false;
    std::vector<int32_t> h_bins;
    // mixers (reference src/mixer.cpp)
    int n_mixers = 0;
    DevBuf<int32_t> mix_offsets;
    DevBuf<MixInput> mix_inputs;
    DevBuf<float> mix_sums;     // [nbmax][n_mixers][2][B]
    DevBuf<int32_t> mix_flags;  // [nbmax][n_mixers]
    std::deque<std::pair<int, int>> mix_ready;  // (slot, batch-in-run), same for every mixer
    std::vector<int> mix_fetched;               // per mixer: entries of mix_ready already popped by that mixer

    K2Launch k2_launch(int cur) const {
        K2Launch L{};
        L.G = G; L.Gp = Gp; L.P = P; L.wave_batch = B; L.fm_demod = fm_demod; L.iq_stride = nbmax * B;
        L.lanes_per_warp = k2_lpw;
        L.nfm_blocks = any_nfm ? 1 : 0;
        L.params = params.p; L.state = state.p; L.devs = d_k2; L.bins = bins.p; L.base_bins = base_bins.p;
        L.win = win[cur].p; L.iqin = iqin[cur].p; L.win_next = win[cur ^ 1].p; L.iqin_next = iqin[cur ^ 1].p; L.wout = wout.p; L.iqout = any_iq_out ? iqout.p : nullptr;
        L.sqbuf = sqbuf.p; L.tone_coeff = tone_coeff.p; L.tone_q1 = tone_q1.p; L.tone_q2 = tone_q2.p; L.tone_mag = tone_mag.p;
        L.axc = axc.p; L.sincos_lut = lut.p;
        return L;
    }
};

namespace {

// result slot memory: page-locked host memory, or HBM in device mode
cudaError_t result_alloc(const abg_engine* e, void** p, size_t bytes) {
    return e->results_where == ABG_RESULTS_DEVICE ? cudaMalloc(p, bytes) : cudaMallocHost(p, bytes);
}
template <typename T>
void result_free(const abg_engine* e, T*& p) {
    if (p) {
        if (e->results_where == ABG_RESULTS_DEVICE) cudaFree(p);
        else cudaFreeHost(p);
    }
    p = nullptr;
}
int alloc_slot_results(abg_engine* e) {
    const size_t GB = (size_t)std::max(e->G, 1) * e->nbmax * e->B;
    for (auto& s : e->slots) {
        CU(result_alloc(e, (void**)&s.wout, sizeof(float) * GB));
        if (e->any_iq_out) CU(result_alloc(e, (void**)&s.iqout, sizeof(float2) * GB));
        CU(result_alloc(e, (void**)&s.axc, (size_t)e->nbmax * e->Gp));
    }
    return ABG_OK;
}
int alloc_slot_mixers(abg_engine* e) {
    const size_t nsum = (size_t)e->nbmax * e->n_mixers * 2 * e->B;
    for (auto& s : e->slots) {
        CU(result_alloc(e, (void**)&s.mix, sizeof(float) * nsum));
        CU(result_alloc(e, (void**)&s.mixflag, sizeof(int32_t) * (size_t)e->nbmax * e->n_mixers));
    }
    return ABG_OK;
}
void free_slot_results(abg_engine* e) {
    for (auto& s : e->slots) {
        result_free(e, s.wout); result_free(e, s.iqout); result_free(e, s.axc); result_free(e, s.mix); result_free(e, s.mixflag);
    }
}

void engine_free(abg_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cuda_dev);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->stream_b) cudaStreamSynchronize(e->stream_b);
    for (auto& s : e->slots)  // device fetches still reading a slot on a caller's stream
        if (s.release_pending) cudaEventSynchronize(s.released);
    for (auto& d : e->dev) {
        for (int i = 0; i < 2; i++)
            if (d.raw[i]) cudaFree(d.raw[i]);
        if (d.res) cudaFree(d.res);
        if (d.spec) cudaFree(d.spec);
    }
    for (auto& g : e->groups) {
        g.wsc.free();
        g.tc_btab.free(); g.tc_sq.free(); g.tc_tab_of_dev.free();
        if (g.d_k1) cudaFree(g.d_k1);
    }
    if (e->tc_status) cudaFreeHost(e->tc_status);
    e->params.free(); e->state.free(); e->bins.free(); e->base_bins.free(); e->win[0].free(); e->win[1].free(); e->wout.free(); e->sqbuf.free();
    e->tone_coeff.free(); e->tone_q1.free(); e->tone_q2.free(); e->tone_mag.free(); e->lut.free(); e->iqin[0].free(); e->iqin[1].free(); e->iqout.free();
    e->tw1.free(); e->tw2.free(); e->twn.free(); e->axc.free(); e->mix_sums.free(); e->mix_flags.free(); e->mix_offsets.free(); e->mix_inputs.free();
    if (e->d_k2) cudaFree(e->d_k2);
    for (auto& sc : e->scan)
        if (sc.stash) cudaFree(sc.stash);
    free_slot_results(e);
    for (auto& s : e->slots) {
        if (s.done) cudaEventDestroy(s.done);
        if (s.released) cudaEventDestroy(s.released);
    }
    for (auto& row : e->tl)
        for (auto& ev : row)
            if (ev) cudaEventDestroy(ev);
    for (int k = 0; k < 2; k++) {
        if (e->ev_k1[k]) cudaEventDestroy(e->ev_k1[k]);
        if (e->ev_k2[k]) cudaEventDestroy(e->ev_k2[k]);
    }
    if (e->stream_b) cudaStreamDestroy(e->stream_b);
    if (e->stream_c) {
        cudaStreamSynchronize(e->stream_c);
        cudaStreamDestroy(e->stream_c);
    }
    if (e->ev_ingest) cudaEventDestroy(e->ev_ingest);
    if (e->ev_caller) cudaEventDestroy(e->ev_caller);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

int frames_available(const abg_engine* e, const Device& d, size_t fill, size_t consumed) {
    // reference src/rtl_airband.cpp:394-400: a frame is taken only while available >= bps + fft_size*bytes_per_sample*2
    const size_t avail = fill - consumed;
    const size_t need = (size_t)d.hop_bytes + (size_t)e->N * d.bpc;
    if (avail < need) return 0;
    return (int)((avail - need) / d.hop_bytes) + 1;
}

// The freq_t part of one channel as parse_channels() sets it up (config.cpp:437-619): Squelch, NotchFilter,
// LowpassFilter, CTCSS banks, ampfactor, modulation, agcavgfast.  Used for channels[] at abg_create() and for every
// entry of a scan-mode frequency list (abg_scan_configure).  Channel-level fields of p / s are left alone.
int build_freq(int W, const abg_channel_cfg& cc, ChanParams& p, ChanState& s, std::vector<float> banks[2], const char* what) {
    if (cc.modulation != ABG_MOD_AM && cc.modulation != ABG_MOD_NFM) return fail(ABG_EINVAL, "%s: unknown modulation", what);
    p.modulation = cc.modulation;
    p.ampfactor = cc.ampfactor;
    p.notch_on = p.lp_on = p.ctcss_on = 0;
    p.n_tones[0] = p.n_tones[1] = 0;
    banks[0].clear();
    banks[1].clear();
    // ---- Squelch::Squelch(), squelch.cpp:36-82 ----
    s.noise_floor = 5.0f;
    s.manual = 0;
    s.normal_ratio = pow(10.0, 9.54f / 20.0);
    s.flappy_ratio = s.normal_ratio * 0.9f;
    s.avg_cap = 1.5f * s.normal_ratio * s.noise_floor;
    s.manual_level = -1.0;
    s.pre_full = s.pre_capped = s.post_full = s.post_capped = 0.001f;
    s.level_cache = 0.0f;
    s.using_post = 0;
    s.next_state = s.cur_state = SQ_CLOSED;
    s.delay = 0;
    s.sample_count_mod16 = 15u;  // sample_count_ = (size_t)-1: the first sample makes it 0 (squelch.cpp:58,204)
    s.head = 0;
    // ---- config.cpp:437-515: level first, then SNR ----
    if (cc.squelch_level > 0) {  // set_squelch_level_threshold, squelch.cpp:84-96
        s.manual = 1;
        s.manual_level = cc.squelch_level;
        s.avg_cap = 1.5f * s.manual_level;
    }
    if (cc.squelch_snr_db >= 0) {  // set_squelch_snr_threshold, squelch.cpp:98-108
        s.manual = 0;
        s.normal_ratio = pow(10.0, cc.squelch_snr_db / 20.0);
        s.flappy_ratio = s.normal_ratio * 0.9f;
        s.avg_cap = 1.5f * s.normal_ratio * s.noise_floor;
    }
    // ---- NotchFilter, filters.cpp:30-47 ----
    if (cc.notch_hz > 0) {
        float sample_freq = W, q = cc.notch_q;
        float wo = 2 * M_PI * (cc.notch_hz / sample_freq);
        float en = 1 / (1 + tan(wo / (q * 2)));
        float pn = cos(wo);
        p.notch_on = 1;
        p.nd0 = en;
        p.nd1 = 2 * en * pn;
        p.nd2 = (2 * en - 1);
    }
    // ---- LowpassFilter, filters.cpp:67-96 ----
    if (cc.lowpass_hz > 0) {
        if (!lowpass_design(cc.lowpass_hz, (float)W, &p.lp_gain, &p.lp_yc0, &p.lp_yc1))
            return fail(ABG_EINVAL, "%s: lowpass design failed (poles not conjugate)", what);
        p.lp_on = 1;
    }
    // ---- CTCSS, squelch.cpp:110-116 ----
    if (cc.ctcss_hz > 0) {
        const float sr = W;
        p.ctcss_on = 1;
        p.window[0] = sr * 0.05;
        p.window[1] = sr * 0.4;
        for (int w = 0; w < 2; w++) {
            std::vector<float> bank = tone_bank(cc.ctcss_hz, sr, p.window[w]);
            if ((int)bank.size() > ABG_MAX_TONES) return fail(ABG_EINVAL, "CTCSS bank too large");
            p.n_tones[w] = (int)bank.size();
            banks[w] = bank;
        }
    }
    s.agcavgfast = 0.5f;  // mk_freqlist / parse_channels, config.cpp:265-281
    return ABG_OK;
}

// 7-term Blackman-Harris window: float literals held in double, evaluated in double, stored float (rtl_airband.cpp:335-351)
std::vector<float> make_window(int N) {
    std::vector<float> window(N);
    const double a0 = 0.27105140069342f, a1 = 0.43329793923448f, a2 = 0.21812299954311f, a3 = 0.06592544638803f;
    const double a4 = 0.01081174209837f, a5 = 0.00077658482522f, a6 = 0.00001388721735f;
    const size_t fft_size = N;
    for (size_t i = 0; i < fft_size; i++) {
        double x = a0 - (a1 * cos((2.0 * M_PI * i) / (fft_size - 1))) + (a2 * cos((4.0 * M_PI * i) / (fft_size - 1))) - (a3 * cos((6.0 * M_PI * i) / (fft_size - 1))) +
                   (a4 * cos((8.0 * M_PI * i) / (fft_size - 1))) - (a5 * cos((10.0 * M_PI * i) / (fft_size - 1))) + (a6 * cos((12.0 * M_PI * i) / (fft_size - 1)));
        window[i] = (float)x;
    }
    return window;
}
float sample_scale(int sfmt, float fullscale) {
    // U8 levels are (i-127.5)/127.5, S8 i/128 (rtl_airband.cpp:319-324); S16/F32 scale = 1/fullscale (:403,421)
    return sfmt == ABG_SFMT_U8 ? 1.0f / 127.5f : sfmt == ABG_SFMT_S8 ? 1.0f / 128.0f : 1.0f / fullscale;
}

// (Re)build the tensor-core K1's coefficient tables of one launch group from the host copy of bins[]: one table per
// distinct list of bins (synthetic many-device configs share one), tab_of_dev[] maps the group's devices to tables.
int rebuild_tc_tables(abg_engine* e, Group& g) {
    std::vector<std::vector<int32_t>> keys;
    std::vector<int32_t> tab_of_dev(g.devs.size());
    for (size_t k = 0; k < g.devs.size(); k++) {
        const Device& d = e->dev[g.devs[k]];
        std::vector<int32_t> key(e->h_bins.begin() + d.g0, e->h_bins.begin() + d.g0 + d.C);
        size_t t = 0;
        while (t < keys.size() && keys[t] != key) t++;
        if (t == keys.size()) keys.push_back(key);
        tab_of_dev[k] = (int32_t)t;
    }
    const size_t nt = keys.size();
    std::vector<signed char> tab(nt * g.tc.table_bytes);
    std::vector<long long> sq(nt * g.tc.C2p);
    for (size_t t = 0; t < nt; t++)
        abg_k1tc_build_table(g.tc, e->N, g.sfmt, g.h_wsc.data(), keys[t].data(), (int)keys[t].size(), tab.data() + t * g.tc.table_bytes,
                             sq.data() + t * g.tc.C2p, &g.tc_cscale);
    if ((int)nt != g.tc_tables) {
        g.tc_btab.free(); g.tc_sq.free();
        if (g.tc_btab.alloc(tab.size()) || g.tc_sq.alloc(sq.size())) return fail(ABG_ENOMEM, "Out of device memory for the tensor-core coefficient tables");
        g.tc_tables = (int)nt;
    }
    if (!g.tc_tab_of_dev.p && g.tc_tab_of_dev.alloc(tab_of_dev.size())) return fail(ABG_ENOMEM, "Out of device memory for the tensor-core coefficient tables");
    CU(cudaMemcpy(g.tc_btab.p, tab.data(), tab.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(g.tc_sq.p, sq.data(), sizeof(long long) * sq.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(g.tc_tab_of_dev.p, tab_of_dev.data(), sizeof(int32_t) * tab_of_dev.size(), cudaMemcpyHostToDevice));
    return ABG_OK;
}

int build(abg_engine* e, const abg_config* cfg, const abg_options* opt) {
    Plan plan;
    if (!plan_for(cfg->fft_size, &plan)) return fail(ABG_EINVAL, "fft_size=%d not supported. Try a power of two between 256 and 8192.", cfg->fft_size);
    if (cfg->wave_rate < 8 || cfg->wave_rate % 8) return fail(ABG_EINVAL, "wave_rate=%d must be a positive multiple of 8", cfg->wave_rate);
    if (cfg->n_devices < 1 || !cfg->devices) return fail(ABG_EINVAL, "no devices configured");
    e->N = cfg->fft_size;
    e->W = cfg->wave_rate;
    e->B = cfg->wave_rate / 8;  // WAVE_BATCH, rtl_airband.h:73
    if (e->B < ABG_AGC_EXTRA) return fail(ABG_EINVAL, "wave_rate too small: WAVE_BATCH must be >= AGC_EXTRA");
    e->fm_demod = cfg->fm_demod;
    e->nbmax = (opt && opt->max_batches_per_run > 0) ? opt->max_batches_per_run : 4;
    e->fft_mode = opt ? opt->fft_mode : 0;
    if (const char* ev = getenv("ABG_K1_TC_DIGITS")) e->tc_digits = atoi(ev) == 3 ? 3 : 4;
    if (const char* ev = getenv("ABG_K1_TC_AUTO")) e->tc_auto = atoi(ev) != 0;
    const int in_cap_batches = (opt && opt->input_capacity_batches > 0) ? opt->input_capacity_batches : e->nbmax + 2;
    e->P = ABG_AGC_EXTRA + e->nbmax * e->B;
    const int N = e->N, B = e->B;

    // ---- devices, channel index space ------------------------------------------------------------------------
    e->dev.resize(cfg->n_devices);
    int G = 0;
    for (int i = 0; i < cfg->n_devices; i++) {
        const abg_device_cfg& dc = cfg->devices[i];
        Device& d = e->dev[i];
        d.sfmt = dc.sfmt;
        switch (dc.sfmt) {
            case ABG_SFMT_U8: case ABG_SFMT_S8: d.bpc = 2; break;
            case ABG_SFMT_S16: d.bpc = 4; break;
            case ABG_SFMT_F32: d.bpc = 8; break;
            default: return fail(ABG_EINVAL, "devices[%d]: unknown sample format %d", i, dc.sfmt);
        }
        if (dc.n_channels < 1 || !dc.channels) return fail(ABG_EINVAL, "devices[%d]: no channels configured", i);
        if (dc.sample_rate <= cfg->wave_rate) return fail(ABG_EINVAL, "devices[%d]: sample_rate must be greater than %d", i, cfg->wave_rate);
        if ((dc.sfmt == ABG_SFMT_S16 || dc.sfmt == ABG_SFMT_F32) && !(dc.fullscale > 0)) return fail(ABG_EINVAL, "devices[%d]: fullscale must be > 0", i);
        d.sample_rate = dc.sample_rate;
        d.fullscale = dc.fullscale;
        d.hop = (int)round((double)dc.sample_rate / (double)cfg->wave_rate);  // rtl_airband.cpp:394
        d.hop_bytes = d.hop * d.bpc;
        d.g0 = G;
        d.C = dc.n_channels;
        G += dc.n_channels;
    }
    e->G = G;
    e->Gp = (G + 31) & ~31;
    const int Gp = e->Gp;

    // ---- per-channel parameters and initial state ----------------------------------------------------------------
    std::vector<ChanParams> hp(Gp);
    std::vector<ChanState> hs(Gp);
    std::vector<int32_t> hb(Gp, 0);
    std::vector<float> h_coeff((size_t)2 * ABG_MAX_TONES * Gp, 0.0f);
    memset(hp.data(), 0, sizeof(ChanParams) * Gp);
    memset(hs.data(), 0, sizeof(ChanState) * Gp);
    for (int i = 0; i < cfg->n_devices; i++) {
        const abg_device_cfg& dc = cfg->devices[i];
        Device& d = e->dev[i];
        for (int c = 0; c < dc.n_channels; c++) {
            const abg_channel_cfg& cc = dc.channels[c];
            const int g = d.g0 + c;
            if (cc.bin < 0 || cc.bin >= N) return fail(ABG_EINVAL, "devices[%d].channels[%d]: bin %d outside 0..%d", i, c, cc.bin, N - 1);
            ChanParams& p = hp[g];
            ChanState& s = hs[g];
            hb[g] = cc.bin;
            p.dev = i;
            p.needs_raw_iq = cc.needs_raw_iq ? 1 : 0;
            p.has_iq_outputs = cc.has_iq_outputs ? 1 : 0;
            if (p.has_iq_outputs) e->any_iq_out = true;
            p.dm_dphi = cc.dm_dphi;
            p.alpha = cc.alpha;
            p.afc = cc.afc & 0xff;
            if (p.afc) d.has_afc = true;
            {
                char what[64];
                snprintf(what, sizeof(what), "devices[%d].channels[%d]", i, c);
                std::vector<float> banks[2];
                const int rc = build_freq(e->W, cc, p, s, banks, what);
                if (rc != ABG_OK) return rc;
                for (int w = 0; w < 2; w++)
                    for (size_t t = 0; t < banks[w].size(); t++) h_coeff[((size_t)w * ABG_MAX_TONES + t) * Gp + g] = banks[w][t];
            }
            // ---- mk_freqlist / parse_channels initial values, config.cpp:265-281,313-331 ----
            s.dm_phi = 0;
            s.pr = s.pj = 0.0f;
            s.prev_waveout = 0.5f;
            s.axc_prev = ABG_NO_SIGNAL;
        }
    }
    e->h_params = hp;
    for (int g = 0; g < G; g++)
        if (hp[g].modulation == ABG_MOD_NFM) e->any_nfm = true;
    e->h_bins = hb;

    // ---- tables -----------------------------------------------------------------------------------------------------
    const std::vector<float> window = make_window(N);
    std::vector<float> h_lut(2 * 257);
    for (uint32_t i = 0; i < 256; i++) sincosf(2.0F * M_PI * (float)i / 256.0f, &h_lut[i], &h_lut[257 + i]);  // util.cpp:105-110
    h_lut[256] = h_lut[0];
    h_lut[257 + 256] = h_lut[257];
    const int M1 = N / plan.r1;
    std::vector<float2> h_tw1((size_t)N);
    for (int k1 = 0; k1 < plan.r1; k1++)
        for (int n2 = 0; n2 < M1; n2++) {
            double ang = -2.0 * M_PI * (double)(((long)k1 * n2) % N) / (double)N;
            h_tw1[(size_t)k1 * M1 + n2] = make_float2((float)cos(ang), (float)sin(ang));
        }
    std::vector<float2> h_tw2;
    if (plan.r3) {
        const int M2 = plan.r3;
        h_tw2.resize((size_t)plan.r2 * M2);
        for (int k = 0; k < plan.r2; k++)
            for (int n3 = 0; n3 < M2; n3++) {
                double ang = -2.0 * M_PI * (double)(k * n3) / (double)M1;
                h_tw2[(size_t)k * M2 + n3] = make_float2((float)cos(ang), (float)sin(ang));
            }
    }

    std::vector<float2> h_twn((size_t)N);
    for (int m = 0; m < N; m++) {
        double ang = -2.0 * M_PI * (double)m / (double)N;
        h_twn[m] = make_float2((float)cos(ang), (float)sin(ang));
    }

    // ---- groups (one K1 launch per sample format / full-scale / hop) ------------------------------------------------------
    for (int i = 0; i < (int)e->dev.size(); i++) {
        Device& d = e->dev[i];
        int gi = -1;
        for (int k = 0; k < (int)e->groups.size(); k++)
            if (e->groups[k].sfmt == d.sfmt && e->groups[k].hop_bytes == d.hop_bytes &&
                (d.sfmt == ABG_SFMT_U8 || d.sfmt == ABG_SFMT_S8 || e->groups[k].fullscale == d.fullscale))
                gi = k;
        if (gi < 0) {
            Group g;
            g.sfmt = d.sfmt;
            g.hop_bytes = d.hop_bytes;
            g.fullscale = d.fullscale;
            e->groups.push_back(g);
            gi = (int)e->groups.size() - 1;
        }
        d.group = gi;
        e->groups[gi].devs.push_back(i);
    }

    // ---- CUDA resources ----------------------------------------------------------------------------------------------------
    {
        const char* pe = getenv("ABG_K2_PRIO");  // measurement knob: -1 = K1's stream above K2's
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(cudaStreamCreateWithPriority(&e->stream, cudaStreamNonBlocking, (pe && atoi(pe) < 0) ? hi : lo));
    }
    e->own_stream = true;
    CU(cudaHostAlloc((void**)&e->tc_status, 64, cudaHostAllocMapped));
    memset(e->tc_status, 0, 64);
    CU(cudaHostGetDevicePointer((void**)&e->tc_status_dev, e->tc_status, 0));
    {
        // K2's few long-running warps must get their SM slots ahead of the next run's K1 blocks
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        const char* pe = getenv("ABG_K2_PRIO");  // measurement knob: 0 = K2's stream at the default priority
        CU(cudaStreamCreateWithPriority(&e->stream_b, cudaStreamNonBlocking, (pe && atoi(pe) <= 0) ? lo : hi));
    }
    for (int k = 0; k < 2; k++) {
        CU(cudaEventCreateWithFlags(&e->ev_k1[k], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&e->ev_k2[k], cudaEventDisableTiming));
    }
    for (auto& row : e->tl)
        for (auto& ev : row) CU(cudaEventCreate(&ev));
    CU(cudaStreamCreateWithFlags(&e->stream_c, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&e->ev_ingest, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_caller, cudaEventDisableTiming));
    for (auto& d : e->dev)
        if (d.has_afc) e->any_afc = true;
    {
        // K2 is a sequential recurrence per channel.  One channel per warp (lane-parallel tiles, no divergence between
        // channels in different squelch states) as long as that is at most 8 warps per SM sub-partition (measured on
        // 4096 channels: K2 0.66 ms against 0.80 ms with 8 channels per warp); beyond that as few channels per warp as
        // keeps the warp count near two per sub-partition.
        int lpw = 1;
        if (e->G > 8 * 592)
            while (lpw < 32 && (e->G + lpw - 1) / lpw > 2 * 592) lpw <<= 1;
        const char* env = getenv("ABG_K2_LPW");
        if (env && atoi(env) > 0) {
            lpw = 1;
            while (lpw < 32 && lpw < atoi(env)) lpw <<= 1;
        }
        e->k2_lpw = lpw;
    }
    for (auto& g : e->groups) {
        g.frames_per_tile = abg_k1_tile_frames(N, g.sfmt, g.hop_bytes, &g.tile_bytes_cap);
        if (g.frames_per_tile < 1) return fail(ABG_EINVAL, "fft_size=%d with this sample format does not fit shared memory", N);
        bool group_afc = false;
        for (int di : g.devs) {
            g.max_channels = std::max(g.max_channels, e->dev[di].C);
            if (e->dev[di].has_afc) group_afc = true;
        }
        g.p_frames_per_tile = abg_k1p_tile_frames(N, g.sfmt, g.hop_bytes, g.max_channels, &g.p_tile_bytes_cap);
        // fft_mode: 0 auto; 1 = full spectrum every frame; 2 = output-pruned last pass on the FP32 pipes; 3 = the bins' DFT as an
        // integer GEMM on the tensor cores (8-bit formats; other groups fall back to 2).  Groups with AFC need whole spectra.
        g.pruned = (e->fft_mode != 1) && !group_afc && g.p_frames_per_tile >= 1;
        const bool want_tc = e->fft_mode == 3 || (e->fft_mode == 0 && e->tc_auto);
        g.use_tc = want_tc && !group_afc && abg_k1tc_plan(N, g.sfmt, g.hop_bytes, g.max_channels, e->tc_digits, &g.tc) == 1;
        const float scale = sample_scale(g.sfmt, g.fullscale);  // window * 1/full-scale
        std::vector<float> wsc(N);
        for (int i = 0; i < N; i++) wsc[i] = window[i] * scale;
        g.h_wsc = wsc;
        CU(g.wsc.alloc(N));
        CU(cudaMemcpy(g.wsc.p, wsc.data(), N * sizeof(float), cudaMemcpyHostToDevice));
        CU(cudaMalloc((void**)&g.d_k1, sizeof(K1Dev) * (g.devs.size() + 1)));
        g.h_k1.assign(g.devs.size() + 1, K1Dev{});
        if (g.use_tc) {
            const int rc = rebuild_tc_tables(e, g);
            if (rc != ABG_OK) return rc;
        }
    }
    for (auto& d : e->dev) {
        // room for in_cap_batches batches + the AGC_EXTRA priming frames + one window, + slack for 16-byte TMA rounding
        d.cap = ((size_t)(in_cap_batches * B + ABG_AGC_EXTRA) * d.hop_bytes + (size_t)N * d.bpc + (size_t)d.hop_bytes + 255) & ~(size_t)255;
        for (int k = 0; k < 2; k++) {
            cudaError_t er = cudaMalloc((void**)&d.raw[k], d.cap + 256);
            if (er != cudaSuccess) return fail(ABG_ENOMEM, "Out of device memory for input buffers (%s)", cudaGetErrorString(er));
            CU(cudaMemsetAsync(d.raw[k], 0, d.cap + 256, e->stream));
        }
        if (d.has_afc) CU(cudaMalloc((void**)&d.spec, sizeof(float2) * (size_t)e->nbmax * N));
    }
    const size_t PG = (size_t)e->P * Gp;
    if (e->params.alloc(Gp) || e->state.alloc(Gp) || e->bins.alloc(Gp) || e->base_bins.alloc(Gp) || e->win[0].alloc(PG) || e->win[1].alloc(PG) || e->iqin[0].alloc(PG) || e->iqin[1].alloc(PG) ||
        e->wout.alloc(PG) || e->sqbuf.alloc((size_t)ABG_SQ_BUF * Gp) || e->tone_coeff.alloc(h_coeff.size()) || e->tone_q1.alloc(h_coeff.size()) ||
        e->tone_q2.alloc(h_coeff.size()) || e->tone_mag.alloc(h_coeff.size()) || e->lut.alloc(h_lut.size()) || e->tw1.alloc(h_tw1.size()) ||
        e->tw2.alloc(std::max<size_t>(h_tw2.size(), 1)) || e->twn.alloc(h_twn.size()) || e->axc.alloc((size_t)e->nbmax * Gp) ||
        (e->any_iq_out && e->iqout.alloc((size_t)Gp * e->nbmax * B)))
        return fail(ABG_ENOMEM, "Out of device memory. Try fewer devices per GPU or a smaller max_batches_per_run.");
    CU(cudaMemcpy(e->params.p, hp.data(), sizeof(ChanParams) * Gp, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->state.p, hs.data(), sizeof(ChanState) * Gp, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->bins.p, hb.data(), sizeof(int32_t) * Gp, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->base_bins.p, hb.data(), sizeof(int32_t) * Gp, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->tone_coeff.p, h_coeff.data(), sizeof(float) * h_coeff.size(), cudaMemcpyHostToDevice));
    CU(cudaMemset(e->tone_q1.p, 0, sizeof(float) * h_coeff.size()));
    CU(cudaMemset(e->tone_q2.p, 0, sizeof(float) * h_coeff.size()));
    CU(cudaMemset(e->tone_mag.p, 0, sizeof(float) * h_coeff.size()));
    CU(cudaMemset(e->sqbuf.p, 0, sizeof(float) * ABG_SQ_BUF * Gp));  // calloc, squelch.cpp:70
    CU(cudaMemcpy(e->lut.p, h_lut.data(), sizeof(float) * h_lut.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->tw1.p, h_tw1.data(), sizeof(float2) * h_tw1.size(), cudaMemcpyHostToDevice));
    if (!h_tw2.empty()) CU(cudaMemcpy(e->tw2.p, h_tw2.data(), sizeof(float2) * h_tw2.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->twn.p, h_twn.data(), sizeof(float2) * h_twn.size(), cudaMemcpyHostToDevice));
    CU(cudaMemset(e->iqin[0].p, 0, sizeof(float2) * PG));
    CU(cudaMemset(e->iqin[1].p, 0, sizeof(float2) * PG));
    if (e->any_iq_out) CU(cudaMemset(e->iqout.p, 0, sizeof(float2) * (size_t)Gp * e->nbmax * B));
    {
        // config.cpp:313-316: wavein[0..AGC_EXTRA) = 20, waveout[0..AGC_EXTRA) = 0.5.  (wavein's priming values are
        // overwritten by the first AGC_EXTRA frames because waveend starts at 0, config.cpp:805; kept for fidelity.)
        std::vector<float> hw(PG, 0.0f), ho(PG, 0.0f);
        for (int k = 0; k < ABG_AGC_EXTRA; k++)
            for (int g = 0; g < Gp; g++) hw[(size_t)k * Gp + g] = 20.0f;
        for (int g = 0; g < Gp; g++)
            for (int k = 0; k < ABG_AGC_EXTRA; k++) ho[(size_t)g * e->P + k] = 0.5f;
        CU(cudaMemcpy(e->win[0].p, hw.data(), sizeof(float) * PG, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(e->win[1].p, hw.data(), sizeof(float) * PG, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(e->wout.p, ho.data(), sizeof(float) * PG, cudaMemcpyHostToDevice));
    }
    CU(cudaMalloc((void**)&e->d_k2, sizeof(K2Dev) * e->dev.size() + 16));
    e->h_k2.assign(e->dev.size(), K2Dev{});
    e->slots.resize(3);
    for (auto& s : e->slots) {
        CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.released, cudaEventDisableTiming));
    }
    {
        const int rc = alloc_slot_results(e);
        if (rc != ABG_OK) return rc;
    }
    CU(cudaStreamSynchronize(e->stream));
    return ABG_OK;
}

// enqueue K1 (+K2) for the per-device batch counts in nb[]; `resident` selects the replay buffers.
int enqueue_run(abg_engine* e, const std::vector<int>& nb, bool resident, bool queue_outputs, int* n_enqueued, bool skip_k1 = false) {
    const int B = e->B, N = e->N;
    int total = 0, nbrun = 0;
    for (int v : nb) {
        total += v;
        nbrun = std::max(nbrun, v);
    }
    *n_enqueued = total;
    if (total == 0) return ABG_OK;
    int slot = -1;
    if (queue_outputs) {
        slot = e->next_slot;
        if (e->slots[slot].pending > 0 || e->slots[slot].mix_pending > 0)
            return fail(ABG_EOVERFLOW, "output overrun: %d finished device batches and %d mixer batches of an earlier run not fetched yet (every configured mixer has to be drained with abg_fetch_mixer_batch)",
                        e->slots[slot].pending, e->slots[slot].mix_pending);
        e->next_slot = (e->next_slot + 1) % (int)e->slots.size();
    }
    cudaStream_t sa = e->stream, sb = e->stream_b;
    const uint64_t ri = e->run_index;
    const int cur = (int)(ri & 1);
    // K1 of this run overwrites win/iqin[cur], last read by K2 of run ri-2; with AFC it also needs the bins K2 of
    // run ri-1 chose.  (ev_k2[x] is re-recorded by every run of that parity; the wait binds to the latest record.)
    if (ri >= 2) CU(cudaStreamWaitEvent(sa, e->ev_k2[cur], 0));
    if (ri >= 1 && e->any_afc) CU(cudaStreamWaitEvent(sa, e->ev_k2[cur ^ 1], 0));
    if (!resident && e->ingest_dirty) {  // K1 reads what abg_push copied on the ingest stream
        CU(cudaEventRecord(e->ev_ingest, e->stream_c));
        CU(cudaStreamWaitEvent(sa, e->ev_ingest, 0));
        e->ingest_dirty = false;
    }
    cudaEvent_t* tl = e->tl[ri % abg_engine::TL_RUNS];
    CU(cudaEventRecord(tl[0], sa));
    // ---- K1 per group (stream A) ----
    for (auto& g : e->groups) {
        if (skip_k1) break;  // abg_debug_inject_wavein: the magnitudes were written into win[cur] directly
        int max_frames = 0;
        for (size_t k = 0; k < g.devs.size(); k++) {
            const int di = g.devs[k];
            Device& d = e->dev[di];
            K1Dev& a = g.h_k1[k];
            const bool primed = resident ? d.res_primed : d.primed;
            a.raw = resident ? d.res : d.raw[d.cur];
            a.n_frames = nb[di] > 0 ? nb[di] * B + (primed ? 0 : ABG_AGC_EXTRA) : 0;
            a.pos0 = primed ? ABG_AGC_EXTRA : 0;
            a.start_byte = resident ? (primed ? (unsigned long long)ABG_AGC_EXTRA * d.hop_bytes : 0ull) : (unsigned long long)d.consumed;
            a.g0 = d.g0;
            a.n_channels = d.C;
            a.hop_bytes = d.hop_bytes;
            a.sfmt = d.sfmt;
            a.spec = d.has_afc ? d.spec : nullptr;
            a.spec_first_pos = ABG_AGC_EXTRA + B - 1;  // the frame that completes batch 0 of the run (waveend hits B+100)
            a.wave_batch = B;
            max_frames = std::max(max_frames, a.n_frames);
        }
        if (max_frames == 0) continue;
        {
            // (the trailing all-zero entry resets the tensor-core kernel's tile counter)
            const int nl = upload_small(g.d_k1, g.h_k1.data(), sizeof(K1Dev) * (g.devs.size() + (g.use_tc ? 1 : 0)), sa);
            if (nl < 0) return fail(ABG_ECUDA, "K1 parameter upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            e->launches += (uint64_t)nl;
        }
        K1Launch L{};
        L.fft_size = N; L.n_devices = (int)g.devs.size(); L.max_frames = max_frames;
        L.frames_per_tile = g.pruned ? g.p_frames_per_tile : g.frames_per_tile;
        L.tile_bytes_cap = g.pruned ? g.p_tile_bytes_cap : g.tile_bytes_cap;
        L.devs = g.d_k1; L.bins = e->bins.p; L.window_scaled = g.wsc.p; L.tw1 = e->tw1.p;
        L.tw2 = e->tw2.p; L.win = e->win[cur].p; L.iqin = e->iqin[cur].p; L.Gp = e->Gp; L.sfmt = g.sfmt;
        cudaError_t er1;
        if (g.use_tc) {
            K1TcTables T{};
            T.tab_of_dev = g.tc_tab_of_dev.p; T.btab = g.tc_btab.p; T.sq = g.tc_sq.p;
            T.counter = reinterpret_cast<int*>(g.d_k1 + g.devs.size());
            T.status = e->tc_status_dev; T.cscale = g.tc_cscale;
            er1 = abg_launch_k1_tc(L, g.tc, T, e->sm_count, sa);
        } else {
            er1 = g.pruned ? abg_launch_k1_pruned(L, e->twn.p, g.max_channels, sa) : abg_launch_k1(L, sa);
        }
        if (er1 != cudaSuccess) return fail(ABG_ECUDA, "K1 launch failed: %s", cudaGetErrorString(er1));
        e->launches += g.use_tc ? 1 : g.pruned ? (uint64_t)((g.max_channels + 31) / 32) : 1;
    }
    CU(cudaEventRecord(tl[1], sa));
    CU(cudaEventRecord(e->ev_k1[cur], sa));
    // ---- K2 (stream B, after this run's K1; overlaps the next run's K1) ----
    CU(cudaStreamWaitEvent(sb, e->ev_k1[cur], 0));
    for (size_t i = 0; i < e->dev.size(); i++) {
        e->h_k2[i].n_batches = nb[i];
        e->h_k2[i].fft_size = N;
        e->h_k2[i].spec = e->dev[i].has_afc ? e->dev[i].spec : nullptr;
    }
    {
        const int nl = upload_small(e->d_k2, e->h_k2.data(), sizeof(K2Dev) * e->dev.size(), sb);
        if (nl < 0) return fail(ABG_ECUDA, "K2 parameter upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        e->launches += (uint64_t)nl;
    }
    CU(cudaEventRecord(tl[2], sb));
    K2Launch L2 = e->k2_launch(cur);
    cudaError_t er = abg_launch_k2(L2, sb);
    if (er != cudaSuccess) return fail(ABG_ECUDA, "K2 launch failed: %s", cudaGetErrorString(er));
    e->launches++;
    CU(cudaEventRecord(tl[3], sb));
    // device mode: a device fetch may still be copying this slot's previous contents on the caller's stream
    if (queue_outputs && e->slots[slot].release_pending) CU(cudaStreamWaitEvent(sb, e->slots[slot].released, 0));
    // ---- mixers: sums over the just-finished batches, before the tail copy (output.cpp:533-535 -> mixer.cpp) ----
    if (e->n_mixers > 0) {
        MixLaunch M{};
        M.n_mixers = e->n_mixers; M.n_batches = nbrun; M.wave_batch = B; M.P = e->P; M.Gp = e->Gp; M.offsets = e->mix_offsets.p;
        M.inputs = e->mix_inputs.p; M.devs = e->d_k2; M.wout = e->wout.p; M.axc = e->axc.p; M.sums = e->mix_sums.p; M.flags = e->mix_flags.p;
        if (queue_outputs) {
            M.host_sums = e->slots[slot].mix;
            M.host_flags = e->slots[slot].mixflag;
        }
        er = abg_launch_mix(M, sb);
        if (er != cudaSuccess) return fail(ABG_ECUDA, "mixer launch failed: %s", cudaGetErrorString(er));
        e->launches++;
    }
    // ---- results: the end-of-run kernel writes them straight into the pinned slot, then does the consumer's tail copy ----
    K2Export X{};
    if (queue_outputs) {
        Slot& s = e->slots[slot];
        X.host_wout = s.wout;
        X.host_iqout = e->any_iq_out ? reinterpret_cast<float2*>(s.iqout) : nullptr;
        X.host_axc = s.axc;
        X.stride = (size_t)e->nbmax * B;
    }
    er = abg_launch_k2_tail(L2, X, sb);
    if (er != cudaSuccess) return fail(ABG_ECUDA, "export/tail-copy launch failed: %s", cudaGetErrorString(er));
    e->launches++;
    if (queue_outputs) {
        Slot& s = e->slots[slot];
        CU(cudaEventRecord(s.done, sb));
        for (size_t i = 0; i < e->dev.size(); i++)
            for (int b = 0; b < nb[i]; b++) {
                e->dev[i].ready.emplace_back(slot, b);
                s.pending++;
            }
        if (e->n_mixers > 0)
            for (int b = 0; b < nbrun; b++) {
                e->mix_ready.emplace_back(slot, b);
                s.mix_pending += e->n_mixers;
            }
    }
    CU(cudaEventRecord(tl[4], sb));
    CU(cudaEventRecord(e->ev_k2[cur], sb));
    e->tev_valid = true;
    e->run_index++;
    // ---- bookkeeping ----
    for (size_t i = 0; i < e->dev.size(); i++) {
        if (nb[i] <= 0) continue;
        Device& d = e->dev[i];
        if (skip_k1) {
            // nothing was consumed from the raw stream
        } else if (resident) {
            d.res_primed = true;
        } else {
            const int frames = nb[i] * B + (d.primed ? 0 : ABG_AGC_EXTRA);
            d.consumed += (size_t)frames * d.hop_bytes;
            d.primed = true;
            d.runs_since_compaction++;
        }
    }
    return ABG_OK;
}

// Append nbytes at the end of a device's raw stream on the ingest stream (stream C), compacting first when they do
// not fit behind the buffered bytes.  abg_push (host source) and abg_push_device (device source) differ only in `kind`.
int push_bytes(abg_engine* e, int dev, const void* iq, size_t nbytes, cudaMemcpyKind kind, const char* who) {
    Device& d = e->dev[dev];
    if (d.fill + nbytes > d.cap) {
        // compact: move the unconsumed tail to the front of the other buffer.  Ingest runs on its own stream so that
        // host->device copies overlap K1; the other buffer may still be read by the most recent K1, so wait for it.
        const size_t keep_from = d.consumed & ~(size_t)15;  // keep the copy 16-byte aligned on both sides
        const size_t rem = d.fill - keep_from;
        if (rem + nbytes > d.cap) {
            return fail(ABG_EOVERFLOW, "%s: device %d input buffer overflow (%zu buffered + %zu new > %zu)", who, dev, d.fill - d.consumed, nbytes, d.cap);
        }
        // the destination buffer was last read by a K1 launched before the previous compaction: with at least one run since
        // then that is run_index-2 or older, so the copy overlaps the K1 that is reading the current buffer right now
        if (d.runs_since_compaction >= 1) {
            if (e->run_index >= 2) CU(cudaStreamWaitEvent(e->stream_c, e->ev_k1[(e->run_index - 2) & 1], 0));
        } else if (e->run_index >= 1) {
            CU(cudaStreamWaitEvent(e->stream_c, e->ev_k1[(e->run_index - 1) & 1], 0));
        }
        d.runs_since_compaction = 0;
        CU(cudaMemcpyAsync(d.raw[d.cur ^ 1], d.raw[d.cur] + keep_from, rem, cudaMemcpyDeviceToDevice, e->stream_c));
        d.cur ^= 1;
        d.fill = rem;
        d.consumed -= keep_from;
    }
    CU(cudaMemcpyAsync(d.raw[d.cur] + d.fill, iq, nbytes, kind, e->stream_c));
    e->ingest_dirty = true;
    d.fill += nbytes;
    return ABG_OK;
}

// ---- device-resident result fetches -------------------------------------------------------------------------------
// The blocks of one batch: channels [g_begin, g_begin + nch) of batch b (of its run) in slot s go to channel offset dst_ch
// of the caller's batch-major buffers (audio and I/Q rows of WAVE_BATCH samples, one flag byte per channel).
void gather_batch(const abg_engine* e, std::vector<GatherCopy>& cps, const Slot& s, int b, int g_begin, int nch, size_t dst_ch, float* d_wo,
                  float* d_iq, char* d_axc) {
    const size_t B = (size_t)e->B, stride = (size_t)e->nbmax * e->B;
    const size_t src0 = (size_t)g_begin * stride + (size_t)b * B;
    if (d_wo)
        cps.push_back({reinterpret_cast<const unsigned char*>(s.wout + src0), reinterpret_cast<unsigned char*>(d_wo + dst_ch * B),
                       (long long)(sizeof(float) * stride), (long long)(sizeof(float) * B), nch, (int32_t)(sizeof(float) * B)});
    if (d_iq)  // no channel with I/Q outputs: zeros, like the host path
        cps.push_back({s.iqout ? reinterpret_cast<const unsigned char*>(s.iqout + 2 * src0) : nullptr, reinterpret_cast<unsigned char*>(d_iq + dst_ch * 2 * B),
                       (long long)(sizeof(float2) * stride), (long long)(sizeof(float2) * B), nch, (int32_t)(sizeof(float2) * B)});
    if (d_axc)
        cps.push_back({s.axc + (size_t)b * e->Gp + g_begin, reinterpret_cast<unsigned char*>(d_axc + dst_ch), nch, nch, 1, nch});
}

// Enqueue the gather on the caller's stream.  It first waits for the runs that filled the slots, and for earlier device
// fetches from them (so that the release event recorded afterwards covers every reader of the slot, whatever stream it
// used); enqueue_run makes the export of a later run into one of these slots wait for that release event.
int gather_launch(abg_engine* e, const std::vector<GatherCopy>& cps, const std::vector<int>& slots, cudaStream_t cs) {
    for (int k : slots) {
        const Slot& s = e->slots[k];
        CU(cudaStreamWaitEvent(cs, s.done, 0));
        if (s.release_pending) CU(cudaStreamWaitEvent(cs, s.released, 0));
    }
    for (size_t i0 = 0; i0 < cps.size(); i0 += ABG_GATHER_MAX) {
        GatherList L;
        L.n = (int32_t)std::min<size_t>(ABG_GATHER_MAX, cps.size() - i0);
        L.max_rows = 0;
        for (int i = 0; i < L.n; i++) {
            L.c[i] = cps[i0 + i];
            L.max_rows = std::max(L.max_rows, L.c[i].rows);
        }
        const cudaError_t er = abg_launch_gather(L, cs);
        if (er != cudaSuccess) return fail(ABG_ECUDA, "result gather launch failed: %s", cudaGetErrorString(er));
        e->launches++;
    }
    for (int k : slots) {
        Slot& s = e->slots[k];
        CU(cudaEventRecord(s.released, cs));
        s.release_pending = true;
    }
    return ABG_OK;
}

void note_slot(std::vector<int>& used, int slot) {
    if (std::find(used.begin(), used.end(), slot) == used.end()) used.push_back(slot);
}

int need_device_results(const abg_engine* e, const char* who) {
    if (e->results_where == ABG_RESULTS_DEVICE) return ABG_OK;
    return fail(ABG_EINVAL, "%s: results are in host memory; call abg_set_result_location(ABG_RESULTS_DEVICE) before the first run", who);
}

}  // namespace

// =========================================================================================================================
// C ABI
// =========================================================================================================================
extern "C" {

const char* abg_last_error(void) { return g_err.c_str(); }
const char* abg_version(void) { return "airband-b200 0.1 (sm_100a)"; }

int abg_create(const abg_config* cfg, const abg_options* opt, abg_engine** out) {
    if (!cfg || !out) return fail(ABG_EINVAL, "abg_create: null argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t er = cudaGetDeviceCount(&ndev);
    if (er != cudaSuccess || ndev < 1)
        return fail(ABG_ENODEV, "Unable to find a CUDA device (%s). This engine has no CPU fallback.", er == cudaSuccess ? "device count is 0" : cudaGetErrorString(er));
    abg_engine* e = new abg_engine();
    if (opt && opt->cuda_device >= 0) {
        e->cuda_dev = opt->cuda_device;
        if (cudaSetDevice(e->cuda_dev) != cudaSuccess) {
            delete e;
            return fail(ABG_ENODEV, "cudaSetDevice(%d) failed", opt->cuda_device);
        }
    } else {
        cudaGetDevice(&e->cuda_dev);
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, e->cuda_dev) != cudaSuccess || prop.major < 10) {
        int major = prop.major;
        delete e;
        return fail(ABG_ENODEV, "CUDA device has compute capability %d.x; this library contains sm_100a code only", major);
    }
    e->sm_count = prop.multiProcessorCount;
    int rc = build(e, cfg, opt);
    if (rc != ABG_OK) {
        std::string keep = g_err;
        engine_free(e);
        g_err = keep;
        return rc;
    }
    *out = e;
    return ABG_OK;
}

void abg_destroy(abg_engine* e) { engine_free(e); }
int abg_wave_batch(const abg_engine* e) { return e->B; }
int abg_hop(const abg_engine* e, int dev) { return (dev < 0 || dev >= (int)e->dev.size()) ? ABG_ERANGE : e->dev[dev].hop; }

int abg_push(abg_engine* e, int dev, const void* iq, size_t nbytes) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_push: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (nbytes == 0) return ABG_OK;
    if (nbytes % d.bpc) return fail(ABG_EINVAL, "abg_push: %zu bytes is not a whole number of complex samples", nbytes);
    cudaSetDevice(e->cuda_dev);
    return push_bytes(e, dev, iq, nbytes, cudaMemcpyHostToDevice, "abg_push");
}

int abg_push_device(abg_engine* e, int dev, const void* d_iq, size_t nbytes, void* cuda_stream) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_push_device: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (nbytes == 0) return ABG_OK;
    if (nbytes % d.bpc) return fail(ABG_EINVAL, "abg_push_device: %zu bytes is not a whole number of complex samples", nbytes);
    if (!d_iq) return fail(ABG_EINVAL, "abg_push_device: null source");
    cudaSetDevice(e->cuda_dev);
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, d_iq) != cudaSuccess) {
        cudaGetLastError();
        return fail(ABG_EINVAL, "abg_push_device: %p is not a CUDA allocation", d_iq);
    }
    if (a.type != cudaMemoryTypeDevice || a.device != e->cuda_dev)
        return fail(ABG_EINVAL, "abg_push_device: source must be device memory on GPU %d (memory type %d on device %d)", e->cuda_dev, (int)a.type, a.device);
    // what the caller enqueued on its stream so far (e.g. the kernel that produced the samples) comes first
    CU(cudaEventRecord(e->ev_caller, (cudaStream_t)cuda_stream));
    CU(cudaStreamWaitEvent(e->stream_c, e->ev_caller, 0));
    return push_bytes(e, dev, d_iq, nbytes, cudaMemcpyDeviceToDevice, "abg_push_device");
}

int abg_ingest_join(abg_engine* e, void* cuda_stream) {
    cudaSetDevice(e->cuda_dev);
    CU(cudaEventRecord(e->ev_ingest, e->stream_c));
    CU(cudaStreamWaitEvent((cudaStream_t)cuda_stream, e->ev_ingest, 0));
    return ABG_OK;
}

int abg_batches_available(const abg_engine* e, int dev) {
    if (dev < 0 || dev >= (int)e->dev.size()) return ABG_ERANGE;
    const Device& d = e->dev[dev];
    const int frames = frames_available(e, d, d.fill, d.consumed) - (d.primed ? 0 : ABG_AGC_EXTRA);
    return frames <= 0 ? 0 : frames / e->B;
}

int abg_run(abg_engine* e, int max_batches) {
    cudaSetDevice(e->cuda_dev);
    if (max_batches < 0 || max_batches > e->nbmax) max_batches = e->nbmax;
    // AFC moves bins[] between batches (rtl_airband.cpp:629): with any AFC channel the run advances one batch at a
    // time so that K1 of batch k+1 sees the bins K2 chose at the end of batch k.
    // (only the AFC devices: the others still advance by up to max_batches in the same run)
    std::vector<int> nb(e->dev.size());
    for (size_t i = 0; i < e->dev.size(); i++) nb[i] = std::min(e->dev[i].has_afc ? 1 : max_batches, abg_batches_available(e, (int)i));
    int n = 0;
    int rc = enqueue_run(e, nb, false, true, &n);
    return rc != ABG_OK ? rc : n;
}

int abg_sync(abg_engine* e) {
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream_c));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    if (e->tc_status && e->tc_status[0]) return fail(ABG_ECUDA, "tensor-core K1 pipeline stalled (wait code %d); results of that run are invalid", e->tc_status[0]);
    return ABG_OK;
}

int abg_join(abg_engine* e) {
    cudaSetDevice(e->cuda_dev);
    if (e->run_index > 0) CU(cudaStreamWaitEvent(e->stream, e->ev_k2[(e->run_index - 1) & 1], 0));
    return ABG_OK;
}

int abg_batches_ready(abg_engine* e, int dev) {
    if (dev < 0 || dev >= (int)e->dev.size()) return ABG_ERANGE;
    return (int)e->dev[dev].ready.size();
}

int abg_fetch_batch(abg_engine* e, int dev, float* waveout, float* iq_out, char* axcindicate) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_fetch_batch: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (d.ready.empty()) return 0;
    const std::pair<int, int> r = d.ready.front();
    Slot& s = e->slots[r.first];
    cudaSetDevice(e->cuda_dev);
    CU(cudaEventSynchronize(s.done));
    if (e->tc_status && e->tc_status[0]) return fail(ABG_ECUDA, "tensor-core K1 pipeline stalled (wait code %d); results of that run are invalid", e->tc_status[0]);
    const int B = e->B;
    const size_t stride = (size_t)e->nbmax * B;
    if (e->results_where == ABG_RESULTS_DEVICE) {  // the same bytes, copied out of the slot in HBM
        const size_t g0 = (size_t)d.g0, off = (size_t)r.second * B;
        if (waveout) CU(cudaMemcpy2D(waveout, sizeof(float) * B, s.wout + g0 * stride + off, sizeof(float) * stride, sizeof(float) * B, d.C, cudaMemcpyDeviceToHost));
        if (iq_out) {
            if (s.iqout)
                CU(cudaMemcpy2D(iq_out, sizeof(float2) * B, s.iqout + 2 * (g0 * stride + off), sizeof(float2) * stride, sizeof(float2) * B, d.C, cudaMemcpyDeviceToHost));
            else
                memset(iq_out, 0, sizeof(float) * 2 * B * d.C);
        }
        if (axcindicate) CU(cudaMemcpy(axcindicate, s.axc + (size_t)r.second * e->Gp + g0, d.C, cudaMemcpyDeviceToHost));
        d.ready.pop_front();
        s.pending--;
        return 1;
    }
    for (int c = 0; c < d.C; c++) {
        const size_t g = (size_t)d.g0 + c;
        if (waveout) memcpy(waveout + (size_t)c * B, s.wout + g * stride + (size_t)r.second * B, sizeof(float) * B);
        if (iq_out) {
            if (s.iqout)
                memcpy(iq_out + (size_t)c * 2 * B, s.iqout + 2 * (g * stride + (size_t)r.second * B), sizeof(float) * 2 * B);
            else
                memset(iq_out + (size_t)c * 2 * B, 0, sizeof(float) * 2 * B);
        }
        if (axcindicate) axcindicate[c] = (char)s.axc[(size_t)r.second * e->Gp + g];
    }
    d.ready.pop_front();
    s.pending--;
    return 1;
}

int abg_fetch_batches(abg_engine* e, int dev, int max_batches, float* waveout, float* iq_out, char* axcindicate) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_fetch_batches: device %d out of range", dev);
    const Device& d = e->dev[dev];
    const size_t C = (size_t)d.C, B = (size_t)e->B;
    int n = 0;
    while (n < max_batches) {
        int rc = abg_fetch_batch(e, dev, waveout ? waveout + (size_t)n * C * B : nullptr, iq_out ? iq_out + (size_t)n * C * 2 * B : nullptr,
                                 axcindicate ? axcindicate + (size_t)n * C : nullptr);
        if (rc < 0) return rc;
        if (rc == 0) break;
        n++;
    }
    return n;
}

int abg_get_stats(abg_engine* e, int dev, int chan, abg_squelch_stats* out) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_get_stats: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (chan < 0 || chan >= d.C || !out) return fail(ABG_ERANGE, "abg_get_stats: channel %d out of range", chan);
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    ChanState s;
    int32_t bin;
    CU(cudaMemcpy(&s, e->state.p + d.g0 + chan, sizeof(s), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&bin, e->bins.p + d.g0 + chan, sizeof(bin), cudaMemcpyDeviceToHost));
    out->noise_level = s.noise_floor;
    out->signal_level = s.pre_full;
    // Squelch::squelch_level(), squelch.cpp:164-177 (read-only evaluation)
    if (s.manual)
        out->squelch_level = s.manual_level;
    else if (s.level_cache != 0.0f)
        out->squelch_level = s.level_cache;
    else
        out->squelch_level = ((s.recent_open_count >= 3u && s.flappy_ratio < s.normal_ratio) ? s.flappy_ratio : s.normal_ratio) * s.noise_floor;
    out->open_count = s.open_count;
    out->flappy_count = s.flappy_count;
    out->ctcss_count = s.ct_found[1];
    out->no_ctcss_count = s.ct_not_found[1];
    out->agcavgfast = s.agcavgfast;
    out->dm_phi = s.dm_phi;
    out->bin = bin;
    out->active_counter = s.active_counter;
    // level_to_dBFS(), util.cpp:169-180: min(0, 20*log10f(level / fft_size) + 7.54f + 10*log10f(fft_size / 2) - 2.38f)
    const size_t fft_size = (size_t)e->N;
    const float offset = 7.54f + 10.0f * log10f(fft_size / 2) - 2.38f;
    auto to_dbfs = [&](float level) { return std::min(0.0f, 20.0f * log10f(level / fft_size) + offset); };
    out->noise_level_dbfs = to_dbfs(out->noise_level);
    out->signal_level_dbfs = to_dbfs(out->signal_level);
    out->squelch_level_dbfs = to_dbfs(out->squelch_level);
    return ABG_OK;
}

int abg_set_bin(abg_engine* e, int dev, int chan, int bin) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_set_bin: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (chan < 0 || chan >= d.C) return fail(ABG_ERANGE, "abg_set_bin: channel %d out of range", chan);
    if (bin < 0 || bin >= e->N) return fail(ABG_EINVAL, "abg_set_bin: bin %d outside 0..%d", bin, e->N - 1);
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream_b));
    int32_t v = bin;
    CU(cudaMemcpyAsync(e->bins.p + d.g0 + chan, &v, sizeof(v), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(e->base_bins.p + d.g0 + chan, &v, sizeof(v), cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    e->h_bins[d.g0 + chan] = bin;
    Group& g = e->groups[d.group];
    if (g.use_tc) return rebuild_tc_tables(e, g);  // the coefficient table carries the bin
    return ABG_OK;
}

int abg_fft_path(const abg_engine* e, int dev) {
    if (dev < 0 || dev >= (int)e->dev.size()) return ABG_ERANGE;
    const Group& g = e->groups[e->dev[dev].group];
    return g.use_tc ? 3 : (g.pruned ? 2 : 1);
}

// ---- scan mode -------------------------------------------------------------------------------------------------------
static ScanView scan_view(abg_engine* e) {
    ScanView v;
    v.params = e->params.p; v.state = e->state.p; v.sqbuf = e->sqbuf.p; v.tone_coeff = e->tone_coeff.p;
    v.tone_q1 = e->tone_q1.p; v.tone_q2 = e->tone_q2.p; v.tone_mag = e->tone_mag.p; v.Gp = e->Gp;
    return v;
}

int abg_scan_configure(abg_engine* e, int dev, int chan, int n_freqs, const abg_channel_cfg* freqs) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_scan_configure: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (chan < 0 || chan >= d.C) return fail(ABG_ERANGE, "abg_scan_configure: channel %d out of range", chan);
    if (n_freqs < 1 || !freqs) return fail(ABG_EINVAL, "abg_scan_configure: empty frequency list");
    const int g = d.g0 + chan;
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    std::vector<FreqSet> sets((size_t)n_freqs);
    for (int i = 0; i < n_freqs; i++) {
        FreqSet& f = sets[i];
        memset(&f, 0, sizeof(f));
        char what[64];
        snprintf(what, sizeof(what), "abg_scan_configure: freqs[%d]", i);
        std::vector<float> banks[2];
        const int rc = build_freq(e->W, freqs[i], f.p, f.s, banks, what);
        if (rc != ABG_OK) return rc;
        if (f.p.modulation == ABG_MOD_NFM) e->any_nfm = true;
        for (int w = 0; w < 2; w++)
            for (size_t t = 0; t < banks[w].size(); t++) f.tone_coeff[w][t] = banks[w][t];
    }
    abg_engine::ScanChan* sc = nullptr;
    for (auto& x : e->scan)
        if (x.g == g) sc = &x;
    if (!sc) {
        e->scan.emplace_back();
        sc = &e->scan.back();
        sc->g = g;
    }
    if (sc->stash) cudaFree(sc->stash);
    sc->stash = nullptr;
    // one extra entry: scratch that receives the state being replaced below
    if (cudaMalloc((void**)&sc->stash, sizeof(FreqSet) * (size_t)(n_freqs + 1)) != cudaSuccess) return fail(ABG_ENOMEM, "Out of device memory for the scan frequency list");
    CU(cudaMemcpy(sc->stash, sets.data(), sizeof(FreqSet) * (size_t)n_freqs, cudaMemcpyHostToDevice));
    sc->n_freqs = n_freqs;
    sc->cur = 0;
    scan_swap_kernel<<<1, 128, 0, e->stream_b>>>(scan_view(e), g, sc->stash + n_freqs, sc->stash + 0);  // entry 0 goes live, fresh
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(e->stream_b));
    return ABG_OK;
}

int abg_scan_select(abg_engine* e, int dev, int chan, int freq_idx) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_scan_select: device %d out of range", dev);
    Device& d = e->dev[dev];
    if (chan < 0 || chan >= d.C) return fail(ABG_ERANGE, "abg_scan_select: channel %d out of range", chan);
    const int g = d.g0 + chan;
    abg_engine::ScanChan* sc = nullptr;
    for (auto& x : e->scan)
        if (x.g == g) sc = &x;
    if (!sc) return fail(ABG_EINVAL, "abg_scan_select: devices[%d].channels[%d] has no frequency list (abg_scan_configure)", dev, chan);
    if (freq_idx < 0 || freq_idx >= sc->n_freqs) return fail(ABG_ERANGE, "abg_scan_select: frequency index %d outside 0..%d", freq_idx, sc->n_freqs - 1);
    if (freq_idx == sc->cur) return ABG_OK;
    cudaSetDevice(e->cuda_dev);
    // stream B: after every K2 already enqueued, before the next one = between two batches (rtl_airband.cpp:498)
    scan_swap_kernel<<<1, 128, 0, e->stream_b>>>(scan_view(e), g, sc->stash + sc->cur, sc->stash + freq_idx);
    CU(cudaGetLastError());
    e->launches++;
    sc->cur = freq_idx;
    return ABG_OK;
}

// Pin (page-lock) a host buffer the caller keeps pushing from - in the reference that is input_t.buffer, the ring the
// SDR driver threads fill (input-helpers.cpp:27-36) - so that abg_push's host->device copies are real asynchronous DMA
// instead of being staged through the driver's bounce buffer.  Optional: abg_push works with pageable memory too.
int abg_host_register(void* ptr, size_t nbytes) {
    if (!ptr || nbytes == 0) return fail(ABG_EINVAL, "abg_host_register: empty range");
    cudaError_t er = cudaHostRegister(ptr, nbytes, cudaHostRegisterPortable);
    if (er == cudaErrorHostMemoryAlreadyRegistered) {
        cudaGetLastError();
        return ABG_OK;
    }
    if (er != cudaSuccess) {
        cudaGetLastError();
        return fail(ABG_ECUDA, "abg_host_register: %s", cudaGetErrorString(er));
    }
    return ABG_OK;
}

// Returns once every abg_push so far has been read out of the caller's buffers (needed before reusing page-locked
// memory that was pushed from: with abg_host_register the copies are asynchronous).  Does not wait for kernels.
int abg_ingest_sync(abg_engine* e) {
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream_c));
    return ABG_OK;
}

int abg_host_unregister(void* ptr) {
    if (!ptr) return ABG_OK;
    cudaError_t er = cudaHostUnregister(ptr);
    if (er != cudaSuccess) {
        cudaGetLastError();
        return fail(ABG_ECUDA, "abg_host_unregister: %s", cudaGetErrorString(er));
    }
    return ABG_OK;
}

int abg_resident_load(abg_engine* e, int dev, const void* iq, size_t nbytes) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_resident_load: device %d out of range", dev);
    Device& d = e->dev[dev];
    const size_t need = (size_t)(e->nbmax * e->B + ABG_AGC_EXTRA - 1) * d.hop_bytes + (size_t)e->N * d.bpc;
    if (nbytes < need) return fail(ABG_EINVAL, "abg_resident_load: need at least %zu bytes for %d batches, got %zu", need, e->nbmax, nbytes);
    cudaSetDevice(e->cuda_dev);
    if (d.res) cudaFree(d.res);
    d.res = nullptr;
    if (cudaMalloc((void**)&d.res, need + 256) != cudaSuccess) return fail(ABG_ENOMEM, "Out of device memory for the resident stream");
    d.res_bytes = need;
    CU(cudaMemsetAsync(d.res + need, 0, 256, e->stream));
    CU(cudaMemcpyAsync(d.res, iq, need, cudaMemcpyHostToDevice, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return ABG_OK;
}

int abg_run_resident(abg_engine* e, int n_batches) {
    cudaSetDevice(e->cuda_dev);
    if (n_batches < 1 || n_batches > e->nbmax) return fail(ABG_EINVAL, "abg_run_resident: n_batches must be 1..%d", e->nbmax);
    std::vector<int> nb(e->dev.size(), n_batches);
    for (auto& d : e->dev)
        if (!d.res) return fail(ABG_EINVAL, "abg_run_resident: abg_resident_load() was not called for every device");
    int n = 0;
    int rc = enqueue_run(e, nb, true, false, &n);
    return rc != ABG_OK ? rc : n;
}

int abg_set_stream(abg_engine* e, void* cuda_stream) {
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    if (e->own_stream) cudaStreamDestroy(e->stream);
    e->stream = (cudaStream_t)cuda_stream;
    e->own_stream = false;
    return ABG_OK;
}

uint64_t abg_launch_count(const abg_engine* e) { return e->launches; }

int abg_last_run_times(abg_engine* e, float* ms4) {
    if (!e->tev_valid) return fail(ABG_EINVAL, "abg_last_run_times: no run yet");
    cudaSetDevice(e->cuda_dev);
    cudaEvent_t* tl = e->tl[(e->run_index - 1) % abg_engine::TL_RUNS];
    CU(cudaEventSynchronize(tl[4]));
    CU(cudaEventElapsedTime(&ms4[0], tl[0], tl[1]));  // K1 on stream A
    CU(cudaEventElapsedTime(&ms4[1], tl[2], tl[3]));  // K2 on stream B
    CU(cudaEventElapsedTime(&ms4[2], tl[3], tl[4]));  // mixers + result export + tail copy
    CU(cudaEventElapsedTime(&ms4[3], tl[0], tl[4]));  // first K1 launch to end of run
    return ABG_OK;
}

// Timeline of the last n_runs (<= 8) runs: 5 timestamps per run (K1 start, K1 end, K2 start, K2 end, end of run) in ms
// relative to the oldest run's K1 start.  Measurement aid: shows how runs overlap inside the stream pipeline.
int abg_debug_timeline(abg_engine* e, int n_runs, float* ms) {
    if (!ms || n_runs < 1 || n_runs > abg_engine::TL_RUNS || (uint64_t)n_runs > e->run_index)
        return fail(ABG_EINVAL, "abg_debug_timeline: bad arguments");
    cudaSetDevice(e->cuda_dev);
    cudaEvent_t* last = e->tl[(e->run_index - 1) % abg_engine::TL_RUNS];
    CU(cudaEventSynchronize(last[4]));
    cudaEvent_t origin = e->tl[(e->run_index - n_runs) % abg_engine::TL_RUNS][0];
    for (int r = 0; r < n_runs; r++) {
        cudaEvent_t* tl = e->tl[(e->run_index - n_runs + r) % abg_engine::TL_RUNS];
        for (int k = 0; k < 5; k++) CU(cudaEventElapsedTime(&ms[r * 5 + k], origin, tl[k]));
    }
    return ABG_OK;
}

int abg_mixers_configure(abg_engine* e, int n_mixers, const int32_t* input_offsets, const abg_mixer_input* inputs) {
    if (n_mixers < 0 || (n_mixers > 0 && (!input_offsets || !inputs))) return fail(ABG_EINVAL, "abg_mixers_configure: bad arguments");
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    if (!e->mix_ready.empty()) return fail(ABG_EINVAL, "abg_mixers_configure: unfetched mixer batches pending");
    const int total = n_mixers ? input_offsets[n_mixers] : 0;
    std::vector<MixInput> mi(total);
    for (int i = 0; i < total; i++) {
        const abg_mixer_input& in = inputs[i];
        if (in.dev < 0 || in.dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "mixer input %d: device %d out of range", i, in.dev);
        if (in.chan < 0 || in.chan >= e->dev[in.dev].C) return fail(ABG_ERANGE, "mixer input %d: channel %d out of range", i, in.chan);
        mi[i].g = e->dev[in.dev].g0 + in.chan;
        mi[i].dev = in.dev;
        const float ampl = fminf(1.0f, 1.0f - in.balance), ampr = fminf(1.0f, 1.0f + in.balance);  // mixer.cpp:82-83
        mi[i].mult_l = in.ampfactor * ampl;  // mixer.cpp:203,206
        mi[i].mult_r = in.ampfactor * ampr;
    }
    e->mix_offsets.free(); e->mix_inputs.free(); e->mix_sums.free(); e->mix_flags.free();
    for (auto& s : e->slots) {
        if (s.release_pending) CU(cudaEventSynchronize(s.released));
        result_free(e, s.mix);
        result_free(e, s.mixflag);
    }
    e->n_mixers = n_mixers;
    e->mix_fetched.assign(n_mixers, 0);
    if (n_mixers == 0) return ABG_OK;
    const size_t nsum = (size_t)e->nbmax * n_mixers * 2 * e->B;
    if (e->mix_offsets.alloc(n_mixers + 1) || e->mix_inputs.alloc(total) || e->mix_sums.alloc(nsum) || e->mix_flags.alloc((size_t)e->nbmax * n_mixers))
        return fail(ABG_ENOMEM, "Out of device memory for mixers");
    CU(cudaMemcpy(e->mix_offsets.p, input_offsets, sizeof(int32_t) * (n_mixers + 1), cudaMemcpyHostToDevice));
    if (total) CU(cudaMemcpy(e->mix_inputs.p, mi.data(), sizeof(MixInput) * total, cudaMemcpyHostToDevice));
    CU(cudaMemset(e->mix_sums.p, 0, sizeof(float) * nsum));
    CU(cudaMemset(e->mix_flags.p, 0, sizeof(int32_t) * (size_t)e->nbmax * n_mixers));
    return alloc_slot_mixers(e);
}

int abg_fetch_mixer_batch(abg_engine* e, int mixer, float* left, float* right, int* has_signal) {
    if (mixer < 0 || mixer >= e->n_mixers) return fail(ABG_ERANGE, "abg_fetch_mixer_batch: mixer %d out of range", mixer);
    const int idx = e->mix_fetched[mixer];
    if (idx >= (int)e->mix_ready.size()) return 0;
    const std::pair<int, int> r = e->mix_ready[idx];
    Slot& s = e->slots[r.first];
    cudaSetDevice(e->cuda_dev);
    CU(cudaEventSynchronize(s.done));
    const int B = e->B;
    const float* base = s.mix + (((size_t)r.second * e->n_mixers + mixer) * 2) * B;
    const int32_t* flag = s.mixflag + (size_t)r.second * e->n_mixers + mixer;
    if (e->results_where == ABG_RESULTS_DEVICE) {
        if (left) CU(cudaMemcpy(left, base, sizeof(float) * B, cudaMemcpyDeviceToHost));
        if (right) CU(cudaMemcpy(right, base + B, sizeof(float) * B, cudaMemcpyDeviceToHost));
        if (has_signal) CU(cudaMemcpy(has_signal, flag, sizeof(int32_t), cudaMemcpyDeviceToHost));
    } else {
        if (left) memcpy(left, base, sizeof(float) * B);
        if (right) memcpy(right, base + B, sizeof(float) * B);
        if (has_signal) *has_signal = *flag;
    }
    e->mix_fetched[mixer]++;
    s.mix_pending--;
    // drop queue entries every mixer has consumed
    int mn = e->mix_fetched[0];
    for (int v : e->mix_fetched) mn = std::min(mn, v);
    while (mn > 0) {
        e->mix_ready.pop_front();
        for (int& v : e->mix_fetched) v--;
        mn--;
    }
    return 1;
}

int abg_mixer_device_buffers(abg_engine* e, float** dev_sums, int32_t** dev_flags) {
    if (e->n_mixers <= 0) return fail(ABG_EINVAL, "abg_mixer_device_buffers: no mixers configured");
    if (dev_sums) *dev_sums = e->mix_sums.p;
    if (dev_flags) *dev_flags = e->mix_flags.p;
    return ABG_OK;
}

// ---- GPU-resident I/O ---------------------------------------------------------------------------------------------------
int abg_set_result_location(abg_engine* e, int where) {
    if (where != ABG_RESULTS_HOST && where != ABG_RESULTS_DEVICE) return fail(ABG_EINVAL, "abg_set_result_location: unknown location %d", where);
    if (e->run_index > 0) return fail(ABG_EINVAL, "abg_set_result_location: only valid before the first run");
    if (where == e->results_where) return ABG_OK;
    cudaSetDevice(e->cuda_dev);
    free_slot_results(e);
    e->results_where = where;
    int rc = alloc_slot_results(e);
    if (rc == ABG_OK && e->n_mixers > 0) rc = alloc_slot_mixers(e);
    return rc;
}

int abg_fetch_batches_device(abg_engine* e, int dev, int max_batches, float* d_waveout, float* d_iq_out, char* d_axcindicate, void* cuda_stream) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_fetch_batches_device: device %d out of range", dev);
    const int rc0 = need_device_results(e, "abg_fetch_batches_device");
    if (rc0 != ABG_OK) return rc0;
    if (max_batches < 0) return fail(ABG_EINVAL, "abg_fetch_batches_device: max_batches %d < 0", max_batches);
    Device& d = e->dev[dev];
    const int n = std::min(max_batches, (int)d.ready.size());
    if (n == 0) return 0;
    cudaSetDevice(e->cuda_dev);
    std::vector<GatherCopy> cps;
    std::vector<int> used;
    for (int i = 0; i < n; i++) {
        const std::pair<int, int> r = d.ready[i];
        gather_batch(e, cps, e->slots[r.first], r.second, d.g0, d.C, (size_t)i * d.C, d_waveout, d_iq_out, d_axcindicate);
        note_slot(used, r.first);
    }
    const int rc = gather_launch(e, cps, used, (cudaStream_t)cuda_stream);
    if (rc != ABG_OK) return rc;
    for (int i = 0; i < n; i++) {
        e->slots[d.ready.front().first].pending--;
        d.ready.pop_front();
    }
    return n;
}

int abg_fetch_all_device(abg_engine* e, int n_batches, float* d_waveout, float* d_iq_out, char* d_axcindicate, void* cuda_stream) {
    const int rc0 = need_device_results(e, "abg_fetch_all_device");
    if (rc0 != ABG_OK) return rc0;
    if (n_batches < 0) return fail(ABG_EINVAL, "abg_fetch_all_device: n_batches %d < 0", n_batches);
    const size_t nd = e->dev.size();
    for (size_t k = 0; k < nd; k++)
        if ((int)e->dev[k].ready.size() < n_batches)
            return fail(ABG_EINVAL, "abg_fetch_all_device: device %zu has %zu finished batches, fewer than %d", k, e->dev[k].ready.size(), n_batches);
    if (n_batches == 0) return 0;
    cudaSetDevice(e->cuda_dev);
    std::vector<GatherCopy> cps;
    std::vector<int> used;
    for (int i = 0; i < n_batches; i++) {
        // consecutive devices whose i-th batch sits at the same place of the same slot are one block: their channels are
        // adjacent in the slot and in the output (with every device in step, one block per batch and array)
        for (size_t k = 0; k < nd;) {
            const std::pair<int, int> r = e->dev[k].ready[i];
            const int g_begin = e->dev[k].g0;
            int g_end = g_begin + e->dev[k].C;
            size_t j = k + 1;
            while (j < nd && e->dev[j].ready[i] == r) g_end += e->dev[j++].C;
            gather_batch(e, cps, e->slots[r.first], r.second, g_begin, g_end - g_begin, (size_t)i * e->G + g_begin, d_waveout, d_iq_out, d_axcindicate);
            note_slot(used, r.first);
            k = j;
        }
    }
    const int rc = gather_launch(e, cps, used, (cudaStream_t)cuda_stream);
    if (rc != ABG_OK) return rc;
    for (auto& d : e->dev)
        for (int i = 0; i < n_batches; i++) {
            e->slots[d.ready.front().first].pending--;
            d.ready.pop_front();
        }
    return n_batches;
}

int abg_fetch_mixer_batches_device(abg_engine* e, int max_batches, float* d_left_right, int32_t* d_has_signal, void* cuda_stream) {
    const int rc0 = need_device_results(e, "abg_fetch_mixer_batches_device");
    if (rc0 != ABG_OK) return rc0;
    if (e->n_mixers <= 0) return fail(ABG_EINVAL, "abg_fetch_mixer_batches_device: no mixers configured");
    if (max_batches < 0) return fail(ABG_EINVAL, "abg_fetch_mixer_batches_device: max_batches %d < 0", max_batches);
    for (int v : e->mix_fetched)
        if (v != 0) return fail(ABG_EINVAL, "abg_fetch_mixer_batches_device: mixers were popped one by one (abg_fetch_mixer_batch) and are not at the same batch");
    const int M = e->n_mixers, n = std::min(max_batches, (int)e->mix_ready.size());
    if (n == 0) return 0;
    cudaSetDevice(e->cuda_dev);
    const size_t B = (size_t)e->B, row = (size_t)M * 2 * B;
    std::vector<GatherCopy> cps;
    std::vector<int> used;
    for (int i = 0; i < n; i++) {
        const std::pair<int, int> r = e->mix_ready[i];
        const Slot& s = e->slots[r.first];
        if (d_left_right)  // [M][2] rows of WAVE_BATCH floats, contiguous on both sides
            cps.push_back({reinterpret_cast<const unsigned char*>(s.mix + (size_t)r.second * row), reinterpret_cast<unsigned char*>(d_left_right + (size_t)i * row),
                           (long long)(sizeof(float) * B), (long long)(sizeof(float) * B), 2 * M, (int32_t)(sizeof(float) * B)});
        if (d_has_signal)
            cps.push_back({reinterpret_cast<const unsigned char*>(s.mixflag + (size_t)r.second * M), reinterpret_cast<unsigned char*>(d_has_signal + (size_t)i * M),
                           (long long)(sizeof(int32_t) * M), (long long)(sizeof(int32_t) * M), 1, (int32_t)(sizeof(int32_t) * M)});
        note_slot(used, r.first);
    }
    const int rc = gather_launch(e, cps, used, (cudaStream_t)cuda_stream);
    if (rc != ABG_OK) return rc;
    for (int i = 0; i < n; i++) {
        e->slots[e->mix_ready.front().first].mix_pending -= M;
        e->mix_ready.pop_front();
    }
    return n;
}

// Host-only (no device needed): the tensor-core K1's plan and coefficient table for one device, exactly as abg_create
// builds them.  plan[13] = {eligible, K, HC, S, NC, ND, C2p, KBS, NSTB, tmem_cols, smem_bytes, halo, nacc}.  tab may be null to
// query the plan; otherwise tab_cap >= K*NC bytes and sq has C2p entries.
int abg_debug_tc_table(int fft_size, int sfmt, int hop_bytes, float fullscale, int n_channels, const int32_t* bins, int digits, int32_t* plan,
                       signed char* tab, size_t tab_cap, long long* sq, double* cscale) {
    K1TcPlan p;
    abg_k1tc_plan(fft_size, sfmt, hop_bytes, n_channels, digits, &p);
    const int32_t v[13] = {p.eligible, p.K, p.HC, p.S, p.NC, p.ND, p.C2p, p.KBS, p.NSTB, p.tmem_cols, p.smem_bytes, p.halo, p.nacc};
    if (plan) memcpy(plan, v, sizeof(v));
    if (!p.eligible) return fail(ABG_EINVAL, "abg_debug_tc_table: configuration not eligible for the tensor-core K1");
    if (!tab) return ABG_OK;
    if (tab_cap < p.table_bytes || !sq || !cscale || !bins) return fail(ABG_EINVAL, "abg_debug_tc_table: buffers too small");
    std::vector<float> wsc = make_window(fft_size);
    const float scale = sample_scale(sfmt, fullscale);
    for (auto& w : wsc) w = w * scale;
    abg_k1tc_build_table(p, fft_size, sfmt, wsc.data(), bins, n_channels, tab, sq, cscale);
    return ABG_OK;
}

// Stage tap for the upstream squelch / CTCSS behavioural tests (reference src/test_squelch.cpp, src/test_ctcss.cpp): feed
// |X[bin]| values straight into the demodulation state machine.  wavein[C][n_batches * WAVE_BATCH] becomes
// channel_t.wavein[AGC_EXTRA ...] of the device's channels (the AGC look-back keeps its initial 20.0, config.cpp:313-316, on
// the first call and the previous tail afterwards), K1 is skipped, K2 runs n_batches batches, results are fetched as usual.
// A device driven this way must not be fed with abg_push, and its channels must not need raw I/Q or AFC.
int abg_debug_inject_wavein(abg_engine* e, int dev, int n_batches, const float* wavein) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_debug_inject_wavein: device %d out of range", dev);
    if (n_batches < 1 || n_batches > e->nbmax || !wavein) return fail(ABG_EINVAL, "abg_debug_inject_wavein: n_batches must be 1..%d", e->nbmax);
    Device& d = e->dev[dev];
    for (int c = 0; c < d.C; c++)
        if (e->h_params[d.g0 + c].needs_raw_iq || e->h_params[d.g0 + c].afc) return fail(ABG_EINVAL, "abg_debug_inject_wavein: channel %d needs raw I/Q or AFC", c);
    cudaSetDevice(e->cuda_dev);
    CU(cudaStreamSynchronize(e->stream_c));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    const int B = e->B, cur = (int)(e->run_index & 1);
    const size_t rows = (size_t)n_batches * B;
    std::vector<float> tm(rows * d.C);  // time-major like win[][]
    for (int c = 0; c < d.C; c++)
        for (size_t r = 0; r < rows; r++) tm[r * d.C + c] = wavein[(size_t)c * rows + r];
    CU(cudaMemcpy2D(e->win[cur].p + (size_t)ABG_AGC_EXTRA * e->Gp + d.g0, sizeof(float) * e->Gp, tm.data(), sizeof(float) * d.C, sizeof(float) * d.C, rows,
                    cudaMemcpyHostToDevice));
    std::vector<int> nb(e->dev.size(), 0);
    nb[dev] = n_batches;
    int n = 0;
    int rc = enqueue_run(e, nb, false, true, &n, true);
    return rc != ABG_OK ? rc : n;
}

// measurement aid: clock64 stamps of the tensor-core K1's roles for the first 16 tiles of every CTA (set ABG_K1_TC_TRACE before
// abg_create); out[256][4 roles][16 tiles][4 events]
int abg_debug_k2_stats(unsigned long long* out) { return abg_k2_stats_dump(out) == 0 ? ABG_OK : fail(ABG_EINVAL, "no counters: not an ABG_K2_STATS build (make stats)"); }
int abg_debug_k1tc_trace(long long* out) { return abg_k1tc_trace_dump(out) == 0 ? ABG_OK : fail(ABG_EINVAL, "no trace: ABG_K1_TC_TRACE was not set"); }

int abg_debug_frame(abg_engine* e, int dev, const void* iq_frame, float* fftout) {
    if (dev < 0 || dev >= (int)e->dev.size()) return fail(ABG_ERANGE, "abg_debug_frame: device %d out of range", dev);
    cudaSetDevice(e->cuda_dev);
    Device& d = e->dev[dev];
    Group& g = e->groups[d.group];
    const int N = e->N;
    unsigned char* raw = nullptr;
    float2* spec = nullptr;
    K1Dev* dk = nullptr;
    const size_t bytes = (size_t)N * d.bpc;
    CU(cudaMalloc((void**)&raw, bytes + 256));
    CU(cudaMalloc((void**)&spec, sizeof(float2) * N));
    CU(cudaMalloc((void**)&dk, sizeof(K1Dev)));
    CU(cudaMemset(raw, 0, bytes + 256));
    CU(cudaMemcpy(raw, iq_frame, bytes, cudaMemcpyHostToDevice));
    K1Dev a{};
    a.raw = raw; a.start_byte = 0; a.n_frames = 1; a.pos0 = 0; a.g0 = d.g0; a.n_channels = 0; a.hop_bytes = d.hop_bytes; a.sfmt = d.sfmt;
    a.spec = spec; a.spec_first_pos = 0; a.wave_batch = e->B;
    CU(cudaMemcpy(dk, &a, sizeof(a), cudaMemcpyHostToDevice));
    K1Launch L{};
    L.fft_size = N; L.n_devices = 1; L.max_frames = 1; L.frames_per_tile = g.frames_per_tile; L.tile_bytes_cap = g.tile_bytes_cap; L.devs = dk;
    L.bins = e->bins.p; L.window_scaled = g.wsc.p; L.tw1 = e->tw1.p; L.tw2 = e->tw2.p; L.win = e->win[0].p; L.iqin = e->iqin[0].p; L.Gp = e->Gp; L.sfmt = g.sfmt;
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->stream_b));
    cudaError_t er = abg_launch_k1(L, e->stream);
    if (er != cudaSuccess) return fail(ABG_ECUDA, "K1 launch failed: %s", cudaGetErrorString(er));
    e->launches++;
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaMemcpy(fftout, spec, sizeof(float2) * N, cudaMemcpyDeviceToHost));
    cudaFree(raw); cudaFree(spec); cudaFree(dk);
    return ABG_OK;
}

}  // extern "C"
