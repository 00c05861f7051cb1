// Internal layouts shared by the host engine and the two sm_100a kernels.
//
// Data layout in HBM (per engine = one GPU's share of devices[]):
//   raw[d]            ring-format bytes of device d, linear, frames overlap in place (never expanded to float in HBM)
//   win[P][Gp]        |X[bin]| per (frame position, channel)  — channel_t.wavein, time-major so that the K2 warp
//   iqin[P][Gp]       X[bin]                                     (32 channels) reads one 128/256-byte line per sample
//   wout[Gp][P]       channel_t.waveout, channel-major (what the output thread consumes, contiguous per channel)
//   iqout[Gp][nb*B]   channel_t.iq_out
//   state[Gp]         per-channel scalars (Squelch, filters, AGC, NFM) — ChanState
//   sqbuf[102][Gp]    Squelch::buffer_ delay line
//   tone_*[2][NT][Gp] Goertzel banks of the fast / slow CTCSS detectors
// P = AGC_EXTRA + max_batches_per_run * WAVE_BATCH positions; position j of a run is exactly index j of the
// reference's wavein[]/waveout[] arrays when max_batches_per_run == 1.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

// Kernel function attributes (dynamic shared-memory opt-in, carveout) are per CUDA device: several engines may live on
// different GPUs of one process and several demod threads may launch concurrently.  One slot per device ordinal keeps the
// largest size configured so far for a kernel instantiation; `apply` runs (under the lock) only when it has to grow.
struct AbgPerDeviceSize {
    std::mutex m;
    size_t v[64] = {};
    template <class F>
    cudaError_t ensure(size_t want, F&& apply) {
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 63;
        std::lock_guard<std::mutex> lock(m);
        if (want > v[dev]) {
            cudaError_t e = apply();
            if (e != cudaSuccess) return e;
            v[dev] = want;
        }
        return cudaSuccess;
    }
};

#define ABG_AGC_EXTRA 100     // reference src/rtl_airband.h:74
#define ABG_SQ_BUF 102        // Squelch::buffer_size_, reference src/squelch.cpp:67
#define ABG_MAX_TONES 52      // wanted tone + 51 standard tones, reference src/ctcss.cpp:89-111

// Squelch::State, reference src/squelch.h:104-110
enum { SQ_CLOSED = 0, SQ_OPENING = 1, SQ_CLOSING = 2, SQ_LOW_SIGNAL_ABORT = 3, SQ_OPEN = 4 };

// Per-channel constants, resolved on the host at abg_create() (reference config.cpp / filters.cpp / squelch.cpp ctor maths).
struct ChanParams {
    int32_t dev;            // owning device index (engine-local)
    int32_t modulation;     // ABG_MOD_*
    int32_t needs_raw_iq, has_iq_outputs;
    uint32_t dm_dphi;
    float alpha, ampfactor;
    int32_t afc;
    // NotchFilter (filters.cpp:30-47)
    int32_t notch_on;
    float nd0, nd1, nd2;
    // LowpassFilter (filters.cpp:67-96)
    int32_t lp_on;
    float lp_gain, lp_yc0, lp_yc1;
    // CTCSS (ctcss.cpp:92-111, squelch.cpp:110-116)
    int32_t ctcss_on;
    int32_t n_tones[2];     // detectors in the fast / slow bank (bank entry 0 is the wanted tone)
    int32_t window[2];      // window sizes: wave_rate*0.05, wave_rate*0.4
};

// Per-channel mutable state: Squelch (squelch.h:117-158), filters' delay elements, freq_t / channel_t scalars.
struct ChanState {
    // --- Squelch ---
    float noise_floor;
    int32_t manual;
    float manual_level, normal_ratio, flappy_ratio, avg_cap;
    float pre_full, pre_capped, post_full, post_capped;
    float level_cache;
    int32_t using_post;
    int32_t next_state, cur_state, delay;
    uint32_t sample_count_mod16;     // only sample_count_ % 16 is ever observed (squelch.cpp:213)
    int32_t low_signal_count;
    uint32_t recent_open_count, closed_sample_count;
    int32_t head;                    // buffer_head_; buffer_tail_ == (head + 1) % 102 always (squelch.cpp:69,457-458)
    unsigned long long open_count, flappy_count;
    // --- CTCSS fast [0] / slow [1] (ctcss.h:78-95) ---
    int32_t ct_enough[2], ct_count[2], ct_has_tone[2];
    unsigned long long ct_found[2], ct_not_found[2];
    // --- NotchFilter x[1],x[2],y[1],y[2] (filters.cpp:49-64) ---
    float nx1, nx2, ny1, ny2;
    // --- LowpassFilter xv[1],xv[2],yv[1],yv[2] (filters.cpp:146-163) ---
    float lx1r, lx1i, lx2r, lx2i, ly1r, ly1i, ly2r, ly2i;
    // --- freq_t / channel_t ---
    float agcavgfast;
    uint32_t dm_phi;
    float pr, pj, prev_waveout;
    unsigned long long active_counter;
    int32_t axc_prev;                // axcindicate of the previous batch (AFC edge detect, rtl_airband.cpp:222)
};

// Per-device, per-launch arguments of K1 (uploaded before every run).
struct K1Dev {
    const unsigned char* raw;  // base of the device's raw byte buffer (16-byte aligned)
    unsigned long long start_byte;  // byte offset of this launch's first frame
    int32_t n_frames;          // frames this launch computes for the device
    int32_t pos0;              // position (row of win/iqin) of the first frame
    int32_t g0, n_channels;    // channel index range [g0, g0 + n_channels)
    int32_t hop_bytes;         // bytes between consecutive frames (bps in the reference, rtl_airband.cpp:394)
    int32_t sfmt;
    float2* spec;              // when non-null: full spectrum of the last frame of every batch goes here (AFC)
    int32_t spec_first_pos;    // position of the first batch-final frame; then every WAVE_BATCH positions
    int32_t wave_batch;
};

// Per-device, per-launch arguments of K2.
struct K2Dev {
    int32_t n_batches;         // batches this launch demodulates for the device (0 = skip)
    int32_t fft_size;
    const float2* spec;        // spectra of batch-final frames [n_batches][fft_size] (AFC) or null
};

// ---- kernel launchers (defined in k1_fft.cu / k2_demod.cu) -------------------------------------------------------
struct K1Launch {
    int fft_size;
    int n_devices;             // grid.y
    int max_frames;            // max n_frames over devices
    int frames_per_tile;
    int tile_bytes_cap;        // dynamic smem reserved for the raw tile
    const K1Dev* devs;         // device memory
    const int32_t* bins;       // [Gp] current bin per channel
    const float* window_scaled;// [N] window * (1/fullscale-type factor) per sample format -> see engine
    const float2* tw1;         // inter-pass twiddles, layout [k1][n2]
    const float2* tw2;         // second inter-pass table for 3-pass sizes (N = 8192) or null
    float* win;                // [P][Gp]
    float2* iqin;              // [P][Gp]
    int Gp;
    int sfmt;                  // all devices of one launch share a format (the engine groups launches by format)
};
cudaError_t abg_launch_k1(const K1Launch& L, cudaStream_t s);
int abg_k1_tile_frames(int fft_size, int sfmt, int hop_bytes, int* tile_bytes_cap);
// output-pruned variant (k1_pruned.cu): only the configured bins are evaluated in the last pass
cudaError_t abg_launch_k1_pruned(const K1Launch& L, const float2* twn, int max_channels, cudaStream_t s);
int abg_k1p_tile_frames(int fft_size, int sfmt, int hop_bytes, int max_channels, int* tile_bytes_cap);

// tensor-core variant (k1_tc.cu): the bins' DFT as an integer GEMM on tcgen05 (8-bit formats, hop_bytes % 32 == 0)
struct K1TcPlan {
    int eligible;
    int K, HC, S, NC, ND, C2p, KBS, NSTB, tmem_cols, smem_bytes, halo, nacc;
    size_t table_bytes;
};
struct K1TcTables {
    const int32_t* tab_of_dev;  // [n_devices of the group] coefficient table of each device
    const signed char* btab;    // [n_tables][K * NC]
    const long long* sq;        // [n_tables][C2p]
    int* counter;               // tile queue head, zero at launch
    int32_t* status;            // != 0 after a pipeline stall inside the kernel (bounded waits, never hangs)
    double cscale;
};
int abg_k1tc_plan(int fft_size, int sfmt, int hop_bytes, int max_channels, int digits, K1TcPlan* p);
void abg_k1tc_build_table(const K1TcPlan& p, int fft_size, int sfmt, const float* wsc, const int32_t* bins, int n_channels, signed char* tab,
                          long long* sq, double* cscale);
cudaError_t abg_launch_k1_tc(const K1Launch& L, const K1TcPlan& p, const K1TcTables& T, int sm_count, cudaStream_t s);
int abg_k1tc_trace_dump(long long* out);  // measurement aid (ABG_K1_TC_TRACE): 256*4*16*4 clock64 stamps

struct K2Launch {
    int G, Gp, P, wave_batch, fm_demod, iq_stride;  // iq_stride = nbmax * B
    int lanes_per_warp;       // channels handled by one warp of K2: 1, 2, 4, 8, 16 or 32
    int nfm_blocks;           // some channel (or scan-list entry) is NFM: run the kernel build with the NFM steady-state blocks
    const ChanParams* params;
    ChanState* state;
    const K2Dev* devs;
    int32_t* bins;
    const int32_t* base_bins;
    float* win;               // [P][Gp] buffer K1 filled for THIS run
    float2* iqin;
    float* win_next;          // buffer the next run's K1 fills: receives the AGC_EXTRA look-back rows
    float2* iqin_next;
    float* wout;
    float2* iqout;            // may be null when no channel has I/Q outputs
    float* sqbuf;             // [102][Gp]
    const float* tone_coeff;  // [2][NT][Gp]
    float* tone_q1;           // [2][NT][Gp]
    float* tone_q2;
    float* tone_mag;
    unsigned char* axc;       // [nbmax][Gp]
    const float* sincos_lut;  // [2][257] sin then cos (util.cpp:103-111)
};
cudaError_t abg_launch_k2(const K2Launch& L, cudaStream_t s);
int abg_k2_stats_dump(unsigned long long* out);  // event counters of the ABG_K2_STATS build (k2_demod.cu)

// mixer sums (reference src/mixer.cpp:133-140,189-214), defined in k2_demod.cu (compiled without FMA contraction)
struct MixInput {
    int32_t g;          // global channel index of the input
    int32_t dev;
    float mult_l, mult_r;  // ampfactor * ampl, ampfactor * ampr
};
struct MixLaunch {
    int n_mixers, n_batches, wave_batch, P, Gp;
    const int32_t* offsets;   // [n_mixers + 1]
    const MixInput* inputs;
    const K2Dev* devs;
    const float* wout;        // [Gp][P]
    const unsigned char* axc; // [nbmax][Gp]
    float* sums;              // [nbmax][n_mixers][2][B]
    int32_t* flags;           // [nbmax][n_mixers]
    float* host_sums;         // same layout in the pinned result slot, or null
    int32_t* host_flags;
};
cudaError_t abg_launch_mix(const MixLaunch& L, cudaStream_t s);
// host-visible (pinned, mapped) result slot the end-of-run kernel writes; all null = no export (resident benchmark runs)
struct K2Export {
    float* host_wout;          // [G][stride]
    float2* host_iqout;        // [G][stride] or null
    unsigned char* host_axc;   // [nbmax][Gp]
    size_t stride;             // nbmax * WAVE_BATCH
};
cudaError_t abg_launch_k2_tail(const K2Launch& L, const K2Export& X, cudaStream_t s);

// device-resident result fetches (export_device.cu): one launch copies a list of rectangular blocks out of the
// channel-major result slots in HBM into the caller's batch-major buffers.  Block k copies rows x row_bytes from
// src (row pitch src_pitch) to dst (row pitch dst_pitch); src == null writes zeros.
struct GatherCopy {
    const unsigned char* src;
    unsigned char* dst;
    long long src_pitch, dst_pitch;
    int32_t rows, row_bytes;
};
#define ABG_GATHER_MAX 96  // blocks per launch: the list is passed by value and stays below the 4 KB parameter limit
struct GatherList {
    int32_t n, max_rows;
    GatherCopy c[ABG_GATHER_MAX];
};
cudaError_t abg_launch_gather(const GatherList& L, cudaStream_t s);
