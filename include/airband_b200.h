/*
 * airband_b200.h — C ABI of the B200 (sm_100a) multichannel demodulation engine.
 *
 * Drop-in boundary for ONE path of RTLSDR-Airband: the body of demodulate()
 * (reference src/rtl_airband.cpp:286-672) — sample conversion + Blackman-Harris window + sliding FFT + per-channel
 * bin extraction + AM / NFM demodulation with squelch, CTCSS, low-pass and notch.  Everything around it
 * (config.cpp, input-*.cpp ring producers, output.cpp / mixer.cpp consumers) stays reference code and talks to this
 * library through plain pointers and sizes.  INTEGRATION.md shows the WITH_B200 branch a maintainer adds next to
 * the existing WITH_BCM_VC branch (reference src/rtl_airband.cpp:293-314,404-412,457-481), whose C API
 * gpu_fft_prepare / gpu_fft_execute / gpu_fft_release (reference src/hello_fft/gpu_fft.h:66-74) is the precedent
 * for this one.
 *
 * Conventions: every function returns 0 on success and a negative ABG_E* code on failure (the VideoCore engine
 * uses -1/-2/-3 the same way, reference src/rtl_airband.cpp:296-310); abg_last_error() gives the text the caller
 * passes to log(LOG_CRIT, ...) before error().  All buffers are caller-owned host memory unless named dev_* or d_*.
 * No CPU fallback exists: without a CUDA device abg_create() fails with ABG_ENODEV.
 */
#ifndef AIRBAND_B200_H
#define AIRBAND_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABG_API __attribute__((visibility("default")))

/* sample_format_t, reference src/input-common.h:31 (same numeric values) */
enum { ABG_SFMT_U8 = 1, ABG_SFMT_S8 = 2, ABG_SFMT_S16 = 3, ABG_SFMT_F32 = 4 };
/* enum modulations, reference src/rtl_airband.h:193-199 */
enum { ABG_MOD_AM = 0, ABG_MOD_NFM = 1 };
/* enum fm_demod_algo, reference src/rtl_airband.cpp:88 (-Q command line switch, :728-730) */
enum { ABG_FM_FAST_ATAN2 = 0, ABG_FM_QUADRI_DEMOD = 1 };
/* enum status (channel_t.axcindicate), reference src/rtl_airband.h:101 */
enum { ABG_NO_SIGNAL = ' ', ABG_SIGNAL = '*', ABG_AFC_UP = '<', ABG_AFC_DOWN = '>' };

enum {
    ABG_OK = 0,
    ABG_ENODEV = -1,   /* no CUDA device / driver (cf. "Unable to enable V3D", rtl_airband.cpp:299) */
    ABG_EINVAL = -2,   /* unsupported configuration (cf. "log2_N=%d not supported", rtl_airband.cpp:303) */
    ABG_ENOMEM = -3,   /* device or host allocation failed (cf. "Out of memory", rtl_airband.cpp:307) */
    ABG_ECUDA = -4,    /* a CUDA call or kernel failed; abg_last_error() has cudaGetErrorString() */
    ABG_ERANGE = -5,   /* device / channel index out of range */
    ABG_EOVERFLOW = -6 /* abg_push: device-side input buffer full (cf. input_t.overflow_count, input-helpers.cpp:56-60) */
};

/* What demodulate() reads from channel_t + freq_t for one channel (reference src/rtl_airband.h:223-263), after
 * parse_channels() has resolved the config file (reference src/config.cpp:306-726). */
typedef struct abg_channel_cfg {
    int32_t bin;            /* dev->bins[i] == dev->base_bins[i], reference src/config.cpp:666-667 */
    int32_t modulation;     /* freq_t.modulation */
    int32_t needs_raw_iq;   /* channel_t.needs_raw_iq */
    int32_t has_iq_outputs; /* channel_t.has_iq_outputs */
    uint32_t dm_dphi;       /* channel_t.dm_dphi, reference src/config.cpp:679-712 */
    float alpha;            /* channel_t.alpha (NFM de-emphasis, reference src/rtl_airband.cpp:87, config.cpp:636-638) */
    float ampfactor;        /* freq_t.ampfactor */
    float squelch_level;    /* > 0: Squelch::set_squelch_level_threshold(level) (config.cpp:437-472) */
    float squelch_snr_db;   /* >= 0: Squelch::set_squelch_snr_threshold(db) afterwards (config.cpp:473-515) */
    float lowpass_hz;       /* > 0: LowpassFilter(lowpass_hz, WAVE_RATE); config passes bandwidth/2 (config.cpp:604,615) */
    float notch_hz;         /* > 0: NotchFilter(notch_hz, WAVE_RATE, notch_q) (config.cpp:541,557) */
    float notch_q;
    float ctcss_hz;         /* > 0: Squelch::set_ctcss_freq(ctcss_hz, WAVE_RATE) (config.cpp:575,584) */
    int32_t afc;            /* channel_t.afc, 0 = off */
} abg_channel_cfg;

/* What demodulate() reads from device_t + input_t (reference src/rtl_airband.h:266-286, src/input-common.h:39-57). */
typedef struct abg_device_cfg {
    int32_t sfmt;        /* input_t.sfmt */
    float fullscale;     /* input_t.fullscale (used by the S16 / F32 branches only, rtl_airband.cpp:403,421) */
    int32_t sample_rate; /* input_t.sample_rate */
    int32_t n_channels;  /* device_t.channel_count */
    const abg_channel_cfg* channels;
} abg_device_cfg;

/* Process-wide settings: globals fft_size and fm_demod (reference src/rtl_airband.cpp:83-90) and the compile-time
 * WAVE_RATE (8000, or 16000 in an -DNFM=ON build, reference src/rtl_airband.h:65-71) as a run-time value. */
typedef struct abg_config {
    int32_t fft_size;
    int32_t wave_rate;
    int32_t fm_demod;
    int32_t n_devices; /* devices[device_start .. device_end) of one demod thread (demod_params_t, rtl_airband.h:310-320) */
    const abg_device_cfg* devices;
} abg_config;

/* Squelch getters the stats file / TUI read (reference src/squelch.h:89-96, src/output.cpp:606-766) plus the
 * channel scalars tests compare. */
typedef struct abg_squelch_stats {
    float noise_level, signal_level, squelch_level;
    uint64_t open_count, flappy_count, ctcss_count, no_ctcss_count;
    float agcavgfast;        /* freq_t.agcavgfast */
    uint32_t dm_phi;         /* channel_t.dm_phi */
    int32_t bin;             /* current dev->bins[i] */
    uint64_t active_counter; /* freq_t.active_counter, reference src/rtl_airband.cpp:645-647 */
    /* the three levels as the stats file and the TUI print them: level_to_dBFS(), reference src/util.cpp:169-180
     * (output.cpp:624-700 channel_dbfs_*_level gauges, rtl_airband.cpp:632-643) */
    float noise_level_dbfs, signal_level_dbfs, squelch_level_dbfs;
} abg_squelch_stats;

/* Engine tuning (0 = default everywhere). */
typedef struct abg_options {
    int32_t cuda_device;        /* ordinal; -1 = current device */
    int32_t max_batches_per_run;/* capacity of one abg_run() per device, in WAVE_BATCH units (default 4) */
    int32_t input_capacity_batches; /* device-side raw sample buffer per device, in batches of input (default max_batches_per_run + 2) */
    int32_t fft_mode;           /* 0 auto, 1 full spectrum every frame, 2 output-pruned last pass (only the configured bins, FP32 pipes),
                                   3 the configured bins' DFT as an integer GEMM on the tensor cores (U8/S8 input whose hop is a
                                   multiple of 16 samples; other devices use 2) */
    int32_t reserved[4];
} abg_options;

typedef struct abg_engine abg_engine;

ABG_API const char* abg_last_error(void);
ABG_API const char* abg_version(void);

/* init_demod() + the engine set-up at the top of demodulate() (reference src/rtl_airband.cpp:253-266,292-351). */
ABG_API int abg_create(const abg_config* cfg, const abg_options* opt, abg_engine** out);
/* gpu_fft_release() analogue (reference src/rtl_airband.cpp:361-364). */
ABG_API void abg_destroy(abg_engine* e);

/* WAVE_BATCH (= wave_rate / 8) and the hop in complex samples for a device (rtl_airband.cpp:394). */
ABG_API int abg_wave_batch(const abg_engine* e);
ABG_API int abg_hop(const abg_engine* e, int dev);

/* Consumer side of the input ring (reference src/rtl_airband.cpp:370-375,402-455,669): hand over `nbytes` of raw
 * ring-format bytes for one device, in order.  The adapter copies [bufs, bufs + n) out of input_t.buffer and advances
 * bufs by what it pushed.  Copies host->device asynchronously on the engine's ingest stream. */
ABG_API int abg_push(abg_engine* e, int dev, const void* iq, size_t nbytes);
/* Batches a device could complete right now under the reference's fill rule
 * `available >= bps + fft_size*bytes_per_sample*2` (rtl_airband.cpp:394-400). */
ABG_API int abg_batches_available(const abg_engine* e, int dev);

/* One pass of the hot path: every device with enough buffered input advances by up to max_batches batches
 * (0 < max_batches <= options.max_batches_per_run; < 0 means the maximum).  Asynchronous; returns the number of
 * device-batches enqueued.  Finished batches are queued per device in order. */
ABG_API int abg_run(abg_engine* e, int max_batches);
/* Wait for everything enqueued so far. */
ABG_API int abg_sync(abg_engine* e);
/* Make the engine's main stream (see abg_set_stream) wait for all demodulation work enqueued so far, without blocking
 * the host: a caller-side event recorded on that stream afterwards covers K1, K2 and the result copies.  (K2 runs on
 * an internal second stream so that it overlaps the next run's K1.) */
ABG_API int abg_join(abg_engine* e);

/* Number of finished, unfetched batches of a device (the reference's dev->waveavail flag, one level deeper). */
ABG_API int abg_batches_ready(abg_engine* e, int dev);
/* What output_thread()/process_outputs() consume for the oldest finished batch of a device
 * (reference src/output.cpp:456-559,903-923): waveout[C][WAVE_BATCH] (= channel_t.waveout[0..WAVE_BATCH) before the
 * AGC_EXTRA tail copy at output.cpp:920, which the engine performs itself), iq_out[C][2*WAVE_BATCH] (may be NULL),
 * axcindicate[C].  Returns 1 if a batch was popped, 0 if none is ready, < 0 on error.  Synchronises as needed. */
ABG_API int abg_fetch_batch(abg_engine* e, int dev, float* waveout, float* iq_out, char* axcindicate);
/* Same for up to max_batches finished batches of one device in one call: waveout[n][C][WAVE_BATCH], iq_out[n][C][2*WAVE_BATCH]
 * (may be NULL), axcindicate[n][C].  Returns the number of batches popped. */
ABG_API int abg_fetch_batches(abg_engine* e, int dev, int max_batches, float* waveout, float* iq_out, char* axcindicate);

ABG_API int abg_get_stats(abg_engine* e, int dev, int chan, abg_squelch_stats* out);
/* Retune a channel's bin between batches: scan mode (controller_thread, reference src/rtl_airband.cpp:101-139) or an
 * external AFC.  Sets both bins[] and base_bins[]. */
ABG_API int abg_set_bin(abg_engine* e, int dev, int chan, int bin);

/* Which K1 implementation a device's frames go through: 1 full-spectrum FFT, 2 output-pruned FFT, 3 tensor-core DFT. */
ABG_API int abg_fft_path(const abg_engine* e, int dev);

/* ---- benchmark / multi-GPU helpers (not part of the reference surface) -------------------------------------- */
/* Upload a raw stream that stays resident in HBM and is replayed by abg_run_resident(): the timed region of the
 * throughput benchmark then starts with inputs already on the device. `nbytes` must cover max_batches_per_run batches. */
ABG_API int abg_resident_load(abg_engine* e, int dev, const void* iq, size_t nbytes);
/* Process n_batches batches of every device from its resident stream (channel state carries over between calls). */
ABG_API int abg_run_resident(abg_engine* e, int n_batches);
/* Use an existing CUDA stream (cudaStream_t as void*) as the engine's main stream, e.g. torch's current stream, so
 * that caller-side CUDA events bracket the engine's work. */
ABG_API int abg_set_stream(abg_engine* e, void* cuda_stream);
/* Kernel launches issued by this engine since creation (bench.py reports it as gpu_launches). */
ABG_API uint64_t abg_launch_count(const abg_engine* e);

/* Device time of the most recent run, from CUDA events recorded on the engine's stream around its kernels:
 * ms4[0] = K1 (convert+window+FFT+bins, all groups), ms4[1] = K2 (demodulation), ms4[2] = mixers + result copies + tail
 * copy, ms4[3] = whole run.  Waits for that run to finish. */
/* Optional: page-lock a host buffer that abg_push will be fed from (in the reference: input_t.buffer, the ring filled by
   the SDR threads, src/input-helpers.cpp:27-36; buf_size + 2*bytes_per_sample*fft_size bytes) so the host->device copies
   are asynchronous DMA.  Unregister before freeing the buffer. */
ABG_API int abg_host_register(void* ptr, size_t nbytes);
ABG_API int abg_host_unregister(void* ptr);
/* Returns once every abg_push so far has been read out of the caller's memory (with page-locked memory the copies are
   asynchronous): call it before letting a producer overwrite ring space that was pushed from.  Does not wait for kernels. */
ABG_API int abg_ingest_sync(abg_engine* e);

/* Scan mode.  Reference: an R_SCAN device has one channel with freqlist[freq_count] (src/rtl_airband.h:250-252); every
   freq_t owns its Squelch, NotchFilter, LowpassFilter, agcavgfast, ampfactor, modulation and active_counter
   (src/rtl_airband.h:223-233).  controller_thread switches channels[0].freq_idx and retunes the input
   (src/rtl_airband.cpp:101-139); demodulate() picks fparms = freqlist + freq_idx at the start of every batch (:498).
   abg_scan_configure installs the list for a channel: freqs[i] supplies the freq_t part of entry i (modulation,
   ampfactor, squelch_*, lowpass_hz, notch_*, ctcss_hz; the channel_t part - bin, dm_dphi, alpha, afc, needs_raw_iq,
   has_iq_outputs - stays what abg_create was given).  Every entry starts from a fresh freq_t; entry 0 becomes current.
   abg_scan_select makes entry freq_idx current for all batches demodulated by later abg_run calls; the state of the
   entry it replaces is kept on the device and resumes when that entry is selected again. */
ABG_API int abg_scan_configure(abg_engine* e, int dev, int chan, int n_freqs, const abg_channel_cfg* freqs);
ABG_API int abg_scan_select(abg_engine* e, int dev, int chan, int freq_idx);

ABG_API int abg_last_run_times(abg_engine* e, float* ms4);
/* Measurement aid: 5 timestamps (K1 start, K1 end, K2 start, K2 end, end of run; ms since the oldest run's K1 start) for
   each of the last n_runs (1..8) runs into ms[5*n_runs]; shows how consecutive runs overlap on the device. */
ABG_API int abg_debug_timeline(abg_engine* e, int n_runs, float* ms);

/* Mixer path (reference src/mixer.cpp:82-83,114-140,189-214): mixer m's output for a batch is, per sample,
 * sum over its inputs (in input order) of waveout * (ampfactor * ampl) [left] and * (ampfactor * ampr) [right], taken
 * over the inputs whose channel had axcindicate != NO_SIGNAL in that batch (mixer_put_samples' has_signal), where
 * ampl = fminf(1, 1 - balance), ampr = fminf(1, 1 + balance).  The reference paces this with wall-clock intervals
 * (mixer.cpp:142-156); here it is deterministic: batch b of a run mixes every input whose device produced batch b in
 * that run.  The sums are computed on the device right after demodulation. */
typedef struct abg_mixer_input {
    int32_t dev, chan;
    float ampfactor; /* mixinput_t.ampfactor */
    float balance;   /* -1..1 (mixer.cpp:82-83) */
} abg_mixer_input;
/* Define all mixers at once: mixer m owns inputs[input_offsets[m] .. input_offsets[m+1]). */
ABG_API int abg_mixers_configure(abg_engine* e, int n_mixers, const int32_t* input_offsets, const abg_mixer_input* inputs);
/* Pop the oldest finished batch of one mixer: left[WAVE_BATCH], right[WAVE_BATCH] (may be NULL), has_signal
 * (channel->axcindicate of the mixer channel: 1 = SIGNAL).  Returns 1 if popped, 0 if none. */
ABG_API int abg_fetch_mixer_batch(abg_engine* e, int mixer, float* left, float* right, int* has_signal);
/* Device pointers to the partial sums of the LATEST run, for a cross-GPU reduction when a mixer's inputs are sharded
 * over several engines: sums float[max_batches_per_run][n_mixers][2][WAVE_BATCH], flags int32[max_batches_per_run][n_mixers]. */
ABG_API int abg_mixer_device_buffers(abg_engine* e, float** dev_sums, int32_t** dev_flags);

/* ---- GPU-resident I/O (not part of the reference surface) ---------------------------------------------------------
 * For callers whose IQ is already in GPU memory (GPUDirect capture, a GPU-side DDC) and whose consumers run on the GPU.
 * Every call here is ordered on the caller's CUDA stream (cudaStream_t passed as void*, NULL = the legacy default
 * stream) and none of them blocks the host.  All d_* pointers are device memory on the engine's GPU. */
enum { ABG_RESULTS_HOST = 0, ABG_RESULTS_DEVICE = 1 };
/* abg_push with a device-memory source: same ring-format bytes, whole complex samples, ABG_EOVERFLOW rule and buffer
 * compaction.  The engine's ingest stream first waits for the work enqueued so far on cuda_stream, then copies device to
 * device.  Host pointers and memory on another GPU are rejected with ABG_EINVAL.  abg_push and abg_push_device may be
 * mixed on one device; the bytes follow each other in call order.  The source must stay unmodified until
 * abg_ingest_join (or abg_ingest_sync) has covered the push. */
ABG_API int abg_push_device(abg_engine* e, int dev, const void* d_iq, size_t nbytes, void* cuda_stream);
/* Make cuda_stream wait until every push so far has been read out of the caller's memory: the non-blocking
 * counterpart of abg_ingest_sync.  Work the caller enqueues on cuda_stream afterwards may overwrite pushed sources. */
ABG_API int abg_ingest_join(abg_engine* e, void* cuda_stream);
/* Where the result slots live: ABG_RESULTS_HOST (default, page-locked host memory) or ABG_RESULTS_DEVICE (HBM).  Only
 * before the first run (ABG_EINVAL afterwards).  abg_fetch_batch(es) and abg_fetch_mixer_batch keep working in device
 * mode (they copy out of the device slot); the *_device fetches below need it. */
ABG_API int abg_set_result_location(abg_engine* e, int where);
/* Pop up to max_batches finished batches of one device (count taken from the engine's bookkeeping, no wait for the GPU)
 * and write them on cuda_stream in abg_fetch_batches' layouts: d_waveout[n][C][WAVE_BATCH], d_iq_out[n][C][2*WAVE_BATCH]
 * (may be NULL; zero-filled when no channel has I/Q outputs), d_axcindicate[n][C] (may be NULL).  Returns n. */
ABG_API int abg_fetch_batches_device(abg_engine* e, int dev, int max_batches, float* d_waveout, float* d_iq_out, char* d_axcindicate,
                                     void* cuda_stream);
/* Pop n_batches batches of EVERY device in one launch, in engine-global channel order: d_waveout[n][G][WAVE_BATCH],
 * d_iq_out[n][G][2*WAVE_BATCH], d_axcindicate[n][G] (G = all channels of the engine).  ABG_EINVAL, popping nothing, if
 * some device has fewer than n_batches finished batches. */
ABG_API int abg_fetch_all_device(abg_engine* e, int n_batches, float* d_waveout, float* d_iq_out, char* d_axcindicate, void* cuda_stream);
/* Pop up to max_batches finished batches of ALL mixers at once: d_left_right[n][n_mixers][2][WAVE_BATCH],
 * d_has_signal[n][n_mixers] (may be NULL).  ABG_EINVAL if a mixer was popped on its own (abg_fetch_mixer_batch) and the
 * mixers are not at the same batch.  Returns n. */
ABG_API int abg_fetch_mixer_batches_device(abg_engine* e, int max_batches, float* d_left_right, int32_t* d_has_signal, void* cuda_stream);

/* ---- stage taps for tests ---------------------------------------------------------------------------------- */
/* Run conversion + window + FFT on one frame of `dev`'s format and return the full spectrum in natural bin order
 * (fftout[2*fft_size]); exercises the same kernel code as abg_run. */
ABG_API int abg_debug_frame(abg_engine* e, int dev, const void* iq_frame, float* fftout);
/* Feed |X[bin]| values straight into the demodulation state machine of one device (K1 skipped): wavein[C][n_batches *
 * WAVE_BATCH] becomes channel_t.wavein[AGC_EXTRA ...]; results are fetched as usual.  For the ports of the reference's own
 * Squelch / CTCSS unit tests (reference src/test_squelch.cpp:51-281, src/test_ctcss.cpp:122-155).  The device must not be
 * fed with abg_push and its channels must not need raw I/Q or AFC.  Returns the number of batches enqueued. */
ABG_API int abg_debug_inject_wavein(abg_engine* e, int dev, int n_batches, const float* wavein);
/* Measurement aid: per-role clock64 stamps of the tensor-core K1 (environment variable ABG_K1_TC_TRACE set at launch time);
 * out[256 CTAs][4 roles: producer, epilogue, loader, MMA][16 tiles][4 events]. */
ABG_API int abg_debug_k1tc_trace(long long* out);
/* Measurement aid: 64 event counters of the K2 tile paths (copied and cleared); only the `make stats` build counts. */
ABG_API int abg_debug_k2_stats(unsigned long long* out);
/* Host-only: plan and coefficient table of the tensor-core K1 (fft_mode 3) for one device, as abg_create builds them
 * (window * twiddle quantised to `digits` signed 8-bit digits, in the shared-memory image the MMA reads).
 * plan[13] = {eligible, K, HC, S, NC, ND, C2p, KBS, NSTB, tmem_cols, smem_bytes, halo, nacc}; tab == NULL queries the plan only. */
ABG_API int abg_debug_tc_table(int fft_size, int sfmt, int hop_bytes, float fullscale, int n_channels, const int32_t* bins, int digits,
                               int32_t* plan, signed char* tab, size_t tab_cap, long long* sq, double* cscale);

#ifdef __cplusplus
}
#endif
#endif /* AIRBAND_B200_H */
