// Host-side mirror of the reference structures the demodulation path touches, and the replacement thread function.
//
// The reference's own rtl_airband.h cannot be included here (it pulls lame/shout/libconfig++/fftw3 headers that are
// not installed), so this header restates ONLY the fields demodulate() reads or writes, with the reference's names:
//   input_t           reference src/input-common.h:39-57   (ring: buffer, buf_size, bufs, bufe, buffer_lock, state, sfmt ...)
//   freq_t            reference src/rtl_airband.h:223-233  (the Squelch / filter objects appear as their config values)
//   channel_t         reference src/rtl_airband.h:234-263
//   device_t          reference src/rtl_airband.h:266-286
//   demod_params_t    reference src/rtl_airband.h:310-320  (no FFTW plan: the engine owns the transform)
//   Signal            reference src/rtl_airband.h:201-221
// In the reference tree the WITH_B200 branch uses the real structs (INTEGRATION.md); this mirror exists so that the
// adapter logic is compiled and tested in this repository.
#pragma once
#include <pthread.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/airband_b200.h"
#include "../../include/airband_b200_host.h"

#define AGC_EXTRA 100  // reference src/rtl_airband.h:74

typedef enum { SFMT_UNDEF = 0, SFMT_U8, SFMT_S8, SFMT_S16, SFMT_F32 } sample_format_t;  // input-common.h:31
typedef enum { INPUT_UNKNOWN = 0, INPUT_INITIALIZED, INPUT_RUNNING, INPUT_FAILED, INPUT_STOPPED, INPUT_DISABLED } input_state_t;
enum status { NO_SIGNAL = ' ', SIGNAL = '*', AFC_UP = '<', AFC_DOWN = '>' };  // rtl_airband.h:101
enum modulations { MOD_AM, MOD_NFM };                                          // rtl_airband.h:193-199

typedef struct input_t input_t;
struct input_t {
    unsigned char* buffer;  // buf_size + 2 * bytes_per_sample * fft_size bytes (wrap tail, input-helpers.cpp:27-36)
    void* dev_data;         // plugin-private (input-common.h:41)
    size_t buf_size, bufs, bufe;
    size_t overflow_count;
    input_state_t state;
    sample_format_t sfmt;
    float fullscale;
    int bytes_per_sample;
    int sample_rate;
    int centerfreq;
    // plugin entry points (input-common.h:50-54; parse_config is libconfig++-typed and not mirrored)
    int (*init)(input_t* const input);
    void* (*run_rx_thread)(void* input_ptr);  // to be launched via pthread_create()
    int (*set_centerfreq)(input_t* const input, int const centerfreq);
    int (*stop)(input_t* const input);
    pthread_t rx_thread;
    pthread_mutex_t buffer_lock;
};

// "pattern" input plugin (host/input_pattern.cpp): replays a block of ring-format bytes, paced like a live SDR or
// lossless like input-file.cpp.  Found by input_new("pattern") in the reference tree (input-common.cpp:35-54 looks up
// <type>_input_new with dlsym).
struct pattern_dev_data_t {
    const unsigned char* block;  // whole complex samples
    size_t block_len;
    long repeat;                 // the block is sent this many times, then the input reports INPUT_FAILED (end of stream)
    double speedup;              // > 0: paced by the wall clock at speedup x sample_rate, never waits (a full ring
                                 // overflows, input-helpers.cpp:56-60); 0: as fast as the ring drains, lossless
    size_t written;              // end of the stream bytes appended so far, stored before each append: stream byte s sits in
                                 // ring slot s % buf_size, so a reader of byte s knows it intact while written <= s + buf_size
};
extern "C" ABG_API input_t* pattern_input_new(void);

class Signal {  // rtl_airband.h:201-221
   public:
    Signal() {
        pthread_cond_init(&cond_, NULL);
        pthread_mutex_init(&mutex_, NULL);
    }
    void send() {
        pthread_mutex_lock(&mutex_);
        pthread_cond_signal(&cond_);
        pthread_mutex_unlock(&mutex_);
    }
    void wait_ms(int ms);  // the reference waits without timeout; tests must not hang on a lost wake-up

   private:
    pthread_cond_t cond_;
    pthread_mutex_t mutex_;
};

// b200_freq_cfg / b200_freq_stats: what the WITH_B200 patch adds to the reference's freq_t (include/airband_b200_host.h)
struct freq_t {
    int frequency;
    float agcavgfast;  // mirrored back from the engine for the stats file
    float ampfactor;
    size_t active_counter;
    enum modulations modulation;
    b200_freq_cfg b200_cfg;
    b200_freq_stats b200_stats;
};

enum ch_states { CH_DIRTY, CH_WORKING, CH_READY };  // rtl_airband.h:102
enum mix_modes { MM_MONO, MM_STEREO };               // rtl_airband.h:103
enum output_type { O_ICECAST, O_FILE, O_RAWFILE, O_MIXER, O_UDP_STREAM };  // rtl_airband.h:104-115
struct output_t {  // rtl_airband.h:180-185
    enum output_type type;
    bool enabled;
    bool active;
    void* data;
};
struct mixer_data {  // rtl_airband.h:175-178
    struct mixer_t* mixer;
    int input;
};

struct channel_t {
    float* waveout;    // [WAVE_LEN]; the consumer reads [0, WAVE_BATCH)
    float* waveout_r;  // [WAVE_LEN] right channel of a stereo mixer (mixer channels only)
    float* iq_out;     // [2 * WAVE_LEN]
    float alpha;
    uint32_t dm_dphi;
    enum mix_modes mode;
    enum status axcindicate;
    unsigned char afc;
    freq_t* freqlist;
    int freq_count, freq_idx;
    int needs_raw_iq, has_iq_outputs;
    enum ch_states state;  // mixer channel state flag (mixer.cpp:157-261 <-> output.cpp:888-896)
    int output_count;
    output_t* outputs;
};

struct device_t {
    input_t* input;
    int channel_count;
    size_t *base_bins, *bins;
    channel_t* channels;
    int waveavail;
    size_t output_overrun_count;
};

struct mixinput_t {  // rtl_airband.h:288-296 (the fields the hand-off reads)
    float ampfactor;
    float ampl, ampr;
};
struct mixer_t {  // rtl_airband.h:298-308
    const char* name;
    bool enabled;
    int interval;
    size_t output_overrun_count;
    int input_count;
    mixinput_t* inputs;
    bool* input_mask;
    channel_t channel;
};

struct demod_params_t {
    Signal* mp3_signal;
    int device_start;
    int device_end;
};

// process-wide state the reference keeps in globals (rtl_airband.cpp:71-90)
struct b200_globals {
    device_t* devices;
    int device_count;
    mixer_t* mixers;          // rtl_airband.cpp:72
    int mixer_count;
    void (*on_device_failed)(device_t* dev);  // stands in for disable_device_outputs(dev), rtl_airband.cpp:386
    size_t fft_size;
    int wave_rate;            // WAVE_RATE as a run-time value
    int fm_demod;
    volatile int do_exit;
    volatile int devices_running;
    volatile int engine_ready;  // set by demodulate_b200() once its engine exists (load-test sources start their clock then)
    int wait_for_consumer;    // offline use (file input faster than real time): deliver a batch only once waveavail == 0
    int max_batches_per_run;
    char last_error[512];
};
extern b200_globals g_b200;

// Drop-in for `void* demodulate(void* params)` (reference src/rtl_airband.cpp:286, started at :1111).
extern "C" ABG_API void* demodulate_b200(void* params);

// circbuffer_append (reference src/input-helpers.cpp:37-63): producer-side reference code, restated for the TEST feeders only
// (host_harness.cpp); in the reference tree the real one is used and nothing here duplicates its symbol.
void circbuffer_append(input_t* const input, unsigned char* buf, size_t len);

// b200_refresh_stats / b200_deliver_mixers / b200_write_rawfile: see b200_adapter.h
