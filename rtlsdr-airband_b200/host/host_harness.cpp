// Test harness around demodulate_b200(): builds devices[] / channels / input rings the way parse_devices() does
// (reference src/config.cpp:793-815), runs one feeder thread per device that behaves like file_rx_thread()
// (reference src/input-file.cpp:82-147: reads buf_size/2 - 1 bytes at a time, waits for ring space, flags
// INPUT_FAILED at end of data), the demod thread under test, and a consumer that does what output_thread() does with a
// finished batch (reference src/output.cpp:903-923: read waveout[0..WAVE_BATCH), clear waveavail).  Exposed through a
// small C ABI so pytest can drive it.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "b200_adapter.h"

#define MIN_BUF_SIZE 2560000  // reference src/rtl_airband.h:61

// reference src/input-helpers.cpp:37-63, restated for the test feeders (the producer side is reference code; in the
// reference tree its own definition is the one that links)
void circbuffer_append(input_t* const input, unsigned char* buf, size_t len) {
    if (len == 0) return;
    pthread_mutex_lock(&input->buffer_lock);
    const size_t tail = 2 * input->bytes_per_sample * g_b200.fft_size;
    size_t space_left = input->buf_size - input->bufe;
    if (space_left >= len) {
        memcpy(input->buffer + input->bufe, buf, len);
        if (input->bufe == 0) memcpy(input->buffer + input->buf_size, input->buffer, std::min(len, tail));
    } else {
        memcpy(input->buffer + input->bufe, buf, space_left);
        memcpy(input->buffer, buf + space_left, len - space_left);
        memcpy(input->buffer + input->buf_size, input->buffer, std::min(len - space_left, tail));
    }
    size_t old_end = input->bufe;
    input->bufe = (input->bufe + len) % input->buf_size;
    if (old_end < input->bufs && input->bufe >= input->bufs) input->overflow_count++;
    pthread_mutex_unlock(&input->buffer_lock);
}

namespace {
struct Feeder {
    input_t* input;
    const unsigned char* data;
    size_t len;
};
void* feeder_thread(void* p) {
    Feeder* f = (Feeder*)p;
    input_t* input = f->input;
    const size_t buf_len = (input->buf_size / 2) - 1;
    size_t pos = 0;
    input->state = INPUT_RUNNING;
    while (!g_b200.do_exit) {
        if (pos >= f->len) {  // feof(): "hit end of file, disabling"
            // let the demod thread drain the ring first (the reference drops what is left; see DESIGN.md §7)
            input->state = INPUT_FAILED;
            break;
        }
        size_t space_left;
        pthread_mutex_lock(&input->buffer_lock);
        if (input->bufe >= input->bufs)
            space_left = input->bufs + (input->buf_size - input->bufe);
        else
            space_left = input->bufs - input->bufe;
        pthread_mutex_unlock(&input->buffer_lock);
        if (space_left > buf_len) {
            size_t n = std::min(buf_len, f->len - pos);
            // keep whole complex samples per append so the consumer never sees half a sample at the ring end
            const size_t bpc = 2 * (size_t)input->bytes_per_sample;
            if (n < f->len - pos) n -= n % bpc;
            circbuffer_append(input, const_cast<unsigned char*>(f->data + pos), n);
            pos += n;
        } else {
            usleep(1000);
        }
    }
    return NULL;
}

struct Harness {
    std::vector<device_t> devs;
    std::vector<input_t> inputs;
    std::vector<std::vector<channel_t>> chans;
    std::vector<std::vector<freq_t>> freqs;
    std::vector<std::vector<freq_t>> scan_lists;  // frequency lists installed with abh_set_freqlist
    std::vector<std::vector<size_t>> bins, base_bins;
    std::vector<std::vector<float>> bufs_wave, bufs_iq;
    std::vector<std::vector<unsigned char>> rings;
    // results
    std::vector<std::vector<float>> out_wave;   // per device: batches x C x B
    std::vector<std::vector<float>> out_iq;     // per device: batches x C x 2B
    std::vector<std::vector<char>> out_axc;     // per device: batches x C
    std::vector<int> n_batches;
    int B = 0, wave_len = 0;
    Signal sig;
    // mixers (mixer_t + the O_MIXER outputs of the input channels, as parse_mixers()/parse_outputs() leave them)
    std::vector<mixer_t> mixers;
    std::vector<std::vector<mixinput_t>> mix_inputs;
    std::vector<std::vector<float>> mix_wave, mix_wave_r;
    std::vector<std::vector<std::vector<output_t>>> outputs;      // [dev][chan][k]
    std::vector<std::vector<std::vector<mixer_data>>> mix_data;   // storage behind output_t.data
    std::vector<std::vector<float>> out_mix_l, out_mix_r;        // per mixer: batches x B
    std::vector<std::vector<char>> out_mix_axc;
    std::vector<int> n_mix_batches;
    std::vector<int> mix_was_gpu;                                 // b200_mixer_is_gpu() as seen while the demod thread was alive
    std::vector<int> failed_calls;                                // disable_device_outputs stand-in: calls per device
    // O_RAWFILE stand-in: (dev, chan) -> FILE*
    struct Raw {
        int dev, chan;
        FILE* f;
    };
    std::vector<Raw> rawfiles;
};
Harness* g_harness = nullptr;
void on_device_failed(device_t* dev) {
    if (g_harness) g_harness->failed_calls[dev - g_harness->devs.data()]++;
}
struct Consumer {
    Harness* h;
    volatile int stop;
};
void consume_ready(Harness* h) {
    // output_thread(): mixers first (output.cpp:888-896), then the devices (:903-923)
    for (size_t m = 0; m < h->mixers.size(); m++) {
        channel_t* channel = &h->mixers[m].channel;
        if (!h->mixers[m].enabled || channel->state != CH_READY) continue;
        h->out_mix_l[m].insert(h->out_mix_l[m].end(), channel->waveout, channel->waveout + h->B);
        h->out_mix_r[m].insert(h->out_mix_r[m].end(), channel->waveout_r, channel->waveout_r + h->B);
        h->out_mix_axc[m].push_back((char)channel->axcindicate);
        h->n_mix_batches[m]++;
        h->mix_was_gpu[m] |= b200_mixer_is_gpu(&h->mixers[m]);
        channel->state = CH_DIRTY;
    }
    for (const Harness::Raw& r : h->rawfiles) {  // process_outputs(), O_RAWFILE branch (output.cpp:519-522)
        device_t* dev = &h->devs[r.dev];
        if (dev->waveavail) b200_write_rawfile(r.f, dev->channels + r.chan, h->B);
    }
    for (size_t i = 0; i < h->devs.size(); i++) {
        device_t* dev = &h->devs[i];
        if (!dev->waveavail) continue;
        for (int c = 0; c < dev->channel_count; c++) {
            channel_t* ch = dev->channels + c;
            h->out_wave[i].insert(h->out_wave[i].end(), ch->waveout, ch->waveout + h->B);
            h->out_iq[i].insert(h->out_iq[i].end(), ch->iq_out, ch->iq_out + 2 * h->B);
            h->out_axc[i].push_back((char)ch->axcindicate);
        }
        h->n_batches[i]++;
        dev->waveavail = 0;  // output.cpp:922 (the AGC_EXTRA tail copy of :920 is done inside the engine)
    }
}
void* consumer_thread(void* p) {
    Consumer* c = (Consumer*)p;
    while (!c->stop) {
        c->h->sig.wait_ms(5);
        consume_ready(c->h);
    }
    consume_ready(c->h);
    return NULL;
}
}  // namespace

extern "C" {

ABG_API void* abh_create(const abg_config* cfg, int max_batches_per_run) {
    Harness* h = new Harness();
    const int D = cfg->n_devices;
    h->B = cfg->wave_rate / 8;
    h->wave_len = 2 * h->B + AGC_EXTRA;
    h->devs.resize(D); h->inputs.resize(D); h->chans.resize(D); h->freqs.resize(D); h->bins.resize(D); h->base_bins.resize(D);
    h->bufs_wave.resize(D); h->bufs_iq.resize(D); h->rings.resize(D);
    h->out_wave.resize(D); h->out_iq.resize(D); h->out_axc.resize(D); h->n_batches.assign(D, 0);
    memset(&g_b200, 0, sizeof(g_b200));
    g_b200.fft_size = cfg->fft_size;
    g_b200.wave_rate = cfg->wave_rate;
    g_b200.fm_demod = cfg->fm_demod;
    g_b200.wait_for_consumer = 1;
    g_b200.max_batches_per_run = max_batches_per_run;
    for (int i = 0; i < D; i++) {
        const abg_device_cfg& dc = cfg->devices[i];
        input_t& in = h->inputs[i];
        memset(&in, 0, sizeof(in));
        in.sfmt = (sample_format_t)dc.sfmt;
        in.fullscale = dc.fullscale;
        in.bytes_per_sample = dc.sfmt == ABG_SFMT_S16 ? 2 : (dc.sfmt == ABG_SFMT_F32 ? 4 : 1);
        in.sample_rate = dc.sample_rate;
        // config.cpp:793-803: MIN_BUF_SIZE rounded up to a multiple of one hop (ceil variant), + the wrap tail
        size_t fft_batch_len = 2 * in.bytes_per_sample * (size_t)ceil((double)dc.sample_rate / (double)cfg->wave_rate);
        in.buf_size = MIN_BUF_SIZE;
        if (in.buf_size % fft_batch_len != 0) in.buf_size += fft_batch_len - in.buf_size % fft_batch_len;
        h->rings[i].assign(in.buf_size + 2 * in.bytes_per_sample * (size_t)cfg->fft_size, 0);
        in.buffer = h->rings[i].data();
        in.state = INPUT_INITIALIZED;
        pthread_mutex_init(&in.buffer_lock, NULL);
        const int C = dc.n_channels;
        h->chans[i].resize(C); h->freqs[i].resize(C); h->bins[i].resize(C); h->base_bins[i].resize(C);
        h->bufs_wave[i].assign((size_t)C * h->wave_len, 0.0f);
        h->bufs_iq[i].assign((size_t)C * 2 * h->wave_len, 0.0f);
        for (int c = 0; c < C; c++) {
            const abg_channel_cfg& cc = dc.channels[c];
            channel_t& ch = h->chans[i][c];
            freq_t& f = h->freqs[i][c];
            memset(&ch, 0, sizeof(ch));
            memset(&f, 0, sizeof(f));
            ch.waveout = &h->bufs_wave[i][(size_t)c * h->wave_len];
            ch.iq_out = &h->bufs_iq[i][(size_t)c * 2 * h->wave_len];
            ch.alpha = cc.alpha;
            ch.dm_dphi = cc.dm_dphi;
            ch.axcindicate = NO_SIGNAL;
            ch.afc = (unsigned char)cc.afc;
            ch.freqlist = &f;
            ch.freq_count = 1;
            ch.needs_raw_iq = cc.needs_raw_iq;
            ch.has_iq_outputs = cc.has_iq_outputs;
            f.agcavgfast = 0.5f;
            f.ampfactor = cc.ampfactor;
            f.modulation = cc.modulation == ABG_MOD_NFM ? MOD_NFM : MOD_AM;
            f.b200_cfg = b200_freq_cfg{cc.squelch_level, cc.squelch_snr_db, cc.notch_hz, cc.notch_q, cc.ctcss_hz, cc.lowpass_hz};
            h->bins[i][c] = h->base_bins[i][c] = (size_t)cc.bin;
        }
        device_t& d = h->devs[i];
        memset(&d, 0, sizeof(d));
        d.input = &in;
        d.channel_count = C;
        d.bins = h->bins[i].data();
        d.base_bins = h->base_bins[i].data();
        d.channels = h->chans[i].data();
    }
    g_b200.devices = h->devs.data();
    g_b200.device_count = D;
    g_b200.devices_running = D;
    h->failed_calls.assign(D, 0);
    h->outputs.resize(D);
    h->mix_data.resize(D);
    for (int i = 0; i < D; i++) {
        h->outputs[i].resize(h->chans[i].size());
        h->mix_data[i].resize(h->chans[i].size());
    }
    g_harness = h;
    g_b200.on_device_failed = on_device_failed;
    return h;
}

// mixers as parse_mixers() + mixer_connect_input() leave them (mixer.cpp:55-96): mixer m owns inputs
// [offsets[m], offsets[m+1]); every input is an O_MIXER output of its channel.  Call before abh_run.
ABG_API int abh_set_mixers(void* hp, int n_mixers, const int32_t* offsets, const abg_mixer_input* inputs) {
    Harness* h = (Harness*)hp;
    h->mixers.resize(n_mixers);
    h->mix_inputs.resize(n_mixers);
    h->mix_wave.resize(n_mixers); h->mix_wave_r.resize(n_mixers);
    h->out_mix_l.resize(n_mixers); h->out_mix_r.resize(n_mixers); h->out_mix_axc.resize(n_mixers);
    h->n_mix_batches.assign(n_mixers, 0);
    h->mix_was_gpu.assign(n_mixers, 0);
    // reserve the per-channel output arrays first: output_t.data points into mix_data
    std::vector<std::vector<int>> count(h->devs.size());
    for (size_t i = 0; i < h->devs.size(); i++) count[i].assign(h->chans[i].size(), 0);
    for (int k = 0; k < offsets[n_mixers]; k++) {
        if (inputs[k].dev < 0 || inputs[k].dev >= (int)h->devs.size() || inputs[k].chan < 0 || inputs[k].chan >= h->devs[inputs[k].dev].channel_count) return -1;
        count[inputs[k].dev][inputs[k].chan]++;
    }
    for (size_t i = 0; i < h->devs.size(); i++)
        for (size_t c = 0; c < h->chans[i].size(); c++) {
            h->outputs[i][c].clear(); h->outputs[i][c].reserve(count[i][c]);
            h->mix_data[i][c].clear(); h->mix_data[i][c].reserve(count[i][c]);
        }
    for (int m = 0; m < n_mixers; m++) {
        mixer_t& mx = h->mixers[m];
        memset(&mx, 0, sizeof(mx));
        mx.name = "mixer";
        mx.enabled = true;
        mx.interval = 2;  // MIX_DIVISOR
        const int n_in = offsets[m + 1] - offsets[m];
        h->mix_inputs[m].assign(n_in, mixinput_t{});
        h->mix_wave[m].assign(h->wave_len, 0.0f);
        h->mix_wave_r[m].assign(h->wave_len, 0.0f);
        mx.channel.waveout = h->mix_wave[m].data();
        mx.channel.waveout_r = h->mix_wave_r[m].data();
        mx.channel.mode = MM_MONO;
        mx.channel.state = CH_DIRTY;
        mx.channel.axcindicate = NO_SIGNAL;
        for (int j = 0; j < n_in; j++) {
            const abg_mixer_input& in = inputs[offsets[m] + j];
            mixinput_t& mi = h->mix_inputs[m][j];
            mi.ampfactor = in.ampfactor;
            mi.ampl = fminf(1.0f, 1.0f - in.balance);  // mixer_connect_input(), mixer.cpp:82-83
            mi.ampr = fminf(1.0f, 1.0f + in.balance);
            if (in.balance != 0.0f) mx.channel.mode = MM_STEREO;
            h->mix_data[in.dev][in.chan].push_back(mixer_data{&mx, j});
            output_t o;
            o.type = O_MIXER; o.enabled = true; o.active = false; o.data = &h->mix_data[in.dev][in.chan].back();
            h->outputs[in.dev][in.chan].push_back(o);
        }
        mx.input_count = n_in;
        mx.inputs = h->mix_inputs[m].data();
    }
    for (size_t i = 0; i < h->devs.size(); i++)
        for (size_t c = 0; c < h->chans[i].size(); c++) {
            h->chans[i][c].output_count = (int)h->outputs[i][c].size();
            h->chans[i][c].outputs = h->outputs[i][c].data();
        }
    g_b200.mixers = h->mixers.data();
    g_b200.mixer_count = n_mixers;
    return 0;
}

// O_RAWFILE stand-in: every delivered batch of devices[dev].channels[chan] is appended to `path` the way process_outputs()
// writes a .cf32 file (output.cpp:519-522).  Call before abh_run; the file is closed by abh_destroy.
ABG_API int abh_add_rawfile(void* hp, int dev, int chan, const char* path) {
    Harness* h = (Harness*)hp;
    FILE* f = fopen(path, "wb");
    if (!f) return -1;
    h->rawfiles.push_back(Harness::Raw{dev, chan, f});
    return 0;
}

// scan mode: give devices[dev].channels[chan] a frequency list (freq_t part of every entry from freqs[]) and the entry
// controller_thread would have selected; call before abh_run
ABG_API int abh_set_freqlist(void* hp, int dev, int chan, int n_freqs, const abg_channel_cfg* freqs, int freq_idx) {
    Harness* h = (Harness*)hp;
    if (dev < 0 || dev >= (int)h->devs.size() || chan < 0 || chan >= h->devs[dev].channel_count || n_freqs < 1 || freq_idx < 0 || freq_idx >= n_freqs) return -1;
    h->scan_lists.emplace_back((size_t)n_freqs);
    std::vector<freq_t>& list = h->scan_lists.back();
    for (int k = 0; k < n_freqs; k++) {
        const abg_channel_cfg& cc = freqs[k];
        freq_t& f = list[k];
        memset(&f, 0, sizeof(f));
        f.agcavgfast = 0.5f;
        f.ampfactor = cc.ampfactor;
        f.modulation = cc.modulation == ABG_MOD_NFM ? MOD_NFM : MOD_AM;
        f.b200_cfg = b200_freq_cfg{cc.squelch_level, cc.squelch_snr_db, cc.notch_hz, cc.notch_q, cc.ctcss_hz, cc.lowpass_hz};
    }
    channel_t& ch = h->chans[dev][chan];
    ch.freqlist = list.data();
    ch.freq_count = n_freqs;
    ch.freq_idx = freq_idx;
    return 0;
}

// feed one raw stream per device through the rings, demodulate with demodulate_b200(), consume; returns 0 on success
static int run_with_inputs(Harness* h, std::vector<pthread_t>& fth, int timeout_s);

ABG_API int abh_run(void* hp, const unsigned char* const* raws, const size_t* raw_bytes, int timeout_s) {
    Harness* h = (Harness*)hp;
    const int D = (int)h->devs.size();
    std::vector<Feeder> feeders(D);
    std::vector<pthread_t> fth(D);
    for (int i = 0; i < D; i++) {
        feeders[i] = {&h->inputs[i], raws[i], raw_bytes[i]};
        pthread_create(&fth[i], NULL, feeder_thread, &feeders[i]);
    }
    return run_with_inputs(h, fth, timeout_s);
}

// the same, but every device is fed by the "pattern" input plugin (host/input_pattern.cpp) started the way input_start()
// starts any plugin (input-common.cpp:67-83): block[i] is replayed `repeat` times, paced at speedup x real time
// (speedup > 0, may overflow like a live SDR) or lossless (speedup == 0)
ABG_API int abh_run_pattern(void* hp, const unsigned char* const* blocks, const size_t* block_bytes, long repeat, double speedup, int timeout_s) {
    Harness* h = (Harness*)hp;
    const int D = (int)h->devs.size();
    std::vector<pthread_t> fth(D);
    std::vector<pattern_dev_data_t> dd(D);
    input_t* proto = pattern_input_new();  // the plugin's vtable
    if (!proto) return -3;
    for (int i = 0; i < D; i++) {
        input_t& in = h->inputs[i];
        dd[i] = {blocks[i], block_bytes[i], repeat, speedup};
        in.dev_data = &dd[i];
        in.init = proto->init;
        in.run_rx_thread = proto->run_rx_thread;
        in.set_centerfreq = proto->set_centerfreq;
        in.stop = proto->stop;
        if (in.init(&in) < 0) {
            free(proto->dev_data);
            free(proto);
            return -3;
        }
    }
    free(proto->dev_data);
    free(proto);
    for (int i = 0; i < D; i++) pthread_create(&fth[i], NULL, h->inputs[i].run_rx_thread, &h->inputs[i]);
    return run_with_inputs(h, fth, timeout_s);
}

static int run_with_inputs(Harness* h, std::vector<pthread_t>& fth, int timeout_s) {
    const int D = (int)h->devs.size();
    for (int t = 0; t < 5000; t++) {  // "wait for INPUT_RUNNING", rtl_airband.cpp:1024-1032
        bool all = true;
        for (int i = 0; i < D; i++) all = all && h->inputs[i].state != INPUT_INITIALIZED;
        if (all) break;
        usleep(1000);
    }
    demod_params_t dp = {&h->sig, 0, D};
    pthread_t dth, cth;
    Consumer cons = {h, 0};
    pthread_create(&cth, NULL, consumer_thread, &cons);
    pthread_create(&dth, NULL, demodulate_b200, &dp);
    // finished when every feeder has ended, every ring is (nearly) empty and nothing new arrived for a while
    int idle_ms = 0, last_total = -1, waited_ms = 0;
    while (!g_b200.do_exit && waited_ms < timeout_s * 1000) {
        usleep(20 * 1000);
        waited_ms += 20;
        bool fed = true;
        for (int i = 0; i < D; i++) fed = fed && (h->inputs[i].state == INPUT_FAILED || h->inputs[i].state == INPUT_DISABLED);
        int total = 0;
        for (int i = 0; i < D; i++) total += h->n_batches[i];
        if (fed && total == last_total)
            idle_ms += 20;
        else
            idle_ms = 0;
        last_total = total;
        if (fed && idle_ms >= 400) break;
    }
    const bool timed_out = waited_ms >= timeout_s * 1000;
    g_b200.do_exit = 1;
    pthread_join(dth, NULL);
    cons.stop = 1;
    pthread_join(cth, NULL);
    for (int i = 0; i < D; i++) pthread_join(fth[i], NULL);
    if (g_b200.last_error[0]) return -2;
    return timed_out ? -1 : 0;
}

// CPU-only self-test of the ingest side (no engine involved): the "pattern" plugin fills an input ring through
// circbuffer_append() while a consumer drains it the way demodulate() does (available bytes under buffer_lock, bufs
// advanced without it) and checks every byte against the replayed block.
// consumer_delay_us > 0 makes the consumer slower than a paced source so that the ring overflows (overflow_count).
// Returns the number of mismatching bytes (-1: set-up failure); *consumed / *overflows report what happened.
ABG_API long abh_pattern_selftest(int sfmt, int sample_rate, size_t fft_size, const unsigned char* block, size_t block_len, long repeat,
                                  double speedup, int consumer_delay_us, size_t* consumed, size_t* overflows) {
    memset(&g_b200, 0, sizeof(g_b200));
    g_b200.fft_size = fft_size;
    g_b200.engine_ready = 1;
    input_t* in = pattern_input_new();
    if (!in) return -1;
    in->sfmt = (sample_format_t)sfmt;
    in->bytes_per_sample = sfmt == ABG_SFMT_S16 ? 2 : (sfmt == ABG_SFMT_F32 ? 4 : 1);
    in->sample_rate = sample_rate;
    pattern_dev_data_t* dd = (pattern_dev_data_t*)in->dev_data;
    *dd = {block, block_len, repeat, speedup};
    const size_t bpc = 2 * (size_t)in->bytes_per_sample, tail = bpc * fft_size;
    in->buf_size = 256 * 1024;  // a small ring so that it wraps many times
    in->buf_size -= in->buf_size % bpc;
    std::vector<unsigned char> ring(in->buf_size + tail, 0);
    in->buffer = ring.data();
    pthread_mutex_init(&in->buffer_lock, NULL);
    in->state = INPUT_INITIALIZED;
    if (in->init(in) < 0) {
        free(in->dev_data);
        free(in);
        return -1;
    }
    pthread_create(&in->rx_thread, NULL, in->run_rx_thread, in);
    long bad = 0;
    size_t pos = 0;
    const size_t total = block_len * (size_t)repeat;
    int idle_ms = 0;
    bool lapped = false;  // the source has overwritten bytes not yet read: from then on the byte positions no longer line up
    while (idle_ms < 2000) {
        size_t available;
        pthread_mutex_lock(&in->buffer_lock);
        available = in->bufe >= in->bufs ? in->bufe - in->bufs : in->buf_size - in->bufs + in->bufe;
        pthread_mutex_unlock(&in->buffer_lock);
        if (available == 0) {
            if (in->state != INPUT_RUNNING && in->state != INPUT_INITIALIZED) break;  // source finished and ring drained
            usleep(1000);
            idle_ms++;
            continue;
        }
        idle_ms = 0;
        if (!lapped) {
            long miss = 0;
            for (size_t k = 0; k < available; k++) {
                const unsigned char got = in->buffer[(in->bufs + k) % in->buf_size];
                if (got != block[(pos + k) % block_len]) miss++;
            }
            // A paced source may lap the ring while the bytes are compared, and overflow_count misses a lap past slot 0.
            // An append that overwrote any of them stored `written` before it took the ring lock, so it is seen under that lock.
            pthread_mutex_lock(&in->buffer_lock);
            lapped = in->overflow_count > 0 || __atomic_load_n(&dd->written, __ATOMIC_ACQUIRE) > pos + in->buf_size;
            pthread_mutex_unlock(&in->buffer_lock);
            if (!lapped) bad += miss;
        }
        pos += available;
        in->bufs = (in->bufs + available) % in->buf_size;  // not under the lock, like rtl_airband.cpp:669
        if (consumer_delay_us > 0) usleep(consumer_delay_us);
    }
    g_b200.do_exit = 1;
    pthread_join(in->rx_thread, NULL);
    if (consumed) *consumed = pos;
    if (overflows) *overflows = in->overflow_count;
    if (in->overflow_count == 0 && pos != total) bad += 1000000;
    pthread_mutex_destroy(&in->buffer_lock);
    free(in->dev_data);
    free(in);
    g_b200.do_exit = 0;
    return bad;
}

ABG_API int abh_batches(void* hp, int dev) { return ((Harness*)hp)->n_batches[dev]; }
ABG_API const float* abh_waveout(void* hp, int dev) { return ((Harness*)hp)->out_wave[dev].data(); }
ABG_API const float* abh_iq_out(void* hp, int dev) { return ((Harness*)hp)->out_iq[dev].data(); }
ABG_API const char* abh_axc(void* hp, int dev) { return ((Harness*)hp)->out_axc[dev].data(); }
ABG_API size_t abh_overflows(void* hp, int dev) { return ((Harness*)hp)->inputs[dev].overflow_count; }
ABG_API size_t abh_overruns(void* hp, int dev) { return ((Harness*)hp)->devs[dev].output_overrun_count; }
ABG_API size_t abh_active_counter(void* hp, int dev, int chan) {
    const channel_t& ch = ((Harness*)hp)->chans[dev][chan];
    return ch.freqlist[ch.freq_idx].active_counter;
}
ABG_API const char* abh_last_error(void) { return g_b200.last_error; }
ABG_API int abh_mixer_batches(void* hp, int m) { return ((Harness*)hp)->n_mix_batches[m]; }
ABG_API const float* abh_mixer_left(void* hp, int m) { return ((Harness*)hp)->out_mix_l[m].data(); }
ABG_API const float* abh_mixer_right(void* hp, int m) { return ((Harness*)hp)->out_mix_r[m].data(); }
ABG_API const char* abh_mixer_axc(void* hp, int m) { return ((Harness*)hp)->out_mix_axc[m].data(); }
ABG_API size_t abh_mixer_overruns(void* hp, int m) { return ((Harness*)hp)->mixers[m].output_overrun_count; }
ABG_API int abh_mixer_is_gpu(void* hp, int m) { return ((Harness*)hp)->mix_was_gpu[m]; }
ABG_API int abh_failed_calls(void* hp, int dev) { return ((Harness*)hp)->failed_calls[dev]; }
ABG_API void abh_destroy(void* hp) {
    Harness* h = (Harness*)hp;
    for (auto& r : h->rawfiles)
        if (r.f) fclose(r.f);
    if (g_harness == h) g_harness = nullptr;
    g_b200.mixers = nullptr;
    g_b200.mixer_count = 0;
    delete h;
}

}  // extern "C"
