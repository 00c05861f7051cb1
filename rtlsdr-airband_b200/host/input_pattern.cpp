// "pattern" input plugin: a synthetic SDR for load tests of the ingest bridge (SURVEY.md §8f rank 1).
// Shape of a reference input plugin (reference src/input-common.h:39-57, e.g. src/input-file.cpp): <type>_input_new()
// returns an input_t with init / run_rx_thread / set_centerfreq / stop filled in; the rx thread appends ring-format bytes
// with circbuffer_append() (reference src/input-helpers.cpp:37-63) and flips input->state.
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include <algorithm>

#include "b200_adapter.h"

namespace {
double now_s() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

int pattern_init(input_t* const input) {
    pattern_dev_data_t* dd = (pattern_dev_data_t*)input->dev_data;
    if (!dd || !dd->block || dd->block_len == 0 || dd->repeat < 1) return -1;
    if (dd->block_len % (2 * (size_t)input->bytes_per_sample)) return -1;  // whole complex samples only
    return 0;
}

void* pattern_rx_thread(void* ctx) {
    input_t* input = (input_t*)ctx;
    pattern_dev_data_t* dd = (pattern_dev_data_t*)input->dev_data;
    const size_t bpc = 2 * (size_t)input->bytes_per_sample;
    const size_t total = dd->block_len * (size_t)dd->repeat;
    const size_t max_chunk = ((input->buf_size / 2 - 1) / bpc) * bpc;  // like input-file.cpp:95
    const double rate = dd->speedup > 0 ? dd->speedup * (double)input->sample_rate * (double)bpc : 0.0;  // bytes per second
    size_t sent = 0;
    input->state = INPUT_RUNNING;
    // paced mode: the clock starts when the demodulator is up, so that its start-up time (CUDA context, allocations) is not
    // counted as half a second of lost samples; a real SDR is started the same way, after init_demod (rtl_airband.cpp:1024-1060)
    while (rate > 0 && !g_b200.engine_ready && !g_b200.do_exit) usleep(1000);
    const double t0 = now_s();
    while (!g_b200.do_exit && sent < total && input->state == INPUT_RUNNING) {
        size_t n;
        if (rate > 0) {  // live source: what the clock says is due, whether or not the consumer kept up
            size_t due = (size_t)((now_s() - t0) * rate);
            due -= due % bpc;
            due = std::min(due, total);
            if (due <= sent) {
                usleep(2000);
                continue;
            }
            n = std::min(due - sent, max_chunk);
        } else {  // lossless: wait for ring space like file_rx_thread (input-file.cpp:104-116)
            size_t space_left;
            pthread_mutex_lock(&input->buffer_lock);
            if (input->bufe >= input->bufs)
                space_left = input->bufs + (input->buf_size - input->bufe);
            else
                space_left = input->bufs - input->bufe;
            pthread_mutex_unlock(&input->buffer_lock);
            if (space_left <= max_chunk + bpc) {
                usleep(1000);
                continue;
            }
            n = std::min(max_chunk, total - sent);
        }
        const size_t off = sent % dd->block_len;
        n = std::min(n, dd->block_len - off);  // one append never straddles the block end
        __atomic_store_n(&dd->written, sent + n, __ATOMIC_RELEASE);
        circbuffer_append(input, const_cast<unsigned char*>(dd->block + off), n);
        sent += n;
    }
    if (input->state == INPUT_RUNNING) input->state = INPUT_FAILED;  // end of stream, like feof() in input-file.cpp:119-123
    return NULL;
}

int pattern_set_centerfreq(input_t* const input, int const centerfreq) {
    input->centerfreq = centerfreq;  // nothing to retune
    return 0;
}

int pattern_stop(input_t* const input) {
    if (input->state == INPUT_RUNNING) input->state = INPUT_STOPPED;
    return 0;
}
}  // namespace

extern "C" ABG_API input_t* pattern_input_new(void) {
    input_t* input = (input_t*)calloc(1, sizeof(input_t));
    if (!input) return NULL;
    input->dev_data = calloc(1, sizeof(pattern_dev_data_t));
    input->state = INPUT_UNKNOWN;
    input->sfmt = SFMT_U8;
    input->fullscale = 127.5f;
    input->bytes_per_sample = 1;
    input->sample_rate = 2560000;
    input->init = &pattern_init;
    input->run_rx_thread = &pattern_rx_thread;
    input->set_centerfreq = &pattern_set_centerfreq;
    input->stop = &pattern_stop;
    return input;
}
