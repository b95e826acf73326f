/*
 * demodulate_cuda.cpp — the thread body that takes the place of demodulate() (boondock_airband.cpp:308-738) when the
 * reference is built to run its hot path on a B200 through libba_cuda.so.  Same signature, same parameter block
 * (demod_params_t), same shared structures: the rx threads of the unmodified input drivers keep appending with
 * circbuffer_append() (input-helpers.cpp:37-63) under buffer_lock, the output thread keeps waiting on mp3_signal and
 * reading channel_t::waveout / iq_out / axcindicate while waveavail is set (output.cpp:931-951).
 *
 * Compiles two ways, unchanged:
 *   inside the reference tree     -DBA_WITH_REFERENCE_HEADERS   includes boondock_airband.h
 *   stand-alone (this repository)  include/ba_ref_layout.h       the same structures restated; tests/shim plays the rx
 *                                                                thread and the output thread around it
 * Host code only (C++11); everything CUDA sits behind include/ba_cuda.h.
 *
 * What it needs from the reference beyond its headers:
 *   - `devices_running` (boondock_airband.cpp:74) without `static`, or this file appended to boondock_airband.cpp;
 *   - the raw configuration values of each channel, which parse_channels() reads and then folds into the Squelch / filter
 *     objects (config.cpp:437-622): ba_ref_channel_cfg(device, channel) returns them.  INTEGRATION.md section 3 shows where
 *     they come from without touching config.cpp (libba_host.so's configuration front-end reads the same file).
 */
#ifdef BA_WITH_REFERENCE_HEADERS
#include "boondock_airband.h"
extern int devices_running;
enum fm_demod_algo { FM_FAST_ATAN2, FM_QUADRI_DEMOD };
extern enum fm_demod_algo fm_demod;
#else
#include "../../include/ba_ref_layout.h"
#endif

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <vector>

#include "../../include/ba_cuda.h"

/* filled by the host program: the values parse_channels() read for channel `channel` of device `device` (config.cpp:437-652):
 * squelch_threshold_dbfs, squelch_snr_threshold, notch, notch_q, ctcss, bandwidth, tau_us, and for scan mode the frequency
 * list.  frequency / modulation / ampfactor / afc / has_iq_outputs may be left zero: they are taken from channel_t. */
extern "C" const ba_channel_desc* ba_ref_channel_cfg(int device, int channel);
/* likewise the device's own settings; only tau_us is read (the device-level "tau", config.cpp:777-781: the reference keeps
 * exp(-1 / (WAVE_RATE * tau)) in device_t::alpha, from which the integer cannot be recovered exactly).  May return NULL. */
extern "C" const ba_device_desc* ba_ref_device_cfg(int device);
/* output.cpp: disable_device_outputs(dev), called when an input has failed (boondock_airband.cpp:407-412) */
void disable_device_outputs(device_t* dev);

namespace {

/* how many WAVE_BATCH batches one pass may hand over.  1 = the reference's cadence (one hand-off per batch); a replay far
 * above real time raises it (BA_CUDA_MAX_BATCHES in the environment). */
int max_batches_from_env() {
    const char* s = getenv("BA_CUDA_MAX_BATCHES");
    const int v = s ? atoi(s) : 1;
    return v < 1 ? 1 : (v > 64 ? 64 : v);
}

/* BA_CUDA_DEVICES: the GPUs the demodulator threads use.  Unset: GPU 0 alone (empty list).  "all": every visible GPU.
 * "0,2,3": those CUDA ordinals.  False on anything else. */
bool gpus_from_env(std::vector<int32_t>& gpus) {
    gpus.clear();
    const char* s = getenv("BA_CUDA_DEVICES");
    if (!s)
        return true;
    if (!strcmp(s, "all")) {
        const int n = ba_cuda_visible_devices();
        for (int i = 0; i < n; i++)
            gpus.push_back(i);
        return n > 0;
    }
    for (;;) {
        char* end;
        const long v = strtol(s, &end, 10);
        if (end == s || v < 0 || v > 1023 || (*end != ',' && *end != 0))
            return false;
        gpus.push_back((int32_t)v);
        if (*end == 0)
            return true;
        s = end + 1;
    }
}

void describe(int devno, device_t* dev, ba_device_desc* d, std::vector<ba_channel_desc>& ch) {
    input_t* in = dev->input;
    memset(d, 0, sizeof(*d));
    d->sample_format = (int)in->sfmt; /* the same numbering: SFMT_U8 = 1 .. SFMT_F32 = 4 (input-common.h:32) */
    d->bytes_per_sample = in->bytes_per_sample;
    d->fullscale = in->fullscale;
    d->sample_rate = in->sample_rate;
    d->centerfreq = in->centerfreq;
    const ba_device_desc* rawdev = ba_ref_device_cfg(devno);
    d->tau_us = rawdev ? rawdev->tau_us : -1;
    d->channel_count = dev->channel_count;
    for (int i = 0; i < dev->channel_count; i++) {
        channel_t* c = dev->channels + i;
        freq_t* f = c->freqlist + c->freq_idx;
        ba_channel_desc x;
        const ba_channel_desc* raw = ba_ref_channel_cfg(devno, i);
        if (raw)
            x = *raw;
        else
            memset(&x, 0, sizeof(x)), x.squelch_snr_threshold = -1.0f, x.tau_us = -1;
        x.frequency = f->frequency;
        x.modulation = (int)f->modulation; /* MOD_AM = 0, MOD_NFM = 1 (boondock_airband.h:202-208) */
        x.ampfactor = f->ampfactor;
        x.afc = c->afc;
        x.has_iq_outputs = c->has_iq_outputs;
        ch.push_back(x);
    }
}

}  // namespace

void* demodulate_cuda(void* params) { /* void* demodulate(void* params), boondock_airband.cpp:308 */
    demod_params_t* dp = (demod_params_t*)params;
    const int first = dp->device_start, n = dp->device_end - dp->device_start;
    std::vector<ba_device_desc> dd(n);
    std::vector<std::vector<ba_channel_desc> > ch(n);
    for (int i = 0; i < n; i++) {
        describe(first + i, devices + first + i, &dd[i], ch[i]);
        dd[i].channels = ch[i].data();
    }
    ba_engine_desc ed;
    memset(&ed, 0, sizeof(ed));
    ed.abi_version = BA_CUDA_ABI_VERSION;
    ed.fft_size = (int)fft_size; /* global, boondock_airband.cpp:83 */
    ed.wave_rate = WAVE_RATE;    /* boondock_airband.h:66-71 */
    ed.fm_demod = (int)fm_demod; /* boondock_airband.cpp:88-89 */
    ed.cuda_device = 0;
    ed.device_count = n;
    ed.devices = dd.data();
    ed.max_batches_per_step = max_batches_from_env();
    if (getenv("BA_CUDA_SKIP_SILENT_ROWS")) /* replays far above real time: silence does not cross the link (see ba_cuda.h) */
        ed.flags |= BA_FLAG_SKIP_SILENT_ROWS;
    std::vector<int32_t> gpus;
    if (!gpus_from_env(gpus)) {
        fprintf(stderr, "BA_CUDA_DEVICES=%s: expected \"all\" or a comma-separated list of CUDA ordinals\n", getenv("BA_CUDA_DEVICES"));
        do_exit = 1;
        return NULL;
    }
    /* a thread of several devices (the reference's default: one thread for all) spreads them over the GPUs as one engine;
     * a thread of one device (multiple_demod_threads) takes the GPU its first device number picks from the list */
    ba_engine* eng = NULL;
    int ret;
    if (gpus.empty() || n == 1) {
        if (!gpus.empty())
            ed.cuda_device = gpus[first % gpus.size()];
        ret = ba_cuda_create(&ed, &eng);
    } else {
        ret = ba_cuda_create_multi(&ed, gpus.data(), (int32_t)gpus.size(), NULL, &eng);
    }
    if (ret != BA_OK) { /* the reference's reaction to a failing gpu_fft_prepare(), boondock_airband.cpp:319-332 */
        fprintf(stderr, "%s: %d (%s)\n", gpus.size() > 0 && n > 1 ? "ba_cuda_create_multi" : "ba_cuda_create", ret, ba_cuda_last_error());
        do_exit = 1;
        return NULL;
    }
    /* The rx threads append into the engine's pinned ring: same size arithmetic as config.cpp:796-805, so input_t::buffer
     * simply points there.  (In the reference this runs before input_start(); a buffer already allocated is released by the
     * caller.)  What was appended before this point is re-published below from bufs. */
    std::vector<size_t> published(n, 0); /* bufe as last handed to the engine, per input */
    for (int i = 0; i < n; i++) {
        input_t* in = devices[first + i].input;
        unsigned char* ring;
        size_t buf_size, mirror;
        ba_cuda_input_ring(eng, i, &ring, &buf_size, &mirror);
        pthread_mutex_lock(&in->buffer_lock);
        if (in->buffer != ring) {
            in->buffer = ring;
            in->buf_size = buf_size;
            in->bufs = in->bufe = 0;
        }
        pthread_mutex_unlock(&in->buffer_lock);
    }
    const size_t B = WAVE_BATCH;
    while (!do_exit) {
        if (devices_running == 0) { /* boondock_airband.cpp:401-405 */
            fprintf(stderr, "All receivers failed, exiting\n");
            do_exit = 1;
            continue;
        }
        bool fresh_any = false;
        for (int i = 0; i < n; i++) { /* ring availability, boondock_airband.cpp:394-399, for every device of this thread */
            device_t* dev = devices + first + i;
            input_t* in = dev->input;
            if (in->state != INPUT_RUNNING) {
                if (in->state == INPUT_FAILED) { /* boondock_airband.cpp:407-412 */
                    in->state = INPUT_DISABLED;
                    disable_device_outputs(dev);
                    devices_running--;
                }
                continue;
            }
            pthread_mutex_lock(&in->buffer_lock);
            const size_t bufe = in->bufe;
            pthread_mutex_unlock(&in->buffer_lock);
            const size_t fresh = (bufe + in->buf_size - published[i]) % in->buf_size;
            if (fresh) {
                if (ba_cuda_commit(eng, i, fresh) == BA_OK) {
                    published[i] = bufe;
                    fresh_any = true;
                } /* BA_ERR_OVERRUN: the copy of an earlier pass still holds the bytes; they are offered again next time */
            }
        }
        const int ticket = ba_cuda_process(eng);
        if (ticket < 0) {
            fprintf(stderr, "ba_cuda_process: %d (%s)\n", ticket, ba_cuda_last_error());
            do_exit = 1;
            break;
        }
        int batches = 0;
        for (int i = 0; i < n; i++) {
            device_t* dev = devices + first + i;
            input_t* in = dev->input;
            ba_step_out out;
            if (ba_cuda_collect(eng, ticket, i, &out) != BA_OK)
                continue;
            /* bufs = (bufs + bps) % buf_size, boondock_airband.cpp:735: the engine says how far the ring has been read */
            size_t consumed;
            if (ba_cuda_input_consumed(eng, i, &consumed) == BA_OK) {
                pthread_mutex_lock(&in->buffer_lock);
                in->bufs = consumed;
                pthread_mutex_unlock(&in->buffer_lock);
            }
            for (int b = 0; b < out.n_batches; b++) {
                /* the single-slot hand-off of boondock_airband.cpp:673-679: at real time the output thread has long cleared
                 * waveavail; in a replay above real time this thread waits for it instead of dropping the batch */
                while (dev->waveavail && !do_exit) {
                    if (getenv("BA_CUDA_DROP_ON_OVERRUN")) {
                        dev->output_overrun_count++;
                        break;
                    }
                    usleep(50);
                }
                if (dev->waveavail)
                    continue;
                for (int c = 0; c < dev->channel_count; c++) {
                    channel_t* chn = dev->channels + c;
                    const ba_channel_status* st = out.status + (size_t)b * out.channel_count + c;
                    if (out.waveout) {
                        memcpy(chn->waveout, out.waveout + (size_t)c * out.wave_stride + (size_t)b * B, B * sizeof(float));
                    } else { /* BA_FLAG_SKIP_SILENT_ROWS: the row, or silence */
                        const int32_t row = out.row_of[(size_t)c * out.row_of_stride + b];
                        if (row >= 0)
                            memcpy(chn->waveout, out.rows + (size_t)row * B, B * sizeof(float));
                        else
                            memset(chn->waveout, 0, B * sizeof(float));
                    }
                    if (out.iq_out && chn->has_iq_outputs)
                        memcpy(chn->iq_out, out.iq_out + 2 * ((size_t)c * out.wave_stride + (size_t)b * B), 2 * B * sizeof(float));
                    chn->axcindicate = (status)st->axcindicate;
                    dev->bins[c] = st->bin; /* AFC result, boondock_airband.cpp:238-249 */
                    chn->freqlist[chn->freq_idx].active_counter = st->active_counter;
                }
                dev->waveavail = 1;       /* boondock_airband.cpp:677 */
                dp->mp3_signal->send();   /* boondock_airband.cpp:728 */
                batches++;
            }
        }
        if (!fresh_any && batches == 0)
            usleep(10000); /* SLEEP(10), boondock_airband.cpp:419-424 */
    }
    ba_cuda_destroy(eng);
    return NULL;
}
