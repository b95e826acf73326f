/*
 * ba_engine.cu — host side of the B200 channelize-and-demodulate engine: the extern "C" boundary of include/ba_cuda.h.
 *
 * It plays the role of the body of demodulate() (boondock_airband.cpp:383-737) for the inputs handed to it:
 *   ring availability + hop arithmetic   .cpp:394-399, 418-424, 735   -> plan_step()
 *   circbuffer_append()                  input-helpers.cpp:37-63      -> ba_cuda_submit() / ba_cuda_commit()
 *   convert + window + FFT + bin pick    .cpp:426-516                 -> K1 (channelize.cu), one launch for all inputs
 *   per-channel loop                     .cpp:518-672                 -> K2 (demod.cu), one launch for all channels
 *   hand-off waveavail / Signal::send    .cpp:673-679, 728            -> ba_cuda_collect()
 * One CUDA stream; every step's descriptors go up in one copy, its results come back in a few large ones.
 * With AFC enabled on an input (channel_t.afc > 0, .cpp:650-654) that input's bins can move after every batch, so
 * its K1/K2 launches alternate batch by batch ("phases"); all other inputs run a whole step in one K1 + one K2.
 *
 * There is no CPU implementation behind this file: without a CUDA device ba_cuda_create() returns BA_ERR_NO_DEVICE.
 */
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <deque>
#include <mutex>
#include <new>
#include <vector>

#include "ba_kernels.h"
#include "host_model.h"

#define BA_MIN_BUF_SIZE 2560000 /* MIN_BUF_SIZE, boondock_airband.h:64 */
#define BA_SLOTS 3               /* tickets that may be outstanding: copies in, kernels and copies out of three passes overlap */

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (cudaError_t)(call);                                                          \
        if (e_ != cudaSuccess)                                                                         \
            return fail(BA_ERR_CUDA, "%s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

/* Every entry point that issues CUDA work first makes the engine's GPU the calling thread's current device: a process may
 * hold one engine per GPU, each driven by its own demodulator thread (multiple_demod_threads, boondock_airband.cpp:1088-1122),
 * and the current device is per-thread state that ba_cuda_create() set only on the thread that created the engine. */
#define USE_DEVICE(e)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = cudaSetDevice((e)->cuda_device);                                               \
        if (e_ != cudaSuccess)                                                                          \
            return fail(BA_ERR_CUDA, "cudaSetDevice(%d) -> %s", (e)->cuda_device, cudaGetErrorString(e_)); \
    } while (0)

/* A group (ba_cuda_create_multi) hands a per-device or per-mixer call to the member that holds that device or mixer, under
 * the member's own index, and returns what the member returns; `call` is the entry point itself, which then sees a plain
 * engine. */
#define FORWARD(e, idx, owner, local, what, call)                                      \
    do {                                                                                \
        if ((e) && !(e)->members.empty()) {                                             \
            ba_engine* g_ = (e);                                                        \
            if (g_->broken)                                                             \
                return group_broken();                                                  \
            if ((idx) < 0 || (idx) >= (int)g_->owner.size())                            \
                return fail(BA_ERR_BAD_ARG, "no " what " %d", (int)(idx));              \
            e = g_->members[g_->owner[idx]];                                            \
            idx = g_->local[idx];                                                       \
            return group_rc(g_, (call));                                                \
        }                                                                               \
    } while (0)
#define FORWARD_DEV(e, dev, call) FORWARD(e, dev, dev_member, dev_local, "device", call)
#define FORWARD_MIXER(e, mixer, call) FORWARD(e, mixer, mix_member, mix_local, "mixer", call)

uint32_t pow2_at_least(uint64_t v) {
    uint32_t p = 1;
    while (p < v)
        p <<= 1;
    return p;
}

struct ExtChunk {
    const unsigned char* p;
    size_t n;
};

struct Dev {
    ba_device_desc cfg;
    std::vector<ba_channel_desc> chans;
    std::vector<std::vector<ba_freq_desc>> freqs; /* per channel: its freqlist (one entry in multichannel mode) */
    std::vector<int> freq_idx;                    /* channel_t.freq_idx */
    std::vector<size_t> bank0;                    /* per channel: first entry of its freq bank (scan channels), else SIZE_MAX */
    int C = 0, c_pad = 0;
    size_t sample_bytes = 0; /* one complex sample */
    size_t hop_bytes = 0, frame_bytes = 0;
    bool any_afc = false, any_iq = false, any_raw = false;
    int first_chan = 0;
    /* host ring = input_t.buffer */
    std::mutex lock;
    unsigned char* ring = nullptr;
    size_t buf_size = 0, mirror = 0, bufs = 0, bufe = 0;
    size_t rpos = 0; /* the engine's read position: bytes in [bufs, rpos) have been queued for copying but the copy engine may still be
                        reading them; bufs (what the producer sees, .cpp:735) follows once the copies have completed */
    uint64_t overflow_count = 0;
    std::vector<ExtChunk> ext;
    /* stream in HBM */
    unsigned char* d_buf[2] = {nullptr, nullptr};
    size_t d_cap = 0;
    int cur = 0;
    size_t have = 0;       /* bytes valid in d_buf[cur] */
    uint64_t base_off = 0; /* stream offset of d_buf[cur][0] */
    const unsigned char* attached = nullptr;
    size_t attached_cap = 0, attached_valid = 0;
    uint64_t frames_done = 0, batches_done = 0;
    bool injected = false;
    /* picks, bins */
    float2* d_picks = nullptr;
    float* d_mags = nullptr;
    uint32_t ring_len = 0;
    uint32_t* d_bins = nullptr;
    float2* d_spectrum = nullptr;
    std::vector<uint32_t> base_bins;
    std::vector<int> feeds; /* flat mixer-input indices fed by channels of this input */
    /* arena offsets (elements) */
    size_t wave_off = 0, iq_off = 0, status_off = 0;
    /* plan of the current step */
    int step_frames = 0, step_batches = 0;
    uint64_t step_frame0 = 0, step_batch0 = 0;
};

/* mixer_t / mixinput_t as the engine keeps them (row f-4) */
struct MixInput {
    int dev = 0, ch = 0;
    float mult_l = 0.f, mult_r = 0.f;
    bool enabled = true; /* input_mask, mixer.cpp:96-112 */
};
struct Mixer {
    int first_in = 0, n_in = 0;
    bool stereo = false;
    uint64_t emitted = 0; /* batches handed out so far */
    size_t out_off = 0;   /* floats into the slot's mixer arena: left plane, then right if stereo */
};

struct Slot {
    float* d_mix = nullptr;
    float* h_mix = nullptr;
    int32_t* d_mix_sig = nullptr;
    int32_t* h_mix_sig = nullptr;
    std::vector<int> mix_emit;        /* per mixer: batches mixed by this ticket */
    std::vector<uint64_t> mix_first;  /* and the number of the first of them */
    float* d_wave = nullptr;
    float* h_wave = nullptr;
    /* BA_FLAG_SKIP_SILENT_ROWS: packed non-silent rows, the row map, the row counter, the per-device row table the pack kernel reads */
    float* d_pack = nullptr;
    float* h_pack = nullptr;
    int32_t* d_rowmap = nullptr;
    int32_t* h_rowmap = nullptr;
    uint32_t* d_rowcount = nullptr;
    uint32_t* h_rowcount = nullptr;
    ba::K3PackDev* h_packdev = nullptr;
    bool pack_pending = false; /* the rows of this ticket have not been fetched yet (the first ba_cuda_collect() does it) */
    uint32_t pack_rows = 0;
    float2* d_iq = nullptr;
    float2* h_iq = nullptr;
    uint8_t* d_trace = nullptr;
    uint8_t* h_trace = nullptr;
    ba_channel_status* d_status = nullptr;
    ba_channel_status* h_status = nullptr;
    unsigned char* d_desc = nullptr;
    unsigned char* h_desc = nullptr;
    ba::K1Carry* h_carry = nullptr; /* pinned; the carry kernel reads it in place */
    cudaEvent_t ev_in2 = nullptr;   /* the second host->device stream has finished its share */
    cudaEvent_t ev_ring = nullptr;  /* the copies out of the pinned input rings have completed */
    std::vector<size_t> ring_taken; /* per device: ring bytes this ticket queued */
    cudaEvent_t ev_begin = nullptr, ev_done = nullptr; /* first operation of the ticket / results are in pinned host memory */
    cudaEvent_t ev_in = nullptr, ev_kdone = nullptr;    /* inputs and descriptors are in HBM / kernels have finished */
    cudaEvent_t ev_k1 = nullptr;                        /* the channelizer of the last phase has finished */
    cudaEvent_t ev_out0 = nullptr;                      /* the device->host stream starts on this ticket's results */
    bool used = false;
    std::vector<cudaEvent_t> ev_k; /* 4 per phase: before/after K1, before/after K2 */
    int phases = 0;
    int ticket = -1;
    bool busy = false;
    std::vector<int> n_batches; /* per device */
    std::vector<uint64_t> frames_done;
    uint64_t h2d_bytes = 0, d2h_bytes = 0;
};

/* ring bytes a ticket queued for copying: given back to the producers (bufs) once `ev` has fired */
struct RingRelease {
    cudaEvent_t ev;
    std::vector<size_t> taken; /* per device */
};

}  // namespace

struct ba_engine {
    std::mutex rel_lock;
    std::deque<RingRelease> rel;
    int fft_size = 0, wave_rate = 0, B = 0, fm_demod = 0, cuda_device = 0, max_batches = 0;
    uint32_t flags = 0;
    int sm_count = 0, smem_optin = 0;
    std::vector<Dev*> dev;
    int total_channels = 0, max_channels = 0;
    int stride = 0; /* max_batches*B + E */
    bool any_iq = false, any_afc = false;
    bool serial_k2 = false; /* demodulator on the channelizer's stream (AFC needs it: the bins feed back) */
    cudaStream_t stream = nullptr; /* = s_k: kernels; debug helpers run here */
    cudaStream_t s_in = nullptr, s_k = nullptr, s_k2 = nullptr, s_out = nullptr; /* host->device, K1, K2, device->host */
    cudaStream_t s_k2b = nullptr; /* the plain-AM demodulator runs here beside the general one */
    cudaStream_t s_pack = nullptr; /* BA_FLAG_SKIP_SILENT_ROWS: ba_cuda_collect() fetches a ticket's packed rows here (its own stream: later tickets queue on s_out) */
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t s_in2 = nullptr; /* second host->device stream: alternate inputs, so that one copy's set-up hides behind the other's transfer */
    int h2d_streams = 2;
    cudaEvent_t ev_tmp[2] = {nullptr, nullptr};
    float* d_window = nullptr;
    float2* d_twiddle = nullptr;
    float* d_sincos = nullptr;
    std::vector<float> window;
    ba::K2Chan* d_chan = nullptr;
    ba::K2State* d_state = nullptr;
    ba::K2Ctcss* d_ctcss = nullptr;
    int32_t* d_order = nullptr;
    uint32_t* d_tile_counter = nullptr;
    int n_plain = 0; /* slots [0, n_plain) of the launch order are plain AM channels */
    std::vector<ba::K2Chan> h_chan;
    std::vector<ba_channel_info> info;
    Slot slot[BA_SLOTS];
    int next_ticket = 0;
    uint64_t launches = 0;
    int tile_frames = 0, raw_bytes = 0, k1_ctas_per_sm = 2;
    size_t desc_bytes = 0;
    int max_phases = 1;
    cudaEvent_t marks[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    /* mixers (K3) */
    std::vector<Mixer> mixers;
    std::vector<MixInput> mix_in;
    /* scan mode: per frequency of every scan channel, the constants and the parked freq_t state */
    ba::K2Chan* d_bank_chan = nullptr;
    ba::K2State* d_bank_state = nullptr;
    ba::K3In* d_mix_in = nullptr;
    ba::K3Mixer* d_mixer = nullptr;
    float* d_fifo = nullptr;
    uint8_t* d_fifo_sig = nullptr;
    int fifo_depth = 0;
    size_t mix_floats = 0;   /* floats of one slot's mixer arena */
    size_t mix_desc_off = 0; /* where the K3 part of the per-ticket descriptor blob starts */
    /* ba_cuda_create_multi(): a group holds nothing but its members (ordinary engines) and where each device and mixer went */
    std::vector<ba_engine*> members;
    std::vector<int> dev_member, dev_local; /* per device of the group's descriptor */
    std::vector<int> mix_member, mix_local; /* per mixer */
    bool broken = false;                    /* a member failed in a way that may leave the members out of step */
};

namespace {

void free_engine(ba_engine* e) {
    if (!e)
        return;
    if (!e->members.empty()) {
        for (ba_engine* m : e->members)
            free_engine(m);
        delete e;
        return;
    }
    cudaSetDevice(e->cuda_device);
    for (cudaStream_t q : {e->s_in, e->s_in2, e->s_k, e->s_k2, e->s_k2b, e->s_out, e->s_pack})
        if (q)
            cudaStreamSynchronize(q);
    for (Dev* d : e->dev) {
        if (!d)
            continue;
        if (d->ring)
            cudaFreeHost(d->ring);
        cudaFree(d->d_buf[0]);
        cudaFree(d->d_buf[1]);
        cudaFree(d->d_picks);
        cudaFree(d->d_mags);
        cudaFree(d->d_bins);
        cudaFree(d->d_spectrum);
        delete d;
    }
    cudaFree(e->d_bank_chan);
    cudaFree(e->d_bank_state);
    cudaFree(e->d_mix_in);
    cudaFree(e->d_mixer);
    cudaFree(e->d_fifo);
    cudaFree(e->d_fifo_sig);
    for (Slot& s : e->slot) {
        cudaFree(s.d_mix);
        cudaFree(s.d_mix_sig);
        if (s.h_mix)
            cudaFreeHost(s.h_mix);
        if (s.h_mix_sig)
            cudaFreeHost(s.h_mix_sig);
        cudaFree(s.d_wave);
        cudaFree(s.d_pack);
        cudaFree(s.d_rowmap);
        cudaFree(s.d_rowcount);
        if (s.h_pack)
            cudaFreeHost(s.h_pack);
        if (s.h_rowmap)
            cudaFreeHost(s.h_rowmap);
        if (s.h_rowcount)
            cudaFreeHost(s.h_rowcount);
        if (s.h_packdev)
            cudaFreeHost(s.h_packdev);
        cudaFree(s.d_iq);
        cudaFree(s.d_trace);
        cudaFree(s.d_status);
        cudaFree(s.d_desc);
        if (s.h_wave)
            cudaFreeHost(s.h_wave);
        if (s.h_iq)
            cudaFreeHost(s.h_iq);
        if (s.h_trace)
            cudaFreeHost(s.h_trace);
        if (s.h_status)
            cudaFreeHost(s.h_status);
        if (s.h_desc)
            cudaFreeHost(s.h_desc);
        if (s.h_carry)
            cudaFreeHost(s.h_carry);
        if (s.ev_in2)
            cudaEventDestroy(s.ev_in2);
        if (s.ev_ring)
            cudaEventDestroy(s.ev_ring);
        if (s.ev_begin)
            cudaEventDestroy(s.ev_begin);
        if (s.ev_done)
            cudaEventDestroy(s.ev_done);
        if (s.ev_in)
            cudaEventDestroy(s.ev_in);
        if (s.ev_kdone)
            cudaEventDestroy(s.ev_kdone);
        if (s.ev_k1)
            cudaEventDestroy(s.ev_k1);
        if (s.ev_out0)
            cudaEventDestroy(s.ev_out0);
        for (cudaEvent_t ev : s.ev_k)
            cudaEventDestroy(ev);
    }
    for (cudaEvent_t ev : e->marks)
        if (ev)
            cudaEventDestroy(ev);
    cudaFree(e->d_window);
    cudaFree(e->d_twiddle);
    cudaFree(e->d_sincos);
    cudaFree(e->d_chan);
    cudaFree(e->d_state);
    cudaFree(e->d_ctcss);
    cudaFree(e->d_order);
    cudaFree(e->d_tile_counter);
    for (cudaStream_t q : {e->s_in, e->s_in2, e->s_k, e->s_k2, e->s_k2b, e->s_out, e->s_pack})
        if (q)
            cudaStreamDestroy(q);
    for (cudaEvent_t ev : {e->ev_tmp[0], e->ev_tmp[1], e->ev_fork, e->ev_join})
        if (ev)
            cudaEventDestroy(ev);
    delete e;
}

/* A member's error that may have left it out of step with the others (a CUDA failure, a half-made pass) ends the group's
 * useful life; refusals (bad arguments, a full ring, a call out of sequence) change nothing and are just returned. */
int group_rc(ba_engine* g, int rc) {
    if (rc == BA_ERR_CUDA || rc == BA_ERR_NOMEM)
        g->broken = true;
    return rc;
}

int group_broken() {
    return fail(BA_ERR_STATE, "a member of this multi-GPU engine failed; the handle is only good for ba_cuda_destroy()");
}

/* Runs f on every member of a group in member order; stops at the first error. */
template <class F>
int each_member(ba_engine* g, F f) {
    if (g->broken)
        return group_broken();
    for (ba_engine* m : g->members) {
        const int rc = group_rc(g, f(m));
        if (rc < 0)
            return rc;
    }
    return BA_OK;
}

/* For the per-ticket timings that come in pairs: each element is the maximum over the members. */
int max_pair_over_members(ba_engine* g, int ticket, float ms[2], int (*get)(ba_engine*, int, float*)) {
    if (!ms)
        return fail(BA_ERR_BAD_ARG, "null argument");
    ms[0] = ms[1] = 0.0f;
    return each_member(g, [&](ba_engine* m) {
        float v[2] = {0.0f, 0.0f};
        const int r = get(m, ticket, v);
        ms[0] = std::max(ms[0], v[0]);
        ms[1] = std::max(ms[1], v[1]);
        return r;
    });
}

/* frames the reference's availability test admits for a stream of `total` bytes (.cpp:418-424 with FFT_BATCH 1):
 * frame f runs while total - f*bps >= bps + fft_size*bytes_per_sample*2 */
uint64_t frames_admitted(const Dev& d, uint64_t total) {
    const uint64_t need = d.hop_bytes + d.frame_bytes;
    if (total < need)
        return 0;
    return (total - need) / d.hop_bytes + 1;
}

/* fills K2Chan constants + initial K2State of one channel; mirrors parse_channels (config.cpp:312-729) */
/* the channel descriptor one entry of the frequency list amounts to */
ba_channel_desc with_freq(const ba_channel_desc& c, const ba_freq_desc& f) {
    ba_channel_desc r = c;
    r.frequency = f.frequency;
    r.modulation = f.modulation;
    r.ampfactor = f.ampfactor;
    r.squelch_threshold_dbfs = f.squelch_threshold_dbfs;
    r.squelch_snr_threshold = f.squelch_snr_threshold;
    r.notch = f.notch;
    r.notch_q = f.notch_q;
    r.ctcss = f.ctcss;
    r.bandwidth = f.bandwidth;
    return r;
}

/* cd: the channel with the fields of ONE frequency; frequency0 / needs_raw_iq: what the channel as a whole derives from
 * freqlist[0] (bin, dm_dphi: config.cpp:669,684) and from all its frequencies (needs_raw_iq: config.cpp:162,596,674-680) */
int setup_channel(ba_engine* e, Dev& d, int ci, const ba_channel_desc& cd, int frequency0, int needs_raw_iq, ba::K2Chan& k, ba::K2State& st, ba::K2Ctcss* ctcss_pool,
                  int& n_ctcss, ba_channel_info& in) {
    using namespace ba;
    const int R = e->wave_rate, N = e->fft_size;
    memset(&k, 0, sizeof(k));
    memset(&st, 0, sizeof(st));
    memset(&in, 0, sizeof(in));
    if (cd.modulation != BA_MOD_AM && cd.modulation != BA_MOD_NFM)
        return fail(BA_ERR_BAD_ARG, "channel %d: unknown modulation %d", ci, cd.modulation);
    k.col = (uint32_t)ci;
    k.picks = d.d_picks ? d.d_picks + (size_t)ci * d.ring_len : nullptr;
    k.mags = d.d_mags + (size_t)ci * d.ring_len;
    k.ring_mask = d.ring_len - 1;
    k.bin = d.d_bins + ci;
    k.fft_size = N;
    k.modulation = cd.modulation;
    k.afc = cd.afc & 0xff;
    k.has_iq_outputs = cd.has_iq_outputs ? 1 : 0;
    k.needs_raw_iq = needs_raw_iq;
    k.fm_demod = e->fm_demod;
    k.ampfactor = cd.ampfactor;
    float alpha = model::alpha_default(R);
    if (d.cfg.tau_us >= 0)
        alpha = model::alpha_from_tau_us(R, d.cfg.tau_us);
    if (cd.tau_us >= 0)
        alpha = model::alpha_from_tau_us(R, cd.tau_us);
    k.alpha = alpha;
    /* Squelch defaults (squelch.cpp:36-70), then the settings in the order parse_channels applies them (config.cpp:437-515) */
    k.manual = 0;
    k.manual_level = -1.0f;
    k.ratio = model::snr_ratio(9.54f);
    if (cd.squelch_threshold_dbfs < 0) {
        const float level = model::dbfs_to_level((float)cd.squelch_threshold_dbfs, N);
        if (level > 0) {
            k.manual = 1;
            k.manual_level = level;
        }
    }
    if (cd.squelch_snr_threshold >= 0) {
        k.manual = 0;
        k.ratio = model::snr_ratio(cd.squelch_snr_threshold);
    }
    k.flappy_ratio = k.ratio * 0.9f;
    if (cd.notch > 0) {
        float dd[3];
        const float q = cd.notch_q == 0.0f ? 10.0f : cd.notch_q;
        if (model::notch_design(cd.notch, (float)R, q, dd)) {
            k.notch_on = 1;
            k.nd0 = dd[0], k.nd1 = dd[1], k.nd2 = dd[2];
        }
    }
    if (cd.bandwidth > 0) {
        float yc[2], gain;
        if (model::lowpass_design((float)cd.bandwidth / 2, (float)R, yc, &gain)) {
            k.lp_on = 1;
            k.lp_c0 = yc[0], k.lp_c1 = yc[1], k.lp_gain = gain;
        }
    }
    k.base_bin = model::bin_index(frequency0, d.cfg.sample_rate, d.cfg.centerfreq, N);
    d.base_bins[ci] = k.base_bin;
    if (k.needs_raw_iq)
        k.dm_dphi = model::derotation_step(frequency0, d.cfg.centerfreq, d.cfg.sample_rate, R);
    if (cd.ctcss > 0) { /* Squelch::set_ctcss_freq, squelch.cpp:106-116 */
        K2Ctcss& c = ctcss_pool[n_ctcss];
        memset(&c, 0, sizeof(c));
        c.win_fast = (int)((float)R * 0.05);
        c.win_slow = (int)((float)R * 0.4);
        c.n_fast = model::tone_bank(cd.ctcss, (float)R, c.win_fast, c.coeff_fast);
        c.n_slow = model::tone_bank(cd.ctcss, (float)R, c.win_slow, c.coeff_slow);
        k.ctcss = e->d_ctcss + n_ctcss;
        n_ctcss++;
        in.ctcss_fast_tones = c.n_fast;
        in.ctcss_slow_tones = c.n_slow;
        in.ctcss_fast_window = c.win_fast;
        in.ctcss_slow_window = c.win_slow;
    }
    /* initial state: Squelch constructor (squelch.cpp:36-70), channel_t/freq_t defaults (config.cpp:276-286,319-334) */
    st.noise = 5.0f;
    st.pre_full = st.pre_cap = st.post_full = st.post_cap = 0.001f;
    st.next = st.cur = BA_SQ_CLOSED;
    st.count16 = 15; /* sample_count_ starts at (size_t)-1: the very first sample updates the noise floor */
    st.head = 0;
    st.tail = 1;
    st.prev_waveout = 0.5f;
    st.agcavgfast = 0.5f;
    st.axcindicate = BA_NO_SIGNAL;
    for (int i = 0; i < BA_E; i++)
        st.waveout_tail[i] = 0.5f;

    in.bin = k.base_bin;
    in.dm_dphi = k.dm_dphi;
    in.needs_raw_iq = k.needs_raw_iq;
    in.alpha = k.alpha;
    in.squelch_ratio = k.ratio;
    in.manual_level = k.manual ? k.manual_level : 0.0f;
    in.notch_enabled = k.notch_on;
    in.notch_d[0] = k.nd0, in.notch_d[1] = k.nd1, in.notch_d[2] = k.nd2;
    in.lowpass_enabled = k.lp_on;
    in.lowpass_ycoeffs[0] = k.lp_c0, in.lowpass_ycoeffs[1] = k.lp_c1;
    in.lowpass_gain = k.lp_gain;
    return BA_OK;
}

/* tile shape of K1 for this engine: as many frames per tile as fit the shared-memory budget, bounded so that
 * a step still spreads over the SMs */
int choose_tiles(ba_engine* e) {
    const int N = e->fft_size;
    size_t max_hop = 0, max_frame = 0;
    for (Dev* d : e->dev) {
        max_hop = std::max(max_hop, d->hop_bytes);
        max_frame = std::max(max_frame, d->frame_bytes);
    }
    const int groups = ba::k1_groups(N);
    const int fixed = ba::k1_smem_bytes(N, 0, e->max_channels);
    /* budget: under half an SM's shared memory so that two CTAs are resident (registers allow it) with room left for the
     * demodulator's warps; the byte span of a tile is double-buffered */
    /* experiment knobs (tuning runs only): resident channelizer CTAs per SM and frames per tile */
    e->k1_ctas_per_sm = ba::k1_ctas_per_sm(N);
    if (const char* v = getenv("BA_CUDA_K1_CTAS"))
        e->k1_ctas_per_sm = std::max(1, atoi(v));
    const int budget = std::min(e->smem_optin, (e->k1_ctas_per_sm > 2 ? 216 * 1024 / e->k1_ctas_per_sm : 96 * 1024));
    auto raw_of = [&](int tf) { return (((size_t)(tf - 1) * max_hop + max_frame + 32) + 15) & ~(size_t)15; };
    /* four rounds of FFT groups per tile; six when a full step still leaves every resident CTA sixteen tiles or more
     * (fewer tile hand-overs: 2 % on the 512-input workload), never so many that a small step no longer covers the SMs */
    int tf = 4 * groups;
    {
        const uint64_t frames_per_step = (uint64_t)e->dev.size() * e->max_batches * e->B;
        if (frames_per_step / (6 * (uint64_t)groups) >= 16ull * e->sm_count * e->k1_ctas_per_sm)
            tf = 6 * groups;
    }
    if (const char* v = getenv("BA_CUDA_K1_TILE"))
        tf = std::max(groups, atoi(v) / groups * groups);
    if (ba::k1_direct(N)) { /* frames are read straight from global memory: a tile only amortises the hand-over */
        e->tile_frames = getenv("BA_CUDA_K1_TILE") ? tf : 4;
        e->raw_bytes = 0;
        return BA_OK;
    }
    while (tf > groups && (size_t)fixed + 2 * raw_of(tf) > (size_t)budget)
        tf -= groups;
    while (tf > 1 && (size_t)fixed + 2 * raw_of(tf) > (size_t)e->smem_optin)
        tf--;
    if (tf > 1)
        tf &= ~1; /* tiles start on even frames of their launch (channelize.cu ties a rotation to the frame's parity) */
    const size_t raw = raw_of(tf);
    if ((size_t)fixed + 2 * raw > (size_t)e->smem_optin)
        return fail(BA_ERR_NOMEM, "K1 needs %zu bytes of shared memory per CTA, the device offers %d", (size_t)fixed + 2 * raw, e->smem_optin);
    e->tile_frames = tf;
    e->raw_bytes = (int)raw;
    return BA_OK;
}

}  // namespace

extern "C" {

const char* ba_cuda_last_error(void) {
    return g_err;
}

int ba_cuda_visible_devices(void) {
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess)
        return fail(BA_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(err));
    return n;
}

void ba_cuda_destroy(ba_engine* e) {
    free_engine(e);
}

int ba_cuda_create(const ba_engine_desc* desc, ba_engine** out) {
    using namespace ba;
    if (!desc || !out)
        return fail(BA_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    if (desc->abi_version != BA_CUDA_ABI_VERSION)
        return fail(BA_ERR_BAD_ARG, "ABI version %d, library speaks %d", desc->abi_version, BA_CUDA_ABI_VERSION);
    const int n_mixers = desc->mixer_count;
    if (n_mixers < 0 || (n_mixers > 0 && !desc->mixers))
        return fail(BA_ERR_BAD_ARG, "mixer_count %d without mixers", n_mixers);
    const int N = desc->fft_size;
    if (N < 256 || N > 8192 || (N & (N - 1)))
        return fail(BA_ERR_BAD_SIZE, "fft_size %d is not a power of two in 256..8192", N);
    if (desc->wave_rate <= 0 || desc->wave_rate % 32) /* WAVE_BATCH = wave_rate / 8 samples move in quads */
        return fail(BA_ERR_BAD_ARG, "wave_rate %d is not a positive multiple of 32", desc->wave_rate);
    if (desc->device_count <= 0 || !desc->devices)
        return fail(BA_ERR_BAD_ARG, "no devices");
    int visible = 0;
    cudaError_t ce = cudaGetDeviceCount(&visible);
    if (ce != cudaSuccess || visible <= 0)
        return fail(BA_ERR_NO_DEVICE, "no CUDA device (%s); this engine has no CPU path", ce != cudaSuccess ? cudaGetErrorString(ce) : "count 0");
    if (desc->cuda_device < 0 || desc->cuda_device >= visible)
        return fail(BA_ERR_NO_DEVICE, "cuda_device %d of %d", desc->cuda_device, visible);
    if (cudaSetDevice(desc->cuda_device) != cudaSuccess)
        return fail(BA_ERR_NO_DEVICE, "cudaSetDevice(%d) failed", desc->cuda_device);

    ba_engine* e = new (std::nothrow) ba_engine();
    if (!e)
        return fail(BA_ERR_NOMEM, "host allocation");
    struct Guard {
        ba_engine* e;
        ~Guard() {
            if (e)
                free_engine(e);
        }
    } guard{e};

    e->fft_size = N;
    e->wave_rate = desc->wave_rate;
    e->B = desc->wave_rate / 8;
    e->fm_demod = desc->fm_demod;
    e->cuda_device = desc->cuda_device;
    e->max_batches = desc->max_batches_per_step > 0 ? desc->max_batches_per_step : 8;
    e->flags = desc->flags;
    e->stride = e->max_batches * e->B + BA_E;
    CU(cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, desc->cuda_device));
    CU(cudaDeviceGetAttribute(&e->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, desc->cuda_device));
    CU(cudaStreamCreateWithFlags(&e->s_in, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->s_in2, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->s_k2b, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    if (const char* v = getenv("BA_CUDA_H2D_STREAMS"))
        e->h2d_streams = atoi(v) >= 2 ? 2 : 1;
    CU(cudaStreamCreateWithFlags(&e->s_k, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->s_k2, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->s_out, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->s_pack, cudaStreamNonBlocking));
    e->stream = e->s_k;
    CU(cudaEventCreateWithFlags(&e->ev_tmp[0], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_tmp[1], cudaEventDisableTiming));

    /* window, twiddles, sine/cosine table */
    e->window.resize(N);
    model::window7(N, e->window.data());
    std::vector<float2> tw(N);
    model::twiddles(N, tw.data());
    float sc[514];
    model::sincos_table(sc);
    CU(cudaMalloc((void**)&e->d_window, sizeof(float) * N));
    CU(cudaMalloc((void**)&e->d_twiddle, sizeof(float2) * N));
    CU(cudaMalloc((void**)&e->d_sincos, sizeof(sc)));
    CU(cudaMemcpy(e->d_window, e->window.data(), sizeof(float) * N, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_twiddle, tw.data(), sizeof(float2) * N, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_sincos, sc, sizeof(sc), cudaMemcpyHostToDevice));

    const size_t ring_min = desc->ring_bytes > 0 ? (size_t)desc->ring_bytes : (size_t)BA_MIN_BUF_SIZE;
    const uint64_t frames_cap = (uint64_t)(e->max_batches + 1) * e->B + BA_E;
    int n_ctcss = 0;
    for (int di = 0; di < desc->device_count; di++) {
        const ba_device_desc& dd = desc->devices[di];
        if (dd.channel_count <= 0 || !dd.channels)
            return fail(BA_ERR_BAD_ARG, "device %d has no channels", di);
        int want_bps = dd.sample_format == BA_SFMT_S16 ? 2 : (dd.sample_format == BA_SFMT_F32 ? 4 : 1);
        if (dd.sample_format < BA_SFMT_U8 || dd.sample_format > BA_SFMT_F32 || dd.bytes_per_sample != want_bps)
            return fail(BA_ERR_BAD_ARG, "device %d: sample format %d with %d bytes per sample", di, dd.sample_format, dd.bytes_per_sample);
        if (dd.sample_rate <= e->wave_rate || !(dd.fullscale > 0))
            return fail(BA_ERR_BAD_ARG, "device %d: sample_rate %d, fullscale %g", di, dd.sample_rate, (double)dd.fullscale);
        Dev* d = new (std::nothrow) Dev();
        if (!d)
            return fail(BA_ERR_NOMEM, "host allocation");
        e->dev.push_back(d);
        d->cfg = dd;
        d->chans.assign(dd.channels, dd.channels + dd.channel_count);
        d->cfg.channels = nullptr;
        for (ba_channel_desc& c : d->chans) { /* freqlist: named in scan mode, else the channel's own fields (mk_freqlist(1)) */
            if (c.freq_count < 0 || (c.freq_count > 0 && !c.freqs))
                return fail(BA_ERR_BAD_ARG, "device %d: freq_count %d without freqs", di, c.freq_count);
            if (c.freq_count > 0)
                d->freqs.emplace_back(c.freqs, c.freqs + c.freq_count);
            else
                d->freqs.emplace_back(1, ba_freq_desc{c.frequency, c.modulation, c.ampfactor, c.squelch_threshold_dbfs, c.squelch_snr_threshold, c.notch, c.notch_q, c.ctcss, c.bandwidth});
            c.freqs = nullptr;
        }
        d->freq_idx.assign(dd.channel_count, 0);
        d->bank0.assign(dd.channel_count, SIZE_MAX);
        d->C = dd.channel_count;
        d->c_pad = (d->C + 3) & ~3;
        d->sample_bytes = 2 * (size_t)dd.bytes_per_sample;
        d->hop_bytes = d->sample_bytes * (size_t)round((double)dd.sample_rate / (double)e->wave_rate); /* .cpp:418 */
        d->frame_bytes = d->sample_bytes * (size_t)N;
        d->first_chan = e->total_channels;
        e->total_channels += d->C;
        e->max_channels = std::max(e->max_channels, d->C);
        for (size_t ci = 0; ci < d->chans.size(); ci++) {
            const ba_channel_desc& c = d->chans[ci];
            if (c.afc & 0xff)
                d->any_afc = true;
            if (c.has_iq_outputs)
                d->any_iq = d->any_raw = true;
            for (const ba_freq_desc& f : d->freqs[ci]) {
                if (f.modulation == BA_MOD_NFM || f.bandwidth != 0) /* needs_raw_iq, config.cpp:162,596,674-680 */
                    d->any_raw = true;
                if (f.ctcss > 0)
                    n_ctcss++;
            }
        }
        e->any_afc |= d->any_afc;
        e->any_iq |= d->any_iq;
        /* host ring, config.cpp:796-805 */
        d->buf_size = model::ring_bytes(ring_min, dd.bytes_per_sample, dd.sample_rate, e->wave_rate);
        d->mirror = d->frame_bytes;
        if (cudaHostAlloc((void**)&d->ring, d->buf_size + d->mirror, cudaHostAllocDefault) != cudaSuccess)
            return fail(BA_ERR_NOMEM, "pinned ring of %zu bytes", d->buf_size + d->mirror);
        memset(d->ring, 0, d->buf_size + d->mirror);
        /* HBM: stream window (two halves), pick ring, bins */
        d->d_cap = (size_t)(frames_cap + 2) * d->hop_bytes + 2 * d->frame_bytes + 64;
        /* two tickets may be in flight on the pick ring: the demodulator of one reads behind the channelizer of the next */
        d->ring_len = pow2_at_least((uint64_t)(2 * e->max_batches + 1) * e->B + 2 * BA_E);
        /* picked-bin IQ is kept only where a demodulator reads it (or a test asked for it); magnitudes always */
        const bool keep_picks = d->any_raw || (e->flags & BA_FLAG_KEEP_PICKS);
        if (cudaMalloc((void**)&d->d_buf[0], d->d_cap) != cudaSuccess || cudaMalloc((void**)&d->d_buf[1], d->d_cap) != cudaSuccess ||
            (keep_picks && cudaMalloc((void**)&d->d_picks, sizeof(float2) * (size_t)d->ring_len * d->C) != cudaSuccess) ||
            cudaMalloc((void**)&d->d_mags, sizeof(float) * (size_t)d->ring_len * d->C) != cudaSuccess ||
            cudaMalloc((void**)&d->d_bins, sizeof(uint32_t) * d->c_pad) != cudaSuccess)
            return fail(BA_ERR_NOMEM, "device memory for input %d", di);
        if (d->d_picks)
            CU(cudaMemset(d->d_picks, 0, sizeof(float2) * (size_t)d->ring_len * d->C));
        CU(cudaMemset(d->d_mags, 0, sizeof(float) * (size_t)d->ring_len * d->C));
        if (d->any_afc) {
            if (cudaMalloc((void**)&d->d_spectrum, sizeof(float2) * N) != cudaSuccess)
                return fail(BA_ERR_NOMEM, "device memory for input %d", di);
            CU(cudaMemset(d->d_spectrum, 0, sizeof(float2) * N));
        }
        d->base_bins.resize(d->C);
    }
    if (e->any_afc)
        e->max_phases = e->max_batches + 1;
    e->serial_k2 = e->any_afc;

    /* per-channel constants and state */
    const int TC = e->total_channels;
    e->h_chan.resize(TC);
    e->info.resize(TC);
    std::vector<K2State> h_state(TC);
    std::vector<K2Ctcss> h_ctcss(std::max(1, n_ctcss));
    CU(cudaMalloc((void**)&e->d_chan, sizeof(K2Chan) * TC));
    CU(cudaMalloc((void**)&e->d_state, sizeof(K2State) * TC));
    CU(cudaMalloc((void**)&e->d_ctcss, sizeof(K2Ctcss) * std::max(1, n_ctcss)));
    CU(cudaMalloc((void**)&e->d_order, sizeof(int32_t) * TC));
    CU(cudaMalloc((void**)&e->d_tile_counter, sizeof(uint32_t)));
    int used_ctcss = 0;
    std::vector<K2Chan> bank_chan; /* scan channels: constants and initial state of every frequency, in list order */
    std::vector<K2State> bank_state;
    for (size_t di = 0; di < e->dev.size(); di++) {
        Dev& d = *e->dev[di];
        for (int ci = 0; ci < d.C; ci++) {
            const int gi = d.first_chan + ci;
            const std::vector<ba_freq_desc>& fl = d.freqs[ci];
            int raw = d.chans[ci].has_iq_outputs ? 1 : 0;
            for (const ba_freq_desc& f : fl)
                if (f.modulation == BA_MOD_NFM || f.bandwidth != 0)
                    raw = 1;
            int rc = setup_channel(e, d, ci, with_freq(d.chans[ci], fl[0]), fl[0].frequency, raw, e->h_chan[gi], h_state[gi], h_ctcss.data(), used_ctcss, e->info[gi]);
            if (rc != BA_OK)
                return rc;
            e->h_chan[gi].dev = (int32_t)di;
            if (fl.size() > 1) {
                d.bank0[ci] = bank_chan.size();
                bank_chan.push_back(e->h_chan[gi]);
                bank_state.push_back(h_state[gi]);
                for (size_t f = 1; f < fl.size(); f++) {
                    K2Chan k;
                    K2State st;
                    ba_channel_info unused;
                    rc = setup_channel(e, d, ci, with_freq(d.chans[ci], fl[f]), fl[0].frequency, raw, k, st, h_ctcss.data(), used_ctcss, unused);
                    if (rc != BA_OK)
                        return rc;
                    k.dev = (int32_t)di;
                    bank_chan.push_back(k);
                    bank_state.push_back(st);
                }
            }
        }
        std::vector<uint32_t> bins(d.c_pad, 0);
        std::copy(d.base_bins.begin(), d.base_bins.end(), bins.begin());
        CU(cudaMemcpy(d.d_bins, bins.data(), sizeof(uint32_t) * d.c_pad, cudaMemcpyHostToDevice));
    }
    /* launch order: group channels of one kind together (plain AM, other AM, filtered/NFM, CTCSS) so that the lanes of a warp
     * run the same code; plain AM channels come first and go to their own kernel */
    {
        std::vector<int32_t> order(TC);
        for (int i = 0; i < TC; i++)
            order[i] = i;
        auto plain = [&](int i) {
            const K2Chan& k = e->h_chan[i];
            const Dev& dv = *e->dev[k.dev];
            if (dv.freqs[k.col].size() > 1) /* a scan channel changes kind with its frequency: the general kernel reads the options at run time */
                return false;
            return k.modulation == BA_MOD_AM && !k.needs_raw_iq && !k.notch_on && !k.ctcss && !k.has_iq_outputs && !k.afc && !(e->flags & BA_FLAG_TRACE);
        };
        auto kind = [&](int i) {
            const K2Chan& k = e->h_chan[i];
            return (plain(i) ? 0 : 1) + (k.ctcss ? 8 : 0) + (k.modulation == BA_MOD_NFM ? 4 : 0) + (k.needs_raw_iq ? 2 : 0);
        };
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return kind(a) < kind(b); });
        e->n_plain = 0;
        for (int i = 0; i < TC; i++)
            e->n_plain += plain(i) ? 1 : 0;
        CU(cudaMemcpy(e->d_order, order.data(), sizeof(int32_t) * TC, cudaMemcpyHostToDevice));
    }
    CU(cudaMemcpy(e->d_chan, e->h_chan.data(), sizeof(K2Chan) * TC, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_state, h_state.data(), sizeof(K2State) * TC, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_ctcss, h_ctcss.data(), sizeof(K2Ctcss) * std::max(1, n_ctcss), cudaMemcpyHostToDevice));
    if (!bank_chan.empty()) {
        CU(cudaMalloc((void**)&e->d_bank_chan, sizeof(K2Chan) * bank_chan.size()));
        CU(cudaMalloc((void**)&e->d_bank_state, sizeof(K2State) * bank_state.size()));
        CU(cudaMemcpy(e->d_bank_chan, bank_chan.data(), sizeof(K2Chan) * bank_chan.size(), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(e->d_bank_state, bank_state.data(), sizeof(K2State) * bank_state.size(), cudaMemcpyHostToDevice));
    }

    /* output arenas, one per slot */
    {
        size_t wave = 0, status = 0;
        for (Dev* d : e->dev) {
            d->wave_off = wave;
            d->iq_off = wave;
            d->status_off = status;
            wave += (size_t)d->C * e->stride;
            status += (size_t)d->C * e->max_batches;
        }
        const size_t nd = e->dev.size();
        e->desc_bytes = (size_t)e->max_phases * nd * (sizeof(K1Device) + sizeof(K2Dyn));
        /* mixers: inputs connect in descriptor order (mixer_connect_input, mixer.cpp:55-93) */
        for (int m = 0; m < n_mixers; m++) {
            const ba_mixer_desc& md = desc->mixers[m];
            if (md.input_count < 0 || (md.input_count > 0 && !md.inputs))
                return fail(BA_ERR_BAD_ARG, "mixer %d: bad input list", m);
            Mixer mx;
            mx.first_in = (int)e->mix_in.size();
            mx.n_in = md.input_count;
            for (int j = 0; j < md.input_count; j++) {
                const ba_mixer_input_desc& in = md.inputs[j];
                if (in.device < 0 || in.device >= (int)nd || in.channel < 0 || in.channel >= e->dev[in.device]->C)
                    return fail(BA_ERR_BAD_ARG, "mixer %d input %d: no channel %d on device %d", m, j, in.channel, in.device);
                if (!(in.balance >= -1.0f && in.balance <= 1.0f)) /* config.cpp:183-186 */
                    return fail(BA_ERR_BAD_ARG, "mixer %d input %d: balance out of allowed range <-1.0;1.0>", m, j);
                MixInput mi;
                mi.dev = in.device;
                mi.ch = in.channel;
                mi.mult_l = in.ampfactor * fminf(1.0f, 1.0f - in.balance); /* ampfactor * ampl, mixer.cpp:79-80,195 */
                mi.mult_r = in.ampfactor * fminf(1.0f, 1.0f + in.balance);
                if (in.balance != 0.0f)
                    mx.stereo = true; /* MM_STEREO, mixer.cpp:82-83 */
                e->dev[in.device]->feeds.push_back((int)e->mix_in.size());
                e->mix_in.push_back(mi);
            }
            e->mixers.push_back(mx);
        }
        if (n_mixers > 0) {
            e->fifo_depth = 2 * e->max_batches;
            for (Mixer& mx : e->mixers) {
                mx.out_off = e->mix_floats;
                e->mix_floats += (size_t)(mx.stereo ? 2 : 1) * e->max_batches * e->B;
            }
            const size_t ni = std::max<size_t>(1, e->mix_in.size());
            std::vector<K3In> h_in(ni);
            std::vector<K3Mixer> h_mx(n_mixers);
            for (size_t i = 0; i < e->mix_in.size(); i++)
                h_in[i] = K3In{e->mix_in[i].mult_l, e->mix_in[i].mult_r};
            for (int m = 0; m < n_mixers; m++)
                h_mx[m] = K3Mixer{e->mixers[m].first_in, e->mixers[m].n_in, e->mixers[m].stereo ? 1 : 0, 0};
            if (cudaMalloc((void**)&e->d_mix_in, sizeof(K3In) * ni) != cudaSuccess || cudaMalloc((void**)&e->d_mixer, sizeof(K3Mixer) * n_mixers) != cudaSuccess ||
                cudaMalloc((void**)&e->d_fifo, sizeof(float) * ni * e->fifo_depth * e->B) != cudaSuccess || cudaMalloc((void**)&e->d_fifo_sig, ni * e->fifo_depth) != cudaSuccess)
                return fail(BA_ERR_NOMEM, "mixer FIFOs for %zu inputs", ni);
            CU(cudaMemcpy(e->d_mix_in, h_in.data(), sizeof(K3In) * ni, cudaMemcpyHostToDevice));
            CU(cudaMemcpy(e->d_mixer, h_mx.data(), sizeof(K3Mixer) * n_mixers, cudaMemcpyHostToDevice));
            CU(cudaMemset(e->d_fifo, 0, sizeof(float) * ni * e->fifo_depth * e->B));
            CU(cudaMemset(e->d_fifo_sig, 0, ni * e->fifo_depth));
            e->mix_desc_off = (e->desc_bytes + 15) & ~(size_t)15;
            e->desc_bytes = e->mix_desc_off + sizeof(K3InDyn) * ni + sizeof(K3MixDyn) * n_mixers;
        }
        for (Slot& s : e->slot) {
            if (n_mixers > 0) {
                if (cudaMalloc((void**)&s.d_mix, sizeof(float) * e->mix_floats) != cudaSuccess || cudaHostAlloc((void**)&s.h_mix, sizeof(float) * e->mix_floats, cudaHostAllocDefault) != cudaSuccess ||
                    cudaMalloc((void**)&s.d_mix_sig, sizeof(int32_t) * n_mixers * e->max_batches) != cudaSuccess ||
                    cudaHostAlloc((void**)&s.h_mix_sig, sizeof(int32_t) * n_mixers * e->max_batches, cudaHostAllocDefault) != cudaSuccess)
                    return fail(BA_ERR_NOMEM, "mixer output arena");
                s.mix_emit.assign(n_mixers, 0);
                s.mix_first.assign(n_mixers, 0);
            }
            if (cudaMalloc((void**)&s.d_wave, sizeof(float) * wave) != cudaSuccess || cudaHostAlloc((void**)&s.h_wave, sizeof(float) * wave, cudaHostAllocDefault) != cudaSuccess ||
                cudaMalloc((void**)&s.d_status, sizeof(ba_channel_status) * status) != cudaSuccess ||
                cudaHostAlloc((void**)&s.h_status, sizeof(ba_channel_status) * status, cudaHostAllocDefault) != cudaSuccess ||
                cudaMalloc((void**)&s.d_desc, e->desc_bytes) != cudaSuccess || cudaHostAlloc((void**)&s.h_desc, e->desc_bytes, cudaHostAllocDefault) != cudaSuccess)
                return fail(BA_ERR_NOMEM, "output arena of %zu floats", wave);
            CU(cudaMemset(s.d_wave, 0, sizeof(float) * wave));
            memset(s.h_wave, 0, sizeof(float) * wave);
            if (e->flags & BA_FLAG_SKIP_SILENT_ROWS) {
                const size_t rows = (size_t)e->total_channels * e->max_batches;
                if (cudaMalloc((void**)&s.d_pack, sizeof(float) * rows * e->B) != cudaSuccess || cudaHostAlloc((void**)&s.h_pack, sizeof(float) * rows * e->B, cudaHostAllocDefault) != cudaSuccess ||
                    cudaMalloc((void**)&s.d_rowmap, sizeof(int32_t) * rows) != cudaSuccess || cudaHostAlloc((void**)&s.h_rowmap, sizeof(int32_t) * rows, cudaHostAllocDefault) != cudaSuccess ||
                    cudaMalloc((void**)&s.d_rowcount, sizeof(uint32_t)) != cudaSuccess || cudaHostAlloc((void**)&s.h_rowcount, sizeof(uint32_t), cudaHostAllocDefault) != cudaSuccess ||
                    cudaHostAlloc((void**)&s.h_packdev, sizeof(ba::K3PackDev) * e->dev.size(), cudaHostAllocDefault) != cudaSuccess)
                    return fail(BA_ERR_NOMEM, "packed-row arena");
                memset(s.h_rowmap, 0xff, sizeof(int32_t) * rows);
            }
            if (e->any_iq) {
                if (cudaMalloc((void**)&s.d_iq, sizeof(float2) * wave) != cudaSuccess || cudaHostAlloc((void**)&s.h_iq, sizeof(float2) * wave, cudaHostAllocDefault) != cudaSuccess)
                    return fail(BA_ERR_NOMEM, "iq_out arena");
                CU(cudaMemset(s.d_iq, 0, sizeof(float2) * wave));
            }
            if (e->flags & BA_FLAG_TRACE) {
                if (cudaMalloc((void**)&s.d_trace, wave) != cudaSuccess || cudaHostAlloc((void**)&s.h_trace, wave, cudaHostAllocDefault) != cudaSuccess)
                    return fail(BA_ERR_NOMEM, "trace arena");
                CU(cudaMemset(s.d_trace, 0, wave));
            }
            CU(cudaEventCreate(&s.ev_begin));
            CU(cudaEventCreate(&s.ev_done));
            CU(cudaEventCreate(&s.ev_in));
            CU(cudaEventCreate(&s.ev_kdone));
            CU(cudaEventCreate(&s.ev_out0));
            CU(cudaEventCreateWithFlags(&s.ev_in2, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&s.ev_ring, cudaEventDisableTiming));
            s.ring_taken.assign(nd, 0);
            if (cudaHostAlloc((void**)&s.h_carry, sizeof(ba::K1Carry) * std::max<size_t>(1, nd), cudaHostAllocDefault) != cudaSuccess)
                return fail(BA_ERR_NOMEM, "pinned carry list");
            CU(cudaEventCreateWithFlags(&s.ev_k1, cudaEventDisableTiming));
            s.ev_k.resize(4 * (size_t)e->max_phases);
            for (cudaEvent_t& ev : s.ev_k)
                CU(cudaEventCreate(&ev));
            s.n_batches.assign(nd, 0);
            s.frames_done.assign(nd, 0);
        }
    }
    int rc = choose_tiles(e);
    if (rc != BA_OK)
        return rc;
    /* kernel attributes are per device: set them for this engine's GPU (the current device since cudaSetDevice above) */
    {
        int ke = k1_configure(N, e->raw_bytes, e->max_channels);
        if (ke == 0)
            ke = k2_configure();
        if (ke != 0)
            return fail(BA_ERR_CUDA, "kernel attributes on device %d: %s", e->cuda_device, cudaGetErrorString((cudaError_t)ke));
    }
    /* The demodulator of ticket t may run beside the channelizer of ticket t+1 (two streams) or behind it (one stream).  A
     * channelizer that fills every SM for milliseconds stretches the plain demodulator's serial chain beside it fourfold
     * (measured: 0.87 ms alone, 1.1-4.2 ms beside K1), and the device->host copy of ticket t waits for that; with nothing but
     * plain channels and a large step, one stream is faster (cfg5: 4.91 vs 5.07 ms per step at fft 512, 7.41 vs 7.71 at
     * 1024).  Small steps and the long general demodulator keep the two streams (cfg3: 0.90 vs 0.96, cfg2 x 64: 8.56 vs 8.79). */
    {
        const uint64_t frames_per_step = (uint64_t)e->dev.size() * e->max_batches * e->B;
        const bool big_step = frames_per_step / (uint64_t)std::max(1, e->tile_frames) >= 16ull * e->sm_count * e->k1_ctas_per_sm;
        if (e->n_plain == e->total_channels && big_step && !(e->flags & BA_FLAG_RESULTS_ON_DEVICE)) /* with no copy waiting for K2, beside K1 is the shorter schedule */
            e->serial_k2 = true;
        if (const char* v = getenv("BA_CUDA_SERIAL_K2")) /* tuning runs only: 0 / 1 overrides the rule (AFC always serialises) */
            e->serial_k2 = e->any_afc || atoi(v) != 0;
    }
    CU(cudaStreamSynchronize(e->stream));
    guard.e = nullptr;
    *out = e;
    return BA_OK;
}

int ba_cuda_create_multi(const ba_engine_desc* desc, const int32_t* gpus, int32_t n_gpus, const int32_t* gpu_of_device, ba_engine** out) {
    if (!desc || !out || !gpus)
        return fail(BA_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    if (n_gpus < 1)
        return fail(BA_ERR_BAD_ARG, "n_gpus %d: a multi-GPU engine needs at least one GPU", n_gpus);
    const int nd = desc->device_count, n_mixers = desc->mixer_count;
    if (nd <= 0 || !desc->devices)
        return fail(BA_ERR_BAD_ARG, "no devices");
    if (n_mixers < 0 || (n_mixers > 0 && !desc->mixers))
        return fail(BA_ERR_BAD_ARG, "mixer_count %d without mixers", n_mixers);
    int visible = 0;
    cudaError_t ce = cudaGetDeviceCount(&visible);
    if (ce != cudaSuccess || visible <= 0)
        return fail(BA_ERR_NO_DEVICE, "no CUDA device (%s); this engine has no CPU path", ce != cudaSuccess ? cudaGetErrorString(ce) : "count 0");
    for (int k = 0; k < n_gpus; k++)
        if (gpus[k] < 0 || gpus[k] >= visible)
            return fail(BA_ERR_BAD_ARG, "gpus[%d] = %d is not a visible CUDA device (%d visible)", k, gpus[k], visible);
    for (int m = 0; m < n_mixers; m++) {
        const ba_mixer_desc& md = desc->mixers[m];
        if (md.input_count < 0 || (md.input_count > 0 && !md.inputs))
            return fail(BA_ERR_BAD_ARG, "mixer %d: bad input list", m);
        for (int j = 0; j < md.input_count; j++)
            if (md.inputs[j].device < 0 || md.inputs[j].device >= nd)
                return fail(BA_ERR_BAD_ARG, "mixer %d input %d: no device %d", m, j, md.inputs[j].device);
    }
    /* which entry of gpus every device goes to */
    std::vector<int> where(nd);
    if (gpu_of_device) {
        for (int d = 0; d < nd; d++) {
            if (gpu_of_device[d] < 0 || gpu_of_device[d] >= n_gpus)
                return fail(BA_ERR_BAD_ARG, "gpu_of_device[%d] = %d is not an index into the %d gpus", d, gpu_of_device[d], n_gpus);
            where[d] = gpu_of_device[d];
        }
        for (int m = 0; m < n_mixers; m++) {
            const ba_mixer_desc& md = desc->mixers[m];
            for (int j = 1; j < md.input_count; j++)
                if (where[md.inputs[j].device] != where[md.inputs[0].device])
                    return fail(BA_ERR_BAD_ARG, "mixer %d has inputs on gpus[%d] and gpus[%d]; a mixer's inputs must share one GPU", m,
                                where[md.inputs[0].device], where[md.inputs[j].device]);
        }
    } else {
        /* devices joined by a mixer form one group (union-find, each set rooted at its first device); groups are dealt out
         * round robin in the order of their first device */
        std::vector<int> root(nd);
        for (int d = 0; d < nd; d++)
            root[d] = d;
        auto find = [&](int d) {
            while (root[d] != d)
                d = root[d] = root[root[d]];
            return d;
        };
        for (int m = 0; m < n_mixers; m++) {
            const ba_mixer_desc& md = desc->mixers[m];
            for (int j = 1; j < md.input_count; j++) {
                const int a = find(md.inputs[0].device), b = find(md.inputs[j].device);
                root[std::max(a, b)] = std::min(a, b);
            }
        }
        std::vector<int> group_of_root(nd, -1);
        int groups = 0;
        for (int d = 0; d < nd; d++) {
            const int r = find(d);
            if (group_of_root[r] < 0)
                group_of_root[r] = groups++;
            where[d] = group_of_root[r] % n_gpus;
        }
    }

    ba_engine* g = new (std::nothrow) ba_engine();
    if (!g)
        return fail(BA_ERR_NOMEM, "host allocation");
    g->dev_member.assign(nd, -1);
    g->dev_local.assign(nd, -1);
    g->mix_member.assign(n_mixers, -1);
    g->mix_local.assign(n_mixers, -1);
    /* one member per entry of gpus that received devices, in the order of gpus; a mixer without inputs goes with device 0 */
    for (int k = 0; k < n_gpus; k++) {
        std::vector<ba_device_desc> devs;
        for (int d = 0; d < nd; d++)
            if (where[d] == k) {
                g->dev_member[d] = (int)g->members.size();
                g->dev_local[d] = (int)devs.size();
                devs.push_back(desc->devices[d]);
            }
        if (devs.empty())
            continue;
        std::vector<ba_mixer_desc> mixers;
        std::vector<std::vector<ba_mixer_input_desc>> inputs;
        for (int m = 0; m < n_mixers; m++) {
            const ba_mixer_desc& md = desc->mixers[m];
            if ((md.input_count > 0 ? where[md.inputs[0].device] : where[0]) != k)
                continue;
            g->mix_member[m] = (int)g->members.size();
            g->mix_local[m] = (int)mixers.size();
            inputs.emplace_back(md.inputs, md.inputs + md.input_count);
            for (ba_mixer_input_desc& in : inputs.back())
                in.device = g->dev_local[in.device];
            mixers.push_back(ba_mixer_desc{md.input_count, nullptr});
        }
        for (size_t m = 0; m < mixers.size(); m++)
            mixers[m].inputs = inputs[m].data();
        ba_engine_desc sub = *desc;
        sub.cuda_device = gpus[k];
        sub.device_count = (int32_t)devs.size();
        sub.devices = devs.data();
        sub.mixer_count = (int32_t)mixers.size();
        sub.mixers = mixers.empty() ? nullptr : mixers.data();
        ba_engine* m = nullptr;
        const int rc = ba_cuda_create(&sub, &m);
        if (rc != BA_OK) {
            for (ba_engine* x : g->members)
                free_engine(x);
            delete g;
            return rc;
        }
        g->members.push_back(m);
    }
    *out = g;
    return BA_OK;
}

int ba_cuda_device_gpu(ba_engine* e, int dev, int32_t* cuda_ordinal) {
    if (!cuda_ordinal)
        return fail(BA_ERR_BAD_ARG, "null argument");
    FORWARD_DEV(e, dev, ba_cuda_device_gpu(e, dev, cuda_ordinal));
    if (!e || dev < 0 || dev >= (int)e->dev.size())
        return fail(BA_ERR_BAD_ARG, "bad engine or device index %d", dev);
    *cuda_ordinal = e->cuda_device;
    return BA_OK;
}

static Dev* get_dev(ba_engine* e, int dev) {
    if (!e || dev < 0 || dev >= (int)e->dev.size()) {
        fail(BA_ERR_BAD_ARG, "bad engine or device index %d", dev);
        return nullptr;
    }
    return e->dev[dev];
}

int ba_cuda_input_ring(ba_engine* e, int dev, unsigned char** buffer, size_t* buf_size, size_t* mirror_bytes) {
    FORWARD_DEV(e, dev, ba_cuda_input_ring(e, dev, buffer, buf_size, mirror_bytes));
    Dev* d = get_dev(e, dev);
    if (!d)
        return BA_ERR_BAD_ARG;
    if (buffer)
        *buffer = d->ring;
    if (buf_size)
        *buf_size = d->buf_size;
    if (mirror_bytes)
        *mirror_bytes = d->mirror;
    return BA_OK;
}

/* bytes the producer may not overwrite yet, as demodulate() computes `available` (.cpp:394-399): from bufs to bufe */
static size_t ring_available(const Dev& d) {
    return d.bufe >= d.bufs ? d.bufe - d.bufs : d.buf_size - d.bufs + d.bufe;
}
/* bytes the engine has not queued for copying yet: from its read position to bufe */
static size_t ring_unread(const Dev& d) {
    return d.bufe >= d.rpos ? d.bufe - d.rpos : d.buf_size - d.rpos + d.bufe;
}

/* bufs = (bufs + bps) % buf_size (.cpp:735), deferred: the copy engine reads the pinned ring asynchronously, so the bytes of a
 * ticket go back to the producer only once the event behind its copies has fired.  Called (without blocking) from every entry
 * point a producer or the demodulator thread passes through; `wait` blocks for the oldest pending ticket (a producer that
 * found the ring full). */
static void release_rings(ba_engine* e, bool wait) {
    std::lock_guard<std::mutex> q(e->rel_lock); /* producers and the demodulator thread both come through here */
    while (!e->rel.empty()) {
        RingRelease& r = e->rel.front();
        if (wait) {
            if (cudaEventSynchronize(r.ev) != cudaSuccess)
                return;
            wait = false;
        } else if (cudaEventQuery(r.ev) != cudaSuccess) {
            return; /* copies complete in the order they were queued: nothing behind this one is done either */
        }
        for (size_t di = 0; di < e->dev.size(); di++)
            if (r.taken[di]) {
                Dev& d = *e->dev[di];
                std::lock_guard<std::mutex> g(d.lock);
                d.bufs = (d.bufs + r.taken[di]) % d.buf_size;
            }
        e->rel.pop_front();
    }
}
static bool ring_release_pending(ba_engine* e, cudaEvent_t ev) {
    std::lock_guard<std::mutex> q(e->rel_lock);
    for (const RingRelease& r : e->rel)
        if (r.ev == ev)
            return true;
    return false;
}

int ba_cuda_submit(ba_engine* e, int dev, const void* iq, size_t len) {
    FORWARD_DEV(e, dev, ba_cuda_submit(e, dev, iq, len));
    Dev* d = get_dev(e, dev);
    if (!d || (!iq && len))
        return fail(BA_ERR_BAD_ARG, "bad argument");
    if (len == 0)
        return BA_OK;
    if (d->attached)
        return fail(BA_ERR_STATE, "input %d reads a device-resident stream", dev);
    release_rings(e, false);
    std::lock_guard<std::mutex> g(d->lock);
    if (!d->ext.empty())
        return fail(BA_ERR_STATE, "input %d: external chunks pending; do not mix ring and external submissions within a step", dev);
    /* unlike circbuffer_append (which overwrites unread data and counts an overflow) the caller is told */
    if (len >= d->buf_size - ring_available(*d)) {
        d->overflow_count++;
        return fail(BA_ERR_OVERRUN, "input %d: ring full (%zu bytes waiting, %zu offered)", dev, ring_available(*d), len);
    }
    const unsigned char* buf = (const unsigned char*)iq;
    const size_t space_left = d->buf_size - d->bufe;
    if (space_left >= len) {
        memcpy(d->ring + d->bufe, buf, len);
        if (d->bufe == 0)
            memcpy(d->ring + d->buf_size, d->ring, std::min(len, d->mirror));
    } else {
        memcpy(d->ring + d->bufe, buf, space_left);
        memcpy(d->ring, buf + space_left, len - space_left);
        memcpy(d->ring + d->buf_size, d->ring, std::min(len - space_left, d->mirror));
    }
    d->bufe = (d->bufe + len) % d->buf_size;
    return BA_OK;
}

int ba_cuda_input_space(ba_engine* e, int dev, size_t* free_bytes) {
    FORWARD_DEV(e, dev, ba_cuda_input_space(e, dev, free_bytes));
    Dev* d = get_dev(e, dev);
    if (!d || !free_bytes)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    release_rings(e, false);
    std::lock_guard<std::mutex> g(d->lock);
    /* what ba_cuda_submit() accepts right now: one byte less than the unread gap (bufe may not catch up with bufs) */
    const size_t gap = d->buf_size - ring_available(*d);
    *free_bytes = gap > 0 ? gap - 1 : 0;
    return BA_OK;
}

int ba_cuda_commit(ba_engine* e, int dev, size_t len) {
    FORWARD_DEV(e, dev, ba_cuda_commit(e, dev, len));
    Dev* d = get_dev(e, dev);
    if (!d)
        return BA_ERR_BAD_ARG;
    if (d->attached)
        return fail(BA_ERR_STATE, "input %d reads a device-resident stream", dev);
    release_rings(e, false);
    std::lock_guard<std::mutex> g(d->lock);
    if (!d->ext.empty())
        return fail(BA_ERR_STATE, "input %d: external chunks pending; do not mix ring and external submissions within a step", dev);
    if (len >= d->buf_size - ring_available(*d)) {
        d->overflow_count++;
        return fail(BA_ERR_OVERRUN, "input %d: ring full", dev);
    }
    d->bufe = (d->bufe + len) % d->buf_size;
    return BA_OK;
}

int ba_cuda_input_consumed(ba_engine* e, int dev, size_t* bufs) {
    FORWARD_DEV(e, dev, ba_cuda_input_consumed(e, dev, bufs));
    Dev* d = get_dev(e, dev);
    if (!d || !bufs)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    release_rings(e, false);
    std::lock_guard<std::mutex> g(d->lock);
    *bufs = d->bufs;
    return BA_OK;
}

int ba_cuda_submit_external(ba_engine* e, int dev, const void* iq, size_t len) {
    FORWARD_DEV(e, dev, ba_cuda_submit_external(e, dev, iq, len));
    Dev* d = get_dev(e, dev);
    if (!d || (!iq && len))
        return fail(BA_ERR_BAD_ARG, "bad argument");
    if (d->attached)
        return fail(BA_ERR_STATE, "input %d reads a device-resident stream", dev);
    if (len == 0)
        return BA_OK;
    std::lock_guard<std::mutex> g(d->lock);
    if (ring_unread(*d))
        return fail(BA_ERR_STATE, "input %d: ring data pending; do not mix ring and external submissions within a step", dev);
    d->ext.push_back(ExtChunk{(const unsigned char*)iq, len});
    return BA_OK;
}

int ba_cuda_attach_device_stream(ba_engine* e, int dev, const void* d_iq, size_t capacity_bytes) {
    FORWARD_DEV(e, dev, ba_cuda_attach_device_stream(e, dev, d_iq, capacity_bytes));
    Dev* d = get_dev(e, dev);
    if (!d || !d_iq)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    if (reinterpret_cast<uintptr_t>(d_iq) & 15)
        return fail(BA_ERR_BAD_ARG, "input %d: a device-resident stream must start on a 16-byte boundary", dev);
    if (d->frames_done || d->have)
        return fail(BA_ERR_STATE, "input %d already consumed data", dev);
    d->attached = (const unsigned char*)d_iq;
    d->attached_cap = capacity_bytes;
    d->attached_valid = 0;
    return BA_OK;
}

int ba_cuda_advance_device_stream(ba_engine* e, int dev, size_t bytes) {
    FORWARD_DEV(e, dev, ba_cuda_advance_device_stream(e, dev, bytes));
    Dev* d = get_dev(e, dev);
    if (!d)
        return BA_ERR_BAD_ARG;
    if (!d->attached)
        return fail(BA_ERR_STATE, "input %d has no device-resident stream", dev);
    if (d->attached_valid + bytes > d->attached_cap)
        return fail(BA_ERR_BAD_ARG, "input %d: %zu + %zu bytes exceed the attached %zu", dev, d->attached_valid, bytes, d->attached_cap);
    d->attached_valid += bytes;
    return BA_OK;
}

/* frames this input may run in the coming step without overflowing its pick ring / output rows */
static uint64_t frame_room(const ba_engine* e, const Dev& d) {
    uint64_t batch_limit = d.batches_done + (uint64_t)e->max_batches;
    /* an input may run ahead of the slowest input of a mixer it feeds by what the mixer FIFO holds */
    for (int fi : d.feeds) {
        if (!e->mix_in[fi].enabled)
            continue;
        for (const Mixer& mx : e->mixers)
            if (fi >= mx.first_in && fi < mx.first_in + mx.n_in)
                batch_limit = std::min<uint64_t>(batch_limit, mx.emitted + (uint64_t)e->fifo_depth);
    }
    const uint64_t limit = batch_limit * e->B + BA_E + e->B - 1;
    return limit > d.frames_done ? limit - d.frames_done : 0;
}

int ba_cuda_process(ba_engine* e) {
    if (e && !e->members.empty()) { /* every member's pass; their tickets move in lockstep */
        int ticket = -1;
        const int rc = each_member(e, [&](ba_engine* m) {
            const int t = ba_cuda_process(m);
            if (t >= 0 && ticket >= 0 && t != ticket)
                return fail(BA_ERR_STATE, "member tickets %d and %d differ", ticket, t);
            ticket = t;
            return t;
        });
        if (rc < 0)
            e->broken = true;
        return rc < 0 ? rc : ticket;
    }
    using namespace ba;
    if (!e)
        return fail(BA_ERR_BAD_ARG, "null engine");
    USE_DEVICE(e);
    const int ticket = e->next_ticket;
    Slot& s = e->slot[ticket % BA_SLOTS];
    release_rings(e, false);
    while (ring_release_pending(e, s.ev_ring)) /* this slot's previous ticket (three steps back) still holds ring bytes: its copies finished long ago */
        release_rings(e, true);
    if (s.busy) {
        /* the slot's previous ticket was never collected: its results are about to be replaced */
        CU(cudaEventSynchronize(s.ev_done));
        s.busy = false;
    }
    if (s.used) {
        /* this slot last served ticket - BA_SLOTS: the descriptors its kernels read are rewritten below, its output arena is
         * rewritten by this ticket's demodulator (wait for its device->host copies) */
        CU(cudaStreamWaitEvent(e->s_in, s.ev_kdone, 0));
        CU(cudaStreamWaitEvent(e->serial_k2 ? e->s_k : e->s_k2, s.ev_done, 0));
    }
    if (ticket >= 2) {
        /* ticket - 2: its channelizer read the input half-buffers that are refilled below, and its demodulator reads the
         * stretch of the pick ring this ticket's channelizer is about to overwrite */
        Slot& older = e->slot[(ticket - 2) % BA_SLOTS];
        CU(cudaStreamWaitEvent(e->s_in, older.ev_k1, 0));
        CU(cudaStreamWaitEvent(e->s_k, older.ev_kdone, 0));
    }
    const size_t nd = e->dev.size();
    const int B = e->B;
    s.h2d_bytes = s.d2h_bytes = 0;
    CU(cudaEventRecord(s.ev_begin, e->s_in));

    /* 1. move new bytes to HBM and decide how many frames and batches every input runs */
    std::vector<size_t>& ring_taken = s.ring_taken;
    std::fill(ring_taken.begin(), ring_taken.end(), (size_t)0);
    bool any_ring = false;
    /* host->device pieces are queued behind ALL the device->device carries of the step, so that the copy engine runs the
     * big transfers back to back instead of alternating directions per input */
    struct Piece {
        unsigned char* dst;
        const unsigned char* src;
        size_t n;
    };
    std::vector<Piece> pieces;
    int n_carry = 0;
    for (size_t di = 0; di < nd; di++) {
        Dev& d = *e->dev[di];
        const uint64_t room = frame_room(e, d);
        uint64_t total = 0;
        if (d.injected) {
            total = 0; /* frames arrive through ba_cuda_debug_inject_picks() */
        } else if (d.attached) {
            total = d.attached_valid;
        } else {
            std::lock_guard<std::mutex> g(d.lock);
            const uint64_t next_off = d.frames_done * d.hop_bytes; /* stream offset of the next frame */
            const size_t lo = (size_t)(next_off - d.base_off);
            const size_t carry = d.have - lo;
            /* most bytes this step can use: enough for `room` frames under the availability rule */
            const uint64_t want_total = next_off + room * d.hop_bytes + d.frame_bytes + d.hop_bytes;
            const uint64_t have_total = d.base_off + d.have;
            size_t take_ring = 0;
            std::vector<ExtChunk> take_ext;
            if (have_total < want_total) {
                uint64_t want = want_total - have_total;
                const size_t cap_left = d.d_cap - carry;
                if (want > cap_left)
                    want = cap_left;
                take_ring = (size_t)std::min<uint64_t>(ring_unread(d), want);
                want -= take_ring;
                while (want > 0 && !d.ext.empty()) {
                    ExtChunk& c = d.ext.front();
                    const size_t n = (size_t)std::min<uint64_t>(c.n, want);
                    take_ext.push_back(ExtChunk{c.p, n});
                    c.p += n;
                    c.n -= n;
                    want -= n;
                    if (c.n == 0)
                        d.ext.erase(d.ext.begin());
                }
            }
            if (take_ring || !take_ext.empty()) {
                const int nxt = d.cur ^ 1;
                if (carry)
                    s.h_carry[n_carry++] = K1Carry{d.d_buf[nxt], d.d_buf[d.cur] + lo, (uint32_t)carry, 0u};
                size_t at = carry;
                if (take_ring) {
                    const size_t first = std::min(take_ring, d.buf_size - d.rpos);
                    pieces.push_back(Piece{d.d_buf[nxt] + at, d.ring + d.rpos, first});
                    if (take_ring > first)
                        pieces.push_back(Piece{d.d_buf[nxt] + at + first, d.ring, take_ring - first});
                    at += take_ring;
                    s.h2d_bytes += take_ring;
                    ring_taken[di] = take_ring;
                    d.rpos = (d.rpos + take_ring) % d.buf_size;
                    any_ring = true;
                }
                for (const ExtChunk& c : take_ext) {
                    pieces.push_back(Piece{d.d_buf[nxt] + at, c.p, c.n});
                    at += c.n;
                    s.h2d_bytes += c.n;
                }
                d.cur = nxt;
                d.base_off = next_off;
                d.have = at;
            }
            total = d.base_off + d.have;
        }
        uint64_t nf = frames_admitted(d, total);
        nf = nf > d.frames_done ? nf - d.frames_done : 0;
        if (nf > room)
            nf = room;
        d.step_frame0 = d.frames_done;
        d.step_frames = (int)nf;
        const uint64_t after = d.frames_done + nf;
        uint64_t nb = after >= (uint64_t)BA_E ? (after - BA_E) / B : 0;
        nb = nb > d.batches_done ? nb - d.batches_done : 0;
        if (nb > (uint64_t)e->max_batches)
            nb = e->max_batches;
        d.step_batch0 = d.batches_done;
        d.step_batches = (int)nb;
    }
    if (n_carry) {
        /* one launch moves every input's tail; the list is read from pinned host memory in place */
        int rc = k1_carry_launch(s.h_carry, n_carry, e->s_in);
        if (rc != 0)
            return fail(BA_ERR_CUDA, "carry launch: %s", cudaGetErrorString((cudaError_t)rc));
        e->launches++;
    }
    {
        const bool two = e->h2d_streams >= 2 && pieces.size() >= 2;
        if (two)
            CU(cudaStreamWaitEvent(e->s_in2, s.ev_begin, 0)); /* recorded behind every wait this ticket's input side needs */
        size_t k = 0;
        for (const Piece& pc : pieces)
            CU(cudaMemcpyAsync(pc.dst, pc.src, pc.n, cudaMemcpyHostToDevice, (two && (k++ & 1)) ? e->s_in2 : e->s_in));
        if (two) {
            CU(cudaEventRecord(s.ev_in2, e->s_in2));
            CU(cudaStreamWaitEvent(e->s_in, s.ev_in2, 0));
        }
    }
    if (any_ring) {
        /* the pinned rings are read by the copy engine: the bytes go back to the producers (bufs, .cpp:735) once this event has
         * fired - checked without blocking by release_rings() at the next call of any entry point, so that this thread can go
         * on planning and a producer thread can go on filling the ring while the copies and the kernels run */
        CU(cudaEventRecord(s.ev_ring, e->s_in));
        std::lock_guard<std::mutex> q(e->rel_lock);
        e->rel.push_back(RingRelease{s.ev_ring, ring_taken});
    }

    /* 2. phases: one for ordinary inputs; an AFC input alternates K1/K2 per batch */
    int phases = 1;
    for (Dev* d : e->dev)
        if (d->any_afc)
            phases = std::max(phases, d->step_batches + 1);
    K1Device* h_k1 = reinterpret_cast<K1Device*>(s.h_desc);
    K2Dyn* h_dyn = reinterpret_cast<K2Dyn*>(s.h_desc + (size_t)e->max_phases * nd * sizeof(K1Device));
    K1Device* d_k1 = reinterpret_cast<K1Device*>(s.d_desc);
    K2Dyn* d_dyn = reinterpret_cast<K2Dyn*>(s.d_desc + (size_t)e->max_phases * nd * sizeof(K1Device));
    /* K1 entries of a phase: inputs without AFC first, then the AFC inputs, which need the instantiation that also writes the
     * spectrum (k1_plain / k1_plain_tiles: entries and tiles of the first kind); each kind is one launch */
    std::vector<int> k1_count(phases, 0), k1_tiles(phases, 0), k2_any(phases, 0), k1_plain(phases, 0), k1_plain_tiles(phases, 0);
    std::vector<size_t> order;
    for (int afc = 0; afc < 2; afc++)
        for (size_t di = 0; di < nd; di++)
            if (e->dev[di]->any_afc == (afc == 1))
                order.push_back(di);
    for (int ph = 0; ph < phases; ph++) {
        for (size_t oi = 0; oi < nd; oi++) {
            const size_t di = order[oi];
            Dev& d = *e->dev[di];
            uint64_t f_begin, f_end;
            int nb_here, b_first;
            if (!d.any_afc) {
                f_begin = d.step_frame0;
                f_end = ph == 0 ? d.step_frame0 + d.step_frames : f_begin;
                nb_here = ph == 0 ? d.step_batches : 0;
                b_first = 0;
            } else {
                const uint64_t step_end = d.step_frame0 + d.step_frames;
                auto batch_end = [&](int i) { return std::min<uint64_t>(step_end, (d.step_batch0 + i + 1) * (uint64_t)B + BA_E); };
                f_begin = ph == 0 ? d.step_frame0 : std::max<uint64_t>(d.step_frame0, batch_end(ph - 1));
                if (ph < d.step_batches) {
                    f_end = batch_end(ph);
                    nb_here = 1;
                } else {
                    f_end = ph == d.step_batches ? step_end : f_begin;
                    nb_here = 0;
                }
                if (f_end < f_begin)
                    f_end = f_begin;
                b_first = ph;
            }
            if (f_end > f_begin) {
                K1Device& k = h_k1[(size_t)ph * nd + k1_count[ph]];
                memset(&k, 0, sizeof(k));
                const uint64_t off = f_begin * d.hop_bytes;
                k.iq = d.attached ? d.attached + off : d.d_buf[d.cur] + (size_t)(off - d.base_off);
                k.hop_bytes = (uint32_t)d.hop_bytes;
                k.n_frames = (uint32_t)(f_end - f_begin);
                k.frame0 = f_begin;
                k.picks = d.d_picks;
                k.mags = d.d_mags;
                k.ring_mask = d.ring_len - 1;
                k.n_channels = (uint32_t)d.C;
                k.tile0 = (uint32_t)(k1_tiles[ph] - (d.any_afc ? k1_plain_tiles[ph] : 0)); /* tiles count from 0 in each launch */
                k.bins = d.d_bins;
                k.scale = 1.0f / d.cfg.fullscale;
                k.fmt = d.cfg.sample_format;
                k.spectrum = (d.any_afc && nb_here) ? d.d_spectrum : nullptr;
                const int tiles = (int)((k.n_frames + e->tile_frames - 1) / e->tile_frames);
                k1_tiles[ph] += tiles;
                k1_count[ph]++;
                if (!d.any_afc) {
                    k1_plain[ph]++;
                    k1_plain_tiles[ph] += tiles;
                }
            }
            K2Dyn& y = h_dyn[(size_t)ph * nd + di];
            memset(&y, 0, sizeof(y));
            y.n_batches = nb_here;
            if (nb_here) {
                k2_any[ph] = 1;
                const size_t shift = (size_t)b_first * B;
                y.first_frame = (d.step_batch0 + b_first) * (uint64_t)B + BA_E;
                y.stride = (uint32_t)e->stride;
                y.n_channels = (uint32_t)d.C;
                y.waveout = s.d_wave + d.wave_off + shift;
                y.iq_out = (s.d_iq && d.any_iq) ? s.d_iq + d.iq_off + shift : nullptr;
                y.trace = s.d_trace ? s.d_trace + d.wave_off + shift : nullptr;
                y.status = s.d_status + d.status_off + (size_t)b_first * d.C;
                y.spectrum = d.any_afc ? d.d_spectrum : nullptr;
            }
        }
    }
    /* 2b. mixers: batch k of a mixer is mixed once every unmasked input has delivered its batch k; what an input
     * delivers beyond that is parked in the mixer FIFO */
    int mix_max_emit = 0, mix_max_stash = 0;
    K3InDyn* d_in_dyn = nullptr;
    K3MixDyn* d_mix_dyn = nullptr;
    if (!e->mixers.empty()) {
        const size_t ni = std::max<size_t>(1, e->mix_in.size());
        K3InDyn* h_in_dyn = reinterpret_cast<K3InDyn*>(s.h_desc + e->mix_desc_off);
        K3MixDyn* h_mix_dyn = reinterpret_cast<K3MixDyn*>(s.h_desc + e->mix_desc_off + sizeof(K3InDyn) * ni);
        d_in_dyn = reinterpret_cast<K3InDyn*>(s.d_desc + e->mix_desc_off);
        d_mix_dyn = reinterpret_cast<K3MixDyn*>(s.d_desc + e->mix_desc_off + sizeof(K3InDyn) * ni);
        for (size_t m = 0; m < e->mixers.size(); m++) {
            Mixer& mx = e->mixers[m];
            uint64_t ready = UINT64_MAX;
            for (int j = 0; j < mx.n_in; j++) {
                const MixInput& mi = e->mix_in[mx.first_in + j];
                if (mi.enabled)
                    ready = std::min<uint64_t>(ready, e->dev[mi.dev]->step_batch0 + (uint64_t)e->dev[mi.dev]->step_batches);
            }
            if (ready == UINT64_MAX || ready < mx.emitted)
                ready = mx.emitted; /* every input masked: the mixer is disabled (mixer.cpp:109-111) */
            const int n_emit = (int)std::min<uint64_t>(ready - mx.emitted, (uint64_t)e->max_batches);
            const uint64_t emit_end = mx.emitted + (uint64_t)n_emit;
            K3MixDyn& y = h_mix_dyn[m];
            memset(&y, 0, sizeof(y));
            y.emit0 = mx.emitted;
            y.n_emit = n_emit;
            y.out_l = s.d_mix + mx.out_off;
            y.out_r = mx.stereo ? s.d_mix + mx.out_off + (size_t)e->max_batches * B : nullptr;
            y.sig = s.d_mix_sig + m * (size_t)e->max_batches;
            mix_max_emit = std::max(mix_max_emit, n_emit);
            for (int j = 0; j < mx.n_in; j++) {
                const MixInput& mi = e->mix_in[mx.first_in + j];
                const Dev& d = *e->dev[mi.dev];
                K3InDyn& x = h_in_dyn[mx.first_in + j];
                memset(&x, 0, sizeof(x));
                x.wave = s.d_wave + d.wave_off + (size_t)mi.ch * e->stride;
                x.status = s.d_status + d.status_off + mi.ch;
                x.status_stride = (uint32_t)d.C;
                x.enabled = mi.enabled ? 1 : 0;
                x.batch0 = d.step_batch0;
                const uint64_t avail_end = d.step_batch0 + (uint64_t)d.step_batches;
                x.stash_from = std::max<uint64_t>(d.step_batch0, emit_end);
                x.stash_count = (mi.enabled && avail_end > x.stash_from) ? (int32_t)(avail_end - x.stash_from) : 0;
                mix_max_stash = std::max(mix_max_stash, x.stash_count);
            }
            s.mix_emit[m] = n_emit;
            s.mix_first[m] = mx.emitted;
            mx.emitted = emit_end;
        }
    }
    CU(cudaMemcpyAsync(s.d_desc, s.h_desc, e->desc_bytes, cudaMemcpyHostToDevice, e->s_in));

    CU(cudaEventRecord(s.ev_in, e->s_in));
    CU(cudaStreamWaitEvent(e->s_k, s.ev_in, 0));

    /* 3. launches.  The channelizer (FP32/shared-memory bound, fills the SMs) and the demodulator (a latency-bound serial
     * recurrence, one or two warps per SM) run on two streams: the demodulator of ticket t overlaps the channelizer of
     * ticket t+1, which writes a disjoint stretch of the pick ring.  With AFC the bins feed back, so one stream is used. */
    cudaStream_t k2s = e->serial_k2 ? e->s_k : e->s_k2;
    for (int ph = 0; ph < phases; ph++) {
        CU(cudaEventRecord(s.ev_k[4 * ph + 0], e->s_k));
        /* Inputs without AFC never run the instantiation that also writes the spectrum: the two are compiled apart and may
         * round the FFT differently in the last bit, and an input's audio must not depend on whether another input of its
         * engine has AFC (nor on which member of a multi-GPU group it was placed in). */
        for (int afc = 0; afc < 2; afc++) {
            const int first = afc ? k1_plain[ph] : 0;
            const int n_dev = afc ? k1_count[ph] - k1_plain[ph] : k1_plain[ph];
            if (n_dev == 0)
                continue;
            K1Params p;
            p.dev = d_k1 + (size_t)ph * nd + first;
            p.n_dev = n_dev;
            p.tile_frames = e->tile_frames;
            p.n_tiles = afc ? k1_tiles[ph] - k1_plain_tiles[ph] : k1_plain_tiles[ph];
            p.window = e->d_window;
            p.twiddle = e->d_twiddle;
            p.raw_bytes = e->raw_bytes;
            p.max_channels = e->max_channels;
            p.tile_counter = e->d_tile_counter;
            const int ctas = std::min(p.n_tiles, e->sm_count * e->k1_ctas_per_sm);
            CU(cudaMemsetAsync(e->d_tile_counter, 0, sizeof(uint32_t), e->s_k));
            int rc = k1_launch(e->fft_size, p, ctas, afc != 0, e->s_k);
            if (rc != 0)
                return fail(BA_ERR_CUDA, "channelize launch: %s", cudaGetErrorString((cudaError_t)rc));
            e->launches++;
        }
        CU(cudaEventRecord(s.ev_k[4 * ph + 1], e->s_k));
        CU(cudaEventRecord(s.ev_k1, e->s_k));
        if (k2s != e->s_k)
            CU(cudaStreamWaitEvent(k2s, s.ev_k1, 0));
        CU(cudaEventRecord(s.ev_k[4 * ph + 2], k2s));
        if (k2_any[ph]) {
            K2Params p;
            p.chan = e->d_chan;
            p.state = e->d_state;
            p.dyn = d_dyn + (size_t)ph * nd;
            p.order = e->d_order;
            p.n_channels = e->total_channels;
            p.wave_batch = B;
            p.sincos = e->d_sincos;
            int rc = k2_launch(p, e->n_plain, e->sm_count, k2s, e->s_k2b, e->ev_fork, e->ev_join);
            if (rc != 0)
                return fail(BA_ERR_CUDA, "demod launch: %s", cudaGetErrorString((cudaError_t)rc));
            e->launches += (e->n_plain > 0 ? 1 : 0) + (e->total_channels > e->n_plain ? 1 : 0);
        }
        CU(cudaEventRecord(s.ev_k[4 * ph + 3], k2s));
    }
    s.phases = phases;
    if (mix_max_emit > 0 || mix_max_stash > 0) {
        K3Params p;
        p.in = e->d_mix_in;
        p.in_dyn = d_in_dyn;
        p.mixer = e->d_mixer;
        p.mix_dyn = d_mix_dyn;
        p.fifo = e->d_fifo;
        p.fifo_sig = e->d_fifo_sig;
        p.fifo_depth = e->fifo_depth;
        p.wave_batch = B;
        int rc = k3_launch(p, (int)e->mixers.size(), mix_max_emit, (int)e->mix_in.size(), mix_max_stash, k2s);
        if (rc != 0)
            return fail(BA_ERR_CUDA, "mixer launch: %s", cudaGetErrorString((cudaError_t)rc));
        e->launches += (mix_max_emit > 0 ? 1 : 0) + (mix_max_stash > 0 ? 1 : 0);
    }

    /* 3b. BA_FLAG_SKIP_SILENT_ROWS: pack the rows that are not silence (behind the demodulator and the mixers, which read the arena) */
    s.pack_pending = false;
    s.pack_rows = 0;
    const bool skip_silence = (e->flags & BA_FLAG_SKIP_SILENT_ROWS) && !(e->flags & BA_FLAG_RESULTS_ON_DEVICE);
    if (skip_silence) {
        uint32_t rows = 0, ch0 = 0;
        int n = 0;
        for (Dev* d : e->dev) {
            if (d->step_batches > 0) {
                s.h_packdev[n].first_channel = ch0;
                s.h_packdev[n].n_channels = (uint32_t)d->C;
                s.h_packdev[n].n_batches = (uint32_t)d->step_batches;
                s.h_packdev[n].row0 = rows;
                rows += (uint32_t)d->C * (uint32_t)d->step_batches;
                n++;
            }
            ch0 += (uint32_t)d->C;
        }
        if (rows > 0) {
            CU(cudaMemsetAsync(s.d_rowcount, 0, sizeof(uint32_t), k2s));
            int rc = ba::k3_pack_launch(s.h_packdev, n, (int)rows, s.d_wave, e->stride, B, s.d_pack, s.d_rowmap, e->max_batches, s.d_rowcount, k2s);
            if (rc != 0)
                return fail(BA_ERR_CUDA, "pack launch: %s", cudaGetErrorString((cudaError_t)rc));
            e->launches += 1;
            s.pack_pending = true;
        }
    }

    CU(cudaEventRecord(s.ev_kdone, k2s));
    CU(cudaStreamWaitEvent(e->s_out, s.ev_kdone, 0));
    CU(cudaEventRecord(s.ev_out0, e->s_out));

    /* 4. results to pinned host memory */
    {
        bool uniform = true;
        int nb0 = e->dev[0]->step_batches;
        for (Dev* d : e->dev)
            uniform = uniform && d->step_batches == nb0;
        auto copy_rows = [&](size_t off, size_t rows, int nb) -> int {
            const size_t width = (size_t)nb * B;
            CU(cudaMemcpy2DAsync(s.h_wave + off, sizeof(float) * e->stride, s.d_wave + off, sizeof(float) * e->stride, sizeof(float) * width, rows, cudaMemcpyDeviceToHost,
                                 e->s_out));
            s.d2h_bytes += sizeof(float) * width * rows;
            if (s.d_trace) {
                CU(cudaMemcpy2DAsync(s.h_trace + off, e->stride, s.d_trace + off, e->stride, width, rows, cudaMemcpyDeviceToHost, e->s_out));
                s.d2h_bytes += width * rows;
            }
            return BA_OK;
        };
        const bool to_host = !(e->flags & BA_FLAG_RESULTS_ON_DEVICE); /* else audio, iq_out and trace stay in HBM for a consumer on the GPU */
        if (!to_host) {
        } else if (skip_silence) {
            /* the row map and the number of packed rows now; the rows themselves when ba_cuda_collect() knows how many there are */
            if (s.pack_pending) {
                const size_t rows = (size_t)e->total_channels * e->max_batches;
                CU(cudaMemcpyAsync(s.h_rowmap, s.d_rowmap, sizeof(int32_t) * rows, cudaMemcpyDeviceToHost, e->s_out));
                CU(cudaMemcpyAsync(s.h_rowcount, s.d_rowcount, sizeof(uint32_t), cudaMemcpyDeviceToHost, e->s_out));
                s.d2h_bytes += sizeof(int32_t) * rows + sizeof(uint32_t);
                if (s.d_trace) {
                    for (Dev* d : e->dev)
                        if (d->step_batches > 0) {
                            const size_t width = (size_t)d->step_batches * B;
                            CU(cudaMemcpy2DAsync(s.h_trace + d->wave_off, e->stride, s.d_trace + d->wave_off, e->stride, width, (size_t)d->C, cudaMemcpyDeviceToHost, e->s_out));
                            s.d2h_bytes += width * d->C;
                        }
                }
            }
        } else if (uniform && nb0 == e->max_batches && !s.d_trace) {
            /* a full step everywhere: one linear copy of the arena (the E carried-over samples per row ride along, 1 %) */
            size_t floats = 0;
            for (Dev* d : e->dev)
                floats += (size_t)d->C * e->stride;
            CU(cudaMemcpyAsync(s.h_wave, s.d_wave, sizeof(float) * floats, cudaMemcpyDeviceToHost, e->s_out));
            s.d2h_bytes += sizeof(float) * floats;
        } else if (uniform) {
            if (nb0 > 0) {
                int rc = copy_rows(0, (size_t)e->total_channels, nb0);
                if (rc != BA_OK)
                    return rc;
            }
        } else {
            for (Dev* d : e->dev)
                if (d->step_batches > 0) {
                    int rc = copy_rows(d->wave_off, (size_t)d->C, d->step_batches);
                    if (rc != BA_OK)
                        return rc;
                }
        }
        for (Dev* d : e->dev) {
            if (d->step_batches <= 0 || !to_host)
                continue;
            if (s.d_iq && d->any_iq) {
                const size_t width = (size_t)d->step_batches * B;
                CU(cudaMemcpy2DAsync(s.h_iq + d->iq_off, sizeof(float2) * e->stride, s.d_iq + d->iq_off, sizeof(float2) * e->stride, sizeof(float2) * width, (size_t)d->C,
                                     cudaMemcpyDeviceToHost, e->s_out));
                s.d2h_bytes += sizeof(float2) * width * d->C;
            }
        }
        bool any = false;
        for (Dev* d : e->dev)
            any = any || d->step_batches > 0;
        if (any) {
            size_t total_status = 0;
            for (Dev* d : e->dev)
                total_status += (size_t)d->C * e->max_batches;
            CU(cudaMemcpyAsync(s.h_status, s.d_status, sizeof(ba_channel_status) * total_status, cudaMemcpyDeviceToHost, e->s_out));
            s.d2h_bytes += sizeof(ba_channel_status) * total_status;
        }
    }
    if (mix_max_emit > 0) {
        if (!(e->flags & BA_FLAG_RESULTS_ON_DEVICE))
            CU(cudaMemcpyAsync(s.h_mix, s.d_mix, sizeof(float) * e->mix_floats, cudaMemcpyDeviceToHost, e->s_out));
        CU(cudaMemcpyAsync(s.h_mix_sig, s.d_mix_sig, sizeof(int32_t) * e->mixers.size() * e->max_batches, cudaMemcpyDeviceToHost, e->s_out));
        s.d2h_bytes += ((e->flags & BA_FLAG_RESULTS_ON_DEVICE) ? 0 : sizeof(float) * e->mix_floats) + sizeof(int32_t) * e->mixers.size() * e->max_batches;
    }
    CU(cudaEventRecord(s.ev_done, e->s_out));

    for (size_t di = 0; di < nd; di++) {
        Dev& d = *e->dev[di];
        d.frames_done += (uint64_t)d.step_frames;
        d.batches_done += (uint64_t)d.step_batches;
        s.n_batches[di] = d.step_batches;
        s.frames_done[di] = d.frames_done;
    }
    s.ticket = ticket;
    s.busy = true;
    s.used = true;
    e->next_ticket++;
    return ticket;
}

static Slot* find_slot(ba_engine* e, int ticket) {
    if (!e || ticket < 0) {
        fail(BA_ERR_BAD_ARG, "bad ticket %d", ticket);
        return nullptr;
    }
    Slot& s = e->slot[ticket % BA_SLOTS];
    if (s.ticket != ticket) {
        fail(BA_ERR_STATE, "ticket %d is not outstanding (slot holds %d)", ticket, s.ticket);
        return nullptr;
    }
    return &s;
}

int ba_cuda_collect(ba_engine* e, int ticket, int dev, ba_step_out* out) {
    FORWARD_DEV(e, dev, ba_cuda_collect(e, ticket, dev, out));
    Slot* s = find_slot(e, ticket);
    Dev* d = get_dev(e, dev);
    if (!s || !d || !out)
        return s && d ? fail(BA_ERR_BAD_ARG, "null out") : BA_ERR_BAD_ARG;
    USE_DEVICE(e);
    CU(cudaEventSynchronize(s->ev_done));
    if (s->pack_pending) { /* BA_FLAG_SKIP_SILENT_ROWS: now the number of rows is known; one contiguous copy, once per ticket */
        s->pack_pending = false;
        s->pack_rows = *s->h_rowcount;
        if (s->pack_rows > 0) {
            CU(cudaMemcpyAsync(s->h_pack, s->d_pack, sizeof(float) * (size_t)s->pack_rows * e->B, cudaMemcpyDeviceToHost, e->s_pack));
            CU(cudaStreamSynchronize(e->s_pack));
            s->d2h_bytes += sizeof(float) * (size_t)s->pack_rows * e->B;
        }
    }
    release_rings(e, false);
    s->busy = false;
    memset(out, 0, sizeof(*out));
    out->n_batches = s->n_batches[dev];
    out->wave_batch = e->B;
    out->channel_count = d->C;
    out->wave_stride = e->stride;
    const bool on_dev = (e->flags & BA_FLAG_RESULTS_ON_DEVICE) != 0;
    out->waveout = (on_dev ? s->d_wave : s->h_wave) + d->wave_off;
    if ((e->flags & BA_FLAG_SKIP_SILENT_ROWS) && !on_dev) {
        out->waveout = nullptr;
        out->rows = s->h_pack;
        out->row_of = s->h_rowmap + (d->wave_off / (size_t)e->stride) * (size_t)e->max_batches;
        out->n_rows = s->pack_rows;
        out->row_of_stride = e->max_batches;
    }
    out->iq_out = (s->h_iq && d->any_iq) ? reinterpret_cast<const float*>((on_dev ? s->d_iq : s->h_iq) + d->iq_off) : nullptr;
    out->trace = s->h_trace ? (on_dev ? s->d_trace : s->h_trace) + d->wave_off : nullptr;
    out->status = s->h_status + d->status_off;
    out->frames_done = s->frames_done[dev];
    return BA_OK;
}

int ba_cuda_collect_mixer(ba_engine* e, int ticket, int mixer, ba_mixer_out* out) {
    FORWARD_MIXER(e, mixer, ba_cuda_collect_mixer(e, ticket, mixer, out));
    Slot* s = find_slot(e, ticket);
    if (!s)
        return BA_ERR_BAD_ARG;
    if (!out || mixer < 0 || mixer >= (int)e->mixers.size())
        return fail(BA_ERR_BAD_ARG, "no mixer %d", mixer);
    USE_DEVICE(e);
    CU(cudaEventSynchronize(s->ev_done));
    const Mixer& mx = e->mixers[mixer];
    memset(out, 0, sizeof(*out));
    out->n_batches = s->mix_emit[mixer];
    out->wave_batch = e->B;
    out->stereo = mx.stereo ? 1 : 0;
    out->first_batch = s->mix_first[mixer];
    const float* mix_base = (e->flags & BA_FLAG_RESULTS_ON_DEVICE) ? s->d_mix : s->h_mix;
    out->waveout = mix_base + mx.out_off;
    out->waveout_r = mx.stereo ? mix_base + mx.out_off + (size_t)e->max_batches * e->B : nullptr;
    out->axcindicate = s->h_mix_sig + (size_t)mixer * e->max_batches;
    return BA_OK;
}

int ba_cuda_mixer_input_mask(ba_engine* e, int mixer, int input, int enabled) {
    FORWARD_MIXER(e, mixer, ba_cuda_mixer_input_mask(e, mixer, input, enabled));
    if (!e || mixer < 0 || mixer >= (int)e->mixers.size() || input < 0 || input >= e->mixers[mixer].n_in)
        return fail(BA_ERR_BAD_ARG, "no input %d on mixer %d", input, mixer);
    MixInput& mi = e->mix_in[e->mixers[mixer].first_in + input];
    if (enabled && !mi.enabled) /* the batches it delivered while masked were never parked; the reference has no re-enable either */
        return fail(BA_ERR_STATE, "mixer %d input %d was disabled and cannot be re-enabled", mixer, input);
    mi.enabled = enabled != 0;
    return BA_OK;
}

int ba_cuda_set_freq_idx(ba_engine* e, int dev, int channel, int freq_idx, uint64_t* from_batch) {
    FORWARD_DEV(e, dev, ba_cuda_set_freq_idx(e, dev, channel, freq_idx, from_batch));
    Dev* d = get_dev(e, dev);
    if (!d)
        return BA_ERR_BAD_ARG;
    if (channel < 0 || channel >= d->C || freq_idx < 0 || freq_idx >= (int)d->freqs[channel].size())
        return fail(BA_ERR_BAD_ARG, "input %d channel %d has no frequency %d", dev, channel, freq_idx);
    if (from_batch)
        *from_batch = d->batches_done;
    const int old = d->freq_idx[channel];
    if (old == freq_idx)
        return BA_OK;
    USE_DEVICE(e);
    /* behind every demodulator launch queued so far, ahead of the next one: park the freq_t state of `old`, bring in `freq_idx` */
    cudaStream_t k2s = e->serial_k2 ? e->s_k : e->s_k2;
    const size_t b0 = d->bank0[channel];
    const int gi = d->first_chan + channel;
    int rc = ba::k2_scan_switch_launch(e->d_chan + gi, e->d_state + gi, e->d_bank_chan + b0, e->d_bank_state + b0, old, freq_idx, k2s);
    if (rc != 0)
        return fail(BA_ERR_CUDA, "scan switch launch: %s", cudaGetErrorString((cudaError_t)rc));
    e->launches++;
    d->freq_idx[channel] = freq_idx;
    return BA_OK;
}

int ba_cuda_ticket_ms(ba_engine* e, int ticket, float* ms) {
    if (e && !e->members.empty()) {
        if (!ms)
            return fail(BA_ERR_BAD_ARG, "null argument");
        float worst = 0.0f;
        const int rc = each_member(e, [&](ba_engine* m) {
            float v = 0.0f;
            const int r = ba_cuda_ticket_ms(m, ticket, &v);
            worst = std::max(worst, v);
            return r;
        });
        *ms = worst;
        return rc;
    }
    Slot* s = find_slot(e, ticket);
    if (!s || !ms)
        return BA_ERR_BAD_ARG;
    USE_DEVICE(e);
    CU(cudaEventSynchronize(s->ev_done));
    CU(cudaEventElapsedTime(ms, s->ev_begin, s->ev_done));
    return BA_OK;
}

int ba_cuda_kernel_ms(ba_engine* e, int ticket, float ms[2]) {
    if (e && !e->members.empty())
        return max_pair_over_members(e, ticket, ms, ba_cuda_kernel_ms);
    Slot* s = find_slot(e, ticket);
    if (!s || !ms)
        return BA_ERR_BAD_ARG;
    USE_DEVICE(e);
    CU(cudaEventSynchronize(s->ev_done));
    ms[0] = ms[1] = 0.0f;
    for (int ph = 0; ph < s->phases; ph++) {
        float a = 0, b = 0;
        CU(cudaEventElapsedTime(&a, s->ev_k[4 * ph + 0], s->ev_k[4 * ph + 1]));
        CU(cudaEventElapsedTime(&b, s->ev_k[4 * ph + 2], s->ev_k[4 * ph + 3]));
        ms[0] += a;
        ms[1] += b;
    }
    return BA_OK;
}

int ba_cuda_copy_ms(ba_engine* e, int ticket, float ms[2]) {
    if (e && !e->members.empty())
        return max_pair_over_members(e, ticket, ms, ba_cuda_copy_ms);
    Slot* s = find_slot(e, ticket);
    if (!s || !ms)
        return BA_ERR_BAD_ARG;
    USE_DEVICE(e);
    CU(cudaEventSynchronize(s->ev_done));
    CU(cudaEventElapsedTime(&ms[0], s->ev_begin, s->ev_in));
    CU(cudaEventElapsedTime(&ms[1], s->ev_out0, s->ev_done));
    return BA_OK;
}

int ba_cuda_step_bytes(ba_engine* e, int ticket, uint64_t* h2d, uint64_t* d2h) {
    if (e && !e->members.empty()) {
        uint64_t sum[2] = {0, 0};
        const int rc = each_member(e, [&](ba_engine* m) {
            uint64_t a = 0, b = 0;
            const int r = ba_cuda_step_bytes(m, ticket, &a, &b);
            sum[0] += a, sum[1] += b;
            return r;
        });
        if (h2d)
            *h2d = sum[0];
        if (d2h)
            *d2h = sum[1];
        return rc;
    }
    Slot* s = find_slot(e, ticket);
    if (!s)
        return BA_ERR_BAD_ARG;
    if (h2d)
        *h2d = s->h2d_bytes;
    if (d2h)
        *d2h = s->d2h_bytes;
    return BA_OK;
}

int ba_cuda_mark(ba_engine* e, int which) {
    if (e && !e->members.empty())
        return each_member(e, [&](ba_engine* m) { return ba_cuda_mark(m, which); });
    if (!e || which < 0 || which >= 8)
        return fail(BA_ERR_BAD_ARG, "bad mark %d", which);
    USE_DEVICE(e);
    if (!e->marks[which])
        CU(cudaEventCreate(&e->marks[which]));
    for (cudaStream_t q : {e->s_in, e->s_in2, e->s_k, e->s_k2}) {
        CU(cudaEventRecord(e->ev_tmp[0], q));
        CU(cudaStreamWaitEvent(e->s_out, e->ev_tmp[0], 0));
    }
    CU(cudaEventRecord(e->marks[which], e->s_out));
    return BA_OK;
}

int ba_cuda_mark_ms(ba_engine* e, int from, int to, float* ms) {
    if (e && !e->members.empty()) {
        if (!ms)
            return fail(BA_ERR_BAD_ARG, "null argument");
        float worst = 0.0f;
        const int rc = each_member(e, [&](ba_engine* m) {
            float v = 0.0f;
            const int r = ba_cuda_mark_ms(m, from, to, &v);
            worst = std::max(worst, v);
            return r;
        });
        *ms = worst;
        return rc;
    }
    if (!e || !ms || from < 0 || from >= 8 || to < 0 || to >= 8 || !e->marks[from] || !e->marks[to])
        return fail(BA_ERR_BAD_ARG, "marks %d, %d not recorded", from, to);
    USE_DEVICE(e);
    CU(cudaEventSynchronize(e->marks[from]));
    CU(cudaEventSynchronize(e->marks[to]));
    CU(cudaEventElapsedTime(ms, e->marks[from], e->marks[to]));
    return BA_OK;
}

int ba_cuda_channel_info(ba_engine* e, int dev, int channel, ba_channel_info* out) {
    FORWARD_DEV(e, dev, ba_cuda_channel_info(e, dev, channel, out));
    Dev* d = get_dev(e, dev);
    if (!d || !out || channel < 0 || channel >= d->C)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    *out = e->info[d->first_chan + channel];
    return BA_OK;
}

int ba_cuda_window(ba_engine* e, float* out, size_t count) {
    if (e && !e->members.empty()) /* every member computed the same window */
        return e->broken ? group_broken() : ba_cuda_window(e->members[0], out, count);
    if (!e || !out || count != e->window.size())
        return fail(BA_ERR_BAD_ARG, "bad argument");
    memcpy(out, e->window.data(), count * sizeof(float));
    return BA_OK;
}

int ba_cuda_launch_count(ba_engine* e, uint64_t* launches) {
    if (e && !e->members.empty()) {
        if (!launches)
            return fail(BA_ERR_BAD_ARG, "null argument");
        uint64_t sum = 0;
        const int rc = each_member(e, [&](ba_engine* m) {
            uint64_t n = 0;
            const int r = ba_cuda_launch_count(m, &n);
            sum += n;
            return r;
        });
        *launches = sum;
        return rc;
    }
    if (!e || !launches)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    *launches = e->launches;
    return BA_OK;
}

int ba_cuda_debug_frames(ba_engine* e, int dev, const void* iq, size_t bytes, int n_frames, float* fftin, float* fftout) {
    FORWARD_DEV(e, dev, ba_cuda_debug_frames(e, dev, iq, bytes, n_frames, fftin, fftout));
    using namespace ba;
    Dev* d = get_dev(e, dev);
    if (!d || !iq || n_frames <= 0)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    const size_t N = (size_t)e->fft_size;
    if ((size_t)(n_frames - 1) * d->hop_bytes + d->frame_bytes > bytes)
        return fail(BA_ERR_BAD_ARG, "%d frames need %zu bytes, %zu given", n_frames, (size_t)(n_frames - 1) * d->hop_bytes + d->frame_bytes, bytes);
    USE_DEVICE(e);
    unsigned char* d_iq = nullptr;
    float2 *d_in = nullptr, *d_out = nullptr, *d_picks = nullptr;
    float* d_mags = nullptr;
    K1Device* d_k = nullptr;
    const uint32_t ring_len = pow2_at_least((uint64_t)n_frames);
    int rc = BA_OK;
    auto cleanup = [&]() {
        cudaFree(d_iq);
        cudaFree(d_in);
        cudaFree(d_out);
        cudaFree(d_picks);
        cudaFree(d_mags);
        cudaFree(d_k);
    };
#define CUD(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (cudaError_t)(call);                                                      \
        if (e_ != cudaSuccess) {                                                                   \
            cleanup();                                                                             \
            return fail(BA_ERR_CUDA, "%s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                          \
    } while (0)
    for (cudaStream_t q : {e->s_in, e->s_in2, e->s_k, e->s_k2, e->s_k2b, e->s_out, e->s_pack})
        CUD(cudaStreamSynchronize(q));
    CUD(cudaMalloc((void**)&d_iq, bytes + 16));
    CUD(cudaMalloc((void**)&d_in, sizeof(float2) * N * n_frames));
    CUD(cudaMalloc((void**)&d_out, sizeof(float2) * N * n_frames));
    CUD(cudaMalloc((void**)&d_picks, sizeof(float2) * (size_t)ring_len * d->C));
    CUD(cudaMalloc((void**)&d_mags, sizeof(float) * (size_t)ring_len * d->C));
    CUD(cudaMalloc((void**)&d_k, sizeof(K1Device)));
    CUD(cudaMemcpy(d_iq, iq, bytes, cudaMemcpyHostToDevice));
    K1Device k;
    memset(&k, 0, sizeof(k));
    k.iq = d_iq;
    k.hop_bytes = (uint32_t)d->hop_bytes;
    k.n_frames = (uint32_t)n_frames;
    k.frame0 = 0;
    k.picks = d_picks;
    k.mags = d_mags;
    k.ring_mask = ring_len - 1;
    k.n_channels = (uint32_t)d->C;
    k.tile0 = 0;
    k.bins = d->d_bins;
    k.scale = 1.0f / d->cfg.fullscale;
    k.fmt = d->cfg.sample_format;
    k.dbg_in = fftin ? d_in : nullptr;
    k.dbg_out = fftout ? d_out : nullptr;
    CUD(cudaMemcpy(d_k, &k, sizeof(k), cudaMemcpyHostToDevice));
    K1Params p;
    p.dev = d_k;
    p.n_dev = 1;
    p.tile_frames = e->tile_frames;
    p.n_tiles = (n_frames + e->tile_frames - 1) / e->tile_frames;
    p.window = e->d_window;
    p.twiddle = e->d_twiddle;
    p.raw_bytes = e->raw_bytes;
    p.max_channels = e->max_channels;
    p.tile_counter = e->d_tile_counter;
    CUD(cudaMemsetAsync(e->d_tile_counter, 0, sizeof(uint32_t), e->stream));
    rc = k1_launch(e->fft_size, p, std::min(p.n_tiles, e->sm_count), true, e->stream);
    if (rc != 0) {
        cleanup();
        return fail(BA_ERR_CUDA, "channelize launch: %s", cudaGetErrorString((cudaError_t)rc));
    }
    e->launches++;
    CUD(cudaStreamSynchronize(e->stream));
    if (fftin)
        CUD(cudaMemcpy(fftin, d_in, sizeof(float2) * N * n_frames, cudaMemcpyDeviceToHost));
    if (fftout)
        CUD(cudaMemcpy(fftout, d_out, sizeof(float2) * N * n_frames, cudaMemcpyDeviceToHost));
#undef CUD
    cleanup();
    return BA_OK;
}

int ba_cuda_debug_picks(ba_engine* e, int dev, int channel, uint64_t first, int count, float* out) {
    FORWARD_DEV(e, dev, ba_cuda_debug_picks(e, dev, channel, first, count, out));
    Dev* d = get_dev(e, dev);
    if (!d || !out || channel < 0 || channel >= d->C || count < 0)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    if (!d->d_picks)
        return fail(BA_ERR_STATE, "input %d keeps no picked-bin IQ (create the engine with BA_FLAG_KEEP_PICKS)", dev);
    if (first + (uint64_t)count > d->frames_done || d->frames_done - first > d->ring_len)
        return fail(BA_ERR_BAD_ARG, "frames [%llu, +%d) are not in the pick ring (frames done %llu, ring %u)", (unsigned long long)first, count,
                    (unsigned long long)d->frames_done, d->ring_len);
    USE_DEVICE(e);
    CU(cudaStreamSynchronize(e->s_k));
    CU(cudaStreamSynchronize(e->s_k2));
    const float2* row = d->d_picks + (size_t)channel * d->ring_len;
    uint64_t f = first;
    int left = count;
    while (left > 0) {
        const uint32_t pos = (uint32_t)(f & (d->ring_len - 1));
        const int n = (int)std::min<uint64_t>((uint64_t)left, d->ring_len - pos);
        CU(cudaMemcpy(out + 2 * (f - first), row + pos, sizeof(float2) * (size_t)n, cudaMemcpyDeviceToHost));
        f += n;
        left -= n;
    }
    return BA_OK;
}

int ba_cuda_debug_inject_picks(ba_engine* e, int dev, const float* picks, int n_frames) {
    FORWARD_DEV(e, dev, ba_cuda_debug_inject_picks(e, dev, picks, n_frames));
    Dev* d = get_dev(e, dev);
    if (!d || !picks || n_frames < 0)
        return fail(BA_ERR_BAD_ARG, "bad argument");
    if ((uint64_t)n_frames > frame_room(e, *d))
        return fail(BA_ERR_OVERRUN, "input %d: room for %llu more frames before the next ba_cuda_process()", dev, (unsigned long long)frame_room(e, *d));
    USE_DEVICE(e);
    CU(cudaStreamSynchronize(e->s_k));
    CU(cudaStreamSynchronize(e->s_k2));
    /* [frame][channel] from the caller -> the device's [channel][frame ring]; the magnitudes K1 would have written next to the
     * picks are computed here: sqrtf and the products are IEEE operations in this host code too (no fast-math; the volatile
     * keeps the compiler from contracting them) */
    const size_t C = (size_t)d->C;
    std::vector<float2> row((size_t)n_frames);
    std::vector<float> mrow((size_t)n_frames);
    for (size_t c = 0; c < C; c++) {
        for (size_t f = 0; f < (size_t)n_frames; f++) {
            const float re = picks[2 * (f * C + c)], im = picks[2 * (f * C + c) + 1];
            volatile float rr = re * re;
            volatile float ii = im * im;
            volatile float sum = rr + ii;
            row[f] = make_float2(re, im);
            mrow[f] = sqrtf(sum);
        }
        uint64_t f = d->frames_done;
        size_t at = 0;
        int left = n_frames;
        while (left > 0) {
            const uint32_t pos = (uint32_t)(f & (d->ring_len - 1));
            const int n = (int)std::min<uint64_t>((uint64_t)left, d->ring_len - pos);
            if (d->d_picks)
                CU(cudaMemcpy(d->d_picks + c * d->ring_len + pos, row.data() + at, sizeof(float2) * (size_t)n, cudaMemcpyHostToDevice));
            CU(cudaMemcpy(d->d_mags + c * d->ring_len + pos, mrow.data() + at, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice));
            f += n;
            at += (size_t)n;
            left -= n;
        }
    }
    d->frames_done += (uint64_t)n_frames;
    d->injected = true;
    return BA_OK;
}

}  /* extern "C" */
