/*
 * ba_kernels.h — device-side job descriptors shared by the host engine (ba_engine.cu) and the two kernels:
 *   K1  channelize  (channelize.cu)  expand + window + batched in-shared-memory FFT + per-channel bin pick
 *                                     replaces boondock_airband.cpp:426-516 (and hello_fft + samplefft on the Pi)
 *   K2  demod       (demod.cu)       the per-channel sample loop, boondock_airband.cpp:518-679, with Squelch,
 *                                     CTCSS, NotchFilter, LowpassFilter state resident in HBM between launches
 *   K3  mixer       (mixer.cu)       mixers summed behind the demodulator, mixer.cpp:114-141,166-257
 */
#ifndef BA_KERNELS_H
#define BA_KERNELS_H

#include <stdint.h>

#include "../../include/ba_cuda.h"
#include "ba_port.h"

#define BA_E 100       /* AGC_EXTRA, boondock_airband.h:74 */
#define BA_SQ_RING 102 /* Squelch::buffer_size_, squelch.cpp:67 */
#define BA_MAX_TONES 52 /* 1 target + 51 standard tones, ctcss.cpp:101-118 */

namespace ba {

/* ------------------------------------------------------------------ K1 */

/* one input (device_t) as K1 sees it for one launch */
struct K1Device {
    const unsigned char* iq; /* first byte of frame 0 of this launch (device memory; its allocation is 16-byte aligned and padded) */
    uint32_t hop_bytes;      /* bps, boondock_airband.cpp:418 */
    uint32_t n_frames;       /* frames in this launch */
    uint64_t frame0;         /* stream index of frame 0 */
    float2* picks;           /* [channel][ring_len]: fftout[bins[c]] per frame, ring over frames; NULL when no channel of the input needs raw IQ */
    float* mags;             /* [channel][ring_len]: |fftout[bins[c]]| = wavein[] as the bin pick writes it (.cpp:507-513) */
    uint32_t ring_mask;      /* ring_len - 1 */
    uint32_t pad0;
    uint32_t n_channels;
    uint32_t tile0;          /* first tile index of this device in the launch-wide tile list */
    const uint32_t* bins;    /* device-resident dev->bins[] (AFC may move them between launches) */
    float scale;             /* 1 / fullscale (S16, F32) */
    int32_t fmt;             /* BA_SFMT_* */
    float2* spectrum;        /* AFC: full spectrum of the last frame of the launch (natural bin order) or NULL */
    float2* dbg_in;          /* tests: converted frames [n_frames][N] or NULL */
    float2* dbg_out;         /* tests: spectra [n_frames][N], natural order, or NULL */
};

struct K1Params {
    const K1Device* dev;
    int32_t n_dev;
    int32_t tile_frames;   /* frames per tile */
    int32_t n_tiles;       /* total tiles over all devices */
    const float* window;   /* [N], boondock_airband.cpp:357-373 */
    const float2* twiddle; /* [N], exp(-2 pi i n / N), rounded from double */
    int32_t raw_bytes;     /* shared-memory bytes reserved for the staged byte span of one tile (multiple of 16) */
    int32_t max_channels;  /* largest channel_count of any input (pick table size) */
    uint32_t* tile_counter; /* zeroed before the launch; CTAs take tile indices from it */
};

/* the unconsumed tail of an input's stream (less than one frame + one hop) moves from the half-buffer the last step read to
 * the front of the one the next step reads (the mirrored tail of circbuffer_append, input-helpers.cpp:37-63, done in HBM) */
struct K1Carry {
    unsigned char* dst;
    const unsigned char* src;
    uint32_t n, pad0;
};
/* one launch for all inputs; `list` may live in pinned host memory (read once, n entries) */
int k1_carry_launch(const K1Carry* list, int n, cudaStream_t s);

/* returns 0 or a cudaError_t; dbg selects the instantiation that also serves dbg_in / dbg_out / spectrum */
int k1_launch(int fft_size, const K1Params& p, int n_ctas, bool dbg, cudaStream_t s);
/* sets the kernels' dynamic shared-memory limit on the CURRENT device; once per engine, after cudaSetDevice() */
int k1_configure(int fft_size, int raw_bytes, int max_channels);
int k1_smem_bytes(int fft_size, int raw_bytes, int max_channels);
int k1_threads(int fft_size);
int k1_groups(int fft_size); /* FFTs a CTA works on at a time */
int k1_ctas_per_sm(int fft_size); /* resident CTAs per SM the plan's register cap is chosen for */
int k1_direct(int fft_size);      /* 1: frames are read straight from global memory (no tile staging in shared memory: raw_bytes = 0) */

/* ------------------------------------------------------------------ K2 */

/* Goertzel bank pair of one CTCSS channel: constants and resident state (ctcss.cpp) */
struct K2Ctcss {
    int32_t n_fast, n_slow, win_fast, win_slow;
    float coeff_fast[BA_MAX_TONES], coeff_slow[BA_MAX_TONES];
    /* state */
    int32_t fast_full, fast_fed, fast_tone, slow_full, slow_fed, slow_tone;
    uint32_t slow_hits, slow_misses;
    float fq1[BA_MAX_TONES], fq2[BA_MAX_TONES], sq1[BA_MAX_TONES], sq2[BA_MAX_TONES];
};

/* constants of one channel (channel_t + freq_t + its Squelch/filter configuration) */
struct K2Chan {
    int32_t dev;          /* input index (K2Dyn) */
    uint32_t col;         /* channel index within its input = column of the pick row */
    const float2* picks;  /* this channel's row of its input's pick ring, [ring_len] (NULL when the input keeps no picks) */
    const float* mags;    /* this channel's row of magnitudes, [ring_len] */
    uint32_t ring_mask, pad0;
    uint32_t* bin;        /* &bins[col] (AFC moves it) */
    uint32_t base_bin;
    int32_t fft_size;
    /* channel_t / freq_t */
    int32_t modulation, afc, needs_raw_iq, has_iq_outputs, fm_demod;
    uint32_t dm_dphi;
    float alpha, ampfactor;
    /* Squelch configuration (squelch.cpp:36-116) */
    int32_t manual;
    float manual_level, ratio, flappy_ratio;
    /* filters (filters.cpp) */
    int32_t notch_on, lp_on;
    float nd0, nd1, nd2;
    float lp_gain, lp_c0, lp_c1;
    /* CTCSS */
    K2Ctcss* ctcss; /* NULL when the channel has no ctcss */
};

/* mutable state of one channel, resident in HBM between launches (SURVEY.md appendix B) */
struct alignas(16) K2State {
    float waveout_tail[BA_E];  /* waveout[B..B+E) kept by output_thread for the next batch (output.cpp:948); first: moved in 16-byte pieces */
    /* Squelch */
    float noise, cap, pre_full, pre_cap, post_full, post_cap;
    int32_t post_active, next, cur, delay, low_run;
    uint32_t opens, flappy, recent_opens, closed_run, count16;
    int32_t head, tail;
    /* channel */
    uint32_t dm_phi;
    float pr, pj, prev_waveout, agcavgfast;
    uint32_t active_counter;
    int32_t axcindicate;
    int32_t hist_ready; /* 0 until the first launch has seeded wavein_hist from frames 0..E-1 */
    int32_t hist_pos;   /* slot of wavein_hist the next sample uses (frame index mod E) */
    /* filters */
    float nx0, nx1, nx2, ny0, ny1, ny2;
    float lxr0, lxr1, lxr2, lxi0, lxi1, lxi2, lyr0, lyr1, lyr2, lyi0, lyi1, lyi2;
    float ring[BA_SQ_RING];    /* Squelch::buffer_ */
    float wavein_hist[BA_E];   /* wavein[] as the loop left it for the last E frames (.cpp:548 overwrites it) */
};

/* per input, per launch */
struct K2Dyn {
    uint64_t first_frame; /* stream index of the first frame the squelch sees: batches_done*B + E */
    int32_t n_batches;    /* batches of this input in this launch (0 = nothing to do) */
    uint32_t stride;      /* elements between consecutive channels in waveout / iq_out / trace */
    uint32_t n_channels;  /* channels of this input (row length of status) */
    uint32_t pad0;
    float* waveout;       /* [C][stride]; row positions [0,E) hold the tail carried in, [0, n_batches*B) go to the host */
    float2* iq_out;       /* [C][stride] or NULL */
    uint8_t* trace;       /* [C][stride] or NULL */
    ba_channel_status* status; /* [max_batches][C] */
    const float2* spectrum;    /* AFC: spectrum of the last frame K1 produced (the last frame of the batch) or NULL */
};

struct K2Params {
    const K2Chan* chan;
    K2State* state;
    const K2Dyn* dyn;     /* [n inputs] */
    const int32_t* order; /* channel indices in launch order (grouped by kind so that warps stay convergent) */
    int32_t n_channels;
    int32_t wave_batch;   /* B, a multiple of 4 */
    const float* sincos;  /* [2][257] sin then cos, util.cpp:103-110 */
    int32_t first_slot, end_slot; /* filled by k2_launch: the slots of `order` this kernel covers */
    int32_t plain_lanes;          /* filled by k2_launch: channels per CTA of demod_plain_kernel (1..32) */
};

/* n_plain: the first n_plain slots of `order` are plain AM channels (demod_plain_kernel), the rest is general (one warp per
 * channel); s2/fork/join (optional) let the two kernels run concurrently */
int k2_launch(const K2Params& p, int n_plain, int sm_count, cudaStream_t s, cudaStream_t s2, cudaEvent_t fork, cudaEvent_t join);
/* sets the demodulators' dynamic shared-memory limit on the CURRENT device; once per engine, after cudaSetDevice() */
int k2_configure(void);

/* scan mode (boondock_airband.cpp:101-139,522): `chan`/`st` are the live entries of one channel, bank_* its per-frequency
 * copies.  Parks the freq_t part of the state (Squelch, filters, AGC level, active_counter) under `from`, loads the one
 * parked under `to` together with that frequency's constants; the channel_t part (look-back, phases, tails) stays. */
int k2_scan_switch_launch(K2Chan* chan, K2State* st, const K2Chan* bank_chan, K2State* bank_state, int from, int to, cudaStream_t s);

/* ------------------------------------------------------------------ K3 (mixer.cu) */

/* one mixer input: constants */
struct K3In {
    float mult_l, mult_r; /* ampfactor * ampl, ampfactor * ampr (mixer.cpp:79-81,195-199) */
};
/* one mixer input, per launch */
struct K3InDyn {
    const float* wave;               /* the channel's row of this step's waveout arena */
    const ba_channel_status* status; /* &status[0][channel] of this step */
    uint32_t status_stride;          /* channels of the input's device: entries between consecutive batches */
    int32_t enabled;                 /* input_mask */
    uint64_t batch0;                 /* number of the first batch the device delivers in this step */
    uint64_t stash_from;             /* batches [stash_from, stash_from + stash_count) go to the FIFO */
    int32_t stash_count, pad0;
};
struct K3Mixer {
    int32_t first_in, n_in, stereo, pad0;
};
struct K3MixDyn {
    uint64_t emit0; /* number of the first batch mixed in this step */
    int32_t n_emit, pad0;
    float* out_l;
    float* out_r;
    int32_t* sig;
};
struct K3Params {
    const K3In* in;
    const K3InDyn* in_dyn;
    const K3Mixer* mixer;
    const K3MixDyn* mix_dyn;
    float* fifo;       /* [inputs][fifo_depth][B] */
    uint8_t* fifo_sig; /* [inputs][fifo_depth] */
    int32_t fifo_depth, wave_batch;
};
/* BA_FLAG_SKIP_SILENT_ROWS: the rows of one step, device by device */
struct K3PackDev {
    uint32_t first_channel, n_channels, n_batches, row0; /* row0: rows of the devices before this one */
};
/* one warp per (channel, batch) row of `wave` ([channel][stride], batch b at b * wave_batch): rows holding anything but +0.0f are
 * copied to pack[slot][wave_batch] (slot from an atomic counter) and rowmap[channel][max_batches] = slot, else -1.
 * `devs` may live in pinned host memory (read once). */
int k3_pack_launch(const K3PackDev* devs, int n_dev, int total_rows, const float* wave, int stride, int wave_batch, float* pack, int32_t* rowmap, int max_batches,
                   uint32_t* count, cudaStream_t s);

/* mixes max_emit (largest n_emit of any mixer) batches, then parks max_stash (largest stash_count) */
int k3_launch(const K3Params& p, int n_mixers, int max_emit, int n_inputs, int max_stash, cudaStream_t s);

/* ------------------------------------------------------------------ channel sharding (mixer.cu) */
/* An input whose channels are demodulated on several GPUs is channelized once, on its home GPU.  Both kernels store to the
 * other GPU's memory (peer stores; a plain store when both sides share one GPU).  Their job tables live in device memory. */

/* ship (on the home, behind K1): one channel's magnitudes, and its picked IQ where the follower reads it, for the frames the
 * home channelized in this step, from the home's pick ring to the same ring positions of the follower's */
struct XShip {
    const float* src_mags;
    float* dst_mags;          /* rows of [ring_len] */
    const float2* src_picks;
    float2* dst_picks;        /* NULL: the IQ stays home */
    uint64_t frame0;          /* first frame of the step */
    uint32_t n_frames, ring_mask;
};
/* gather (on the follower, behind K2): one channel's results of the step into the home's result slot */
struct XGather {
    const float* src_wave;
    float* dst_wave;          /* n_samples floats */
    const uint8_t* src_trace;
    uint8_t* dst_trace;       /* or NULL */
    const float2* src_iq;
    float2* dst_iq;           /* or NULL */
    const ba_channel_status* src_status;
    ba_channel_status* dst_status; /* &status[0][channel] */
    uint32_t n_samples, n_batches, src_status_stride, dst_status_stride; /* strides in entries between batches */
};
int x_ship_launch(const XShip* jobs, int n_jobs, uint32_t max_frames, cudaStream_t s);
int x_gather_launch(const XGather* jobs, int n_jobs, uint32_t max_samples, cudaStream_t s);

}  // namespace ba
#endif
