/*
 * ba_cuda.h — C-ABI of the B200 channelize-and-demodulate engine.
 *
 * This is the drop-in boundary for Boondock-Airband's demodulate() path
 * (reference: src/boondock_airband.cpp:308-738).  The reference has no plugin
 * API for its DSP; the two precedents that define the shape of an accelerator
 * boundary in that code base are
 *   - the VideoCore FFT C API  gpu_fft_prepare / gpu_fft_execute / gpu_fft_release
 *     (src/hello_fft/gpu_fft.h:66-74, call sites src/boondock_airband.cpp:316-332,482)
 *     — int return, 0 = ok, negative = reason, opaque handle out-parameter;
 *   - the NEON sample expander  extern "C" samplefft(...)
 *     (src/boondock_airband.h:88-92).
 * Every entry point below says which piece of the reference it replaces.
 *
 * Plain C: pointers and sizes only, no C++/torch types, no exceptions cross
 * this boundary.  All functions return BA_OK (0) or a negative BA_ERR_* code.
 * There is NO CPU fallback behind this API: without a usable CUDA device
 * ba_cuda_create() fails with BA_ERR_NO_DEVICE.
 */
#ifndef BA_CUDA_H
#define BA_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BA_CUDA_ABI_VERSION 3 /* 2: mixers in ba_engine_desc, frequency lists in ba_channel_desc; 3: ba_step_out grew (rows, row_of, n_rows). Older callers are refused */

#if defined(__GNUC__)
#define BA_API __attribute__((visibility("default")))
#else
#define BA_API
#endif

/* sample_format_t of the reference, same numeric values (src/input-common.h:32) */
enum { BA_SFMT_UNDEF = 0, BA_SFMT_U8 = 1, BA_SFMT_S8 = 2, BA_SFMT_S16 = 3, BA_SFMT_F32 = 4 };
/* enum modulations (src/boondock_airband.h:202-208) */
enum { BA_MOD_AM = 0, BA_MOD_NFM = 1 };
/* enum fm_demod_algo (src/boondock_airband.cpp:88), selected by -Q on the reference CLI */
enum { BA_FM_FAST_ATAN2 = 0, BA_FM_QUADRI_DEMOD = 1 };
/* enum status / channel_t.axcindicate (src/boondock_airband.h:101) */
enum { BA_NO_SIGNAL = ' ', BA_SIGNAL = '*', BA_AFC_UP = '<', BA_AFC_DOWN = '>' };
/* Squelch::State numbering (src/squelch.h:104-110), used in the decision trace */
enum { BA_SQ_CLOSED = 0, BA_SQ_OPENING = 1, BA_SQ_CLOSING = 2, BA_SQ_LOW_SIGNAL_ABORT = 3, BA_SQ_OPEN = 4 };

#define BA_AGC_EXTRA 100 /* AGC_EXTRA, src/boondock_airband.h:74 */

/* return codes; -1..-3 keep the meaning gpu_fft_prepare gives them (src/boondock_airband.cpp:319-332) */
#define BA_OK 0
#define BA_ERR_NO_DEVICE (-1) /* accelerator cannot be enabled */
#define BA_ERR_BAD_SIZE (-2)  /* fft_size is not 2^8 .. 2^13 (MIN/MAX_FFT_SIZE_LOG, boondock_airband.h:80-82) */
#define BA_ERR_NOMEM (-3)     /* host or device allocation failed */
#define BA_ERR_BAD_ARG (-4)
#define BA_ERR_CUDA (-5)    /* a CUDA call failed; ba_cuda_last_error() has the text */
#define BA_ERR_OVERRUN (-6) /* output slot not collected yet / input ring full (cf. output_overrun_count, .cpp:673-676) */
#define BA_ERR_STATE (-7)   /* call sequence violated */

/* engine flags */
#define BA_FLAG_TRACE 0x1u /* also return the per-sample squelch decision trace (like -DDEBUG_SQUELCH, squelch.cpp:520-633) */
#define BA_FLAG_KEEP_PICKS 0x2u /* keep the picked-bin IQ of every channel on the device (ba_cuda_debug_picks); without it only
                                 * inputs with a channel that needs raw IQ (NFM, bandwidth, iq outputs) keep it, plain AM needs |X| only */

#define BA_FLAG_RESULTS_ON_DEVICE 0x4u /* for consumers on the GPU (encoders, further DSP): waveout / iq_out / trace of ba_step_out
                                        * and the planes of ba_mixer_out are DEVICE pointers into the ticket's result slot and are not
                                        * copied to the host; status and axcindicate still are.  Valid until three more ba_cuda_process(). */
#define BA_FLAG_SKIP_SILENT_ROWS 0x8u  /* Far above real time the device->host copy of the audio bounds the path, and a squelched channel's
                                        * audio is exact zeros.  With this flag the engine looks at every (channel, batch) row of wave_batch
                                        * samples on the device, packs the rows that hold anything but +0.0f, and copies only those:
                                        * ba_step_out.waveout is NULL, ba_step_out.rows / row_of describe the packed rows (a consumer writes
                                        * silence for row_of < 0, where it would have copied the row).  Decided on the data, never on the
                                        * squelch state; iq_out, trace, status and the mixers are returned as without the flag. */

/* trace byte layout: bits 0-2 Squelch current_state_, bit 3 is_open(), bit 4 should_process_audio(),
 * bit 5 should_filter_sample() && needs_raw_iq (the sample went through derotation/LPF) */
#define BA_TRACE_STATE_MASK 0x07
#define BA_TRACE_OPEN 0x08
#define BA_TRACE_AUDIO 0x10
#define BA_TRACE_FILTERED 0x20

/* One freq_t of a scan-mode channel (src/config.cpp:364-433): what the channel may set once per frequency. */
typedef struct ba_freq_desc {
    int32_t frequency;              /* "freqs"[f] */
    int32_t modulation;             /* "modulations"[f] or the channel's "modulation" */
    float ampfactor;                /* "ampfactor" scalar or list */
    int32_t squelch_threshold_dbfs; /* "squelch_threshold" scalar or list */
    float squelch_snr_threshold;    /* "squelch_snr_threshold" scalar or list; <0 = default */
    float notch, notch_q, ctcss;    /* scalar or list */
    int32_t bandwidth;              /* scalar or list; <0 = present but rejected */
} ba_freq_desc;

/*
 * One channel = channel_t + its single freq_t (multichannel mode, src/config.cpp:312-729).
 * Values are the ones written in the libconfig file; every derived constant
 * (bin, dm_dphi, biquad coefficients, Goertzel coefficients, alpha) is computed
 * by the engine with the reference's formulas.
 */
typedef struct ba_channel_desc {
    int32_t frequency;             /* Hz, freq_t.frequency (config.cpp:357) */
    int32_t modulation;            /* BA_MOD_* (config.cpp:341-353) */
    int32_t afc;                   /* channel_t.afc 0..255 (config.cpp:354) */
    float ampfactor;               /* freq_t.ampfactor (config.cpp:624-650); mk_freqlist default 1.0 */
    int32_t squelch_threshold_dbfs; /* "squelch_threshold": <0 manual level in dBFS, 0 = automatic (config.cpp:437-472) */
    float squelch_snr_threshold;   /* "squelch_snr_threshold" in dB; <0 = leave the default 9.54 dB (config.cpp:473-515, squelch.cpp:38) */
    float notch;                   /* "notch" Hz, 0 = off (config.cpp:516-562) */
    float notch_q;                 /* "notch_q", 0 = default 10.0 */
    float ctcss;                   /* "ctcss" Hz, 0 = off (config.cpp:563-590) */
    int32_t bandwidth;             /* "bandwidth" Hz, 0 = off; low-pass at bandwidth/2 (config.cpp:591-622); <0 = the key was there
                                    * but its value was rejected: needs_raw_iq is set, no filter (config.cpp:592,609-610) */
    int32_t tau_us;                /* "tau" µs; <0 = inherit the device value (config.cpp:652-656) */
    int32_t has_iq_outputs;        /* channel_t.has_iq_outputs: a rawfile output wants iq_out (config.cpp:162) */
    /* scan mode (R_SCAN, config.cpp:364-433): freq_count > 0 makes `freqs` the channel's freqlist and the per-frequency
     * fields above (frequency, modulation, ampfactor, squelch_*, notch*, ctcss, bandwidth) are not read.  The bin and the
     * derotation step come from freqs[0] (config.cpp:669,684); ba_cuda_set_freq_idx() plays controller_thread's part. */
    int32_t freq_count;
    const ba_freq_desc* freqs;
} ba_channel_desc;

/* One device_t + its input_t (src/boondock_airband.h:272-292, src/input-common.h:39-57). */
typedef struct ba_device_desc {
    int32_t sample_format;    /* input_t.sfmt */
    int32_t bytes_per_sample; /* input_t.bytes_per_sample (per I or Q component) */
    float fullscale;          /* input_t.fullscale */
    int32_t sample_rate;      /* input_t.sample_rate, Hz */
    int32_t centerfreq;       /* input_t.centerfreq, Hz */
    int32_t tau_us;           /* device "tau" µs; <0 = global default alpha = exp(-1/(WAVE_RATE*2e-4)) (.cpp:87, config.cpp:777-781) */
    int32_t channel_count;
    const ba_channel_desc* channels;
} ba_device_desc;

/* One mixer input = one channel output of type "mixer" (mixer_connect_input, src/mixer.cpp:55-93; config.cpp:173-194). */
typedef struct ba_mixer_input_desc {
    int32_t device;  /* index into ba_engine_desc.devices */
    int32_t channel; /* index into that device's channels */
    float ampfactor; /* output "ampfactor", default 1.0 */
    float balance;   /* output "balance" -1..1, default 0; any non-zero balance makes the mixer stereo */
} ba_mixer_input_desc;

/* One mixer_t (src/boondock_airband.h mixer_t, src/mixer.cpp).  Inputs are summed in this order. */
typedef struct ba_mixer_desc {
    int32_t input_count;
    const ba_mixer_input_desc* inputs;
} ba_mixer_desc;

/* The globals demodulate() reads (src/boondock_airband.cpp:71-90), passed explicitly. */
typedef struct ba_engine_desc {
    int32_t abi_version;          /* BA_CUDA_ABI_VERSION */
    int32_t fft_size;             /* global fft_size, 256..8192 power of two */
    int32_t wave_rate;            /* WAVE_RATE: 8000 (AM-only build) or 16000 (NFM build), boondock_airband.h:67-71 */
    int32_t fm_demod;             /* BA_FM_* */
    int32_t cuda_device;          /* CUDA ordinal to run on */
    int32_t device_count;         /* devices handled by this engine = one demod thread's device_start..device_end */
    const ba_device_desc* devices;
    int32_t max_batches_per_step; /* capacity: WAVE_BATCH batches per device one ba_cuda_process() may produce; 0 = 8 */
    uint32_t flags;               /* BA_FLAG_* */
    uint64_t ring_bytes;          /* base size of each pinned input ring before rounding; 0 = MIN_BUF_SIZE 2560000 (boondock_airband.h:64) */
    /* mixers summed on the device behind the demodulator (SURVEY.md section 8, row f-4) */
    int32_t mixer_count;
    const ba_mixer_desc* mixers;
} ba_engine_desc;

/* Per-channel scalars observers read after every batch
 * (JSON status .cpp:687-726, stats file output.cpp:634-811, AFC result .cpp:238-249). */
typedef struct ba_channel_status {
    int32_t axcindicate; /* BA_NO_SIGNAL / BA_SIGNAL / BA_AFC_UP / BA_AFC_DOWN */
    uint32_t bin;        /* dev->bins[i] after AFC */
    float signal_level;  /* Squelch::signal_level() */
    float noise_level;   /* Squelch::noise_level() */
    float squelch_level; /* Squelch::squelch_level() */
    uint32_t open_count;
    uint32_t flappy_count;
    uint32_t ctcss_count;
    uint32_t no_ctcss_count;
    uint32_t active_counter; /* freq_t.active_counter (.cpp:669-671) */
} ba_channel_status;

/* Everything one ba_cuda_process() produced for one device, in pinned host memory owned by the engine. */
typedef struct ba_step_out {
    int32_t n_batches;     /* whole batches of wave_batch samples; 0 if not enough input yet */
    int32_t wave_batch;    /* WAVE_BATCH = wave_rate / 8 */
    int32_t channel_count;
    int32_t wave_stride;   /* floats between consecutive channels in waveout (and float pairs in iq_out, bytes in trace) */
    const float* waveout;  /* [channel][n_batches*wave_batch]: what output_thread reads as waveout[0..WAVE_BATCH) per batch */
    const float* iq_out;   /* [channel][n_batches*wave_batch][2] or NULL when no channel has_iq_outputs */
    const uint8_t* trace;  /* [channel][n_batches*wave_batch] decision trace, NULL unless BA_FLAG_TRACE */
    const ba_channel_status* status; /* [batch][channel] */
    uint64_t frames_done;  /* FFT frames consumed from this device's stream so far */
    /* BA_FLAG_SKIP_SILENT_ROWS only (else NULL / 0): */
    const float* rows;     /* [n_rows][wave_batch]: the rows of the whole step (all devices of that GPU) that are not silence, packed */
    const int32_t* row_of; /* [channel][max_batches_per_step] for this device: index into rows, or -1 = wave_batch samples of +0.0f */
    uint32_t n_rows;
    int32_t row_of_stride; /* = max_batches_per_step */
} ba_step_out;

/* What one ba_cuda_process() mixed for one mixer: the batches every unmasked input had delivered by the end of the step
 * (mixer_thread's output, src/mixer.cpp:166-257, with batch numbers taking the place of its 1/16 s timer). */
typedef struct ba_mixer_out {
    int32_t n_batches;      /* whole batches mixed in this step (0..max_batches_per_step) */
    int32_t wave_batch;
    int32_t stereo;         /* channel.mode == MM_STEREO */
    int32_t pad0;
    uint64_t first_batch;   /* number of the first of them (batches count from 0 per mixer) */
    const float* waveout;   /* [n_batches*wave_batch] left (or mono) */
    const float* waveout_r; /* right, NULL for a mono mixer */
    const int32_t* axcindicate; /* [n_batches] BA_SIGNAL if any input had signal in that batch, else BA_NO_SIGNAL */
} ba_mixer_out;

/* Derived per-channel constants, for inspection and parity tests. */
typedef struct ba_channel_info {
    uint32_t bin;          /* config.cpp:669-670 */
    uint32_t dm_dphi;      /* config.cpp:682-715 */
    int32_t needs_raw_iq;
    float alpha;
    float squelch_ratio;   /* normal_signal_ratio_ */
    float manual_level;    /* >0 when a manual threshold is active */
    int32_t notch_enabled;
    float notch_d[3];
    int32_t lowpass_enabled;
    float lowpass_ycoeffs[2];
    float lowpass_gain;
    int32_t ctcss_fast_tones, ctcss_slow_tones; /* detectors after de-duplication (ctcss.cpp:61-72) */
    int32_t ctcss_fast_window, ctcss_slow_window;
} ba_channel_info;

typedef struct ba_engine ba_engine;

/* Replaces init_demod()/gpu_fft_prepare (src/boondock_airband.cpp:253-266,316-332): builds the
 * window (.cpp:357-373), twiddles, per-channel constants and the resident per-channel state. */
BA_API int ba_cuda_create(const ba_engine_desc* desc, ba_engine** out);
/*
 * One engine over several GPUs: a group of ordinary engines ("members"), one per GPU that receives devices, behind one
 * handle.  No data moves between GPUs: every device runs on exactly one of them, and a mixer's inputs stay together.
 *   gpus[0..n_gpus)      CUDA ordinals; one may repeat (two members on one GPU).  desc->cuda_device is ignored.
 *   gpu_of_device        NULL, or desc->device_count indices into gpus.  NULL places devices joined by a mixer (transitively)
 *                        as one group, groups in the order of their first device, group k on gpus[k % n_gpus]; without
 *                        mixers device i goes to gpus[i % n_gpus].  An explicit map may not split a mixer's inputs.
 * A GPU that gets no device gets no member and is not touched.  BA_ERR_BAD_ARG for n_gpus < 1, an ordinal that is not
 * visible, an index out of range or a split mixer.
 * Every entry point below accepts the handle.  Device and mixer indices stay those of desc; per-device and per-mixer
 * calls go to the member that holds the device or mixer.  ba_cuda_process() runs every member's pass, in member order,
 * and returns their common ticket (members' tickets move in lockstep); ba_cuda_collect() waits for the member of the
 * device only.  ticket_ms, copy_ms, kernel_ms and mark_ms give the maximum over members; step_bytes and launch_count the
 * sum; ba_cuda_mark() records on every member.  After an error from any member the handle is only good for
 * ba_cuda_destroy() (a failed ba_cuda_process() or CUDA error makes every later call return BA_ERR_STATE). */
BA_API int ba_cuda_create_multi(const ba_engine_desc* desc, const int32_t* gpus, int32_t n_gpus, const int32_t* gpu_of_device, ba_engine** out);
/* The CUDA ordinal device `dev` runs on (a plain engine: its cuda_device).  Memory given to ba_cuda_attach_device_stream()
 * must be on that GPU, and the BA_FLAG_RESULTS_ON_DEVICE pointers of the device point there. */
BA_API int ba_cuda_device_gpu(ba_engine* e, int dev, int32_t* cuda_ordinal);
/* Replaces gpu_fft_release (src/boondock_airband.cpp:385-388). */
BA_API void ba_cuda_destroy(ba_engine* e);
/* Text of the most recent failure on this thread (never NULL). */
BA_API const char* ba_cuda_last_error(void);
/* Number of CUDA devices visible, or a negative BA_ERR_*. */
BA_API int ba_cuda_visible_devices(void);

/* The pinned host ring that takes the place of input_t.buffer (allocation: src/config.cpp:796-805):
 * buf_size bytes plus a mirror tail of 2*bytes_per_sample*fft_size bytes, same arithmetic. */
BA_API int ba_cuda_input_ring(ba_engine* e, int dev, unsigned char** buffer, size_t* buf_size, size_t* mirror_bytes);

/* Replaces circbuffer_append() for callers that do not own an input_t (src/input-helpers.cpp:37-63):
 * appends `bytes` of interleaved IQ from host memory to the device's stream.  */
BA_API int ba_cuda_submit(ba_engine* e, int dev, const void* iq, size_t bytes);
/* Bytes ba_cuda_submit() would accept right now (the space test of file_rx_thread, src/input-file.cpp:126-133). */
BA_API int ba_cuda_input_space(ba_engine* e, int dev, size_t* free_bytes);
/* Same, for callers that wrote into the ring from ba_cuda_input_ring() themselves
 * (the rx thread of an unmodified input driver): publishes `bytes` more bytes at the ring's write index. */
BA_API int ba_cuda_commit(ba_engine* e, int dev, size_t bytes);
/* The ring's read index as demodulate() would have left it in input_t.bufs (bufs = (bufs + bps) % buf_size,
 * src/boondock_airband.cpp:735): bytes before it have been copied to the device and may be overwritten by the rx thread. */
BA_API int ba_cuda_input_consumed(ba_engine* e, int dev, size_t* bufs);

/* Zero-copy variant for producers that already hold their samples in (ideally pinned) host memory: the bytes are
 * copied host->device straight from `iq` during the next ba_cuda_process() calls, without passing through the ring.
 * The memory must stay valid and unchanged until the ticket that consumed it has been collected. */
BA_API int ba_cuda_submit_external(ba_engine* e, int dev, const void* iq, size_t bytes);

/* Device-resident input (benchmarks, GPUDirect producers): the stream lives in HBM at d_iq (16-byte aligned, as every
 * device allocation is; the channelizer fetches whole 16-byte granules, so the allocation must extend to the next
 * multiple of 16 past capacity_bytes, which cudaMalloc guarantees); ba_cuda_advance_device_stream() says how many more
 * bytes of it are valid. */
BA_API int ba_cuda_attach_device_stream(ba_engine* e, int dev, const void* d_iq, size_t capacity_bytes);
BA_API int ba_cuda_advance_device_stream(ba_engine* e, int dev, size_t bytes);

/* One pass of the hot path over everything submitted so far, for all devices of the engine
 * (replaces the body of the while(true) loop, src/boondock_airband.cpp:383-737): host->device copy,
 * expand+window+FFT+bin pick, fused per-channel demodulation, device->host copy of the results.
 * Asynchronous; returns a ticket >= 0.  At most three tickets may be outstanding (a fourth ba_cuda_process()
 * first waits for the oldest one and reuses its result buffers). */
BA_API int ba_cuda_process(ba_engine* e);
/* Waits for `ticket` and describes what it produced for device `dev` (replaces the hand-off
 * waveavail=1 + Signal::send(), src/boondock_airband.cpp:673-679,728).  Pointers stay valid until
 * three more ba_cuda_process() calls have been made. */
BA_API int ba_cuda_collect(ba_engine* e, int ticket, int dev, ba_step_out* out);
/* Same for mixer `mixer` of the engine descriptor: what mixer_thread would hand to the output thread (src/mixer.cpp:166-257). */
BA_API int ba_cuda_collect_mixer(ba_engine* e, int ticket, int mixer, ba_mixer_out* out);
/* mixer_disable_input() (src/mixer.cpp:96-112): enabled == 0 masks the input - it is neither waited for nor summed from the next
 * ba_cuda_process() on.  There is no way back, as in the reference (it has no mixer_enable_input()): enabled != 0 on an input that is
 * masked returns BA_ERR_STATE; on one that is not it changes nothing. */
BA_API int ba_cuda_mixer_input_mask(ba_engine* e, int mixer, int input, int enabled);
/* Scan mode (row f-3): what controller_thread's `channels[0].freq_idx = i` does (src/boondock_airband.cpp:101-139): from the
 * next ba_cuda_process() on, the channel runs with freqlist[freq_idx] — its own Squelch, filters, AGC level, modulation,
 * ampfactor and counters, which resume where they were left (demodulate() reads freq_idx once per batch, :522).
 * *from_batch (optional) receives the number of the first batch of the device that runs with it.  Retuning the input
 * (input_set_centerfreq) stays the caller's business. */
BA_API int ba_cuda_set_freq_idx(ba_engine* e, int dev, int channel, int freq_idx, uint64_t* from_batch);
/* Device time (ms) between the first and last GPU operation of a finished ticket. */
BA_API int ba_cuda_ticket_ms(ba_engine* e, int ticket, float* ms);

/* Bytes the ticket moved host->device (input samples) and device->host (results). */
BA_API int ba_cuda_step_bytes(ba_engine* e, int ticket, uint64_t* h2d, uint64_t* d2h);

/* Timing marks on the engine's own CUDA stream (torch/CUDA events of the caller do not see that stream):
 * ba_cuda_mark records mark `which` (0..7) behind everything queued so far; ba_cuda_mark_ms waits for both marks
 * and returns the device time between them. */
BA_API int ba_cuda_mark(ba_engine* e, int which);
BA_API int ba_cuda_mark_ms(ba_engine* e, int from, int to, float* ms);

BA_API int ba_cuda_channel_info(ba_engine* e, int dev, int channel, ba_channel_info* out);
/* Window as computed at create time, fft_size floats (src/boondock_airband.cpp:357-373). */
BA_API int ba_cuda_window(ba_engine* e, float* out, size_t count);

/* Parity hooks (used only by tests): run the expand+window stage and the FFT on `n_frames` frames taken
 * `hop_bytes` apart from `iq` (host memory, format of device `dev`) and return the converted frames
 * (fftin, [n_frames][fft_size][2]) and/or full spectra (fftout, same shape).  Either output may be NULL. */
BA_API int ba_cuda_debug_frames(ba_engine* e, int dev, const void* iq, size_t bytes, int n_frames, float* fftin, float* fftout);
/* Copy out the picked-bin IQ series the last finished ticket consumed for one channel:
 * frames [first, first+count) of the device's stream, as (re,im) pairs.  Needs BA_FLAG_KEEP_PICKS (or a raw-IQ channel). */
BA_API int ba_cuda_debug_picks(ba_engine* e, int dev, int channel, uint64_t first, int count, float* out);
/* Parity hook: append `n_frames` rows of externally computed picked-bin IQ ([n_frames][channel_count][2] floats) to the
 * device's pick ring as if the channelizer had produced them; the next ba_cuda_process() demodulates them.  Lets the
 * tests check the demodulator bit for bit on the oracle's own FFT output.  Not to be mixed with byte input. */
BA_API int ba_cuda_debug_inject_picks(ba_engine* e, int dev, const float* picks, int n_frames);
/* Kernel launch counters since create (all kernels are this library's own). */
BA_API int ba_cuda_launch_count(ba_engine* e, uint64_t* launches);
/* Per-kernel accumulated device time of the last finished ticket: ms[0]=channelize (K1), ms[1]=demod (K2). */
BA_API int ba_cuda_kernel_ms(ba_engine* e, int ticket, float ms[2]);

/* Copy legs of a finished ticket: ms[0] = host->device (input bytes + descriptors), ms[1] = device->host (results),
 * each from the first to the last operation of that leg on its own stream. */
BA_API int ba_cuda_copy_ms(ba_engine* e, int ticket, float ms[2]);

#ifdef __cplusplus
}
#endif
#endif /* BA_CUDA_H */
