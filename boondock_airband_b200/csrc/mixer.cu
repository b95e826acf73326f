/*
 * mixer.cu — K3: the mixers of the reference summed on the device, behind the demodulator (SURVEY.md section 8, row f-4).
 *
 * Replaces mixer_put_samples() + the summing part of mixer_thread() (src/mixer.cpp:114-131, 133-141, 166-257) for the
 * channels of one engine: a channel output of type "mixer" hands its batch (waveout[0..WAVE_BATCH) and
 * axcindicate != NO_SIGNAL, output.cpp:562-564) to input `input` of a mixer; the mixer zeroes its own waveout, then adds
 * every input that has signal, in input order, as  sum[s] += in[s] * (ampfactor * ampl)  — and the same with ampr into
 * waveout_r when any input has a balance (MM_STEREO).  The reference pairs batches by wall-clock (a 1/16 s timer with one
 * interval of grace); at many times real time there is no clock to pair by, so batches are paired by number: batch k of a
 * mixer is the sum of batch k of each unmasked input, emitted once all of them have delivered it.  Batches an input
 * delivers ahead of the others wait in a device-resident FIFO (the role of mixinput_t.wavein, one slot deep there).
 *
 * Compiled with -fmad=false: the product and the sum round separately, as the reference's C does.
 * HBM-bound elementwise work: 4 bytes read per input sample with signal, 4 (8 stereo) written per output sample.
 *
 * Also here: ship_kernel and gather_kernel, the copies between the members of a group that spreads one input's channels
 * over several GPUs (ba_cuda_create_multi_split, DESIGN.md section 6).
 */
#include "ba_kernels.h"

namespace ba {
namespace {

/* one thread = four consecutive samples of one batch of one mixer */
__global__ void __launch_bounds__(128) mix_kernel(K3Params p) {
    const int m = blockIdx.z;
    const K3Mixer mx = p.mixer[m];
    const K3MixDyn dy = p.mix_dyn[m];
    const int b = blockIdx.y;
    if (b >= dy.n_emit)
        return;
    const int q = blockIdx.x * 128 + threadIdx.x; /* quad index inside the batch */
    const int B = p.wave_batch;
    if (q * 4 >= B)
        return;
    const uint64_t k = dy.emit0 + (uint64_t)b;
    float4 l = make_float4(0.f, 0.f, 0.f, 0.f), r = make_float4(0.f, 0.f, 0.f, 0.f); /* CH_DIRTY: memset (mixer.cpp:185-191) */
    bool any = false;
    for (int j = 0; j < mx.n_in; j++) {
        const int fi = mx.first_in + j;
        const K3In in = p.in[fi];
        const K3InDyn id = p.in_dyn[fi];
        if (!id.enabled) /* input_mask, mixer.cpp:183 */
            continue;
        const float* src;
        bool sig;
        if (k >= id.batch0) { /* delivered by this step: still in the demodulator's output rows */
            const uint64_t rel = k - id.batch0;
            src = id.wave + rel * B;
            sig = id.status[rel * id.status_stride].axcindicate != BA_NO_SIGNAL; /* output.cpp:564 */
        } else { /* delivered earlier and parked */
            const uint32_t slot = (uint32_t)(k % (uint64_t)p.fifo_depth);
            src = p.fifo + ((size_t)fi * p.fifo_depth + slot) * B;
            sig = p.fifo_sig[(size_t)fi * p.fifo_depth + slot] != 0;
        }
        if (!sig) /* has_signal == false: nothing is added (mixer.cpp:193) */
            continue;
        any = true;
        const float4 v = *reinterpret_cast<const float4*>(src + 4 * q);
        if (in.mult_l != 0.0f) { /* mix_waveforms returns early on a zero factor (mixer.cpp:134-136) */
            l.x = l.x + v.x * in.mult_l;
            l.y = l.y + v.y * in.mult_l;
            l.z = l.z + v.z * in.mult_l;
            l.w = l.w + v.w * in.mult_l;
        }
        if (mx.stereo && in.mult_r != 0.0f) {
            r.x = r.x + v.x * in.mult_r;
            r.y = r.y + v.y * in.mult_r;
            r.z = r.z + v.z * in.mult_r;
            r.w = r.w + v.w * in.mult_r;
        }
    }
    *reinterpret_cast<float4*>(dy.out_l + (size_t)b * B + 4 * q) = l;
    if (mx.stereo)
        *reinterpret_cast<float4*>(dy.out_r + (size_t)b * B + 4 * q) = r;
    if (q == 0)
        dy.sig[b] = any ? BA_SIGNAL : BA_NO_SIGNAL; /* channel->axcindicate, mixer.cpp:190,201 */
}

/* batches an input delivered beyond what its mixer emits in this step are parked: the copy of mixer_put_samples() */
__global__ void __launch_bounds__(128) stash_kernel(K3Params p) {
    const int fi = blockIdx.z;
    const K3InDyn id = p.in_dyn[fi];
    const int b = blockIdx.y;
    if (b >= id.stash_count)
        return;
    const int q = blockIdx.x * 128 + threadIdx.x;
    const int B = p.wave_batch;
    if (q * 4 >= B)
        return;
    const uint64_t k = id.stash_from + (uint64_t)b;
    const uint64_t rel = k - id.batch0;
    const uint32_t slot = (uint32_t)(k % (uint64_t)p.fifo_depth);
    const bool sig = id.status[rel * id.status_stride].axcindicate != BA_NO_SIGNAL;
    if (sig) /* memcpy only when has_signal (mixer.cpp:121-123) */
        *reinterpret_cast<float4*>(p.fifo + ((size_t)fi * p.fifo_depth + slot) * B + 4 * q) = *reinterpret_cast<const float4*>(id.wave + rel * B + 4 * q);
    if (q == 0)
        p.fifo_sig[(size_t)fi * p.fifo_depth + slot] = sig ? 1 : 0;
}

/* BA_FLAG_SKIP_SILENT_ROWS: HBM-bound elementwise work (every audio sample is read once, the rows that are kept written once) */
__global__ void __launch_bounds__(256) pack_rows_kernel(const K3PackDev* devs, int n_dev, int total_rows, const float* wave, int stride, int B, float* pack, int32_t* rowmap,
                                                        int max_batches, uint32_t* count) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= total_rows)
        return;
    int lo = 0, hi = n_dev - 1; /* device that owns row r: last one with row0 <= r */
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (devs[mid].row0 <= (uint32_t)r)
            lo = mid;
        else
            hi = mid - 1;
    }
    const K3PackDev d = devs[lo];
    const uint32_t local = (uint32_t)r - d.row0;
    const uint32_t ch = d.first_channel + local / d.n_batches, b = local % d.n_batches;
    const float4* src = reinterpret_cast<const float4*>(wave + (size_t)ch * stride + (size_t)b * B);
    const int quads = B >> 2;
    float4 v[8];
    unsigned bits = 0u;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int q = lane + 32 * i;
        v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < quads) {
            v[i] = src[q];
            bits |= __float_as_uint(v[i].x) | __float_as_uint(v[i].y) | __float_as_uint(v[i].z) | __float_as_uint(v[i].w);
        }
    }
    for (int q = lane + 256; q < quads; q += 32) { /* (wave_batch above 1024: the rest of the row, checked here, copied below) */
        const float4 x = src[q];
        bits |= __float_as_uint(x.x) | __float_as_uint(x.y) | __float_as_uint(x.z) | __float_as_uint(x.w);
    }
    const bool any = __any_sync(0xffffffffu, bits != 0u);
    int slot = -1;
    if (any) {
        if (lane == 0)
            slot = (int)atomicAdd(count, 1u);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        float4* dst = reinterpret_cast<float4*>(pack + (size_t)slot * B);
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int q = lane + 32 * i;
            if (q < quads)
                dst[q] = v[i];
        }
        for (int q = lane + 256; q < quads; q += 32)
            dst[q] = src[q];
    }
    if (lane == 0)
        rowmap[(size_t)ch * max_batches + b] = slot;
}

/* channel sharding: HBM/NVLink-bound copies, one CTA row per job, threads over the frames (samples) of the step */
__global__ void __launch_bounds__(256) ship_kernel(const XShip* jobs, int n_jobs) {
    for (int jb = blockIdx.y; jb < n_jobs; jb += gridDim.y) {
        const XShip j = jobs[jb];
        for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < j.n_frames; i += gridDim.x * 256) {
            const uint32_t pos = (uint32_t)((j.frame0 + i) & (uint64_t)j.ring_mask);
            j.dst_mags[pos] = j.src_mags[pos];
            if (j.dst_picks)
                j.dst_picks[pos] = j.src_picks[pos];
        }
    }
}

__global__ void __launch_bounds__(256) gather_kernel(const XGather* jobs, int n_jobs) {
    for (int jb = blockIdx.y; jb < n_jobs; jb += gridDim.y) {
        const XGather j = jobs[jb];
        const uint32_t t0 = blockIdx.x * 256 + threadIdx.x, step = gridDim.x * 256;
        for (uint32_t i = t0; i < j.n_samples; i += step) {
            j.dst_wave[i] = j.src_wave[i];
            if (j.dst_trace)
                j.dst_trace[i] = j.src_trace[i];
            if (j.dst_iq)
                j.dst_iq[i] = j.src_iq[i];
        }
        const uint32_t words = (uint32_t)(sizeof(ba_channel_status) / 4);
        for (uint32_t i = t0; i < j.n_batches * words; i += step) {
            const uint32_t b = i / words, w = i % words;
            reinterpret_cast<uint32_t*>(j.dst_status + (size_t)b * j.dst_status_stride)[w] =
                reinterpret_cast<const uint32_t*>(j.src_status + (size_t)b * j.src_status_stride)[w];
        }
    }
}

/* CTAs per job along the frames / samples: enough to cover a short step in one pass, few enough that a long one loops */
inline unsigned x_blocks(uint32_t n) {
    const unsigned b = (n + 255) / 256;
    return b < 1 ? 1 : (b > 8 ? 8 : b);
}

}  // namespace

int x_ship_launch(const XShip* jobs, int n_jobs, uint32_t max_frames, cudaStream_t s) {
    if (n_jobs <= 0 || max_frames == 0)
        return 0;
    BA_LAUNCH(ship_kernel, dim3(x_blocks(max_frames), n_jobs < 65535 ? n_jobs : 65535), 256, 0, s, jobs, n_jobs);
    return (int)cudaGetLastError();
}

int x_gather_launch(const XGather* jobs, int n_jobs, uint32_t max_samples, cudaStream_t s) {
    if (n_jobs <= 0 || max_samples == 0)
        return 0;
    BA_LAUNCH(gather_kernel, dim3(x_blocks(max_samples), n_jobs < 65535 ? n_jobs : 65535), 256, 0, s, jobs, n_jobs);
    return (int)cudaGetLastError();
}

int k3_pack_launch(const K3PackDev* devs, int n_dev, int total_rows, const float* wave, int stride, int wave_batch, float* pack, int32_t* rowmap, int max_batches,
                   uint32_t* count, cudaStream_t s) {
    if (total_rows <= 0)
        return 0;
    BA_LAUNCH(pack_rows_kernel, (total_rows + 7) / 8, 256, 0, s, devs, n_dev, total_rows, wave, stride, wave_batch, pack, rowmap, max_batches, count);
    return (int)cudaGetLastError();
}

int k3_launch(const K3Params& p, int n_mixers, int max_emit, int n_inputs, int max_stash, cudaStream_t s) {
    const int tiles = (p.wave_batch / 4 + 127) / 128;
    if (n_mixers > 0 && max_emit > 0) {
        BA_LAUNCH(mix_kernel, dim3(tiles, max_emit, n_mixers), 128, 0, s, p);
        int rc = (int)cudaGetLastError();
        if (rc)
            return rc;
    }
    if (n_inputs > 0 && max_stash > 0) {
        BA_LAUNCH(stash_kernel, dim3(tiles, max_stash, n_inputs), 128, 0, s, p);
        return (int)cudaGetLastError();
    }
    return 0;
}

}  // namespace ba
