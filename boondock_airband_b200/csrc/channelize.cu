/*
 * channelize.cu — K1: sample expansion + window + batched in-shared-memory FFT + per-channel bin pick (sm_100a).
 *
 * Replaces, for FFT_BATCH-style batches of sliding frames (boondock_airband.h:94, the VideoCore path's shape):
 *   sample expansion tables + window multiply   boondock_airband.cpp:338-346, 426-479   (samplefft on the Pi, rtl_airband_neon.s:28-83)
 *   fftwf_execute / gpu_fft_execute             boondock_airband.cpp:481-485
 *   bin pick                                    boondock_airband.cpp:507-513            (the magnitude is taken in K2)
 *
 * Shape of the kernel
 *   - persistent CTAs pull tiles from a launch-wide counter; a tile = `tile_frames` consecutive frames of one input;
 *   - the byte span of the tile (frames overlap by fft_size - hop samples) is brought into shared memory by ONE bulk
 *     copy (cp.async.bulk -> UBLKCP, completion on an mbarrier) into the idle half of a double buffer while the FFT groups
 *     work on the other half: every input byte is read from HBM/L2 once per tile and no thread waits on a global load;
 *   - an FFT is done by a group of G = N/V threads, V = 16 complex values per thread per pass (32 for N = 512: a half warp
 *     per FFT there and for 256; 2..16 warps above), mixed radix 2/4/8/16/32 decimation in frequency, 2..4 passes;
 *     window values and twiddles of a thread do not depend on the frame, they live in registers;
 *   - between passes the data goes through a per-group shared-memory buffer whose layouts are padded/skewed so that
 *     every 8-byte load and store of a half warp hits 16 distinct bank pairs;
 *   - the last pass leaves the spectrum in a digit-reversed order; only the configured bins are read out
 *     (pick table built per input) and written transposed, picks[channel][frame ring] / mags[channel][frame ring].
 * Sample conversion is exact: u8 levels (i - 127.5f) / 127.5f are reproduced with a two-float reciprocal
 * (verified for all 256 codes by tests), products use round-to-nearest multiplies that are never contracted.
 * No cuFFT, no tensor cores: the work is FP32 butterflies and shared-memory transposes.
 */
#include <stdint.h>

#include <map>
#include <mutex>
#include <utility>

#include "ba_kernels.h"
#include "ba_f32x2.h"

namespace ba {
namespace {

/* V complex values per thread, radices of the passes.  N = 512 keeps 32 values per thread (16 threads per FFT, two FFTs per
 * warp) so that two passes (32 x 16) and ONE trip through shared memory do it: with the arithmetic on packed FP32 pairs the
 * kernel is bound by the shared-memory pipe (profiles/), and the 8 x 8 x 8 plan made two trips.  N = 1024 likewise: 32 x 32,
 * one warp per FFT (cfg5 at fft 1024: 8.1 -> 6.5 ms per launch).  N = 8192: 32 x 16 x 16 with 256 threads, three passes
 * instead of four (cfg4: 2.57 -> 2.35 ms).  2048 and 4096 need three passes either way and stay at 16 values. */
template <int N>
struct Plan;
#define BA_PLAN(N_, V_, T_, REGS_, CTAS_, P_, A, B, C, D)                                          \
    template <>                                                                             \
    struct Plan<N_> {                                                                       \
        static constexpr int V = V_;       /* values per thread */                          \
        static constexpr int THREADS = T_; /* threads per CTA */                            \
        static constexpr int REGS = REGS_; /* register cap */                               \
        static constexpr int CTAS = CTAS_; /* resident CTAs per SM the cap is chosen for */ \
        /* N = 8192: the 32 window values and 2 x 31 twiddles of a thread would take 156 registers and leave room for one CTA of  \
         * eight warps per SM; they are read through L1 where they are used instead, the frames are read straight from global     \
         * memory (a frame is 64 KB of cf32: staging tiles of them in shared memory is what kept a second CTA out), and two CTAs  \
         * are resident */                                                                   \
        static constexpr bool DIRECT = (N_ == 8192);                                         \
        static constexpr int P = P_;                                                        \
        static constexpr int r(int i) { return i == 0 ? A : (i == 1 ? B : (i == 2 ? C : D)); } \
    };
/* 112 registers: two CTAs of 256 threads leave 8192 registers per SM for the demodulator's warps, which run beside this kernel;
 * the 32-value plans run CTAs of 128 threads: two at 224 registers for N = 1024, three at 168 for N = 512 (a few values
 * spill; measured 4.6 % faster on the 512-input workload than two at 224: 3.68 vs 3.85 ms per step) */
BA_PLAN(256, 16, 256, 112, 2, 2, 16, 16, 1, 1)
BA_PLAN(512, 32, 128, 168, 3, 2, 32, 16, 1, 1)
BA_PLAN(1024, 32, 128, 224, 2, 2, 32, 32, 1, 1)
BA_PLAN(2048, 16, 256, 112, 2, 3, 8, 16, 16, 1)
BA_PLAN(4096, 16, 256, 112, 2, 3, 16, 16, 16, 1)
BA_PLAN(8192, 32, 256, 128, 2, 3, 32, 16, 16, 1)

template <int N>
struct Geo {
    using PL = Plan<N>;
    static constexpr int P = PL::P;
    static constexpr int V = PL::V;
    static constexpr int G = N / V; /* threads per FFT */
    static constexpr int THREADS = PL::THREADS;
    static constexpr int W = THREADS / G; /* FFT groups per CTA */
    /* Two FFT groups share a warp when G = 16, and their frames lie a multiple of 128 bytes apart: read in the same order, the
     * two half-warps would load their samples from the same banks.  The odd group therefore reads (and keeps) its samples
     * rotated by one row of the first pass, x'[j] = x[(j + 1) mod R]; a rotation by r multiplies output k of that pass by
     * W_R^(-rk), which the odd group's twiddles take back (they are per-thread constants anyway). */
    static constexpr bool ROT = (G == 16) && (V / PL::r(0) == 1);
    static constexpr int WORK = N + N / 8; /* float2 per group */
    static constexpr int R(int pass) { return PL::r(pass - 1); } /* pass = 1..P */
    static constexpr int Q(int level) { /* blocks after `level` passes */
        int q = 1;
        for (int i = 0; i < level; i++)
            q *= PL::r(i);
        return q;
    }
    static constexpr int M(int level) { return N / Q(level); }
    /* shared-memory position (in float2) of element `pos` of block `q` after `level` passes, 1 <= level <= P-1 */
    static __host__ __device__ constexpr int at(int level, int q, int pos) {
        if (level == P - 1)
            return pos * (Q(level) + 1) + q; /* feeds the last pass: position-major, odd row stride */
        const int next = M(level) / R(level + 1);
        const int stride = M(level) + (next < 16 ? 8 : 0);
        return q * stride + pos;
    }
    /* where the last pass leaves X[bin] */
    static __host__ __device__ constexpr int out_pos(int bin) {
        int q = 0, k = 0;
        for (int pass = 1; pass <= P; pass++) {
            k = bin % R(pass);
            bin /= R(pass);
            if (pass < P)
                q = q * R(pass) + k;
        }
        return k * (N / R(P)) + q;
    }
};

/* Complex arithmetic on Blackwell's packed FP32 pairs: a float2 (re, im) lives in an aligned register pair and
 * add/sub/mul/fma.rn.f32x2 (SASS FADD2/FMUL2/FFMA2) work on both halves at once.  ptxas folds component swaps, per-component
 * sign flips and scalar broadcasts of the operands into the instruction (R.F32x2.LO_HI.NP, R.F32), so a complex add or
 * subtract is ONE instruction, a multiply by -j is free, and a complex multiply is FMUL2 + FFMA2.  The kernel is bound by
 * instruction issue (profiles/): this halves the FP32 instruction count of the butterflies, twiddles and the sample
 * conversion.  Every component is still an individually rounded IEEE operation (the conversions stay bit-exact). */
/* (add2 / sub2 / mul2 / fma2: ba_f32x2.h) */
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return add2(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return sub2(a, b); }
/* (a.x b.x - a.y b.y, a.y b.x + a.x b.y) = (-a.y, a.x) * b.y + a * b.x */
__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return fma2(make_float2(-a.y, a.x), make_float2(b.y, b.y), mul2(a, make_float2(b.x, b.x))); }
__device__ __forceinline__ float2 mul_mj(float2 a) { return make_float2(a.y, -a.x); } /* a * (-j): an operand swizzle of whatever reads it */
/* a * exp(-j pi/4) = c * (a + a*(-j)) and a * exp(-3j pi/4) = c * (a*(-j) - a), c = sqrt(1/2) */
__device__ __forceinline__ float2 rot_m45(float2 a, float c) { return mul2(add2(a, mul_mj(a)), make_float2(c, c)); }
__device__ __forceinline__ float2 rot_m135(float2 a, float c) { return mul2(sub2(mul_mj(a), a), make_float2(c, c)); }

template <int R>
struct Dft;
template <>
struct Dft<1> {
    static __device__ __forceinline__ void run(float2*) {}
};
template <>
struct Dft<2> {
    static __device__ __forceinline__ void run(float2* x) {
        float2 a = x[0], b = x[1];
        x[0] = cadd(a, b);
        x[1] = csub(a, b);
    }
};
template <>
struct Dft<4> {
    static __device__ __forceinline__ void run(float2* x) {
        float2 t0 = cadd(x[0], x[2]), t1 = csub(x[0], x[2]);
        float2 t2 = cadd(x[1], x[3]), t3 = mul_mj(csub(x[1], x[3]));
        x[0] = cadd(t0, t2);
        x[1] = cadd(t1, t3);
        x[2] = csub(t0, t2);
        x[3] = csub(t1, t3);
    }
};
template <>
struct Dft<8> {
    static __device__ __forceinline__ void run(float2* x) {
        const float c = 0.70710678118654752440f;
        float2 a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            a[i] = cadd(x[i], x[i + 4]);
            b[i] = csub(x[i], x[i + 4]);
        }
        b[1] = rot_m45(b[1], c);
        b[2] = mul_mj(b[2]);
        b[3] = rot_m135(b[3], c);
        Dft<4>::run(a);
        Dft<4>::run(b);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            x[2 * i] = a[i];
            x[2 * i + 1] = b[i];
        }
    }
};
template <>
struct Dft<16> {
    static __device__ __forceinline__ void run(float2* x) {
        const float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f, c = 0.70710678118654752440f;
        float2 a[8], b[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            a[i] = cadd(x[i], x[i + 8]);
            b[i] = csub(x[i], x[i + 8]);
        }
        /* b[i] *= exp(-2 pi i * i / 16) */
        b[1] = cmul(b[1], make_float2(c1, -s1));
        b[2] = rot_m45(b[2], c);
        b[3] = cmul(b[3], make_float2(s1, -c1));
        b[4] = mul_mj(b[4]);
        b[5] = cmul(b[5], make_float2(-s1, -c1));
        b[6] = rot_m135(b[6], c);
        b[7] = cmul(b[7], make_float2(-c1, -s1));
        Dft<8>::run(a);
        Dft<8>::run(b);
#pragma unroll
        for (int i = 0; i < 8; i++) {
            x[2 * i] = a[i];
            x[2 * i + 1] = b[i];
        }
    }
};

template <>
struct Dft<32> {
    static __device__ __forceinline__ void run(float2* x) {
        /* exp(-2 pi i k / 32), k = 1..7 (cos, sin); the others follow by symmetry */
        const float c1 = 0.98078528040323044913f, s1 = 0.19509032201612826785f, c2 = 0.92387953251128675613f, s2 = 0.38268343236508977173f;
        const float c3 = 0.83146961230254523708f, s3 = 0.55557023301960222474f, c = 0.70710678118654752440f;
        float2 a[16], b[16];
#pragma unroll
        for (int i = 0; i < 16; i++) {
            a[i] = cadd(x[i], x[i + 16]);
            b[i] = csub(x[i], x[i + 16]);
        }
        b[1] = cmul(b[1], make_float2(c1, -s1));
        b[2] = cmul(b[2], make_float2(c2, -s2));
        b[3] = cmul(b[3], make_float2(c3, -s3));
        b[4] = rot_m45(b[4], c);
        b[5] = cmul(b[5], make_float2(s3, -c3));
        b[6] = cmul(b[6], make_float2(s2, -c2));
        b[7] = cmul(b[7], make_float2(s1, -c1));
        b[8] = mul_mj(b[8]);
        b[9] = cmul(b[9], make_float2(-s1, -c1));
        b[10] = cmul(b[10], make_float2(-s2, -c2));
        b[11] = cmul(b[11], make_float2(-s3, -c3));
        b[12] = rot_m135(b[12], c);
        b[13] = cmul(b[13], make_float2(-c3, -s3));
        b[14] = cmul(b[14], make_float2(-c2, -s2));
        b[15] = cmul(b[15], make_float2(-c1, -s1));
        Dft<16>::run(a);
        Dft<16>::run(b);
#pragma unroll
        for (int i = 0; i < 16; i++) {
            x[2 * i] = a[i];
            x[2 * i + 1] = b[i];
        }
    }
};

template <int N>
__device__ __forceinline__ void group_sync(int grp) {
    constexpr int G = Geo<N>::G;
    if (G <= 32) {
        __syncwarp();
    } else if (Geo<N>::W == 1) {
        __syncthreads();
    } else {
        BA_BAR_SYNC(1 + grp, G);
    }
}

/* exact (i - 127.5f) / 127.5f for the byte `which` (0..3) of `word`, boondock_airband.cpp:341-343.
 * PRMT drops the byte into mantissa bits 8..15 of 2^15, i.e. the float 32768 + v; v - 127.5 is then one exact subtraction.
 * The quotient a / 127.5 is a * (r_hi + r_lo) with the reciprocal split in two floats: fma(a, r_hi, RN(a * r_lo)) equals the
 * correctly rounded quotient for all 256 codes (checked exhaustively by tests/test_gpu_parity.py::test_u8_all_codes and,
 * in exact rational arithmetic, by tests/test_oracle_pins.py::test_u8_level_formula). */
template <int WHICH>
__device__ __forceinline__ float level_u8(unsigned word) {
    const float f = __uint_as_float(__byte_perm(word, 0x47000000u, 0x7604u | (WHICH << 4)));
    const float a = __fadd_rn(f, -32895.5f); /* v - 127.5, exact */
    const float r_hi = 0x1.010102p-7f, r_lo = -0x1.fdfdfep-32f;
    return __fmaf_rn(a, r_hi, __fmul_rn(a, r_lo));
}
/* i / 128.0f, boondock_airband.cpp:344-346 (code 0x80 is left undefined by the reference; -1.0 here) */
__device__ __forceinline__ float level_s8(unsigned v) {
    return __fmul_rn((float)(int)(signed char)v, 0.0078125f);
}

/* both components of one u8 sample at once: the same four individually rounded operations as level_u8, then the window */
__device__ __forceinline__ float2 sample_u8(unsigned v, float w) {
    const float2 f = make_float2(__uint_as_float(__byte_perm(v, 0x47000000u, 0x7604u)), __uint_as_float(__byte_perm(v, 0x47000000u, 0x7614u)));
    const float2 a = add2(f, make_float2(-32895.5f, -32895.5f)); /* v - 127.5, exact */
    const float r_hi = 0x1.010102p-7f, r_lo = -0x1.fdfdfep-32f;
    const float2 q = fma2(a, make_float2(r_hi, r_hi), mul2(a, make_float2(r_lo, r_lo)));
    return mul2(q, make_float2(w, w));
}

template <int N, int FMT>
__device__ __forceinline__ float2 load_sample(const unsigned char* frame, int n, float w, float scale) {
    if (FMT == BA_SFMT_U8) {
        const unsigned v = *reinterpret_cast<const unsigned short*>(frame + 2 * n);
        return sample_u8(v, w);
    } else if (FMT == BA_SFMT_S8) {
        const unsigned v = *reinterpret_cast<const unsigned short*>(frame + 2 * n);
        return make_float2(__fmul_rn(level_s8(v & 0xffu), w), __fmul_rn(level_s8(v >> 8), w));
    } else if (FMT == BA_SFMT_S16) {
        const short2 v = *reinterpret_cast<const short2*>(frame + 4 * n);
        return mul2(mul2(make_float2(scale, scale), make_float2((float)v.x, (float)v.y)), make_float2(w, w));
    } else {
        const float2 v = *reinterpret_cast<const float2*>(frame + 8 * n);
        return mul2(mul2(make_float2(scale, scale), v), make_float2(w, w));
    }
}

/* per-thread constants that do not depend on the frame: in registers, or (Plan::DIRECT) where to read them */
template <int N, bool DIRECT = Plan<N>::DIRECT>
struct ThreadConst {
    float win[Geo<N>::V];
    float2 tw[Geo<N>::P - 1][Geo<N>::V - 1];
};
template <int N>
struct ThreadConst<N, true> {
    const float* window;  /* [N] */
    const float2* table;  /* [N] exp(-2 pi i n / N) */
};

template <int N, int PASS>
__device__ __forceinline__ void twiddle_setup(ThreadConst<N>& tc, const float2* __restrict__ table, int t, int rot) {
    using GE = Geo<N>;
    if constexpr (Plan<N>::DIRECT) {
        tc.table = table;
    } else if constexpr (PASS < GE::P) {
        constexpr int R = GE::R(PASS);
        constexpr int NB = GE::V / R;
        constexpr int Mp = GE::M(PASS);       /* positions per block after this pass */
        constexpr int Qprev = GE::Q(PASS - 1);
#pragma unroll
        for (int i = 0; i < NB; i++) {
            const int u = t + GE::G * i;
            const int m = u % Mp;
#pragma unroll
            for (int k = 1; k < R; k++) {
                float2 w = table[k * m * Qprev];
                if (PASS == 1 && GE::ROT && rot)
                    w = cmul(w, table[(k * (N / R)) & (N - 1)]); /* W_R^k: undoes the rotation of the odd group's inputs */
                tc.tw[PASS - 1][i * (R - 1) + (k - 1)] = w;
            }
        }
        twiddle_setup<N, PASS + 1>(tc, table, t, rot);
    }
}

template <int N, int FMT, int PASS>
__device__ __forceinline__ void fft_pass(const ThreadConst<N>& tc, float2* __restrict__ work, const unsigned char* frame, float scale, int t,
                                         int grp, float2* dbg_in) {
    using GE = Geo<N>;
    constexpr int R = GE::R(PASS);
    constexpr int NB = GE::V / R;
    constexpr int Mp = GE::M(PASS);
    constexpr bool FIRST = PASS == 1, LAST = PASS == GE::P;
    float2 x[NB][R];
#pragma unroll
    for (int i = 0; i < NB; i++) {
        const int u = t + GE::G * i;
        const int q = u / Mp, m = u % Mp;
#pragma unroll
        for (int j = 0; j < R; j++) {
            if (FIRST) {
                int n = j * Mp + m;
                if (GE::ROT) { /* ((j + rot) mod R) * Mp + m */
                    const int rot = grp & 1;
                    n += rot * Mp - ((j == R - 1) ? rot * R * Mp : 0);
                }
                float w;
                if constexpr (Plan<N>::DIRECT)
                    w = __ldg(tc.window + n);
                else
                    w = tc.win[i * R + j];
                x[i][j] = load_sample<N, FMT>(frame, n, w, scale);
                if (dbg_in)
                    dbg_in[n] = x[i][j];
            } else {
                x[i][j] = work[GE::at(PASS - 1, q, j * Mp + m)];
            }
        }
    }
    /* every load of this pass (and every read of the previous frame's spectrum) precedes the stores below */
    group_sync<N>(grp);
    if constexpr (Plan<N>::DIRECT && !LAST) {
        /* Twiddles made in registers: W^(k m), k = 1 .. R-1, is the product of W^(2^b m) over the set bits b of k; the log2 R base
         * powers come from the table (each correctly rounded), so a twiddle is at most log2 R - 1 complex products away from
         * exact values.  Reading all of them through L1 instead made the load/store pipe the bound of this kernel (83 % of its
         * wavefront rate, most of it scattered twiddle sectors) while the FMA pipe idled at 27 %.  The blocks of a thread share
         * m (G is a multiple of the block length), so one set serves them all. */
        static_assert(GE::G % Mp == 0, "the blocks of a thread share their twiddles");
        constexpr int LR = (R == 32) ? 5 : ((R == 16) ? 4 : ((R == 8) ? 3 : ((R == 4) ? 2 : 1)));
        const int m = t % Mp;
        float2 base[LR];
#pragma unroll
        for (int b = 0; b < LR; b++)
            base[b] = __ldg(tc.table + ((m * GE::Q(PASS - 1)) << b));
#pragma unroll
        for (int i = 0; i < NB; i++)
            Dft<R>::run(x[i]);
        float2 pw[R];
#pragma unroll
        for (int k = 1; k < R; k++) {
            const int rest = k & (k - 1); /* k without its lowest set bit */
            const int low = (k & 1) ? 0 : ((k & 2) ? 1 : ((k & 4) ? 2 : ((k & 8) ? 3 : 4))); /* its position */
            pw[k] = rest == 0 ? base[low] : cmul(pw[rest], base[low]);
#pragma unroll
            for (int i = 0; i < NB; i++) {
                const int u = t + GE::G * i;
                work[GE::at(PASS, (u / Mp) * R + k, m)] = cmul(x[i][k], pw[k]);
            }
        }
#pragma unroll
        for (int i = 0; i < NB; i++) {
            const int u = t + GE::G * i;
            work[GE::at(PASS, (u / Mp) * R, m)] = x[i][0];
        }
    } else {
#pragma unroll
        for (int i = 0; i < NB; i++) {
            const int u = t + GE::G * i;
            const int q = u / Mp, m = u % Mp;
            Dft<R>::run(x[i]);
#pragma unroll
            for (int k = 0; k < R; k++) {
                if (LAST) {
                    work[k * (N / R) + q] = x[i][k];
                } else {
                    float2 v = x[i][0];
                    if (k != 0) {
                        if constexpr (Plan<N>::DIRECT)
                            v = cmul(x[i][k], __ldg(tc.table + k * m * GE::Q(PASS - 1)));
                        else
                            v = cmul(x[i][k], tc.tw[PASS - 1][i * (R - 1) + (k - 1)]);
                    }
                    work[GE::at(PASS, q * R + k, m)] = v;
                }
            }
        }
    }
    group_sync<N>(grp);
    if constexpr (!LAST)
        fft_pass<N, FMT, PASS + 1>(tc, work, frame, scale, t, grp, dbg_in);
}

/* what the frame loop needs of a K1Device, read once per tile into registers */
struct TileCtx {
    unsigned hop_bytes, n_frames, ring_mask, ring_len, n_channels;
    unsigned long long frame0;
    float2* picks;
    float* mags;
    float scale;
};

template <int N, int FMT, bool DBG>
__device__ __forceinline__ void run_tile_frames(const ThreadConst<N>& tc, const TileCtx& c, const K1Device* dg, const unsigned char* raw0, float2* work,
                                                const uint16_t* picktab, int f0, int nf, int t, int grp) {
    using GE = Geo<N>;
    /* With rotated odd groups (Geo::ROT) a frame must meet the same rotation however the stream was cut into steps and tiles:
     * the rotation follows the parity of the frame's index in the stream.  Tiles start on even frames of their launch, so
     * swapping the two groups of a warp when the launch starts on an odd frame does it. */
    const int swap = GE::ROT ? (int)(c.frame0 & 1ull) : 0;
    for (int base = 0; base < nf; base += GE::W) {
        const int mine = base + (grp ^ swap);
        const bool live = mine < nf;
        if (GE::G == 32 && !live)
            break; /* a group that is exactly one warp synchronises with nobody else */
        const int fi = live ? mine : nf - 1; /* idle groups redo the last frame so that barriers stay uniform */
        const unsigned char* frame = raw0 + (size_t)fi * c.hop_bytes;
        const int f = f0 + fi;
        float2* dbg_in = nullptr;
        if (DBG) {
            float2* di = dg->dbg_in;
            dbg_in = (live && di) ? di + (size_t)f * N : nullptr;
        }
        fft_pass<N, FMT, 1>(tc, work, frame, c.scale, t, grp, dbg_in);
        if (live) {
            /* picked bins go out transposed, [channel][frame ring], so that the demodulator streams each channel contiguously */
            const unsigned pos = (unsigned)((c.frame0 + (unsigned long long)f) & c.ring_mask);
            for (int ch = t; ch < (int)c.n_channels; ch += GE::G) {
                const float2 v = work[picktab[ch]];
                const size_t at = (size_t)ch * c.ring_len + pos;
                if (c.picks)
                    c.picks[at] = v;
                /* wavein[] = sqrtf(re*re + im*im), boondock_airband.cpp:507-513: three separately rounded operations and an IEEE square root */
                c.mags[at] = __fsqrt_rn(__fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y)));
            }
            if (DBG) {
                float2* dout = dg->dbg_out;
                float2* spec = dg->spectrum;
                if (dout) {
                    float2* o = dout + (size_t)f * N;
                    for (int k = t; k < N; k += GE::G)
                        o[k] = work[GE::out_pos(k)];
                }
                if (spec && f == (int)c.n_frames - 1) {
                    for (int k = t; k < N; k += GE::G)
                        spec[k] = work[GE::out_pos(k)];
                }
            }
        }
    }
}

/* Persistent CTAs pull tiles from a launch-wide counter; the byte span of the next tile is fetched by one bulk copy
 * (cp.async.bulk, completion on an mbarrier) into the other half of a double buffer while the FFT groups work on this one. */
template <int N, bool DBG>
__global__ void __maxnreg__(Plan<N>::REGS) channelize_kernel(K1Params p) {
    using GE = Geo<N>;
    static_assert(!Plan<N>::DIRECT, "this size runs channelize_direct_kernel");
    BA_SHARED(smem);
    float2* work_all = reinterpret_cast<float2*>(smem + 2 * (size_t)p.raw_bytes);
    uint16_t* picktab = reinterpret_cast<uint16_t*>(work_all + GE::W * GE::WORK);
    unsigned char* tail = reinterpret_cast<unsigned char*>(picktab + ((p.max_channels + 7) & ~7));
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(tail); /* [2] */
    int* s_tile = reinterpret_cast<int*>(tail + 16);                        /* [2] tile index staged in each half */
    int* s_dev = s_tile + 2;                                                /* [2] its input */
    int* s_pre = s_dev + 2;                                                 /* [2] bytes between the 16-byte aligned copy start and frame 0 of the tile */
    const int tid = threadIdx.x;
    const int grp = tid / GE::G, t = tid % GE::G;
    float2* work = work_all + grp * GE::WORK;

    ThreadConst<N> tc;
    {
        constexpr int R = GE::R(1);
        constexpr int NB = GE::V / R;
        constexpr int M1 = GE::M(1);
#pragma unroll
        for (int i = 0; i < NB; i++) {
            const int m = (t + GE::G * i) % M1;
#pragma unroll
            for (int j = 0; j < R; j++) {
                int n = j * M1 + m;
                if (GE::ROT)
                    n += (grp & 1) * M1 - ((j == R - 1) ? (grp & 1) * R * M1 : 0);
                tc.win[i * R + j] = p.window[n];
            }
        }
        twiddle_setup<N, 1>(tc, p.twiddle, t, GE::ROT ? (grp & 1) : 0);
    }

    /* thread 0: take the next tile off the counter and start the copy of its bytes into half `half` */
    auto fetch = [&](int half) {
        const int tile = (int)atomicAdd(p.tile_counter, 1u);
        s_tile[half] = tile;
        if (tile >= p.n_tiles)
            return;
        int lo = 0, hi = p.n_dev - 1; /* input that owns this tile: last device with tile0 <= tile */
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (p.dev[mid].tile0 <= (uint32_t)tile)
                lo = mid;
            else
                hi = mid - 1;
        }
        const K1Device& d = p.dev[lo];
        const int f0 = (tile - (int)d.tile0) * p.tile_frames;
        const int nf = min(p.tile_frames, (int)d.n_frames - f0);
        const int bytes_per = (d.fmt == BA_SFMT_S16) ? 4 : (d.fmt == BA_SFMT_F32 ? 8 : 2);
        const unsigned char* g0 = d.iq + (size_t)f0 * d.hop_bytes;
        const size_t span = (size_t)(nf - 1) * d.hop_bytes + (size_t)N * bytes_per;
        /* the copy covers whole 16-byte granules; the granules of the first and last byte of the span lie inside the
         * stream's allocation because device allocations are at least 16-byte aligned and padded */
        const uintptr_t a0 = reinterpret_cast<uintptr_t>(g0) & ~(uintptr_t)15;
        const int pre = (int)(reinterpret_cast<uintptr_t>(g0) - a0);
        const unsigned bytes = (unsigned)((pre + span + 15) & ~(size_t)15);
        s_dev[half] = lo;
        s_pre[half] = pre;
        BA_MBAR_EXPECT_TX(&mbar[half], bytes);
        BA_BULK_G2S(smem + (size_t)half * p.raw_bytes, reinterpret_cast<const void*>(a0), bytes, &mbar[half]);
    };

    if (tid == 0) {
        BA_MBAR_INIT(&mbar[0], 1);
        BA_MBAR_INIT(&mbar[1], 1);
        BA_FENCE_MBAR_INIT();
        fetch(0);
    }
    __syncthreads();

    int half = 0, cur_dev = -1;
    unsigned parity = 0u; /* bit h = phase parity the next wait on mbar[h] looks for */
    for (;;) {
        const int tile = s_tile[half];
        if (tile >= p.n_tiles)
            break;
        if (tid == 0)
            fetch(half ^ 1); /* that half was last read before the barrier that ended the previous tile */
        const int di = s_dev[half];
        const K1Device* dg = p.dev + di;
        TileCtx c;
        c.hop_bytes = dg->hop_bytes;
        c.n_frames = dg->n_frames;
        c.ring_mask = dg->ring_mask;
        c.ring_len = dg->ring_mask + 1;
        c.n_channels = dg->n_channels;
        c.frame0 = dg->frame0;
        c.picks = dg->picks;
        c.mags = dg->mags;
        c.scale = dg->scale;
        const int fmt = dg->fmt;
        const int f0 = (tile - (int)dg->tile0) * p.tile_frames;
        const int nf = min(p.tile_frames, (int)c.n_frames - f0);
        const bool new_dev = di != cur_dev; /* uniform over the CTA */
        if (new_dev) {
            const uint32_t* bins = dg->bins;
            for (int ch = tid; ch < (int)c.n_channels; ch += GE::THREADS)
                picktab[ch] = (uint16_t)GE::out_pos((int)(bins[ch] & (N - 1)));
            cur_dev = di;
        }
        BA_MBAR_WAIT(&mbar[half], (parity >> half) & 1u); /* every thread waits for the bytes itself */
        parity ^= 1u << half;
#ifdef BA_EMU
        __syncthreads(); /* emulation: thread 0's copy has happened */
#else
        if (new_dev)
            __syncthreads(); /* picktab is complete (consecutive tiles of a CTA mostly belong to one input: no barrier then) */
#endif

        const unsigned char* raw0 = smem + (size_t)half * p.raw_bytes + s_pre[half];
        switch (fmt) {
            case BA_SFMT_U8:
                run_tile_frames<N, BA_SFMT_U8, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, grp);
                break;
            case BA_SFMT_S8:
                run_tile_frames<N, BA_SFMT_S8, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, grp);
                break;
            case BA_SFMT_S16:
                run_tile_frames<N, BA_SFMT_S16, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, grp);
                break;
            default:
                run_tile_frames<N, BA_SFMT_F32, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, grp);
                break;
        }
        __syncthreads(); /* every group is done with this half, with picktab and with s_tile/s_dev/s_pre of this half */
        half ^= 1;
    }
}

/* N = 8192 (Plan::DIRECT): one FFT per CTA of 256 threads at a time, frames read straight from global memory (consecutive
 * lanes read consecutive samples of a first-pass row: 256 coalesced bytes of cf32 per load; frames overlap, so all but the
 * first touch of a byte is an L2 hit), window and twiddles through L1.  Shared memory holds only the exchange buffer, 128
 * registers per thread: two or three CTAs per SM instead of one.  Tiles come off the launch-wide counter as above. */
template <int N, bool DBG>
__global__ void __maxnreg__(Plan<N>::REGS) channelize_direct_kernel(K1Params p) {
    using GE = Geo<N>;
    static_assert(GE::W == 1, "one FFT group per CTA");
    BA_SHARED(smem);
    float2* work = reinterpret_cast<float2*>(smem);
    uint16_t* picktab = reinterpret_cast<uint16_t*>(work + GE::WORK);
    int* s_tile = reinterpret_cast<int*>(picktab + ((p.max_channels + 7) & ~7));
    const int t = threadIdx.x;
    ThreadConst<N> tc;
    tc.window = p.window;
    tc.table = p.twiddle;
    int cur_dev = -1;
    for (;;) {
        __syncthreads(); /* everybody is done with s_tile and with the pick table of the tile before */
        if (t == 0)
            *s_tile = (int)atomicAdd(p.tile_counter, 1u);
        __syncthreads();
        const int tile = *s_tile;
        if (tile >= p.n_tiles)
            break;
        int lo = 0, hi = p.n_dev - 1; /* input that owns this tile: last device with tile0 <= tile */
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (p.dev[mid].tile0 <= (uint32_t)tile)
                lo = mid;
            else
                hi = mid - 1;
        }
        const K1Device* dg = p.dev + lo;
        TileCtx c;
        c.hop_bytes = dg->hop_bytes;
        c.n_frames = dg->n_frames;
        c.ring_mask = dg->ring_mask;
        c.ring_len = dg->ring_mask + 1;
        c.n_channels = dg->n_channels;
        c.frame0 = dg->frame0;
        c.picks = dg->picks;
        c.mags = dg->mags;
        c.scale = dg->scale;
        const int fmt = dg->fmt;
        const int f0 = (tile - (int)dg->tile0) * p.tile_frames;
        const int nf = min(p.tile_frames, (int)c.n_frames - f0);
        if (lo != cur_dev) { /* uniform over the CTA */
            const uint32_t* bins = dg->bins;
            for (int ch = t; ch < (int)c.n_channels; ch += GE::THREADS)
                picktab[ch] = (uint16_t)GE::out_pos((int)(bins[ch] & (N - 1)));
            cur_dev = lo;
            __syncthreads();
        }
        const unsigned char* raw0 = dg->iq + (size_t)f0 * c.hop_bytes;
        switch (fmt) {
            case BA_SFMT_U8:
                run_tile_frames<N, BA_SFMT_U8, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, 0);
                break;
            case BA_SFMT_S8:
                run_tile_frames<N, BA_SFMT_S8, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, 0);
                break;
            case BA_SFMT_S16:
                run_tile_frames<N, BA_SFMT_S16, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, 0);
                break;
            default:
                run_tile_frames<N, BA_SFMT_F32, DBG>(tc, c, dg, raw0, work, picktab, f0, nf, t, 0);
                break;
        }
    }
}

template <int N, bool DBG>
int launch_n(const K1Params& p, int n_ctas, cudaStream_t s) {
    using GE = Geo<N>;
    const size_t smem = (size_t)k1_smem_bytes(N, p.raw_bytes, p.max_channels);
    if constexpr (Plan<N>::DIRECT) {
        auto kern = channelize_direct_kernel<N, DBG>;
        BA_LAUNCH(kern, n_ctas, GE::THREADS, smem, s, p);
    } else {
        auto kern = channelize_kernel<N, DBG>;
        BA_LAUNCH(kern, n_ctas, GE::THREADS, smem, s, p);
    }
    return (int)cudaGetLastError();
}

/* The dynamic shared-memory limit of a kernel is an attribute of the (device, function) pair: it is set per device, right
 * after cudaSetDevice() in ba_cuda_create(), for both instantiations an engine may launch there - never through a
 * process-wide flag (one process may drive one engine per GPU, boondock_airband.cpp:1088-1122). */
template <int N>
int configure_n(size_t smem) {
    cudaError_t e;
    if constexpr (Plan<N>::DIRECT) {
        e = cudaFuncSetAttribute(channelize_direct_kernel<N, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(channelize_direct_kernel<N, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    } else {
        e = cudaFuncSetAttribute(channelize_kernel<N, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(channelize_kernel<N, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    return (int)e;
}

template <int N>
int launch_dbg(const K1Params& p, int n_ctas, bool dbg, cudaStream_t s) {
    return dbg ? launch_n<N, true>(p, n_ctas, s) : launch_n<N, false>(p, n_ctas, s);
}

}  // namespace

namespace {
__global__ void __launch_bounds__(128) carry_kernel(const K1Carry* list, int n) {
    const int i = blockIdx.x;
    if (i >= n)
        return;
    const K1Carry c = list[i];
    for (uint32_t b = threadIdx.x; b < c.n; b += blockDim.x)
        c.dst[b] = c.src[b];
}
}  // namespace

int k1_carry_launch(const K1Carry* list, int n, cudaStream_t s) {
    if (n <= 0)
        return 0;
    BA_LAUNCH(carry_kernel, n, 128, 0, s, list, n);
    return (int)cudaGetLastError();
}

namespace {
template <int N>
void plan_of(int* threads, int* v, int* ctas = nullptr) {
    *threads = Plan<N>::THREADS;
    *v = Plan<N>::V;
    if (ctas)
        *ctas = Plan<N>::CTAS;
}
void plan_lookup(int n, int* threads, int* v, int* ctas = nullptr) {
    switch (n) {
        case 256: plan_of<256>(threads, v, ctas); break;
        case 512: plan_of<512>(threads, v, ctas); break;
        case 1024: plan_of<1024>(threads, v, ctas); break;
        case 2048: plan_of<2048>(threads, v, ctas); break;
        case 4096: plan_of<4096>(threads, v, ctas); break;
        default: plan_of<8192>(threads, v, ctas); break;
    }
}
}  // namespace
int k1_threads(int n) {
    int t, v;
    plan_lookup(n, &t, &v);
    return t;
}
int k1_ctas_per_sm(int n) {
    int t, v, c;
    plan_lookup(n, &t, &v, &c);
    return c;
}
int k1_groups(int n) {
    int t, v;
    plan_lookup(n, &t, &v);
    return t / (n / v);
}
/* two halves of raw bytes, the FFT work buffers, the pick table, two mbarriers and the tile bookkeeping */
int k1_smem_bytes(int n, int raw_bytes, int max_channels) {
    return 2 * raw_bytes + 8 * k1_groups(n) * (n + n / 8) + 2 * ((max_channels + 7) & ~7) + 64;
}
/* sizes whose frames are read straight from global memory: no tile staging, raw_bytes = 0 */
int k1_direct(int n) { return n == 8192 ? 1 : 0; }

/* Engines on one GPU share the attribute: one that needs less must not lower it under another's launches, so the limit
 * set per (device, FFT size) only ever goes up. */
int k1_configure(int fft_size, int raw_bytes, int max_channels) {
    static std::mutex lock;
    static std::map<std::pair<int, int>, size_t> limit;
    const size_t smem = (size_t)k1_smem_bytes(fft_size, raw_bytes, max_channels);
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess)
        return (int)e;
    std::lock_guard<std::mutex> g(lock);
    size_t& have = limit[std::make_pair(device, fft_size)];
    if (smem <= have)
        return 0;
    int rc = (int)cudaErrorInvalidValue;
    switch (fft_size) {
        case 256: rc = configure_n<256>(smem); break;
        case 512: rc = configure_n<512>(smem); break;
        case 1024: rc = configure_n<1024>(smem); break;
        case 2048: rc = configure_n<2048>(smem); break;
        case 4096: rc = configure_n<4096>(smem); break;
        case 8192: rc = configure_n<8192>(smem); break;
    }
    if (rc == 0)
        have = smem;
    return rc;
}

int k1_launch(int fft_size, const K1Params& p, int n_ctas, bool dbg, cudaStream_t s) {
    switch (fft_size) {
        case 256:
            return launch_dbg<256>(p, n_ctas, dbg, s);
        case 512:
            return launch_dbg<512>(p, n_ctas, dbg, s);
        case 1024:
            return launch_dbg<1024>(p, n_ctas, dbg, s);
        case 2048:
            return launch_dbg<2048>(p, n_ctas, dbg, s);
        case 4096:
            return launch_dbg<4096>(p, n_ctas, dbg, s);
        case 8192:
            return launch_dbg<8192>(p, n_ctas, dbg, s);
    }
    return (int)cudaErrorInvalidValue;
}

}  // namespace ba
