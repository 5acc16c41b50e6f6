// Hand-written sm_100a kernels of the SDRReceiver channelizer hot path.
//
// Pipeline per process call (all streams of a bank, n_blocks callbacks each); kernels marked (v2) live in
// kernels_v2.cuh:
//   k0_dc_anchor / k0_dc_blocks / k0_dc_walk  DC-removal IIR (sdrj.cpp:277-283) reproduced bit for bit, one callback
//                                           ahead on a side stream
//   k1_v2 (v2)                              u8 -> f32 (sdr.cpp:43-49), DC, per main VFO NCO mix (vfo.cpp:237-245) +
//                                           11-tap half-band cascade (halfbanddecimator.cpp:43-72) -> cf32 main output
//   k1_ingest_main                          the same for cf32 input (vfo::process on a main VFO: no u8, no DC)
//   k2a_v2 (v2)                             all sub VFOs of a main VFO: NCO mix + S half-band stages -> cf32 z
//   k2_late_v2 (v2) / k2_late_fir           /5 or /6 decimating FIR (vfo.cpp:334-387); the second is the fallback
//   k2b_v2 (v2)                             delay62 - Hilbert125 (vfo.cpp:316-324), optional low-pass, gain, int16
//                                           (vfo.cpp:328)
//   k3_carry                                filter tails / raw tail / counters for the next call
//   k_state_io                              the same carried state to / from per-receiver records (outside the call)
//
// Reference quirks reproduced on purpose (SURVEY.md section 0):
//   * FIRQueueBackToFront copies one slot early (dsp.cpp:169): at every callback edge, at
//     every half-band stage, window slots that fall before the callback read one sample
//     further back ("HEAD" path of hb_stage).
//   * NCO = 1-second lookup table with |v| -> sqrt(0.95); stream sample 0 uses entry L-1.
//   * FIR::FIRUpdateAndProcess excludes the newest sample; FIRHilbert includes it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sdrb {

// ------------------------------------------------------------------------------------
// constants
// ------------------------------------------------------------------------------------
// hbcoeff11 (halfbanddecimator.h:66-79)
#define HB_P0 0.0060431029837374152f
#define HB_P2 (-0.049372515458761493f)
#define HB_P4 0.29332944952052842f
#define HB_P5 0.5f

constexpr int DC_BLK = 128;            // samples per DC-recursion block (16 K1 lanes)
constexpr int RAW_TAIL = 256;          // raw samples carried between calls (K1 halo warp)
constexpr int K1_WARPS = 8;            // active warps per K1 CTA (+1 halo warp)
constexpr int K1_THREADS = (K1_WARPS + 1) * 32;
constexpr int K1_TILE = K1_WARPS * 256;
constexpr int HB_PAD = 8;              // leading pad chunks of every smem stage array
constexpr int MAIN_HIST = 512;         // main-output samples kept in front of each call
constexpr int LATE_TILE = 256;
constexpr int MAX_FIR_TAPS = 512;

constexpr int DC_HALO_BLKS = RAW_TAIL / DC_BLK;     // table entries kept from the previous call

// Bank stream of grid index i. MAP = false: streams s0 .. s0+n-1 of the bank (every full-bank and stream-group launch); MAP = true:
// the stream-list calls, where map is the call's device copy of the caller's list and i a list position.
template <bool MAP>
__device__ __forceinline__ int map_stream(const int *__restrict__ map, int s0, int i) { return MAP ? __ldg(map + i) : s0 + i; }
#define DC_A (1.0f - 0.000001f)         /* sdrj.cpp:281, evaluated in float like the reference */
#define DC_C 0.000001f
#define DC_MAGIC 12582912.0f            /* 1.5 * 2^23: (y + M) - M rounds y to nearest-even integer */

// Per call and per (stream, arm): the float neighbourhood the DC state lives in.
// Inside (lo, hi) the state keeps its sign and exponent and the rounded product
// fl(s*a) equals s - r*ulp with r = r0 below the bit pattern T and r0 + 1 from T on.
struct DcAnchor {
    float sgn, inv_u;
    int r0, ok;
    unsigned T, lo, hi, pad;
};
// Per DC block and arm, from the integer increments d_k = Q_k - r0 (ulps of the anchor,
// U_k = their prefix sums, k < DC_BLK): D = U_DC_BLK and three bit-pattern thresholds relative
// to lo + 1 (V = bits(|state|) - (lo + 1)):
//   V < ta            =>  every state of the block stays below T    (translation by D)
//   tb <= V < tb_hi   =>  every state stays in [T, hi)               (translation by D - DC_BLK)
// ta = 0 / tb = 0xFFFFFFFF force real float stepping (no anchor).
struct DcStats { int D; unsigned ta, tb, tb_hi; };

struct MainDev {
    const float2 *lut;      // Oscillator table
    float2 *out;            // [n_streams][out_stride]: MAIN_HIST history + n_blocks*block_out
    long long out_stride;
    int lut_len, decim, block_out;
};

struct K1Params {
    const float2 *cf_in;            // cf32 input variant (vfo::process on already-converted samples)
    const float2 *cf_tail;          // [n_streams][RAW_TAIL]
    size_t cf_stride;
    const long long *blocks_done;   // [n_streams]
    int block, n_main, stream0, b0;
    MainDev mains[SDRB_MAX_MAIN];
};

struct LateDev {
    const float2 *z;                // pre-decimation samples (K2A output) -- or, for a fused mixer-only VFO, the parent's main output
    float2 *d;                      // [n_streams][d_stride]: d_hist + n_blocks*samples_out
    const float *taps;              // ntaps floats
    long long z_stride, d_stride;
    int z_hist, d_hist, block_z, samples_out, late, ntaps;
    // Fused NCO mix (sub VFOs without half-band stages, vfo.cpp:237-245 with decimateCount 0): z is never written; the late
    // kernel reads the parent's output and multiplies by the Oscillator table entry of each sample while it stages them.
    const float2 *mix_lut;          // nullptr: z holds mixed samples already
    const long long *blocks_done;   // [n_streams]: callbacks before this call (table index = (blocks_done*block_z + i) mod lut_len)
    int lut_len, pad;
};

struct UsbDev {
    const float2 *src;              // z (plain path) or d (late path), with history in front
    long long src_stride;
    int src_hist, samples_out, np, pcm_offset;
    const float *hil;               // 64 floats: 0,0, points[1], points[3], ... points[123]
    const float *lpf;               // np floats, leading zeros then the low-pass taps
    float gain;
};

struct CarryItem {
    void *base;                     // per-stream buffers of `stride` bytes
    long long stride;
    int hist_bytes, block_bytes;    // copy [hist + n*block - hist, hist + n*block) -> [0, hist)
};

// ------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// Blackwell packed FP32 pairs (FADD2 / FMUL2 / FFMA2): one issue slot for both arms of a complex
// sample. Each element is rounded exactly like the scalar .rn instruction.
__device__ __forceinline__ unsigned long long f2_bits(float2 v) { return *reinterpret_cast<unsigned long long *>(&v); }
__device__ __forceinline__ float2 bits_f2(unsigned long long v) { return *reinterpret_cast<float2 *>(&v); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
    return bits_f2(r);
}
__device__ __forceinline__ float2 splat2(float v) { return make_float2(v, v); }

// byte k of w -> (float)byte - 127  without the conversion pipe: splice the byte into the
// mantissa of 2^23 and subtract 2^23 + 127.
template <int K>
__device__ __forceinline__ float u8_to_f(uint32_t w) {
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540 | K)) - 8388735.0f;
}

// same, both arms of a sample in one FADD2: bytes 2k (I) and 2k+1 (Q) of w
template <int K>
__device__ __forceinline__ float2 u8_to_f2(uint32_t w) {
    const float2 b = make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540 | (2 * K))),
                                 __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540 | (2 * K + 1))));
    return add2(b, make_float2(-8388735.0f, -8388735.0f));
}
__device__ __forceinline__ void unpack8p(const uint4 raw, float2 (&x)[8]) {
    x[0] = u8_to_f2<0>(raw.x); x[1] = u8_to_f2<1>(raw.x);
    x[2] = u8_to_f2<0>(raw.y); x[3] = u8_to_f2<1>(raw.y);
    x[4] = u8_to_f2<0>(raw.z); x[5] = u8_to_f2<1>(raw.z);
    x[6] = u8_to_f2<0>(raw.w); x[7] = u8_to_f2<1>(raw.w);
}

__device__ __forceinline__ void unpack8(const uint4 raw, float2 (&x)[8]) {
    x[0] = make_float2(u8_to_f<0>(raw.x), u8_to_f<1>(raw.x));
    x[1] = make_float2(u8_to_f<2>(raw.x), u8_to_f<3>(raw.x));
    x[2] = make_float2(u8_to_f<0>(raw.y), u8_to_f<1>(raw.y));
    x[3] = make_float2(u8_to_f<2>(raw.y), u8_to_f<3>(raw.y));
    x[4] = make_float2(u8_to_f<0>(raw.z), u8_to_f<1>(raw.z));
    x[5] = make_float2(u8_to_f<2>(raw.z), u8_to_f<3>(raw.z));
    x[6] = make_float2(u8_to_f<0>(raw.w), u8_to_f<1>(raw.w));
    x[7] = make_float2(u8_to_f<2>(raw.w), u8_to_f<3>(raw.w));
}

template <int N> struct Log2 { static constexpr int v = 1 + Log2<N / 2>::v; };
template <> struct Log2<1> { static constexpr int v = 0; };

// Position of natural sample u (relative to the CTA's first chunk, may be negative down to
// -HB_PAD chunks) inside a padded smem stage array: chunks of CH samples, of which the last
// P are stored, STR float2 apart.
template <int CH, int P, int STR>
__device__ __forceinline__ int hb_pos(int u) {
    return ((u >> Log2<CH>::v) + HB_PAD) * STR + ((u & (CH - 1)) - (CH - P));
}

// One 11-tap half-band stage for the thread that owns input samples in[0..2R-1] (natural
// order, first one at callback coordinate v0) and produces out[0..R-1].
// Window of output m = v0/2 + r is callback coordinates 2m-10 .. 2m, taps at +0,2,4,5,6,8,10
// (dsp.cpp:139-142). Samples the thread does not own come from the previous chunks through
// `sm`. HEAD: for outputs of this callback (m >= 0), window slots with a negative coordinate
// read one sample further back -- the FIRQueueBackToFront off-by-one (dsp.cpp:163-173).
template <int R, int P, int STR, bool HEAD>
__device__ __forceinline__ void hb_stage(const float2 (&in)[2 * R], float2 (&out)[R],
                                         const float2 *__restrict__ sm, int t, int v0) {
    constexpr int CH = 2 * R;
#define HB_TAP(dst, K)                                                          \
    {                                                                           \
        const int p_ = 2 * r - 10 + (K);                                        \
        if (p_ >= 0) {                                                          \
            dst = in[p_ >= 0 ? p_ : 0];                                         \
        } else {                                                                \
            int u_ = t * CH + p_;                                               \
            if (HEAD) { if (m >= 0 && v0 + p_ < 0) u_ -= 1; }                   \
            dst = sm[hb_pos<CH, P, STR>(u_)];                                   \
        }                                                                       \
    }
    const int m0 = v0 >> 1;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int m = m0 + r;
        (void)m;
        float2 w0, w2, w4, w5, w6, w8, w10;
        HB_TAP(w0, 0) HB_TAP(w2, 2) HB_TAP(w4, 4) HB_TAP(w5, 5) HB_TAP(w6, 6) HB_TAP(w8, 8) HB_TAP(w10, 10)
        // both arms at once: 3 FADD2 + 1 FMUL2 + 3 FFMA2 per complex output
        out[r] = fma2(splat2(HB_P5), w5,
                      fma2(splat2(HB_P4), add2(w4, w6),
                           fma2(splat2(HB_P2), add2(w2, w8), mul2(splat2(HB_P0), add2(w0, w10)))));
    }
#undef HB_TAP
}

template <int R, int P, int STR>
__device__ __forceinline__ void hb_run(const float2 (&in)[2 * R], float2 (&out)[R],
                                       const float2 *__restrict__ sm, int t, int v0) {
    const int m0 = v0 >> 1;
    if (m0 >= 0 && m0 < 5) hb_stage<R, P, STR, true>(in, out, sm, t, v0);
    else hb_stage<R, P, STR, false>(in, out, sm, t, v0);
}

// store the last P of a thread's R stage outputs for its right-hand neighbours
template <int R, int P, int STR>
__device__ __forceinline__ void hb_publish(const float2 (&v)[R], float2 *__restrict__ sm, int t) {
#pragma unroll
    for (int k = R - P; k < R; ++k) sm[(t + HB_PAD) * STR + (k - (R - P))] = v[k];
}

// ------------------------------------------------------------------------------------
// K0: DC-removal IIR  avept = fl(fl(avept*a) + fl(c*x)),  a = 1 - 1e-6f  (sdrj.cpp:277-283).
//
// The recursion cannot be replaced by exact arithmetic: the rounded product fl(s*a) removes
// an INTEGER number r = RN(17*M/2^24) of ulps per sample (M = 24-bit mantissa of s, r in 9..17),
// so the state locks onto the nearest mantissa where r steps -- up to 6 % away from the ideal
// low-pass value (0.4853 instead of 0.4934 for a DC of 0.5) -- and wanders there following the
// data. That residual is audible in VFOs whose passband contains the DC line, so it is
// reproduced bit for bit:
//   k0_dc_anchor  per call: sign, ulp, r0 and the threshold T nearest to the carried state
//   k0_dc_blocks  parallel: per 32-sample block the integer increments Q_k = RN(fl(c*x_k)/ulp)
//                 and the block statistics that prove "no step of this block crosses T"
//   k0_dc_walk    one warp per stream: block after block, either a pure translation
//                 (W += D, exact in the integer-ulp domain) or 32 real float steps
// K1 then re-derives every sample's avept from the block-start states.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float dc_step(float s, float x) {
    return __fadd_rn(__fmul_rn(s, DC_A), __fmul_rn(DC_C, x));
}

// Q = RN_even(fl(c*x)/ulp) as an integer-valued float
__device__ __forceinline__ float dc_incr(const DcAnchor &A, float x) {
    const float y = __fmul_rn(__fmul_rn(DC_C, A.sgn * x), A.inv_u);
    return __fadd_rn(__fadd_rn(y, DC_MAGIC), -DC_MAGIC);
}

template <bool MAP = false>
__global__ void __launch_bounds__(128) k0_dc_anchor(const float2 *__restrict__ dc_state, DcAnchor *__restrict__ anchors,
                                                     int n_streams, int stream0, const int *__restrict__ map = nullptr) {
    const int idx = blockIdx.x * 128 + threadIdx.x;
    if (idx >= 2 * n_streams) return;
    const int stream = map_stream<MAP>(map, stream0, idx >> 1), arm = idx & 1;
    const float2 st = dc_state[stream];
    const float s0 = arm ? st.y : st.x;
    DcAnchor A;
    A.sgn = s0 < 0.f ? -1.f : 1.f; A.inv_u = 0.f; A.r0 = 0; A.ok = 0; A.T = 0; A.lo = 0; A.hi = 0; A.pad = 0;
    const float m = fabsf(s0);
    const unsigned bits = __float_as_uint(m);
    const unsigned ef = bits >> 23;
    if (ef >= 40 && ef <= 200) {
        const unsigned base = bits & 0xFF800000u;
        const float u = __uint_as_float(base - (23u << 23));
        A.inv_u = __uint_as_float((254u - (ef - 23u)) << 23);               // exactly 1/u
        const float dec = __fadd_rn(m, -__fmul_rn(m, DC_A));                 // exact: r * u
        const int r = __float2int_rn(__fmul_rn(dec, A.inv_u));
        const double step = 16777216.0 / 17.0;                               // mantissa distance between steps of r
        const double m_cur = (double)((bits & 0x7FFFFFu) + 0x800000u);
        const double m_up = ceil((r + 0.5) * step), m_dn = ceil((r - 0.5) * step);
        int r0; double m_t;
        if (fabs(m_up - m_cur) <= fabs(m_cur - m_dn)) { r0 = r; m_t = m_up; } else { r0 = r - 1; m_t = m_dn; }
        unsigned T;
        if (m_t >= 16777216.0) T = base + 0x800000u;                         // never reached inside the window
        else if (m_t < 8388608.0) T = base;                                  // always above: r = r0 + 1
        else {
            T = base + (unsigned)((long long)m_t - 8388608ll);
            for (int it = 0; it < 6; ++it) {                                 // pin T with the real float product
                const float a1 = __uint_as_float(T), a0 = __uint_as_float(T - 1);
                const float d1 = __fmul_rn(__fadd_rn(a1, -__fmul_rn(a1, DC_A)), A.inv_u);
                const float d0 = __fmul_rn(__fadd_rn(a0, -__fmul_rn(a0, DC_A)), A.inv_u);
                if (d1 >= (float)(r0 + 1) && d0 <= (float)r0) break;
                if (d1 < (float)(r0 + 1)) ++T; else --T;
            }
        }
        // window: same binade, r in {r0, r0+1}, minus the largest excursion one block can make
        double lo = 8388608.0 + 4096.0, hi = 16777216.0 - 65536.0;
        lo = fmax(lo, ceil((r0 - 0.5) * step) + 2.0);
        hi = fmin(hi, ceil((r0 + 1.5) * step) - 2.0);
        // the low side keeps a margin for the largest dip one block can make below its start;
        // the high side is checked exactly per block (DcStats::tb_hi)
        const double qmax = ceil(128.0 * (double)DC_C * (double)A.inv_u) + 18.0;
        lo += DC_BLK * qmax;
        if (hi > lo && qmax < 1.0e5) {
            A.lo = base + (unsigned)((long long)lo - 8388608ll);
            A.hi = base + (unsigned)((long long)hi - 8388608ll);
            A.r0 = r0; A.T = T; A.ok = 1;
            (void)u;
        }
    }
    anchors[2 * stream + arm] = A;
}

// The increment of a sample depends only on its byte (256 values) and on the call's anchor: d(byte) = Q - r0 with
// Q = RN_even(fl(c*x)/ulp). One table of 256 ints per stream and arm, built once per call right after the anchor: the block
// statistics and the walk's integer solves look increments up instead of redoing five float operations per sample.
// Q needs no tie handling: a half-way fl(c*x)/ulp, whose rounding in the real sum would depend on the state's parity, occurs
// only for |state| < 2^-6, where the anchor is never ok (tests/test_dc_model.py::test_no_rounding_tie_is_reachable checks
// every byte against every anchor a uint8 input can produce).
template <bool MAP = false>
__global__ void __launch_bounds__(256) k0_dc_qtab(const DcAnchor *__restrict__ anchors, int *__restrict__ qtab, int stream0,
                                                  const int *__restrict__ map = nullptr) {
    const int sa = MAP ? 2 * map_stream<MAP>(map, 0, blockIdx.x >> 1) + (blockIdx.x & 1) : 2 * stream0 + blockIdx.x;   // (stream, arm)
    const DcAnchor A = anchors[sa];
    int d = 0;
    if (A.ok) d = (int)dc_incr(A, (float)((int)threadIdx.x - 127)) - A.r0;
    qtab[(size_t)sa * 256 + threadIdx.x] = d;
}

template <bool MAP = false>
__global__ void __launch_bounds__(128) k0_dc_blocks(const uint8_t *__restrict__ iq, size_t iq_stride,
                                                     const DcAnchor *__restrict__ anchors, const int *__restrict__ qtab,
                                                     DcStats *__restrict__ stats, int stats_stride, int blk0, int n_blk, int stream0,
                                                     const int *__restrict__ map = nullptr) {
    __shared__ int sq[2][257];                                     // +1: the two arms start in different banks
    const int stream = map_stream<MAP>(map, stream0, blockIdx.y);
    for (int e = threadIdx.x; e < 512; e += 128) sq[e >> 8][e & 255] = qtab[(size_t)stream * 512 + e];
    __syncthreads();
    const int blk = blk0 + blockIdx.x * 128 + threadIdx.x;
    if (blk >= blk0 + n_blk) return;
    const DcAnchor AI = anchors[2 * stream], AQ = anchors[2 * stream + 1];
    DcStats *out = stats + ((size_t)stream * stats_stride + blk) * 2;
    DcStats bad; bad.D = 0; bad.ta = 0u; bad.tb = 0xFFFFFFFFu; bad.tb_hi = 0u;
    if (!AI.ok && !AQ.ok) { out[0] = bad; out[1] = bad; return; }
    const uint4 *src = reinterpret_cast<const uint4 *>(iq + (size_t)stream * iq_stride + (size_t)blk * (2 * DC_BLK));
    // integer ulps: u = prefix of the increments before sample k; amax = max u, bmin/bmax = min/max of u - k
    // (fused add + min/max: one VIADDMNMX each)
    int uI = 0, uQ = 0, amaxI = 0, amaxQ = 0, bminI = 0, bminQ = 0, bmaxI = 0, bmaxQ = 0;
#pragma unroll 2
    for (int v = 0; v < DC_BLK / 8; ++v) {
        const uint4 raw = __ldg(src + v);
        const unsigned w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned pr = w[k >> 1] >> (16 * (k & 1));
            const int kk = 8 * v + k;
            amaxI = max(amaxI, uI); bminI = __viaddmin_s32(uI, -kk, bminI); bmaxI = __viaddmax_s32(uI, -kk, bmaxI);
            amaxQ = max(amaxQ, uQ); bminQ = __viaddmin_s32(uQ, -kk, bminQ); bmaxQ = __viaddmax_s32(uQ, -kk, bmaxQ);
            uI += sq[0][pr & 0xffu];
            uQ += sq[1][(pr >> 8) & 0xffu];
        }
    }
    const bool badI = !AI.ok, badQ = !AQ.ok;
    // amax >= 0 >= bmin by construction (the k = 0 term), so ta <= T - lo1 <= tb
    DcStats sI, sQ;
    long long t;
    const long long lo1I = (long long)AI.lo + 1, lo1Q = (long long)AQ.lo + 1;
    sI.D = uI;
    t = (long long)AI.T - (long long)amaxI - lo1I; sI.ta = t > 0 ? (unsigned)t : 0u;
    t = (long long)AI.T - (long long)bminI - lo1I; sI.tb = t > 0 ? (unsigned)t : 0u;
    t = (long long)AI.hi - (long long)bmaxI - lo1I; sI.tb_hi = t > 0 ? (unsigned)t : 0u;
    sQ.D = uQ;
    t = (long long)AQ.T - (long long)amaxQ - lo1Q; sQ.ta = t > 0 ? (unsigned)t : 0u;
    t = (long long)AQ.T - (long long)bminQ - lo1Q; sQ.tb = t > 0 ? (unsigned)t : 0u;
    t = (long long)AQ.hi - (long long)bmaxQ - lo1Q; sQ.tb_hi = t > 0 ? (unsigned)t : 0u;
    out[0] = badI ? bad : sI;
    out[1] = badQ ? bad : sQ;
}

// Sequential part: one CTA of two warps per stream, warp 0 walks the I arm, warp 1 the Q arm.
// The loop-carried value is V = bit pattern of |state| - (lo + 1), identical in all 32 lanes.
//
//  * 32 blocks at a time, one per lane: a warp prefix sum of the block totals D gives every lane
//    the state its block would start from if all blocks before it were translations ("all below
//    T" and "all at or above T" are both tried); each lane checks its own block's thresholds and
//    a ballot finds the longest provable run. A run of 32 translations costs one scan, not 32
//    dependent steps.
//  * the block that ends a run is retried on its own; if its states really straddle T it is
//    solved by the whole warp in the integer-ulp domain (dc_solve_run): first together with the
//    three (or one) blocks behind it where the batch has them, then alone.
//  * blocks whose states leave the anchor's window fall back to 128 real float steps on lane 0.
// Raw bytes are only needed for straddling blocks; they flow through a cp.async ring anyway so
// that a straddling block never waits for HBM.
// Table entry per block and arm: {V, 0|1} (translations / integer solve), {float bits, 2} (stepped).
constexpr int DCW_BATCH = 32;
constexpr int DCW_SLOT16 = DCW_BATCH * (2 * DC_BLK / 16);                    // uint4 per ring slot
// Ring depth: the raw bytes of DCW_RING batches per arm sit in shared memory (8 KB per batch and arm). Two CTAs of the walk per
// SM next to the filter kernels is what matters: with four slots (66.5 KB) a walk CTA displaced two of the six k1_v2 CTAs of its
// SM for as long as it ran; two slots (33.5 KB) cost the walk nothing -- a batch takes thousands of cycles, HBM latency is hundreds.
constexpr int DCW_RING = 2;
constexpr size_t DCW_SMEM = (size_t)2 * DCW_RING * DCW_SLOT16 * 16 + 2 * DC_BLK * sizeof(float);

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ---- mbarrier + bulk-copy (TMA engine) helpers of k1_v2 ----
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem, const void *gmem, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     (unsigned)__cvta_generic_to_shared(smem)),
                 "l"(gmem), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}

// Integer solve of a RUN of R consecutive blocks (R * 128 samples, 4 R per lane) in one pass. The straddling blocks cluster -- the
// state dwells near its threshold for a few blocks at a time -- and one solve of four blocks costs little more than a solve of one:
// the same warp scan, the same fixed-point structure with 4 R dependent steps per lane and round. V_k = V + U_k - C_k with U the
// prefix sums of the increments and C_{i+1} = C_i + [C_i <= V + U_i - T]; the lanes iterate their indicators against the counts of
// the lanes before them (bit-sliced ballots of the per-lane counts) until nothing changes (the sequential solution is the unique
// fixed point; 2-3 rounds in practice, at most 33). Every state of the run must stay below hiw and the state after it inside
// [0, hiw), otherwise the caller falls back to a shorter run or to float steps. A run of several blocks must also keep every state
// at or above 0; a single block may dip below: the anchor's window keeps a margin of one block's largest dip at its low side.
// On success: the block-start states go to to[0], to[2], .. (one entry per block), V becomes the state after the run.
template <int R>
__device__ __forceinline__ bool dc_solve_run(const unsigned char *raw, int arm, int lane, unsigned lt_mask, const int *sqt, int Tv, int hiw,
                                             unsigned &V, uint2 *to) {
    constexpr int NS = 4 * R;                                   // samples per lane
    constexpr int BITS = R == 1 ? 3 : (R == 2 ? 4 : 5);         // bits of a lane's indicator count (<= NS)
    unsigned w[NS / 2];                                         // one 32-bit word = two IQ pairs
    if (R == 4) {
        const uint4 a = *reinterpret_cast<const uint4 *>(raw + lane * 32), c = *reinterpret_cast<const uint4 *>(raw + lane * 32 + 16);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4 % (NS / 2)] = c.x; w[5 % (NS / 2)] = c.y; w[6 % (NS / 2)] = c.z; w[7 % (NS / 2)] = c.w;
    } else if (R == 2) {
        const uint4 a = *reinterpret_cast<const uint4 *>(raw + lane * 16);
        w[0] = a.x; w[1] = a.y; w[2 % (NS / 2)] = a.z; w[3 % (NS / 2)] = a.w;
    } else {
        const uint2 a = *reinterpret_cast<const uint2 *>(raw + lane * 8);
        w[0] = a.x; w[1] = a.y;
    }
    int p[NS + 1];
    p[0] = 0;
#pragma unroll
    for (int i = 0; i < NS; ++i) p[i + 1] = p[i] + sqt[(w[i >> 1] >> (16 * (i & 1) + 8 * arm)) & 0xffu];
    const int tot = p[NS];
    int inc = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    const int base = (int)V + (inc - tot);                      // V + U at the lane's first sample
    int cin = 0, nl = 0;
    for (int it = 0; it < 34; ++it) {
        int c = cin;
#pragma unroll
        for (int i = 0; i < NS; ++i) c += (c <= base + p[i] - Tv) ? 1 : 0;
        nl = c - cin;
        int nc = 0;
#pragma unroll
        for (int bit = 0; bit < BITS; ++bit) nc += __popc(__ballot_sync(0xffffffffu, (nl >> bit) & 1) & lt_mask) << bit;
        const bool changed = nc != cin;
        cin = nc;
        if (!__any_sync(0xffffffffu, changed)) break;
    }
    // final pass: every state of the lane inside the window?
    bool inside = true;
    {
        int c = cin;
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            const int v = base + p[i] - c;
            inside &= (R == 1 || v >= 0) & (v < hiw);
            c += (c <= base + p[i] - Tv) ? 1 : 0;
        }
    }
    const int total = __shfl_sync(0xffffffffu, inc, 31);
    const int ctot = __shfl_sync(0xffffffffu, cin + nl, 31);
    const int vend = (int)V + total - ctot;
    if (!(__all_sync(0xffffffffu, inside) && vend >= 0 && vend < hiw)) return false;
    constexpr int LPB = 32 / R;                                 // lanes per block
    if ((lane & (LPB - 1)) == 0) to[(size_t)(lane / LPB) * 2] = make_uint2((unsigned)(base - cin), 0u);
    V = (unsigned)vend;
    return true;
}

template <bool MAP = false>
__global__ void __launch_bounds__(64) k0_dc_walk(const uint8_t *__restrict__ iq, size_t iq_stride,
                                                  const DcStats *__restrict__ stats, int stats_stride,
                                                  const DcAnchor *__restrict__ anchors, const int *__restrict__ qtab,
                                                  float2 *__restrict__ dc_state,
                                                  uint2 *__restrict__ table, int table_stride, int blk0, int n_blk,
                                                  int stream0, const int *__restrict__ map = nullptr) {
    extern __shared__ __align__(16) unsigned char dcw_smem[];
    const int stream = map_stream<MAP>(map, stream0, blockIdx.x);
    const int arm = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint4 *ring = reinterpret_cast<uint4 *>(dcw_smem) + (size_t)arm * DCW_RING * DCW_SLOT16;
    float *sq = reinterpret_cast<float *>(dcw_smem + (size_t)2 * DCW_RING * DCW_SLOT16 * 16) + arm * DC_BLK;
    const DcStats *sp = stats + ((size_t)stream * stats_stride + blk0) * 2 + arm;
    const uint4 *rp = reinterpret_cast<const uint4 *>(iq + (size_t)stream * iq_stride) + (size_t)blk0 * (2 * DC_BLK / 16);
    uint2 *tab = table + ((size_t)stream * table_stride + DC_HALO_BLKS + blk0) * 2 + arm;
    const int n_batch = (n_blk + DCW_BATCH - 1) / DCW_BATCH;
    const unsigned lt_mask = (1u << lane) - 1u;
    __shared__ int s_qtab[2][256];                                  // this stream's increment tables (k0_dc_qtab), one per arm
    for (int e = lane; e < 256; e += 32) s_qtab[arm][e] = qtab[((size_t)stream * 2 + arm) * 256 + e];
    __syncwarp();
    const int *sqt = s_qtab[arm];

    auto prefetch = [&](int batch) {
        if (batch < n_batch) {
            uint4 *dst = ring + (size_t)(batch % DCW_RING) * DCW_SLOT16;
            const uint4 *src = rp + (size_t)batch * DCW_SLOT16;
            const int n_valid = min(DCW_BATCH, n_blk - batch * DCW_BATCH) * (2 * DC_BLK / 16);
#pragma unroll
            for (int i = 0; i < DCW_SLOT16 / 32; ++i) {
                const int e = i * 32 + lane;
                if (e < n_valid) cp_async16(dst + e, src + e);
            }
        }
        cp_async_commit();
    };
    auto load_stats = [&](int batch) {
        DcStats S; S.D = 0; S.ta = 0xFFFFFFFFu; S.tb = 0u; S.tb_hi = 0xFFFFFFFFu;          // neutral: passes both ways
        const int j = batch * DCW_BATCH + lane;
        if (j < n_blk) S = sp[(size_t)j * 2];
        return S;
    };

    const DcAnchor A = anchors[2 * stream + arm];
    const unsigned lo1 = A.lo + 1u;
    const unsigned sign_bit = A.sgn < 0.f ? 0x80000000u : 0u;
    const unsigned win = A.ok ? A.hi - lo1 : 0u;                    // V in [0, win): the integer model holds
    const int Tv = (int)(A.T - lo1);
    unsigned V = 0xFFFFFFFFu;                                       // invalid: forces float stepping
    float s;
    {
        const float2 st0 = dc_state[stream];
        s = arm ? st0.y : st0.x;
        if (A.ok && s * A.sgn > 0.f) V = __float_as_uint(fabsf(s)) - lo1;
    }
#pragma unroll
    for (int i = 0; i < DCW_RING - 1; ++i) prefetch(i);
    DcStats Snext = load_stats(0);
    for (int batch = 0; batch < n_batch; ++batch) {
        // the copy into the slot about to be refilled (batch - 1's, consumed) has landed
        cp_async_wait<DCW_RING - 1>();
        __syncwarp();
        prefetch(batch + DCW_RING - 1);
        const DcStats S = Snext;
        if (batch + 1 < n_batch) Snext = load_stats(batch + 1);
        const int nb = min(DCW_BATCH, n_blk - batch * DCW_BATCH);
        const uint4 *slot = ring + (size_t)(batch % DCW_RING) * DCW_SLOT16;
        uint2 *to = tab + (size_t)batch * DCW_BATCH * 2;
        bool raw_ready = false;
        int j0 = 0;
        // exclusive prefix of the block totals, once per batch: a run that restarts at block j0 only rebases it
        unsigned excl;
        {
            unsigned inc = (unsigned)S.D;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += v;
            }
            excl = inc - (unsigned)S.D;
        }
        while (j0 < nb) {
            int n = j0;                                             // block to be handled on its own
            if (V < win) {
                // ---- speculative run of translations from block j0 ----
                const unsigned V0 = V + (excl - __shfl_sync(0xffffffffu, excl, j0));
                const unsigned V1 = V0 - (unsigned)DC_BLK * (unsigned)(lane - j0);
                const bool ok0 = lane < j0 || V0 < S.ta;
                const bool ok1 = lane < j0 || (V1 >= S.tb && V1 < S.tb_hi);
                const unsigned m0 = __ballot_sync(0xffffffffu, ok0), m1 = __ballot_sync(0xffffffffu, ok1);
                const int n0 = m0 == 0xFFFFFFFFu ? 32 : __ffs(~m0) - 1;
                const int n1 = m1 == 0xFFFFFFFFu ? 32 : __ffs(~m1) - 1;
                const bool up = n1 > n0;
                n = up ? n1 : n0;
                const unsigned Vsel = up ? V1 : V0;
                if (lane >= j0 && lane < n && lane < nb) to[(size_t)lane * 2] = make_uint2(Vsel, up ? 1u : 0u);
                if (n >= nb) {                                      // every remaining block translated
                    const unsigned E = Vsel + (unsigned)S.D - (up ? (unsigned)DC_BLK : 0u);
                    V = __shfl_sync(0xffffffffu, E, nb - 1);
                    break;
                }
                V = __shfl_sync(0xffffffffu, Vsel, n);              // state at the start of block n
            }
            // ---- block n on its own ----
            const int Dn = __shfl_sync(0xffffffffu, S.D, n);
            const unsigned tan = __shfl_sync(0xffffffffu, S.ta, n), tbn = __shfl_sync(0xffffffffu, S.tb, n);
            const unsigned tbhn = __shfl_sync(0xffffffffu, S.tb_hi, n);
            const bool fa = V < win && V < tan, fb = V < win && V >= tbn && V < tbhn;
            if (fa | fb) {
                if (lane == 0) to[(size_t)n * 2] = make_uint2(V, fb ? 1u : 0u);
                V = V + (unsigned)Dn - (fb ? (unsigned)DC_BLK : 0u);
                j0 = n + 1;
                continue;
            }
            if (!raw_ready) {
                cp_async_wait<DCW_RING - 1>();
                __syncwarp();
                raw_ready = true;
            }
            const unsigned char *rawn = reinterpret_cast<const unsigned char *>(slot + (size_t)n * (2 * DC_BLK / 16));
            if (V < win) {
                // a run of four (or two) blocks in one solve where the batch has that many left, then the block alone
                if (n + 4 <= nb) {
                    if (dc_solve_run<4>(rawn, arm, lane, lt_mask, sqt, Tv, (int)win, V, to + (size_t)n * 2)) { j0 = n + 4; continue; }
                } else if (n + 2 <= nb) {
                    if (dc_solve_run<2>(rawn, arm, lane, lt_mask, sqt, Tv, (int)win, V, to + (size_t)n * 2)) { j0 = n + 2; continue; }
                }
                if (dc_solve_run<1>(rawn, arm, lane, lt_mask, sqt, Tv, (int)win, V, to + (size_t)n * 2)) { j0 = n + 1; continue; }
            }
            // real float steps (sdrj.cpp:281) on lane 0; the other lanes only provide fl(c*x) of their 4 samples of this arm
            const uint2 rw = *reinterpret_cast<const uint2 *>(rawn + lane * 8);
            const unsigned w0 = arm ? rw.x >> 8 : rw.x, w1 = arm ? rw.y >> 8 : rw.y;
            const float x0 = u8_to_f<0>(w0), x1 = u8_to_f<2>(w0), x2 = u8_to_f<0>(w1), x3 = u8_to_f<2>(w1);
            if (V != 0xFFFFFFFFu) s = __uint_as_float((V + lo1) | sign_bit);
            __syncwarp();
            *reinterpret_cast<float4 *>(sq + 4 * lane) = make_float4(__fmul_rn(DC_C, x0), __fmul_rn(DC_C, x1), __fmul_rn(DC_C, x2), __fmul_rn(DC_C, x3));
            __syncwarp();
            if (lane == 0) {
                to[(size_t)n * 2] = make_uint2(__float_as_uint(s), 2u);
#pragma unroll 1
                for (int c = 0; c < DC_BLK / 32; ++c) {
                    float q[32];
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float4 v = *reinterpret_cast<const float4 *>(sq + 32 * c + 4 * k);
                        q[4 * k] = v.x; q[4 * k + 1] = v.y; q[4 * k + 2] = v.z; q[4 * k + 3] = v.w;
                    }
#pragma unroll
                    for (int k = 0; k < 32; ++k) s = __fadd_rn(__fmul_rn(s, DC_A), q[k]);
                }
            }
            s = __shfl_sync(0xffffffffu, s, 0);
            V = (A.ok && s * A.sgn > 0.f) ? __float_as_uint(fabsf(s)) - lo1 : 0xFFFFFFFFu;
            j0 = n + 1;
        }
        __syncwarp();
    }
    __shared__ float s_end[2];
    if (lane == 0) {
        if (V != 0xFFFFFFFFu) s = __uint_as_float((V + lo1) | sign_bit);
        s_end[arm] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) dc_state[stream] = make_float2(s_end[0], s_end[1]);
}

// ------------------------------------------------------------------------------------
// K1 for cf32 input (vfo::process on a main VFO, vfo.cpp:235: no byte conversion, no DC removal): main VFOs only. The uint8
// path is k1_v2 (kernels_v2.cuh); round 1's uint8 branch of this kernel is gone with its DC consumer.
// CTA = 9 warps: warp 0 recomputes the 256 samples in front of the tile (filter halo, or
// the tail of the previous callback for tile 0), warps 1..8 own 256 samples each; every
// thread owns 8 consecutive samples = one 16-byte load.
// ------------------------------------------------------------------------------------
constexpr int K1_A0_STR = 10, K1_A1_STR = 6, K1_A2_STR = 2;

__global__ void __launch_bounds__(K1_THREADS, 2) k1_ingest_main(const K1Params p) {
    __shared__ __align__(16) float2 sA0[(K1_THREADS + HB_PAD) * K1_A0_STR];
    __shared__ __align__(16) float2 sA1[(K1_THREADS + HB_PAD) * K1_A1_STR];
    __shared__ __align__(16) float2 sA2[(K1_THREADS + HB_PAD) * K1_A2_STR];

    const int stream = p.stream0 + blockIdx.x;
    const int tile = blockIdx.y, b = p.b0 + blockIdx.z;
    const int t = threadIdx.x, lane = t & 31;
    const int B = p.block;
    const int i0 = tile * K1_TILE - 256 + t * 8;          // callback coordinate of the chunk
    const long long blk = p.blocks_done[stream] + b;
    const bool in_block = i0 < B;
    const bool first_ever = (blk == 0);                    // nothing exists before sample 0
    const bool exists = in_block && !(first_ever && i0 < 0);
    const bool halo = t < 32;

    float2 x[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = make_float2(0.f, 0.f);
    if (exists) {
        // cf32 input (what vfo::process receives, vfo.cpp:235): no byte conversion, no DC removal
        const float2 *csrc = (b == 0 && i0 < 0)
            ? p.cf_tail + (size_t)stream * RAW_TAIL + (RAW_TAIL + i0)
            : p.cf_in + (size_t)stream * p.cf_stride + ((size_t)b * B + i0);
        const float4 *c4 = reinterpret_cast<const float4 *>(csrc);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float4 v = __ldg(c4 + k);
            x[2 * k] = make_float2(v.x, v.y);
            x[2 * k + 1] = make_float2(v.z, v.w);
        }
    }
    const long long n_abs = blk * (long long)B + i0;
    // every main VFO table has (int)Fs entries, so one modulo serves them all
    const int lut_idx = exists ? (int)(n_abs % p.mains[0].lut_len) : 0;

    for (int mi = 0; mi < p.n_main; ++mi) {
        const MainDev &M = p.mains[mi];
        float2 mixed[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) mixed[k] = make_float2(0.f, 0.f);
        if (exists) {
            const float4 *lp = reinterpret_cast<const float4 *>(M.lut + lut_idx);
            float4 l01 = __ldg(lp), l23 = __ldg(lp + 1), l45 = __ldg(lp + 2), l67 = __ldg(lp + 3);
            if (n_abs == 0) {                       // Oscillator start-up quirk (oscillator.cpp:26-30)
                const float2 last = __ldg(M.lut + (M.lut_len - 1));
                l01.x = last.x; l01.y = last.y;
            }
            mixed[0] = cmul(make_float2(l01.x, l01.y), x[0]);
            mixed[1] = cmul(make_float2(l01.z, l01.w), x[1]);
            mixed[2] = cmul(make_float2(l23.x, l23.y), x[2]);
            mixed[3] = cmul(make_float2(l23.z, l23.w), x[3]);
            mixed[4] = cmul(make_float2(l45.x, l45.y), x[4]);
            mixed[5] = cmul(make_float2(l45.z, l45.w), x[5]);
            mixed[6] = cmul(make_float2(l67.x, l67.y), x[6]);
            mixed[7] = cmul(make_float2(l67.z, l67.w), x[7]);
        }
        const bool store = in_block && !halo;
        float2 *outp = M.out + (size_t)stream * M.out_stride + MAIN_HIST + (size_t)b * M.block_out;
        if (M.decim == 0) {
            if (store) {
                float4 *o4 = reinterpret_cast<float4 *>(outp + i0);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    o4[k] = make_float4(mixed[2 * k].x, mixed[2 * k].y, mixed[2 * k + 1].x, mixed[2 * k + 1].y);
            }
            continue;
        }
        __syncthreads();                            // previous main done with sA0
        {
            float4 *s4 = reinterpret_cast<float4 *>(sA0 + (t + HB_PAD) * K1_A0_STR);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                s4[k] = make_float4(mixed[2 * k].x, mixed[2 * k].y, mixed[2 * k + 1].x, mixed[2 * k + 1].y);
        }
        __syncthreads();
        float2 o1[4];
        hb_run<4, 8, K1_A0_STR>(mixed, o1, sA0, t, i0);
        if (M.decim == 1) {
            if (store) {
                float4 *o4 = reinterpret_cast<float4 *>(outp + (i0 >> 1));
                o4[0] = make_float4(o1[0].x, o1[0].y, o1[1].x, o1[1].y);
                o4[1] = make_float4(o1[2].x, o1[2].y, o1[3].x, o1[3].y);
            }
            continue;
        }
        hb_publish<4, 4, K1_A1_STR>(o1, sA1, t);
        __syncthreads();
        float2 o2[2];
        hb_run<2, 4, K1_A1_STR>(o1, o2, sA1, t, i0 >> 1);
        if (M.decim == 2) {
            if (store)
                *reinterpret_cast<float4 *>(outp + (i0 >> 2)) = make_float4(o2[0].x, o2[0].y, o2[1].x, o2[1].y);
            continue;
        }
        hb_publish<2, 2, K1_A2_STR>(o2, sA2, t);
        __syncthreads();
        float2 o3[1];
        hb_run<1, 2, K1_A2_STR>(o2, o3, sA2, t, i0 >> 2);
        if (store) outp[i0 >> 3] = o3[0];
    }
}

// ------------------------------------------------------------------------------------
// K2 late: d[m] = sum_i taps[i] * z[late*m - ntaps + i]  on both arms
// (fir_decI/Q FIRUpdateAndProcess on the first sample of each group of `late`, FIRUpdate
// on the others: vfo.cpp:346-384; newest sample excluded: dsp.cpp:59-71).
// ------------------------------------------------------------------------------------
template <bool MAP = false>
__global__ void __launch_bounds__(LATE_TILE) k2_late_fir(const LateDev *__restrict__ devs, int cb0, int ncb, int stream0,
                                                         const int *__restrict__ map = nullptr) {
    __shared__ float2 sz[LATE_TILE * 6 + MAX_FIR_TAPS];
    __shared__ float st[MAX_FIR_TAPS];
    const LateDev &D = devs[blockIdx.y];
    const int stream = map_stream<MAP>(map, stream0, blockIdx.x);
    const int n_total = (cb0 + ncb) * D.samples_out;               // outputs exist up to here
    const int m0 = cb0 * D.samples_out + blockIdx.z * LATE_TILE;
    if (m0 >= n_total) return;
    const int t = threadIdx.x;
    const int span = D.late * LATE_TILE + D.ntaps;
    const long long zlo = (long long)D.late * m0 - D.ntaps;       // may be negative: history
    const long long zmax = (long long)(cb0 + ncb) * D.block_z;
    const float2 *zp = D.z + (size_t)stream * D.z_stride + D.z_hist;
    for (int e = t; e < span; e += LATE_TILE) {
        const long long zi = zlo + e;
        sz[e] = (zi < zmax) ? zp[zi] : make_float2(0.f, 0.f);
    }
    for (int e = t; e < D.ntaps; e += LATE_TILE) st[e] = D.taps[e];
    __syncthreads();
    const int m = m0 + t;
    if (m >= n_total) return;
    const float2 *w = sz + D.late * t;
    float ax = 0.f, ay = 0.f;
    for (int i = 0; i < D.ntaps; ++i) {
        const float c = st[i];
        const float2 v = w[i];
        ax = fmaf(c, v.x, ax);
        ay = fmaf(c, v.y, ay);
    }
    D.d[(size_t)stream * D.d_stride + D.d_hist + m] = make_float2(ax, ay);
}

// ------------------------------------------------------------------------------------
// K3: carry. Copies the trailing `hist` bytes of what this call produced to the front of
// each buffer (main outputs, z, d) and keeps the last RAW_TAIL raw samples.
// ------------------------------------------------------------------------------------
template <bool MAP = false>
__global__ void __launch_bounds__(128) k3_carry(const CarryItem *__restrict__ items, int n_items, int n_blocks,
                                                 const uint8_t *__restrict__ iq, size_t iq_stride, int block,
                                                 uint8_t *__restrict__ tail, long long *__restrict__ blocks_done,
                                                 const uint2 *__restrict__ dc_table, uint2 *__restrict__ dc_table_next,
                                                 const DcAnchor *__restrict__ dc_anchor,
                                                 int dc_table_stride, int n_dcblk, int stream0,
                                                 const float2 *__restrict__ cf_in, size_t cf_stride,
                                                 float2 *__restrict__ cf_tail, const int *__restrict__ map = nullptr) {
    const int stream = map_stream<MAP>(map, stream0, blockIdx.x);
    const int item = blockIdx.y;
    if (item < n_items) {
        const CarryItem it = items[item];
        unsigned char *base = reinterpret_cast<unsigned char *>(it.base) + (size_t)stream * it.stride;
        const uint4 *src = reinterpret_cast<const uint4 *>(base + (size_t)n_blocks * it.block_bytes);
        uint4 *dst = reinterpret_cast<uint4 *>(base);
        // The tail moves towards the front of the same buffer; with a call shorter than the history the two ranges
        // overlap. Chunk by chunk in rising order, every chunk read completely before it is written: a later chunk's
        // source lies above everything written so far, so nothing is clobbered before it has been read.
        const int n16 = it.hist_bytes / 16;
        for (int e0 = 0; e0 < n16; e0 += 128) {
            const int e = e0 + threadIdx.x;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (e < n16) v = src[e];
            __syncthreads();
            if (e < n16) dst[e] = v;
            __syncthreads();
        }
    } else {
        if (iq) {
            const uint4 *src = reinterpret_cast<const uint4 *>(iq + (size_t)stream * iq_stride + ((size_t)n_blocks * block - RAW_TAIL) * 2);
            uint4 *dst = reinterpret_cast<uint4 *>(tail + (size_t)stream * (2 * RAW_TAIL));
            for (int e = threadIdx.x; e < (2 * RAW_TAIL) / 16; e += 128) dst[e] = src[e];
        } else {
            const float2 *src = cf_in + (size_t)stream * cf_stride + ((size_t)n_blocks * block - RAW_TAIL);
            float2 *dst = cf_tail + (size_t)stream * RAW_TAIL;
            for (int e = threadIdx.x; e < RAW_TAIL; e += 128) dst[e] = src[e];
        }
        if (threadIdx.x == 0) blocks_done[stream] += n_blocks;
        // DC table: the last DC_HALO_BLKS block-start states move to the front for the next call's
        // halo warp; they become "stepped" entries because the next call has a new anchor.
        if (dc_table && threadIdx.x < 2 * DC_HALO_BLKS) {
            const uint2 *t = dc_table + (size_t)stream * dc_table_stride * 2;
            uint2 e = t[(size_t)n_dcblk * 2 + threadIdx.x];
            if (e.y < 2u) {                                      // translation entry -> plain float bits
                const DcAnchor A = dc_anchor[2 * stream + (threadIdx.x & 1)];
                e.x = (e.x + A.lo + 1u) | (A.sgn < 0.f ? 0x80000000u : 0u);
            }
            e.y = 2u;
            dc_table_next[(size_t)stream * dc_table_stride * 2 + threadIdx.x] = e;   // the next call owns the other buffer
        }
    }
}

// ------------------------------------------------------------------------------------
// Receiver state records (sdrb_bank_save_state / load_state, layout in include/sdrb200.h): everything k3_carry leaves
// for the next call, for a list of streams, as one fixed-size record per stream. The record holds the carry items'
// history regions (never bank rows, whose strides depend on max_blocks), so banks of one plan exchange records.
// ------------------------------------------------------------------------------------
struct StateHeader {
    unsigned magic, version;
    unsigned long long record_bytes, fingerprint;
    long long blocks_done;
    float2 dc_state;
    unsigned flags, reserved[5];
};
static_assert(sizeof(StateHeader) == 64, "the record header is 64 bytes");
constexpr unsigned STATE_MAGIC = 0x54534253u;                   // "SBST", little endian
constexpr unsigned STATE_VERSION = 1u;
constexpr unsigned STATE_FLAG_DC = 1u, STATE_FLAG_FUSED_LATE = 2u;
constexpr int STATE_HALO_OFF = (int)sizeof(StateHeader);                        // 2*DC_HALO_BLKS uint2
constexpr int STATE_RAW_OFF = STATE_HALO_OFF + 2 * DC_HALO_BLKS * 8;            // 2*RAW_TAIL bytes
constexpr int STATE_CF_OFF = STATE_RAW_OFF + 2 * RAW_TAIL;                      // RAW_TAIL float2
constexpr int STATE_ITEMS_OFF = STATE_CF_OFF + RAW_TAIL * 8;                    // carry items, in bank order
static_assert(STATE_RAW_OFF % 16 == 0 && STATE_CF_OFF % 16 == 0 && STATE_ITEMS_OFF % 16 == 0, "sections start on 16 bytes");

struct StateIoParams {
    const CarryItem *items;         // the bank's carry items (the list k3_carry runs)
    const int2 *item_rec;           // per item: (offset in the record, 1 = some kernel reads it / 0 = saved as zeros)
    int n_items;
    const int *streams;             // record k <-> stream streams[k]
    unsigned char *rec;             // n records of rec_bytes
    size_t rec_bytes;
    long long *blocks_done;
    float2 *dc_state;
    uint8_t *raw_tail;              // [n_streams][2*RAW_TAIL]
    float2 *cf_tail;                // [n_streams][RAW_TAIL]
    uint2 *dc_table;                // table_buf(dc_par): the buffer the next call reads its halo from; nullptr without DC
    int dc_table_stride;
    StateHeader hdr;                // SAVE: magic .. flags of this bank; blocks_done and dc_state are filled per stream
};

// grid (listed streams, n_items + 1): y < n_items copies one carry item's history, the last y-block the header scalars, the DC
// halo and the raw / cf32 tails (as k3_carry splits its work). Every section is a whole number of 16-byte chunks.
template <bool SAVE>
__global__ void __launch_bounds__(128) k_state_io(const __grid_constant__ StateIoParams p) {
    const int stream = p.streams[blockIdx.x];
    unsigned char *rec = p.rec + (size_t)blockIdx.x * p.rec_bytes;
    auto copy16 = [&](void *bank, int rec_off, int bytes, bool live) {
        uint4 *b = reinterpret_cast<uint4 *>(bank);
        uint4 *r = reinterpret_cast<uint4 *>(rec + rec_off);
        for (int e = threadIdx.x; e < bytes / 16; e += 128) {
            if (SAVE) r[e] = live ? b[e] : make_uint4(0u, 0u, 0u, 0u);
            else b[e] = r[e];
        }
    };
    if ((int)blockIdx.y < p.n_items) {
        const CarryItem it = p.items[blockIdx.y];
        const int2 ir = p.item_rec[blockIdx.y];
        copy16(reinterpret_cast<unsigned char *>(it.base) + (size_t)stream * it.stride, ir.x, it.hist_bytes, ir.y != 0);
        return;
    }
    StateHeader *h = reinterpret_cast<StateHeader *>(rec);
    long long done;
    if (SAVE) {
        done = p.blocks_done[stream];
        if (threadIdx.x == 0) {
            StateHeader o = p.hdr;
            o.blocks_done = done;
            o.dc_state = p.dc_state[stream];
            *h = o;
        }
    } else {
        done = h->blocks_done;
        if (threadIdx.x == 0) { p.blocks_done[stream] = done; p.dc_state[stream] = h->dc_state; }
    }
    // the halo entries only exist once a call has run: a fresh stream's record holds zeros
    if (SAVE || p.dc_table)
        copy16(p.dc_table + (size_t)stream * p.dc_table_stride * 2, STATE_HALO_OFF, 2 * DC_HALO_BLKS * 8, p.dc_table && done != 0);
    copy16(p.raw_tail + (size_t)stream * (2 * RAW_TAIL), STATE_RAW_OFF, 2 * RAW_TAIL, true);
    copy16(p.cf_tail + (size_t)stream * RAW_TAIL, STATE_CF_OFF, RAW_TAIL * 8, true);
}

// ------------------------------------------------------------------------------------
// k_compress: vfo::compress (vfo.cpp:389-424), the IQ forwarder of a main VFO without sub VFOs.
//   style 1:  byte = ((signed char)((re/scale)*128) & 0xF0) | (((signed char)((im/scale)*128) & 0xF0) >> 4)
//   else:     bytes = (signed char)(re*128), (signed char)(im*128)
// float -> signed char as the reference's x86 build does it: truncate toward zero to int, keep
// the low 8 bits. Pure streaming: 8 B read + 1 (2) B written per sample, a thread owns 4
// consecutive samples (two 16-byte loads, one 4- or 8-byte store), grid.y = stream.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned comp_s8(float v) { return (unsigned)__float2int_rz(v) & 0xffu; }
__device__ __forceinline__ unsigned comp_pack(float2 v, float scale) {
    const unsigned re = comp_s8((v.x / scale) * 128.0f), im = comp_s8((v.y / scale) * 128.0f);
    return (re & 0xF0u) | ((im & 0xF0u) >> 4);
}

__global__ void __launch_bounds__(256) k_compress(const float2 *__restrict__ in, long long in_stride, uint8_t *__restrict__ out,
                                                  long long out_stride, int n, float scale, int style) {
    const int i0 = (blockIdx.x * 256 + threadIdx.x) * 4;
    if (i0 >= n) return;
    const float2 *src = in + (size_t)blockIdx.y * in_stride + i0;
    uint8_t *dst = out + (size_t)blockIdx.y * out_stride;
    const bool vec = (i0 + 4 <= n) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    float2 v[4];
    if (vec) {
        const float4 a = __ldg(reinterpret_cast<const float4 *>(src)), c = __ldg(reinterpret_cast<const float4 *>(src) + 1);
        v[0] = make_float2(a.x, a.y); v[1] = make_float2(a.z, a.w); v[2] = make_float2(c.x, c.y); v[3] = make_float2(c.z, c.w);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = (i0 + k < n) ? __ldg(src + k) : make_float2(0.f, 0.f);
    }
    if (style == 1) {
        const unsigned w = comp_pack(v[0], scale) | (comp_pack(v[1], scale) << 8) | (comp_pack(v[2], scale) << 16) |
                           (comp_pack(v[3], scale) << 24);
        if (vec && ((reinterpret_cast<uintptr_t>(dst + i0) & 3) == 0)) {
            *reinterpret_cast<unsigned *>(dst + i0) = w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (i0 + k < n) dst[i0 + k] = (uint8_t)(w >> (8 * k));
        }
    } else {
        unsigned w[2];
#pragma unroll
        for (int h = 0; h < 2; ++h)
            w[h] = comp_s8(v[2 * h].x * 128.0f) | (comp_s8(v[2 * h].y * 128.0f) << 8) | (comp_s8(v[2 * h + 1].x * 128.0f) << 16) |
                   (comp_s8(v[2 * h + 1].y * 128.0f) << 24);
        if (vec && ((reinterpret_cast<uintptr_t>(dst + 2 * (size_t)i0) & 7) == 0)) {
            *reinterpret_cast<uint2 *>(dst + 2 * (size_t)i0) = make_uint2(w[0], w[1]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (i0 + k < n) {
                    dst[2 * (size_t)(i0 + k)] = (uint8_t)(w[k >> 1] >> (16 * (k & 1)));
                    dst[2 * (size_t)(i0 + k) + 1] = (uint8_t)(w[k >> 1] >> (16 * (k & 1) + 8));
                }
        }
    }
}

// test/inspection helper: block-start DC states of the last call as float2 (I, Q)
__global__ void __launch_bounds__(256) dc_trace_gather(const uint2 *__restrict__ table, const DcAnchor *__restrict__ anchors,
                                                        int table_stride, int n, float2 *__restrict__ out,
                                                        uint8_t *__restrict__ modes) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const uint2 *t = table + ((size_t)blockIdx.y * table_stride + DC_HALO_BLKS + i) * 2;
    float v[2];
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const DcAnchor A = anchors[2 * blockIdx.y + a];
        v[a] = t[a].y < 2u ? A.sgn * __uint_as_float(t[a].x + A.lo + 1u) : __uint_as_float(t[a].x);
    }
    out[(size_t)blockIdx.y * n + i] = make_float2(v[0], v[1]);
    if (modes) modes[(size_t)blockIdx.y * n + i] = (uint8_t)(t[0].y | (t[1].y << 4));
}

}  // namespace sdrb
