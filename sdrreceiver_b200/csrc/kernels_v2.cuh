// Second-generation channelizer kernels (sm_100a): k1_v2 (ingest + main VFOs) and k2a_v2 (all sub
// VFOs of one main VFO per CTA). Both are the same machine:
//
//   * a thread owns 32 consecutive input samples (+ the 11 in front of them) IN REGISTERS and keeps
//     them there while it loops over every VFO fed by that input (2-3 main VFOs in k1_v2, the 12-15
//     sub VFOs of a main in k2a_v2): the input is read from HBM/L2 once, not once per VFO;
//   * the NCO is not read sample by sample. Past its start-up transient the Oscillator table
//     (oscillator.cpp:9-28) advances by the constant float rotation `rot` per entry, so inside a
//     thread's chunk  lut[k0 + j] = lut[k0] * Rf[j]  with Rf[j] = (rot/|rot|)^j  to 2e-7 rms / 1e-6
//     worst case (tools/rf_error.py; the parity budget is 1e-4). The thread mixes with the 42
//     constants Rf[-10..31] (shared memory broadcast), runs the first half-band stage entirely on its
//     own registers -- no neighbour exchange -- and multiplies the 16 outputs by the one table entry
//     F = lut[k0] it loads. Table traffic drops from 8 B per mixed sample to 8 B per 32;
//   * chunks that touch the first 512 table entries, the table wrap, stream sample 0
//     (oscillator.cpp:26-30,42-48) or the first sample of a callback take the exact path: every
//     rotation comes from the table itself;
//   * later half-band stages exchange only the 10 trailing samples per thread through padded,
//     conflict-free shared memory (one 16-byte load per pair); the thread's own samples never
//     leave registers;
//   * the FIRQueueBackToFront off-by-one (dsp.cpp:163-173) is one rule: a window slot at a
//     negative callback coordinate c holds sample c-1;
//   * 168 registers per thread give 12 warps per SM whatever the CTA size, so the CTA size (64, 96
//     or 128 threads, a template parameter) only trades barrier-domain size against halo threads;
//     k1_v2 additionally walks K1_TPC consecutive tiles per CTA with the next tile's bytes
//     prefetched by cp.async.
// Also here: k2b_v2 (USB demodulation, one warp per tile) and k2_late_v2 (polyphase /5 and /6 FIR).
#pragma once
#include "kernels.cuh"

namespace sdrb {

constexpr int V2_CHUNK = 32;
constexpr int RF_LEN = 48;             // per VFO: Rf[j], j = -10..31 at index j + 10; padded to 48
constexpr int V2_MAX_VFO = 16;         // VFOs per launch (descriptors + Rf tables in the kernel parameters)
constexpr int LUT_STEADY = 512;        // table entries needed by the start-up transient (94 measured)
constexpr int K1V2_HT = 4;             // halo threads of k1_v2: one DC block, covers 3 half-band stages
// CTA size: 168 registers per thread allow 12 warps per SM whatever the CTA size, so a smaller CTA
// costs nothing in occupancy; it shortens every barrier domain (the stage transitions are where the
// warps stall) and costs halo threads: HT of NT threads recompute the previous tile's tail. Measured
// on B200 (25E): ingest 0.87 -> 0.79 ms per step at 64 threads (4 halo threads); the sub-VFO cascade
// gains the same ~9 % per useful thread, which the 11 halo threads of a 5-stage group give back. The
// host picks 64, 96 or 128 threads per launch (api.cu: v2_pick_threads).
template <int NT> constexpr int v2_minb() { return 384 / NT; }    // 12 warps per SM
template <int NT> constexpr int k1v2_adv() { return (NT - K1V2_HT) * V2_CHUNK; }    // host side

struct CascVfo {
    const float2 *lut;          // Oscillator table of this VFO
    float2 *out;                // [n_streams][out_stride]: hist + n_blocks*block_out
    int S;                      // half-band stages
    int block_out, hist, pad;
};
// Rf[j], j = -10..31 at pair index (j + 10) / 2. The tables and the VFO descriptors travel in the
// kernel parameters (constant bank): the VFO index is uniform across the CTA, so the rotation
// operands come through the uniform/constant path and cost the shared-memory pipe nothing
// (they were 21 broadcast LDS.128 per VFO and thread; ncu had k2a at 79 % L1/shared throughput).
// One float4 per rotation: (c, c, -s, s) for Rf[j] = c + j s. A complex product Rf[j] * x is then two packed operations --
// mul2(x, (c, c)) and fma2((x.y, x.x), (-s, s), .) with the half swap folded into the FFMA2 operand by ptxas -- instead of four
// scalar ones; the constants reach the instructions as uniform registers.
struct RfTab { float4 q[RF_LEN]; };
__device__ __forceinline__ float2 rot2(float4 r, float2 x) {
    return fma2(make_float2(x.y, x.x), make_float2(r.z, r.w), mul2(x, make_float2(r.x, r.y)));
}
// the same with a per-thread factor F, prepared once as Fc = (F.x, F.x), Fs = (-F.y, F.y)
__device__ __forceinline__ float2 rotF(float2 Fc, float2 Fs, float2 x) { return fma2(make_float2(x.y, x.x), Fs, mul2(x, Fc)); }

// scratch layout of the array a stage reads: N samples per thread, STR float2 apart, PADT
// never-written thread slots in front (read only by halo threads whose results are dropped)
template <int N> struct StLay;
template <> struct StLay<16> { static constexpr int STR = 18, PADT = 1; };
template <> struct StLay<8> { static constexpr int STR = 10, PADT = 2; };
template <> struct StLay<4> { static constexpr int STR = 6, PADT = 3; };
template <> struct StLay<2> { static constexpr int STR = 2, PADT = 6; };
template <int N, int NT> constexpr int st_elems() { return (NT + StLay<N>::PADT) * StLay<N>::STR; }

template <int NT> struct V2L {                                  // scratch offsets (float2) of a CTA of NT threads
    static constexpr int SA = 0;                                // two copies, alternating from VFO to VFO
    static constexpr int SA_LEN = st_elems<16, NT>();
    static constexpr int SB = SA + 2 * SA_LEN;
    static constexpr int SC = SB + st_elems<8, NT>();
    static constexpr int SD = SC + st_elems<4, NT>();
    static constexpr int SEND = SD + st_elems<2, NT>();         // then 16 bytes of misc
    static constexpr size_t SMEM = (size_t)SEND * sizeof(float2) + 16;
};

template <int N>
__device__ __forceinline__ int st_pos(int c_rel) {              // CTA-relative sample, may be negative
    return ((c_rel >> Log2<N>::v) + StLay<N>::PADT) * StLay<N>::STR + (c_rel & (N - 1));
}

template <int N>
__device__ __forceinline__ void st_publish(const float2 (&v)[N], float2 *__restrict__ s, int t) {
    float4 *p = reinterpret_cast<float4 *>(s + (t + StLay<N>::PADT) * StLay<N>::STR);
#pragma unroll
    for (int k = 0; k < N / 2; ++k) p[k] = make_float4(v[2 * k].x, v[2 * k].y, v[2 * k + 1].x, v[2 * k + 1].y);
}

// hbcoeff11 on a window (halfbanddecimator.h:66-79, dsp.cpp:139-142), both arms packed:
// 3 FADD2 + 1 FMUL2 + 3 FFMA2 per complex output
__device__ __forceinline__ float2 hb11(float2 w0, float2 w2, float2 w4, float2 w5, float2 w6, float2 w8, float2 w10) {
    return fma2(splat2(HB_P5), w5,
                fma2(splat2(HB_P4), add2(w4, w6), fma2(splat2(HB_P2), add2(w2, w8), mul2(splat2(HB_P0), add2(w0, w10)))));
}

// One half-band stage: the thread owns N samples (first one at callback coordinate vs of this
// stage) and needs the 10 samples in front of them from its left neighbours. OWN = the thread's own
// samples are still in registers (`in`); otherwise they are read back from the scratch as well.
template <int N, bool OWN>
__device__ __forceinline__ void st_run(const float2 *in, float2 (&out)[N / 2], const float2 *__restrict__ s, int t, int vs) {
    float2 w[10 + N];
    if (vs >= 0 && vs < 10) {
        // head of a callback: slots at negative coordinates hold the sample one further back
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            int c = vs - 10 + k;
            c -= (c < 0) ? 1 : 0;
            w[k] = s[st_pos<N>(t * N + (c - vs))];
        }
    } else {
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            const float4 v = *reinterpret_cast<const float4 *>(s + st_pos<N>(t * N - 10 + 2 * q));
            w[2 * q] = make_float2(v.x, v.y);
            w[2 * q + 1] = make_float2(v.z, v.w);
        }
    }
    if constexpr (OWN) {
#pragma unroll
        for (int k = 0; k < N; ++k) w[10 + k] = in[k];
    } else {
        const float4 *own = reinterpret_cast<const float4 *>(s + (t + StLay<N>::PADT) * StLay<N>::STR);
#pragma unroll
        for (int q = 0; q < N / 2; ++q) {
            const float4 v = own[q];
            w[10 + 2 * q] = make_float2(v.x, v.y);
            w[11 + 2 * q] = make_float2(v.z, v.w);
        }
    }
#pragma unroll
    for (int r = 0; r < N / 2; ++r)
        out[r] = hb11(w[2 * r], w[2 * r + 2], w[2 * r + 4], w[2 * r + 5], w[2 * r + 6], w[2 * r + 8], w[2 * r + 10]);
}

template <int N>
__device__ __forceinline__ void st_store(const float2 (&v)[N], float2 *__restrict__ dst) {
    if constexpr (N == 1) {
        dst[0] = v[0];
    } else {
        float4 *o4 = reinterpret_cast<float4 *>(dst);
#pragma unroll
        for (int k = 0; k < N / 2; ++k) o4[k] = make_float4(v[2 * k].x, v[2 * k].y, v[2 * k + 1].x, v[2 * k + 1].y);
    }
}

// st_store of the first n of the N outputs (a chunk that runs past the end of its callback: the filters are causal, so the outputs
// inside the callback are complete and the rest belong to nobody). Every stored length is even, so n is even for N >= 2.
template <int N>
__device__ __forceinline__ void st_store_n(const float2 (&v)[N], float2 *__restrict__ dst, int n) {
    if (n >= N) {
        st_store<N>(v, dst);
    } else {
#pragma unroll
        for (int k = 0; k < N; ++k)
            if (k < n) dst[k] = v[k];
    }
}

// Exact first stage for the few chunks the rotating-frame shortcut does not cover (table start-up
// transient and wrap, stream sample 0, first chunk of a callback): every rotation is read from
// the Oscillator table. Deliberately not inlined and not unrolled: it runs for ~1 % of the chunks
// and must not cost the common path registers.
__device__ __noinline__ void stage1_exact(const float2 *xc, const float2 *__restrict__ lut, int k0, int L, long long n_abs,
                                          int head, float4 *pa) {
    float2 rot[41];
#pragma unroll
    for (int i = 0; i < 41; ++i) {                        // all table reads in flight together
        const int j = i - 10;
        const int sh = (j < 0) ? head : 0;                // negative coordinate c holds sample c-1
        int idx = k0 + j - sh;
        if (idx < 0) idx += L;
        if (idx >= L) idx -= L;
        if (n_abs + j - sh == 0) idx = L - 1;             // stream sample 0 uses the last entry (oscillator.cpp:26-30)
        rot[i] = __ldg(lut + idx);
    }
    float2 u[41];
#pragma unroll
    for (int i = 0; i < 41; ++i) u[i] = cmul(rot[i], xc[i + 2 - (i < 10 ? head : 0)]);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int r = 2 * k;
        const float2 a = hb11(u[2 * r], u[2 * r + 2], u[2 * r + 4], u[2 * r + 5], u[2 * r + 6], u[2 * r + 8], u[2 * r + 10]);
        const float2 c = hb11(u[2 * r + 2], u[2 * r + 4], u[2 * r + 6], u[2 * r + 7], u[2 * r + 8], u[2 * r + 10], u[2 * r + 12]);
        pa[k] = make_float4(a.x, a.y, c.x, c.y);
    }
}

// Everything after the input is in registers: for each VFO mix + S half-band stages + store.
//   x[i]      input sample at callback coordinate v0 - 12 + i   (i = 0..43)
//   n_abs     absolute stream index of sample v0 (negative: before the stream began)
//   k0        n_abs mod L
//   P         the kernel's parameter struct (__grid_constant__): P::vfos[], P::rf[]
// RAGGED: the callback is not a whole number of 32-sample chunks; `nin` = samples of the callback from v0 on, and outputs
// past the callback end are not stored (they would overwrite the next callback's first outputs).
template <int MAXS, int NT, class P, bool RAGGED = false>
__device__ __forceinline__ void cascade_loop(const float2 (&x)[44], const P &p, int count,
                                             float2 *__restrict__ sm, int t, int v0, long long n_abs, int k0, int L,
                                             bool store, size_t out_off /* stream*out_stride */, int b, int nin = V2_CHUNK) {
    float2 *sB = sm + V2L<NT>::SB, *sC = sm + V2L<NT>::SC, *sD = sm + V2L<NT>::SD;
    int prevS = 1, flip = 0;
    const bool head = (v0 == 0);
    const bool fast = (k0 >= LUT_STEADY + 10) && (k0 + V2_CHUNK <= L) && !head;
    float2 xc[44];                                        // addressable copy for the exact path only
    if (!fast) {
#pragma unroll
        for (int i = 0; i < 44; ++i) xc[i] = x[i];
    }
    float2 Fnext = make_float2(1.f, 0.f);
    if (fast) Fnext = __ldg(p.vfos[0].lut + k0);
    for (int v = 0; v < count; ++v) {
        const CascVfo V = p.vfos[v];
        const float2 F = Fnext;
        if (fast && v + 1 < count) Fnext = __ldg(p.vfos[v + 1].lut + k0);   // one VFO ahead: never waited for
        float2 *outp = V.out + out_off + V.hist + (size_t)b * V.block_out;
        if (V.S == 0) {                                   // mixer only (vfo.cpp:237-245 with decimateCount 0)
            if (store && fast) {
                // rotating frame like the first half-band stage: lut[k0 + j] = F * Rf[j], no table reads per sample
                // (the per-sample reads are 8-byte loads 256 bytes apart across a warp: 32 sectors per instruction)
#pragma unroll
                const float2 Fc = make_float2(F.x, F.x), Fs = make_float2(-F.y, F.y);
                for (int q = 0; q < V2_CHUNK / 2; ++q) {
                    const float2 a = rotF(Fc, Fs, rot2(p.rf[v].q[2 * q + 10], x[12 + 2 * q]));      // Rf[2q]
                    const float2 c = rotF(Fc, Fs, rot2(p.rf[v].q[2 * q + 11], x[13 + 2 * q]));      // Rf[2q+1]
                    if (!RAGGED || 2 * q < nin) *reinterpret_cast<float4 *>(outp + v0 + 2 * q) = make_float4(a.x, a.y, c.x, c.y);
                }
            } else if (store) {
#pragma unroll
                for (int j = 0; j < V2_CHUNK; j += 2) {
                    int i0 = k0 + j, i1 = k0 + j + 1;
                    if (i0 >= L) i0 -= L;
                    if (i1 >= L) i1 -= L;
                    if (n_abs + j == 0) i0 = L - 1;       // oscillator.cpp:26-30
                    const float2 a = cmul(__ldg(V.lut + i0), x[12 + j]), c = cmul(__ldg(V.lut + i1), x[13 + j]);
                    if (!RAGGED || j < nin) *reinterpret_cast<float4 *>(outp + v0 + j) = make_float4(a.x, a.y, c.x, c.y);
                }
            }
            continue;
        }
        // The stage-1 array alternates between two copies, so a VFO that follows one with >= 2 stages
        // needs no barrier here: whoever still reads the other copy's stage-1 data has not yet passed
        // the previous VFO's first barrier, and everything behind it (sB, sC, sD) is only rewritten
        // after this VFO's own barriers. After a 1-stage VFO (no barrier of its own) one is needed.
        float2 *sA = sm + V2L<NT>::SA + flip * V2L<NT>::SA_LEN;
        flip ^= 1;
        if (prevS < 2) __syncthreads();
        prevS = V.S;
        // stage 1 straight into the scratch (two outputs per 16-byte store): nothing but the input stays in registers
        float4 *pa = reinterpret_cast<float4 *>(sA + (t + StLay<16>::PADT) * StLay<16>::STR);
        if (fast) {
            float2 u[42];
#pragma unroll
            for (int j = 0; j < 42; ++j) u[j] = rot2(p.rf[v].q[j], x[j + 2]);
            const float2 Fc = make_float2(F.x, F.x), Fs = make_float2(-F.y, F.y);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int r = 2 * k;
                const float2 a = rotF(Fc, Fs, hb11(u[2 * r], u[2 * r + 2], u[2 * r + 4], u[2 * r + 5], u[2 * r + 6], u[2 * r + 8], u[2 * r + 10]));
                const float2 c = rotF(Fc, Fs, hb11(u[2 * r + 2], u[2 * r + 4], u[2 * r + 6], u[2 * r + 7], u[2 * r + 8], u[2 * r + 10], u[2 * r + 12]));
                pa[k] = make_float4(a.x, a.y, c.x, c.y);
            }
        } else {
            stage1_exact(xc, V.lut, k0, L, n_abs, head ? 1 : 0, pa);
        }
        if (V.S == 1) {
            if (store) {
                float4 *o4 = reinterpret_cast<float4 *>(outp + (v0 >> 1));
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (!RAGGED || 4 * k < nin) o4[k] = pa[k];
            }
            continue;
        }
        __syncthreads();
        float2 o2[8];
        st_run<16, false>(nullptr, o2, sA, t, v0 >> 1);
        if (V.S == 2) {
            if (store) {
                if (RAGGED) st_store_n<8>(o2, outp + (v0 >> 2), nin >> 2);
                else st_store<8>(o2, outp + (v0 >> 2));
            }
            continue;
        }
        st_publish<8>(o2, sB, t);
        __syncthreads();
        float2 o3[4];
        st_run<8, true>(o2, o3, sB, t, v0 >> 2);
        if (MAXS == 3 || V.S == 3) {
            if (store) {
                if (RAGGED) st_store_n<4>(o3, outp + (v0 >> 3), nin >> 3);
                else st_store<4>(o3, outp + (v0 >> 3));
            }
            continue;
        }
        if constexpr (MAXS > 3) {
            st_publish<4>(o3, sC, t);
            __syncthreads();
            float2 o4[2];
            st_run<4, true>(o3, o4, sC, t, v0 >> 3);
            if (V.S == 4) {
                if (store) {
                    if (RAGGED) st_store_n<2>(o4, outp + (v0 >> 4), nin >> 4);
                    else st_store<2>(o4, outp + (v0 >> 4));
                }
                continue;
            }
            st_publish<2>(o4, sD, t);
            __syncthreads();
            float2 o5[1];
            st_run<2, true>(o4, o5, sD, t, v0 >> 4);
            if (store) {
                if (RAGGED) st_store_n<1>(o5, outp + (v0 >> 5), nin >> 5);
                else st_store<1>(o5, outp + (v0 >> 5));
            }
        }
    }
}

// ------------------------------------------------------------------------------------
// k2a_v2: all sub VFOs (of one group: same parent main VFO, at most V2_MAX_VFO) for one
// (stream, tile, callback). The parent's output chunk is loaded once per thread.
// ------------------------------------------------------------------------------------
struct K2V2Params {
    CascVfo vfos[V2_MAX_VFO];       // this group's sub VFOs
    RfTab rf[V2_MAX_VFO];
    const float2 *in;               // parent main output (MAIN_HIST history in front of each stream)
    const long long *blocks_done;
    long long in_stride, out_stride;
    int count, lut_len, block_in, HT, stream0, b0;
    int blk_off, pad;               // added to the callback counter: -n for a replay of the last call's callbacks after the carry
};

// RAGGED: callbacks that are not a whole number of 32-sample chunks (a 30 000- or 3 600-sample parent): loads stop at the end of
// the callback, stores at the end of each VFO's callback (cascade_loop).
template <int NT, bool RAGGED = false>
__global__ void __launch_bounds__(NT, v2_minb<NT>()) k2a_v2(const __grid_constant__ K2V2Params p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2 *sm = reinterpret_cast<float2 *>(smem_raw);
    int *sBase = reinterpret_cast<int *>(sm + V2L<NT>::SEND);

    const int stream = p.stream0 + blockIdx.x;
    const int tile = blockIdx.y, b = p.b0 + blockIdx.z;
    const int t = threadIdx.x;
    const int B = p.block_in, L = p.lut_len;
    const int v0 = tile * ((NT - p.HT) * V2_CHUNK) - p.HT * V2_CHUNK + t * V2_CHUNK;
    const long long blk = p.blocks_done[stream] + b + p.blk_off;
    if (t == 0) sBase[0] = (int)((blk * (long long)B) % L);
    const bool in_block = v0 < B;
    float2 x[44];
    if (in_block) {
        // history in front of the first callback of a call is the previous call's tail (zeros after a reset)
        const float4 *xp = reinterpret_cast<const float4 *>(p.in + (size_t)stream * p.in_stride + MAIN_HIST + (size_t)b * B + (v0 - 12));
#pragma unroll
        for (int q = 0; q < 22; ++q) {
            const float4 v = (!RAGGED || v0 - 12 + 2 * q < B) ? __ldg(xp + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            x[2 * q] = make_float2(v.x, v.y);
            x[2 * q + 1] = make_float2(v.z, v.w);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 44; ++i) x[i] = make_float2(0.f, 0.f);
    }
    __syncthreads();
    int k0 = sBase[0] + v0;
    if (k0 < 0) k0 += L;
    if (k0 >= L) k0 -= L;
    cascade_loop<5, NT, K2V2Params, RAGGED>(x, p, p.count, sm, t, v0, blk * (long long)B + v0, k0, L, in_block && t >= p.HT,
                                            (size_t)stream * p.out_stride, b, B - v0);
}

// ------------------------------------------------------------------------------------
// k_hb_tail: the half-band stages of a VFO beyond what its mixing kernel runs (a main VFO's stages 4..8 after k1_v2's three, a
// sub VFO's stages 6..8 after the five of k2a_v3 / k2a_v2). No NCO: the input is already mixed and partly decimated, staged
// per callback with a carried history in front. The machine is k2a_v2's without the mixer: a thread owns 32 input samples (+ 12
// in front) in registers and runs the first stage on them, later stages exchange 10 trailing samples through shared memory
// (st_run), HT halo threads per tile recompute what the stages need from in front of the tile. Every stage applies the
// FIRQueueBackToFront rule in its own callback coordinates (st_run's head path; for the first stage here: window slots at negative
// coordinates hold the staged sample one further back, i.e. the previous callback's staged outputs).
// Grid = (stream, channel x tile, callback): all channels of a plan class (mains or subs) and all callbacks of a call in one launch.
// ------------------------------------------------------------------------------------
constexpr int TAIL_NT = 64;
constexpr int TAIL_MAX_STAGES = 5;
constexpr int TAIL_HIST = 512;         // staged samples kept in front of each call (>= the 11 halo chunks + 12 of a 5-stage tail)
struct TailDev {
    const float2 *in;               // staged input: [n_streams][in_stride], in_hist + n_blocks*block_in
    float2 *out;                    // [n_streams][out_stride], out_hist + n_blocks*(block_in >> S)
    long long in_stride, out_stride;
    int in_hist, out_hist, block_in, S, HT, tiles;   // HT halo threads per tile, tiles per callback
};

__global__ void __launch_bounds__(TAIL_NT) k_hb_tail(const TailDev *__restrict__ devs, int max_tiles, int stream0, int b0) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2 *sm = reinterpret_cast<float2 *>(smem_raw);
    const TailDev D = devs[blockIdx.y / max_tiles];
    const int tile = blockIdx.y % max_tiles;
    if (tile >= D.tiles) return;                              // uniform per CTA: a shorter channel of the launch
    const int stream = stream0 + blockIdx.x, b = b0 + blockIdx.z;
    const int t = threadIdx.x;
    const int B = D.block_in, S = D.S;
    const int v0 = tile * ((TAIL_NT - D.HT) * V2_CHUNK) - D.HT * V2_CHUNK + t * V2_CHUNK;
    const bool in_block = v0 < B;
    float2 x[44];                                             // x[i] = staged sample v0 - 12 + i
    {
        // halo chunks reach at most 11 * 32 + 12 samples in front of the callback: the previous callback or the carried history
        const float4 *xp = reinterpret_cast<const float4 *>(D.in + (size_t)stream * D.in_stride + D.in_hist + (size_t)b * B + (v0 - 12));
#pragma unroll
        for (int q = 0; q < 22; ++q) {
            const float4 v = (in_block && v0 - 12 + 2 * q < B) ? __ldg(xp + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            x[2 * q] = make_float2(v.x, v.y);
            x[2 * q + 1] = make_float2(v.z, v.w);
        }
    }
    // first stage on the thread's registers: output r has the window x[2r+2 .. 2r+12] (newest = sample v0 + 2r); at the head of
    // a callback the slots at negative coordinates (x[0..11]) hold the sample one further back
    const int head = (v0 == 0) ? 1 : 0;
    float2 o1[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        float2 w[11];
#pragma unroll
        for (int k = 0; k < 11; ++k) {
            const int i = 2 * r + 2 + k;
            w[k] = (i < 12 && head) ? x[i - 1] : x[i];
        }
        o1[r] = hb11(w[0], w[2], w[4], w[5], w[6], w[8], w[10]);
    }
    const bool store = in_block && t >= D.HT;
    const int nin = B - v0;
    float2 *outp = D.out + (size_t)stream * D.out_stride + D.out_hist + (size_t)b * (B >> S);
    if (S == 1) {
        if (store) st_store_n<16>(o1, outp + (v0 >> 1), nin >> 1);
        return;
    }
    float2 *sA = sm + V2L<TAIL_NT>::SA, *sB = sm + V2L<TAIL_NT>::SB, *sC = sm + V2L<TAIL_NT>::SC, *sD = sm + V2L<TAIL_NT>::SD;
    st_publish<16>(o1, sA, t);
    __syncthreads();
    float2 o2[8];
    st_run<16, true>(o1, o2, sA, t, v0 >> 1);
    if (S == 2) {
        if (store) st_store_n<8>(o2, outp + (v0 >> 2), nin >> 2);
        return;
    }
    st_publish<8>(o2, sB, t);
    __syncthreads();
    float2 o3[4];
    st_run<8, true>(o2, o3, sB, t, v0 >> 2);
    if (S == 3) {
        if (store) st_store_n<4>(o3, outp + (v0 >> 3), nin >> 3);
        return;
    }
    st_publish<4>(o3, sC, t);
    __syncthreads();
    float2 o4[2];
    st_run<4, true>(o3, o4, sC, t, v0 >> 3);
    if (S == 4) {
        if (store) st_store_n<2>(o4, outp + (v0 >> 4), nin >> 4);
        return;
    }
    st_publish<2>(o4, sD, t);
    __syncthreads();
    float2 o5[1];
    st_run<2, true>(o4, o5, sD, t, v0 >> 4);
    if (store) st_store_n<1>(o5, outp + (v0 >> 5), nin >> 5);
}

// ------------------------------------------------------------------------------------
// k1_v2: uint8 IQ -> float (sdr.cpp:43-49) -> DC removal (sdrj.cpp:277-283) -> every main VFO.
// Tile = NT - 4 chunks of 32 samples (a whole number of 128-sample DC blocks); 4 halo threads (one DC block) in front.
//
// DC: the block-start states come bit-exact from the walk kernel (k0_dc_walk). Inside a 128-sample
// block the recursion is continued in real arithmetic: state before the thread's chunk =
// s_blk*(1 - p*c) + c*sum(x[0..p)) (integer prefix sums over the 4 threads of the block; the
// neglected terms are below 2e-8), then avept += c*(x - avept) sample by sample, forwards over
// the chunk and backwards over the 11 samples in front of it. What is lost is only the float
// rounding noise of 128 steps (~1e-7), not the state's lock-in, which lives in the block-start states.
// ------------------------------------------------------------------------------------
struct K1V2Params {
    const uint8_t *iq;
    size_t iq_stride;
    const uint8_t *tail;            // [n_streams][2*RAW_TAIL]
    const uint2 *dc_table;
    const DcAnchor *dc_anchor;
    const long long *blocks_done;
    long long out_stride;
    int dc_stride, block, lut_len, n_main, stream0, b0;
    CascVfo vfos[SDRB_MAX_MAIN];    // the main VFOs
    RfTab rf[SDRB_MAX_MAIN];
};

__device__ __forceinline__ float dc_decode(uint2 e, const DcAnchor &A) {
    return e.y < 2u ? A.sgn * __uint_as_float(e.x + A.lo + 1u) : __uint_as_float(e.x);
}

// Inspection: the `samples` vector of sdrj::demodData (sdrj.cpp:271-294) -- converted and, with
// correct_dc_bias, DC-corrected input -- for the first n samples of one callback. It is what the
// "Main" spectrum shows (sdrj.cpp:296-303). One thread per 128-sample DC block: it starts from the
// block-start state of the walk (bit-exact) and repeats the reference's float steps (no FMA), so
// the result is bit-identical to the reference. table == nullptr: conversion only.
__global__ void __launch_bounds__(64) k_input_samples(const uint8_t *__restrict__ iq, size_t iq_stride, size_t first, int n,
                                                      const uint2 *__restrict__ table, const DcAnchor *__restrict__ anchor,
                                                      int table_stride, int blk0, float2 *__restrict__ out) {
    const int j = blockIdx.x * 64 + threadIdx.x;                 // DC block inside the request
    if (j * DC_BLK >= n) return;
    const int stream = blockIdx.y;
    const uint8_t *src = iq + (size_t)stream * iq_stride + (first + (size_t)j * DC_BLK) * 2;
    float2 *dst = out + (size_t)stream * n + (size_t)j * DC_BLK;
    float sI = 0.f, sQ = 0.f;
    if (table) {
        const uint2 *te = table + ((size_t)stream * table_stride + DC_HALO_BLKS + blk0 + j) * 2;
        sI = dc_decode(__ldg(te), anchor[2 * stream]);
        sQ = dc_decode(__ldg(te + 1), anchor[2 * stream + 1]);
    }
    for (int q = 0; q < DC_BLK / 8; ++q) {
        const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(src) + q);
        const unsigned w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned pr = w[k >> 1] >> (16 * (k & 1));
            float xI = (float)((int)(pr & 0xffu) - 127), xQ = (float)((int)((pr >> 8) & 0xffu) - 127);   // sdr.cpp:48
            if (table) {                                         // sdrj.cpp:281-282, float ops as written
                sI = __fadd_rn(__fmul_rn(sI, DC_A), __fmul_rn(DC_C, xI));
                sQ = __fadd_rn(__fmul_rn(sQ, DC_A), __fmul_rn(DC_C, xQ));
                xI = __fsub_rn(xI, sI);
                xQ = __fsub_rn(xQ, sQ);
            }
            dst[q * 8 + k] = make_float2(xI, xQ);
        }
    }
}

// Tiles per CTA: a CTA walks K1_TPC consecutive tiles of its (stream, callback). While it filters tile i,
// the raw bytes and DC block states of tile i+1 travel global -> shared with cp.async (every thread
// fetches exactly the 96 + 16 bytes it will read back itself, so no barrier is involved); the global
// load latency that used to open every CTA (15 % of the warps' time, profiles/r01_k2a_regions.md) is
// paid once per CTA, and the per-stream constants (callback counter, DC anchors) are read once.
#ifndef SDRB_K1_TPC
#define SDRB_K1_TPC 4
#endif
constexpr int K1_TPC = SDRB_K1_TPC;

// ---- bulk-copy (TMA engine, cp.async.bulk + mbarrier) variant of the tile prefetch: one elected thread moves the whole
// tile's raw bytes and DC block states with two or three bulk copies; everybody waits on the buffer's mbarrier ----
// (mbar_init / mbar_expect_tx / mbar_wait / bulk_g2s live in kernels.cuh)
template <int NT> constexpr int k1_bulk_raw_bytes() { return NT * 64 + 32; }                 // samples v0(0)-16 .. v0(NT-1)+31
template <int NT> constexpr int k1_bulk_buf_bytes() { return k1_bulk_raw_bytes<NT>() + (NT / 4) * 16 + 16; }
template <int NT> constexpr size_t k1v2_smem_bulk() { return V2L<NT>::SMEM + 2 * (size_t)k1_bulk_buf_bytes<NT>(); }
constexpr int K1_PF_BYTES = 112;                          // per thread: 6 x 16 raw bytes + 2 x 8 table bytes
template <int NT> constexpr size_t k1v2_smem() { return V2L<NT>::SMEM + (size_t)NT * K1_PF_BYTES; }

template <bool DC, int NT, bool BULK = false>
__global__ void __launch_bounds__(NT, v2_minb<NT>()) k1_v2(const __grid_constant__ K1V2Params p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2 *sm = reinterpret_cast<float2 *>(smem_raw);
    int *sBase = reinterpret_cast<int *>(sm + V2L<NT>::SEND);

    const int stream = p.stream0 + blockIdx.x;
    const int b = p.b0 + blockIdx.z;
    const int t = threadIdx.x;
    const int B = p.block, L = p.lut_len;
    constexpr int ADV = (NT - K1V2_HT) * V2_CHUNK;
    const int n_tiles = (B + ADV - 1) / ADV;
    const int tile0 = blockIdx.y * K1_TPC;
    unsigned char *pf = smem_raw + V2L<NT>::SMEM + (size_t)t * K1_PF_BYTES;     // this thread's prefetch record
    constexpr int BULK_RAW = NT * 64 + 32, BULK_BUF = BULK_RAW + (NT / 4) * 16 + 16;   // = k1_bulk_raw_bytes / k1_bulk_buf_bytes
    __shared__ __align__(8) unsigned long long pf_bar[2];
    unsigned char *bulk0 = smem_raw + V2L<NT>::SMEM;                            // BULK: two buffers of k1_bulk_buf_bytes
    if (BULK) {
        if (t == 0) {
            mbar_init(&pf_bar[0], 1);
            mbar_init(&pf_bar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        }
        __syncthreads();
    }
    // BULK: thread 0 fetches tile `tile` into buffer `buf`: the raw bytes of samples first-16 .. (clipped to the callback; the
    // part in front of callback 0 of a call comes from the carried tail) and the DC block states of the tile's NT/4 blocks
    auto bulk_issue = [&](int tile, int buf) {
        const int first = tile * ADV - K1V2_HT * V2_CHUNK - 16;                 // first sample of the window of thread 0
        int n = NT * V2_CHUNK + 16;
        if (first + n > B) n = B - first;
        unsigned char *dst = bulk0 + (size_t)buf * BULK_BUF;
        unsigned bytes = 2u * (unsigned)n;
        int ntab = 0;
        if (DC) {
            const int dblk0 = (b * B + first + 16 + RAW_TAIL) / DC_BLK;
            ntab = min(NT / 4, p.dc_stride - dblk0);
            bytes += 16u * (unsigned)ntab;
        }
        mbar_expect_tx(&pf_bar[buf], bytes);
        if (b == 0 && first < 0) {
            bulk_g2s(dst, p.tail + (size_t)stream * (2 * RAW_TAIL) + 2 * (RAW_TAIL + first), 2u * (unsigned)(-first), &pf_bar[buf]);
            bulk_g2s(dst + 2 * (-first), p.iq + (size_t)stream * p.iq_stride, 2u * (unsigned)(n + first), &pf_bar[buf]);
        } else {
            bulk_g2s(dst, p.iq + (size_t)stream * p.iq_stride + ((size_t)b * B + first) * 2, 2u * (unsigned)n, &pf_bar[buf]);
        }
        if (DC && ntab > 0) {
            const int dblk0 = (b * B + first + 16 + RAW_TAIL) / DC_BLK;
            bulk_g2s(dst + BULK_RAW, p.dc_table + ((size_t)stream * p.dc_stride + dblk0) * 2, 16u * (unsigned)ntab, &pf_bar[buf]);
        }
    };

    // fetch of one tile: raw bytes of samples v0-16 .. v0+31 (six 16-byte pieces of 8 samples) and the DC
    // block-start states; pieces that do not exist (past the callback) are simply not fetched
    auto prefetch = [&](int tile) {
        const int v0 = tile * ADV - K1V2_HT * V2_CHUNK + t * V2_CHUNK;
        if (v0 < B) {
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                const int c = v0 - 16 + 8 * q;
                const uint8_t *src = (b == 0 && c < 0) ? p.tail + (size_t)stream * (2 * RAW_TAIL) + 2 * (RAW_TAIL + c)
                                                       : p.iq + (size_t)stream * p.iq_stride + ((size_t)b * B + c) * 2;
                cp_async16(pf + 16 * q, src);
            }
            if (DC) {
                const int dblk = (b * B + v0 + RAW_TAIL) / DC_BLK;   // table index incl. the carried entries
                cp_async16(pf + 96, p.dc_table + ((size_t)stream * p.dc_stride + dblk) * 2);
            }
        }
        cp_async_commit();
    };
    if (BULK) { if (t == 0 && tile0 < n_tiles) bulk_issue(tile0, 0); }
    else if (tile0 < n_tiles) prefetch(tile0);
    const long long blk = p.blocks_done[stream] + b;
    if (t == 0) sBase[0] = (int)((blk * (long long)B) % L);
    const bool first_ever = (blk == 0);
    DcAnchor AI, AQ;
    if (DC) { AI = p.dc_anchor[2 * stream]; AQ = p.dc_anchor[2 * stream + 1]; }
    __syncthreads();
    const int kbase = sBase[0];

    for (int ti = 0; ti < K1_TPC; ++ti) {
        const int tile = tile0 + ti;
        if (tile >= n_tiles) break;
        const int v0 = tile * ADV - K1V2_HT * V2_CHUNK + t * V2_CHUNK;
        const bool in_block = v0 < B;
        if (BULK) {
            mbar_wait(&pf_bar[ti & 1], (unsigned)((ti >> 1) & 1));
            pf = bulk0 + (size_t)(ti & 1) * BULK_BUF + 64 * t;    // this thread's 96 bytes of the shared window
        } else {
            cp_async_wait<0>();
        }
        uint4 raw[6];
        uint2 teI = make_uint2(0u, 2u), teQ = make_uint2(0u, 2u);     // DC block-start states (mode 2 = plain float bits: 0.0f)
#pragma unroll
        for (int q = 0; q < 6; ++q) {
            raw[q] = make_uint4(0x7f7f7f7fu, 0x7f7f7f7fu, 0x7f7f7f7fu, 0x7f7f7f7fu);   // 127 -> 0.0
            if (in_block && !(first_ever && v0 - 16 + 8 * q < 0)) raw[q] = *reinterpret_cast<const uint4 *>(pf + 16 * q);
        }
        if (DC && in_block) {
            const uint4 te = BULK ? *reinterpret_cast<const uint4 *>(bulk0 + (size_t)(ti & 1) * BULK_BUF +
                                                                      BULK_RAW + 16 * (t >> 2))
                                  : *reinterpret_cast<const uint4 *>(pf + 96);
            teI = make_uint2(te.x, te.y);
            teQ = make_uint2(te.z, te.w);
        }
        float2 x[44];                   // x[i] = sample v0 - 12 + i
        {
            float2 y[8];
            unpack8p(raw[0], y);
#pragma unroll
            for (int k = 4; k < 8; ++k) x[k - 4] = y[k];
#pragma unroll
            for (int q = 1; q < 6; ++q) {
                unpack8p(raw[q], y);
#pragma unroll
                for (int k = 0; k < 8; ++k) x[8 * q - 4 + k] = y[k];
            }
        }
        unsigned sI = 0u, sQ = 0u;
        if (DC) {
            // integer sums of the chunk's 32 samples per arm (bytes; I in even, Q in odd positions)
#pragma unroll
            for (int q = 2; q < 6; ++q) {
                sI = __dp4a(raw[q].x, 0x00010001u, sI); sQ = __dp4a(raw[q].x, 0x01000100u, sQ);
                sI = __dp4a(raw[q].y, 0x00010001u, sI); sQ = __dp4a(raw[q].y, 0x01000100u, sQ);
                sI = __dp4a(raw[q].z, 0x00010001u, sI); sQ = __dp4a(raw[q].z, 0x01000100u, sQ);
                sI = __dp4a(raw[q].w, 0x00010001u, sI); sQ = __dp4a(raw[q].w, 0x01000100u, sQ);
            }
        }
        // the record has been consumed (its bytes are in registers): the next tile may overwrite it
        if (ti + 1 < K1_TPC && tile + 1 < n_tiles) {
            if (BULK) { if (t == 0) bulk_issue(tile + 1, (ti + 1) & 1); }     // that buffer was last read two tiles ago (barrier below)
            else prefetch(tile + 1);
        }
        if (DC) {
            const int tot = (int)(sI | (sQ << 16));                 // 32*255 < 65536; prefix of 3 chunks < 65536 too
            const int g = t & 3;                             // position of the chunk inside its DC block
            int inc = tot;
            int up = __shfl_up_sync(0xffffffffu, inc, 1, 4);
            if (g >= 1) inc += up;
            up = __shfl_up_sync(0xffffffffu, inc, 2, 4);
            if (g >= 2) inc += up;
            const int excl = inc - tot;
            const int pcount = 32 * g;
            const float PI_ = (float)((excl & 0xffff) - 127 * pcount), PQ_ = (float)((int)((unsigned)excl >> 16) - 127 * pcount);
            float bI = 0.f, bQ = 0.f;
            if (in_block && !(first_ever && v0 < 0)) {
                bI = dc_decode(teI, AI);
                bQ = dc_decode(teQ, AQ);
            }
            const float decay = 1.0f - DC_C * (float)pcount;
            // negated state after sample v0-1
            const float2 ns0 = make_float2(-(bI * decay + DC_C * PI_), -(bQ * decay + DC_C * PQ_));
            float2 ns = ns0;
#pragma unroll
            for (int i = 12; i < 44; ++i) {                  // forwards: d = x - s, s += c*d, out = x - s
                const float2 d = add2(x[i], ns);
                ns = fma2(splat2(-DC_C), d, ns);
                x[i] = add2(x[i], ns);
            }
            ns = ns0;
#pragma unroll
            for (int i = 11; i >= 1; --i) {                  // backwards: out = x - s_j, s_{j-1} = s_j - c*out
                x[i] = add2(x[i], ns);
                ns = fma2(splat2(DC_C), x[i], ns);
            }
        }
        if (first_ever && v0 <= 0) {                         // nothing exists before stream sample 0
            const int lim = v0 < 0 ? 44 : 12;
#pragma unroll
            for (int i = 0; i < 44; ++i)
                if (i < lim) x[i] = make_float2(0.f, 0.f);
        }
        int k0 = kbase + v0;
        if (k0 < 0) k0 += L;
        if (k0 >= L) k0 -= L;
        cascade_loop<3, NT>(x, p, p.n_main, sm, t, v0, blk * (long long)B + v0, k0, L, in_block && t >= K1V2_HT,
                            (size_t)stream * (size_t)p.out_stride, b);
        __syncthreads();                                     // the scratch arrays are reused by the next tile
    }
}

}  // namespace sdrb

namespace sdrb {

// ------------------------------------------------------------------------------------
// k2b_v2: USB demodulation + optional low-pass + gain + int16, one WARP per tile, no CTA barrier.
//   usb[n] = re[n-62] - sum_{i odd} points[i]*im[n-124+i]      (vfo.cpp:316-324, dsp.cpp:218-231)
//   out[n] = sum_{t<N} lpf[t]*usb[n-N+t]                        (dsp.cpp:59-71: newest sample excluded)
//   pcm    = (short)(out*gain*32768.0)                          (vfo.cpp:328)
// A tile is 1024 usb values (1024 - NP outputs; the first NP are the low-pass history). A lane owns
// 32 consecutive values = 16 packed pairs and keeps 16 FP32x2 accumulators:
//   * Hilbert: only odd taps are non-zero, so usb[2w] and usb[2w+1] use the same 62 coefficients on
//     im[2w-123+2m] and im[2w-122+2m]: the pair (im[2v+1], im[2v+2]) IS the packed operand -- one
//     FFMA2 per tap and output pair, operands straight out of 16-byte shared loads;
//   * low-pass: the pair (out[k], out[k+1]) needs (usb[k+t], usb[k+t+1]): even t from the natural
//     pairs E, odd t from a copy O shifted by one sample;
//   * shared arrays are rows of 32 floats + 4 pad: a lane's row starts 36 words after its
//     neighbour's, so every 16-byte access of a warp is conflict free; E/O overlay the input rows.
// Work per 16 taps: 16 LDS.128 + 256 FFMA2 per lane.
// ------------------------------------------------------------------------------------
constexpr int UV_USB = 1024;                 // usb values per tile
constexpr int UV_ROW = 36;                   // floats per padded row
constexpr int UV_WARPS = 4;                  // warps (= streams) per CTA
constexpr int UV_RE_ROWS = 32, UV_IM_ROWS = 36;
constexpr int UV_IN_FLOATS = (UV_RE_ROWS + UV_IM_ROWS) * UV_ROW;

struct K2bV2Params {
    const UsbDev *devs;
    int16_t *pcm;
    float *tap;
    int n_blocks, cb0, ncb, stream0, stream_end, pcm_per_block;
    int warp_floats;                        // shared floats per warp: max(input rows, 2 * E/O rows)
    int eo_rows;                            // rows of each of E and O
    int np_max;                             // longest (padded) low-pass of the plan
    unsigned short tiles[SDRB_MAX_SUB];     // tiles per callback of each USB VFO: CTAs beyond it leave without touching memory
};

__device__ __forceinline__ constexpr int uv_off(int x) { return (x >> 4) * UV_ROW + (x & 15) * 2; }   // pair index -> float offset

// acc[r] += sum_{s<STEPS} coef[s*CSTR] * W[p0 + r + s],  r = 0..15; W = packed pairs of the lane's rows.
// p0 (even) is a run-time value: the callers loop over tap blocks WITHOUT unrolling, so the hot code
// of the kernel is two bodies of 256 FFMA2 (~10 KB). The fully unrolled version was 103 KB of SASS and
// the warps of a CTA, which run independently here, stalled on instruction fetch ("no instruction"
// 2.9 stalls per issue in ncu) -- see profiles/r01_k2b_icache.md.
template <int STEPS, int CSTR>
__device__ __forceinline__ void uv_fir_block(float2 (&acc)[16], const float *__restrict__ row, int p0, const float2 *__restrict__ coef2) {
    constexpr int NCH = (16 + STEPS) / 2;                    // 16-byte chunks = 2 pairs each (one pair more than needed)
    float2 W[2 * NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const int p = p0 + 2 * c;                            // pair p lives at float 2p + 4*(p/16) of the padded rows
        const float4 v = *reinterpret_cast<const float4 *>(row + 2 * p + 4 * (p >> 4));
        W[2 * c] = make_float2(v.x, v.y);
        W[2 * c + 1] = make_float2(v.z, v.w);
    }
#pragma unroll
    for (int s = 0; s < STEPS; ++s) {
        const float2 c2 = coef2[s * CSTR];
#pragma unroll
        for (int r = 0; r < 16; ++r) acc[r] = fma2(c2, W[r + s], acc[r]);
    }
}

// Ragged end of a tile / callback / call (not taken for the sample plans, whose sizes are multiples
// of 8): element-wise stores. Out of line and rolled so that it costs the hot path nothing.
__device__ __noinline__ void uv_store_ragged(const float *v, int k0, int tile_out, int n0, int n_total, int samples_out, int stream,
                                             int n_blocks, int pcm_per_block, int pcm_offset, int16_t *pcm, float *tap) {
    int nn = n0 + k0;
    int bl = nn / samples_out, ii = nn - bl * samples_out;
#pragma unroll 1
    for (int e = 0; e < 32; ++e, ++nn) {
        if (k0 + e < tile_out && nn < n_total) {
            const size_t a2 = ((size_t)stream * n_blocks + bl) * pcm_per_block + pcm_offset + ii;
            pcm[a2] = (int16_t)__float2int_rz(v[e]);
            if (tap) tap[a2] = v[e];
        }
        if (++ii == samples_out) { ii = 0; ++bl; }
    }
}

#ifndef UV_MINB
#define UV_MINB 4
#endif
__global__ void __launch_bounds__(UV_WARPS * 32, UV_MINB) k2b_v2(const __grid_constant__ K2bV2Params p) {
    extern __shared__ __align__(16) float uv_smem[];
    if (blockIdx.z >= p.tiles[blockIdx.y]) return;          // grid.z is the longest VFO's tile count
    const UsbDev &D = p.devs[blockIdx.y];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int NP = D.np;                                    // multiple of 16 (leading zeros)
    const int tile_out = UV_USB - NP;
    const int n_lo = p.cb0 * D.samples_out, n_total = (p.cb0 + p.ncb) * D.samples_out;
    const int n0 = n_lo + blockIdx.z * tile_out;
    if (n0 >= n_total) return;
    const int stream = p.stream0 + blockIdx.x * UV_WARPS + warp;
    const bool live = stream < p.stream_end;
    // ---- the tile's input, z-local q = 0..1152 (re rows: q - 66, im rows: q - 1): lane l owns q = 32 it + l.
    // All 37 loads of the lane are issued before the coefficient staging and the barrier, so the tile costs
    // one HBM/L2 latency, overlapped with the descriptor-dependent coefficient loads.
    constexpr int NIT = (UV_USB + 128 + 1 + 31) / 32;
    float2 v[NIT];
    {
        const long long zlo = (long long)n0 - NP - 128;
        const long long room = (long long)n_total - zlo;                              // samples that exist from zlo on (> 0)
        const int lim = (int)(room < (long long)(UV_USB + 128 + 1) ? room : (long long)(UV_USB + 128 + 1)) - lane;
        const float2 *zq = D.src + (size_t)(live ? stream : p.stream0) * D.src_stride + D.src_hist + zlo + lane;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            v[it] = make_float2(0.f, 0.f);
            if (live && 32 * it < lim) v[it] = __ldg(zq + 32 * it);
        }
    }
    // coefficient pairs (h, h), shared by the CTA's warps
    float2 *sHil2 = reinterpret_cast<float2 *>(uv_smem);
    float2 *sLpf2 = sHil2 + 64;
    float *wbase = uv_smem + 2 * (64 + p.np_max) + (size_t)warp * p.warp_floats;
    for (int e = threadIdx.x; e < 64; e += UV_WARPS * 32) { const float h = D.hil[e]; sHil2[e] = make_float2(h, h); }
    for (int e = threadIdx.x; e < NP; e += UV_WARPS * 32) { const float c = D.lpf[e]; sLpf2[e] = make_float2(c, c); }
    __syncthreads();                                        // the only CTA-wide barrier
    if (!live) return;

    // ---- input rows: re (z-local 66..1089) and im (z-local 1..1152) ----
    float *sRe = wbase, *sIm = wbase + UV_RE_ROWS * UV_ROW;
    {
        // u = q - 66 = 32 (it - 3) + (lane + 30), k = q - 1 = 32 (it - 1) + (lane + 31): row = it + const(lane),
        // so every store is the lane's base pointer plus a compile-time offset; only the first and last rows
        // depend on the lane
        const int cr = lane + 30, ci = lane + 31;
        const int hr = cr >> 5, hi = ci >> 5;
        float *pr = sRe + (hr - 3) * UV_ROW + (cr & 31);
        float *pi = sIm + (hi - 1) * UV_ROW + (ci & 31);
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            if (it >= 3 && it <= UV_RE_ROWS + 1) pr[it * UV_ROW] = v[it].x;
            else if (it == 2) { if (hr == 1) pr[it * UV_ROW] = v[it].x; }
            else if (it == UV_RE_ROWS + 2) { if (hr == 0) pr[it * UV_ROW] = v[it].x; }
            if (it >= 1 && it <= UV_IM_ROWS - 1) pi[it * UV_ROW] = v[it].y;
            else if (it == 0) { if (hi == 1) pi[it * UV_ROW] = v[it].y; }
            else if (it == UV_IM_ROWS) { if (hi == 0) pi[it * UV_ROW] = v[it].y; }
        }
    }
    __syncwarp();

    // ---- Hilbert: pair (usb[32 lane + 2r], usb[.. + 2r + 1]) = re - sum_j hil[j] * P[16 lane + r + j] ----
    float2 acc[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) acc[r] = make_float2(0.f, 0.f);
    const float *imrow = sIm + lane * UV_ROW;
#pragma unroll 1
    for (int s = 0; s < 4; ++s) uv_fir_block<16, 1>(acc, imrow, 16 * s, sHil2 + 16 * s);
    {
        const float4 *re4 = reinterpret_cast<const float4 *>(sRe + lane * UV_ROW);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const float4 v = re4[c];
            acc[2 * c] = make_float2(v.x - acc[2 * c].x, v.y - acc[2 * c].y);
            acc[2 * c + 1] = make_float2(v.z - acc[2 * c + 1].x, v.w - acc[2 * c + 1].y);
        }
    }
    if (NP > 0) {
        // ---- E/O rows over the (now dead) input rows, then the low-pass ----
        const float nxt = __shfl_down_sync(0xffffffffu, acc[0].x, 1);   // first usb value of the next lane
        __syncwarp();
        float *sE = wbase, *sO = wbase + p.eo_rows * UV_ROW;
        float4 *e4 = reinterpret_cast<float4 *>(sE + lane * UV_ROW), *o4 = reinterpret_cast<float4 *>(sO + lane * UV_ROW);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            e4[c] = make_float4(acc[2 * c].x, acc[2 * c].y, acc[2 * c + 1].x, acc[2 * c + 1].y);
            const float last = c < 7 ? acc[c < 7 ? 2 * c + 2 : 0].x : nxt;
            o4[c] = make_float4(acc[2 * c].y, acc[2 * c + 1].x, acc[2 * c + 1].y, last);
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 16; ++r) acc[r] = make_float2(0.f, 0.f);
        const float *erow = sE + lane * UV_ROW, *orow = sO + lane * UV_ROW;
        const int nb16 = NP >> 4;                             // blocks of 16 taps = 8 pair steps on E and on O
#pragma unroll 1
        for (int b = 0; b < nb16; ++b) {
            const float2 *cf = sLpf2 + 16 * b;
            uv_fir_block<8, 2>(acc, erow, 8 * b, cf);
            uv_fir_block<8, 2>(acc, orow, 8 * b, cf + 1);
        }
    }
    // ---- gain, quantise, store: 32 consecutive outputs per lane ----
    const int k0 = 32 * lane;
    if (k0 >= tile_out) return;
    const int n = n0 + k0;
    if (n >= n_total) return;
    const int blk = n / D.samples_out, i = n - blk * D.samples_out;
    const size_t at = ((size_t)stream * p.n_blocks + blk) * p.pcm_per_block + D.pcm_offset + i;
    const float g = D.gain;
    const int nv = min(32, min(tile_out - k0, n_total - n));      // outputs this lane owns
    if ((nv & 7) == 0 && (i + nv <= D.samples_out) && ((at & 7) == 0)) {   // whole 16-byte groups inside one callback record
        uint4 *dst = reinterpret_cast<uint4 *>(p.pcm + at);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            if (8 * c >= nv) break;
            unsigned w[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const float2 v = acc[4 * c + h];
                const int lo = __float2int_rz((v.x * g) * 32768.0f), hi = __float2int_rz((v.y * g) * 32768.0f);
                w[h] = ((unsigned)lo & 0xffffu) | ((unsigned)hi << 16);
            }
            dst[c] = make_uint4(w[0], w[1], w[2], w[3]);
        }
        if (p.tap) {
            float4 *t4 = reinterpret_cast<float4 *>(p.tap + at);
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (4 * c < nv)
                    t4[c] = make_float4((acc[2 * c].x * g) * 32768.0f, (acc[2 * c].y * g) * 32768.0f,
                                        (acc[2 * c + 1].x * g) * 32768.0f, (acc[2 * c + 1].y * g) * 32768.0f);
        }
    } else {
        float v[32];
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            v[2 * r] = (acc[r].x * g) * 32768.0f;
            v[2 * r + 1] = (acc[r].y * g) * 32768.0f;
        }
        uv_store_ragged(v, k0, tile_out, n0, n_total, D.samples_out, stream, p.n_blocks, p.pcm_per_block, D.pcm_offset, p.pcm, p.tap);
    }
}

}  // namespace sdrb

namespace sdrb {

// ------------------------------------------------------------------------------------
// k2_late_v2: the /5 and /6 decimating FIR of the "late" plans (vfo.cpp:346-384; fir_decI/Q of 49 / 73
// taps on both arms), polyphase:  d[m] = sum_i c[i] z[L m - N + i],  i = L a + r  ->
//   d[m] = sum_r sum_a c[L a + r] * zr[m + a],   zr[j] = z[L j - N + r].
// A thread owns R = 8 consecutive outputs. Per phase r it loads the R + A - 1 samples zr[m0 .. m0+R+A-2]
// once (LDS.64, stride L samples) and runs A x R packed FMAs on them (both arms at once, the tap as
// (c, c)): 1.3 instructions per output and tap instead of the 4 of one-output-per-thread code.
// Shared layout: one pad slot per thread segment of L*R samples, so the segment stride is odd in
// 8-byte units and the strided loads of a warp are conflict free.
// ------------------------------------------------------------------------------------
constexpr int LV_THREADS = 128, LV_R = 8, LV_TILE = LV_THREADS * LV_R;
constexpr int LV_AMAX = 16;                               // taps per phase the coefficient table is padded to
template <int L> constexpr int lv_span() { return L * LV_TILE + L * LV_AMAX; }
template <int L> constexpr size_t lv_smem() {
    return (size_t)(lv_span<L>() + lv_span<L>() / (L * LV_R) + 2) * sizeof(float2) + (size_t)L * LV_AMAX * sizeof(float2);
}

// AT: taps per phase at compile time (10 for the reference's 49 taps / 5, 13 for 73 / 6) when every late VFO of the plan has that
// many; 0 = read from the descriptor (the FIR loops are then predicated per tap: a third more instructions)
#ifndef LV_MINB
#define LV_MINB 4
#endif
template <int L, int AT>
__global__ void __launch_bounds__(LV_THREADS, LV_MINB) k2_late_v2(const LateDev *__restrict__ devs, int cb0, int ncb, int stream0) {
    extern __shared__ __align__(16) unsigned char lv_raw[];
    constexpr int SEG = L * LV_R;                           // samples per thread segment
    float2 *sz = reinterpret_cast<float2 *>(lv_raw);
    constexpr int SPAN_MAX = L * LV_TILE + L * LV_AMAX;     // = lv_span<L>()
    float2 *sc = sz + SPAN_MAX + SPAN_MAX / SEG + 2;        // (c, c) pairs, index L*a + r, zero padded
    const LateDev &D = devs[blockIdx.y];
    const int n_total = (cb0 + ncb) * D.samples_out;               // outputs exist up to here
    const int m0 = cb0 * D.samples_out + blockIdx.z * LV_TILE;
    if (m0 >= n_total) return;
    const int stream = stream0 + blockIdx.x;
    const int t = threadIdx.x;
    const int N = D.ntaps;
    const int A = AT > 0 ? AT : (N + L - 1) / L;            // taps per phase (10 for 49/5, 13 for 73/6)
    const int span = L * LV_TILE + L * A;
    const long long zlo = (long long)L * m0 - N;            // may be negative: history
    const long long zmax = (long long)(cb0 + ncb) * D.block_z;
    const float2 *zp = D.z + (size_t)stream * D.z_stride + D.z_hist;
    if (D.mix_lut == nullptr) {
#pragma unroll 8
        for (int e = t; e < span; e += LV_THREADS) {         // 8 independent loads in flight per thread
            const long long zi = zlo + e;
            sz[e + e / SEG] = (zi < zmax) ? __ldg(zp + zi) : make_float2(0.f, 0.f);
        }
    } else {
        // fused mixer: sample zi of this call is stream sample n0 + zi and uses table entry (n0 + zi) mod len -- entry len-1
        // for stream sample 0 (oscillator.cpp:26-30,42-48). History in front of the call (zi < 0) is the parent's own history.
        const int len = D.lut_len;
        const long long n0 = D.blocks_done[stream] * (long long)D.block_z;
        const long long first = n0 + zlo;                    // stream sample of element 0 of the tile
        if (first > 0 && zlo + span <= zmax && span < len) {
            // the usual tile: every element exists, stream sample 0 is not in it, the table wraps at most once. Per element two
            // 8-byte loads, one compare-and-subtract for the wrap and a complex product as two packed operations -- the staging
            // loop used to cost more instructions than the FIR behind it (16 per element against 13 per element for /5, 49 taps)
            const int k0 = (int)(first % len);
            const float2 *__restrict__ xp = zp + zlo;
            const float2 *__restrict__ lut = D.mix_lut;
            if (AT > 0 && k0 + span <= len) {
                // ... and the table does not wrap inside the tile (all tiles but one per second of signal), tile length known at
                // compile time: a thread's elements are e = t + 128 i. Both loads then are one base pointer plus an immediate, and
                // so is the padded destination e + e / SEG: 128 * P is a whole number of segments for P = SEG / gcd(128, SEG)
                // (5 for /5, 3 for /6), so only the first P destinations are computed, the others are those plus a constant.
                // Per element: two loads, two packed operations, one store (the address arithmetic used to be 12 integer
                // instructions per element, profiles/r02_experiments.md section 5).
                constexpr int SPAN_C = L * LV_TILE + L * AT;
                constexpr int G = (SEG % 16 == 0) ? 16 : 8;      // gcd(128, SEG) for SEG = 40 (8) and 48 (16)
                static_assert(SEG % G == 0 && LV_THREADS % G == 0 && (SEG / G) % 2 == 1, "period of the padded layout");
                constexpr int P = SEG / G;
                constexpr int ADV = LV_THREADS * P + LV_THREADS * P / SEG;
                constexpr int NFULL = SPAN_C / LV_THREADS;
                int dbase[P];
#pragma unroll
                for (int u = 0; u < P; ++u) dbase[u] = (t + LV_THREADS * u) + (t + LV_THREADS * u) / SEG;
                const float2 *__restrict__ xq = xp + t;
                const float2 *__restrict__ lq = lut + k0 + t;
#pragma unroll
                for (int i = 0; i < NFULL; ++i) {
                    const float2 x = __ldg(xq + LV_THREADS * i), r = __ldg(lq + LV_THREADS * i);
                    sz[dbase[i % P] + (i / P) * ADV] = fma2(make_float2(-x.y, x.x), make_float2(r.y, r.y), mul2(x, make_float2(r.x, r.x)));
                }
                const int e = t + LV_THREADS * NFULL;
                if (e < SPAN_C) {
                    const float2 x = __ldg(xp + e), r = __ldg(lut + k0 + e);
                    sz[e + e / SEG] = fma2(make_float2(-x.y, x.x), make_float2(r.y, r.y), mul2(x, make_float2(r.x, r.x)));
                }
            } else {
#pragma unroll 8
                for (int e = t; e < span; e += LV_THREADS) {
                    int k = k0 + e;
                    if (k >= len) k -= len;
                    const float2 x = __ldg(xp + e), r = __ldg(lut + k);
                    sz[e + e / SEG] = fma2(make_float2(-x.y, x.x), make_float2(r.y, r.y), mul2(x, make_float2(r.x, r.x)));
                }
            }
        } else {
            int k = (int)(((first + t) % len + len) % len);
            const int kstep = LV_THREADS % len;
#pragma unroll 4
            for (int e = t; e < span; e += LV_THREADS) {
                const long long zi = zlo + e;
                float2 v = make_float2(0.f, 0.f);
                if (zi < zmax) {
                    const float2 x = __ldg(zp + zi);
                    const float2 r = __ldg(D.mix_lut + ((n0 + zi == 0) ? len - 1 : k));
                    v = fma2(make_float2(-x.y, x.x), make_float2(r.y, r.y), mul2(x, make_float2(r.x, r.x)));
                }
                sz[e + e / SEG] = v;
                k += kstep;
                if (k >= len) k -= len;
            }
        }
    }
    for (int e = t; e < L * LV_AMAX; e += LV_THREADS) {
        const float c = e < N ? D.taps[e] : 0.f;
        sc[e] = make_float2(c, c);
    }
    __syncthreads();
    const int m = m0 + t * LV_R;
    if (m >= n_total) return;
    float2 acc[LV_R];
#pragma unroll
    for (int k = 0; k < LV_R; ++k) acc[k] = make_float2(0.f, 0.f);
    const float2 *base = sz + t * (SEG + 1);                // logical sample L*(t*R) of the tile
#pragma unroll 1
    for (int r = 0; r < L; ++r) {
        constexpr int AU = AT > 0 ? AT : LV_AMAX;             // unrolled extent
        float2 w[LV_R + AU - 1];
#pragma unroll
        for (int j = 0; j < LV_R + AU - 1; ++j)
            if (AT > 0 || j < LV_R + A - 1) w[j] = base[L * j + r + j / LV_R];          // + one pad per segment crossed
#pragma unroll
        for (int a = 0; a < AU; ++a) {
            if (AT > 0 || a < A) {
                const float2 c2 = sc[L * a + r];
#pragma unroll
                for (int k = 0; k < LV_R; ++k) acc[k] = fma2(c2, w[k + a], acc[k]);
            }
        }
    }
    float2 *dst = D.d + (size_t)stream * D.d_stride + D.d_hist + m;
    if (m + LV_R <= n_total && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
        for (int k = 0; k < LV_R; k += 2)
            *reinterpret_cast<float4 *>(dst + k) = make_float4(acc[k].x, acc[k].y, acc[k + 1].x, acc[k + 1].y);
    } else {
        for (int k = 0; k < LV_R; ++k)
            if (m + k < n_total) dst[k] = acc[k];
    }
}

}  // namespace sdrb
