// Third-generation sub-VFO cascade (sm_100a): k2a_v3. One WARP is the unit of work -- no CTA barrier in
// the steady state -- and it alternates between two roles over tiles of 128 parent samples:
//
//   A (time-parallel, first half-band stage): lane l owns parent samples c0+4l .. c0+4l+3 of each of the
//     warp's streams and produces the two first-stage outputs whose newest sample is c0+4l and c0+4l+2.
//     The NCO rotation (vfo.cpp:237-245) is folded into the half-band taps (halfbanddecimator.h:66-79):
//     with lut[k+d] = lut[k] * E^d (E = rot/|rot|, the rotating frame of kernels_v2.cuh) the mixed and
//     filtered sample is
//         y = lut[kc] * ( h5 x[c] + sum_{d=1,3,5} h_d cos(wd) (x[c+d] + x[c-d]) + j h_d sin(wd) (x[c+d] - x[c-d]) ),
//     and the sums and differences do NOT depend on the VFO: they are formed once per tile and stream and
//     reused by all 12-15 sub VFOs. Per VFO and output: 6 FFMA2 + one complex multiply by the table entry
//     (instead of 21 complex multiplies + 7 packed operations per 16 outputs and VFO in k2a_v2); the complex
//     multiplies are two packed operations each (k3_cmul).
//     Taps are doubled (2 h5 = 1: the centre term costs nothing) and the factor 2^-S of the S stages is
//     folded into the rotation table, which is exact in binary floating point.
//   B (VFO-parallel, later stages): lane = (stream, VFO) row. The row's 64 first-stage outputs of the tile
//     pass through shared memory exactly once (A writes, B reads); stages 2..S then run as a streaming
//     filter on the lane's OWN registers, the 11-sample histories of every stage stay in registers from
//     tile to tile: no halo exchange, no neighbour, no barrier. (k2a_v2 spent as many shared-memory
//     wavefronts on halo and own-sample round trips as FMA-pipe cycles on arithmetic.)
//
// A warp walks a span of consecutive tiles of one callback; the histories at the start of a span are
// rebuilt by running the three tiles in front of it (the cascade is feed-forward, so this is exact).
// FIRQueueBackToFront's off-by-one (dsp.cpp:163-173) is one rule again: at callback coordinate 0 every
// stage's history is shifted by one sample (the newest is dropped), and the tile that starts a callback
// -- like tiles that touch the table's start-up transient, its wrap or stream sample 0
// (oscillator.cpp:26-30,42-48) -- takes the exact path: every rotation read from the Oscillator table.
//
// The body is written once as a __host__ __device__ template over an execution environment (lane id,
// warp barrier): tests/cpp/k3_sim.cu runs the very same code on the CPU with 32 host threads per warp.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string.h>

namespace sdrb {

constexpr int K3_TILE = 128;            // parent samples per tile
constexpr int K3_OUT1 = 64;             // first-stage outputs per row and tile
constexpr int K3_ROW = 66;              // float2 per ring row: 64 + 2 pad (row stride 528 B: 16-byte row reads of 8 lanes hit 8 bank groups)
constexpr int K3_WARM = 3;              // warm-up tiles in front of a span (>= 336 samples for 5 stages)
constexpr int K3_MAX_VFO = 16;
constexpr int K3_LUT_STEADY = 512;      // table entries of the start-up transient (94 measured)
constexpr int K3_MAX_SLOTS = K3_MAX_VFO * 32;

#ifndef HB_P0
#define HB_P0 0.0060431029837374152f
#define HB_P2 (-0.049372515458761493f)
#define HB_P4 0.29332944952052842f
#define HB_P5 0.5f
#endif

#define K3_HD __host__ __device__ __forceinline__

struct K3Vfo {
    const float2 *lut;          // Oscillator table
    float2 *out;                // [n_streams][out_stride]: hist + n_blocks*block_out
    int S, block_out, hist, pad;
    float2 A[3];                // (a, a),  a = 2 h_d cos(w d), d = 1, 3, 5
    float2 Bc[3];               // (-b, b), b = 2 h_d sin(w d)
};

struct K3Params {
    K3Vfo v[K3_MAX_VFO];
    const float2 *rrel;         // [count][64]: 2^-S * E^(2j - 5)
    const float2 *in;           // parent main output, hist_in samples of history in front of each stream
    const long long *blocks_done;
    long long in_stride, out_stride;
    int hist_in, count, lut_len, block_in, n_tiles, tiles_per_span, stream0, stream_end, b0, nsw;
    // k2a_v3<MAXS, true>: warp-local stream s of stream group sg is bank stream map[sg * nsw + s]; stream0 is 0 and stream_end is
    // the list length
    const int *map;
};

// Host side: the folded taps and the rotation table of one VFO. w = angle of the float rotation the Oscillator
// table is built from (oscillator.cpp:9-14), so E^d = (cos(w d), sin(w d)) follows the table, not the ideal NCO.
inline void k3_fill_vfo(double sample_rate, double frequency, int S, K3Vfo &V, float2 *rrel64) {
    const double step = 2.0 * 3.14159265358979323846264338327950288 * frequency / sample_rate;
    const float rr = (float)cos(step), ri = (float)sin(step);
    const double w = atan2((double)ri, (double)rr);
    const double h[3] = {(double)HB_P4, (double)HB_P2, (double)HB_P0};       // taps at distance 1, 3, 5 from the centre
    for (int d = 0; d < 3; ++d) {
        const double a = 2.0 * h[d] * cos(w * (2 * d + 1)), b = 2.0 * h[d] * sin(w * (2 * d + 1));
        V.A[d] = make_float2((float)a, (float)a);
        V.Bc[d] = make_float2((float)-b, (float)b);
    }
    const double sc = 1.0 / (double)(1 << S);
    for (int j = 0; j < K3_OUT1; ++j) rrel64[j] = make_float2((float)(sc * cos(w * (2 * j - 5))), (float)(sc * sin(w * (2 * j - 5))));
    V.S = S;
}

// ---- arithmetic helpers: packed FP32 pairs on the device, plain C++ in the host simulation ----
K3_HD float2 k3_add(float2 a, float2 b) {
#ifdef __CUDA_ARCH__
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&r);
#else
    return make_float2(a.x + b.x, a.y + b.y);
#endif
}
K3_HD float2 k3_sub(float2 a, float2 b) {
#ifdef __CUDA_ARCH__
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&r);
#else
    return make_float2(a.x - b.x, a.y - b.y);
#endif
}
K3_HD float2 k3_fma(float2 a, float2 b, float2 c) {
#ifdef __CUDA_ARCH__
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(r)
        : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)),
          "l"(*reinterpret_cast<unsigned long long *>(&c)));
    return *reinterpret_cast<float2 *>(&r);
#else
    return make_float2(a.x * b.x + c.x, a.y * b.y + c.y);
#endif
}
K3_HD float2 k3_splat(float v) { return make_float2(v, v); }
// complex product a * b. Device: two packed operations -- b * (a.x, a.x), then (-b.y, b.x) * (a.y, a.y) added: ptxas folds the
// half swap, the per-half sign and the broadcast of the scalar into the operands of FMUL2 / FFMA2 (no extra registers or moves)
K3_HD float2 k3_cmul(float2 a, float2 b) {
#ifdef __CUDA_ARCH__
    unsigned long long r, bx = *reinterpret_cast<unsigned long long *>(&b);
    float2 sx = make_float2(a.x, a.x), sy = make_float2(a.y, a.y), bs = make_float2(-b.y, b.x);
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(bx), "l"(*reinterpret_cast<unsigned long long *>(&sx)));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(r) : "l"(*reinterpret_cast<unsigned long long *>(&bs)), "l"(*reinterpret_cast<unsigned long long *>(&sy)));
    return *reinterpret_cast<float2 *>(&r);
#else
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
#endif
}
// 16-byte store to GLOBAL memory (the compiler then knows it cannot alias the shared-memory loads around it)
K3_HD void k3_store_global16(float2 *dst, float4 v) {
#ifdef __CUDA_ARCH__
    asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(__cvta_generic_to_global(dst)), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
#else
    *reinterpret_cast<float4 *>(dst) = v;
#endif
}
template <class T> K3_HD T k3_ldg(const T *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// 11-tap half-band with doubled taps (2 h5 = 1): returns 2 * hbcoeff11 . window  (dsp.cpp:139-142)
K3_HD float2 k3_hb(float2 w0, float2 w2, float2 w4, float2 w5, float2 w6, float2 w8, float2 w10) {
    return k3_fma(k3_splat(2.f * HB_P0), k3_add(w0, w10),
                  k3_fma(k3_splat(2.f * HB_P2), k3_add(w2, w8), k3_fma(k3_splat(2.f * HB_P4), k3_add(w4, w6), w5)));
}

// One streaming half-band stage on a lane's own registers. h[0..10] = the 11 samples in front of nw[0]
// (h[10] the newest); outputs o[r] have nw[2r] as their newest sample (window = the 10 samples before it
// and itself). Afterwards h = the last 11 samples of [h | nw].
template <int N>
K3_HD void k3_stage(float2 (&h)[11], const float2 (&nw)[N], float2 (&o)[N / 2]) {
    float2 W[11 + N];
#pragma unroll
    for (int i = 0; i < 11; ++i) W[i] = h[i];
#pragma unroll
    for (int i = 0; i < N; ++i) W[11 + i] = nw[i];
#pragma unroll
    for (int r = 0; r < N / 2; ++r)
        o[r] = k3_hb(W[2 * r + 1], W[2 * r + 3], W[2 * r + 5], W[2 * r + 6], W[2 * r + 7], W[2 * r + 9], W[2 * r + 11]);
#pragma unroll
    for (int i = 0; i < 11; ++i) h[i] = W[N + i];
}

// the FIRQueueBackToFront rule at callback coordinate 0: the sample at coordinate -1 is dropped, slots
// -10..-1 of the next windows hold coordinates -11..-2
K3_HD void k3_head_shift(float2 (&h)[11]) {
#pragma unroll
    for (int i = 10; i >= 1; --i) h[i] = h[i - 1];
}

struct K3Hist {
    float2 h2[11], h3[11], h4[11], h5[11];
};

// Shared memory of a CTA: [rrel: count*64 float2][slot table: K3_MAX_SLOTS ushort][per warp: ring of `rows` rows,
// 32 dst pointers, 2 x 32 table anchors (float2), 32 per-stream table bases (int2)]
K3_HD size_t k3_warp_smem_bytes(int rows) {
    return (size_t)rows * K3_ROW * sizeof(float2) + 32 * sizeof(float2 *) + 64 * sizeof(float2) + 32 * sizeof(int2);
}
K3_HD size_t k3_cta_smem_bytes(int count, int warps, int rows) {
    return (size_t)count * K3_OUT1 * sizeof(float2) + K3_MAX_SLOTS * sizeof(unsigned short) + (size_t)warps * k3_warp_smem_bytes(rows);
}
// 8 bytes global -> shared without passing through a register (LDGSTS); k3_async_wait() makes them visible to the issuing thread
K3_HD void k3_async_copy8(void *smem, const void *gmem) {
#ifdef __CUDA_ARCH__
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(gmem));
#else
    memcpy(smem, gmem, 8);
#endif
}
K3_HD void k3_async_copy16(void *smem, const void *gmem) {
#ifdef __CUDA_ARCH__
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
#else
    memcpy(smem, gmem, 16);
#endif
}
K3_HD void k3_async_wait() {
#ifdef __CUDA_ARCH__
    asm volatile("cp.async.wait_all;\n" ::: "memory");
#endif
}
K3_HD void k3_prefetch_l1(const void *p) {
#ifdef __CUDA_ARCH__
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

// One warp's work: streams sbase .. sbase+nsw-1 (MAP: list entries sg*nsw .. sg*nsw+nsw-1 of p.map), tiles of span `span` of
// callback b.
//   ring    32 rows of K3_ROW float2, private to the warp
//   sdst    32 pointers, private to the warp
//   srrel   the CTA's copy of p.rrel;  stab: slot table (v << 8 | 16-byte chunk), n_slots entries per stream
//   sK      32 entries, private to the warp: 0..nsw-1 hold each stream's table index and start flag, and with MAP entries 16.. the
//           bank index of each stream (every row offset below is then taken from stream 0, not from the warp's first stream)
// The warp plays both roles in turn (role A, warp barrier, role B). The lanes load their windows from global memory, the lines
// prefetched into L1 one tile ahead.
template <int MAXS, bool MAP = false, class Env>
K3_HD void k3_unit(Env &env, const K3Params &p, int sg, int span, int b, float2 *ring, float2 **sdst, float2 *sF, int2 *sK,
                   const float2 *srrel, const unsigned short *stab, int n_slots) {
    const int lane = env.lane;
    const int nv = p.count, nsw = p.nsw, B = p.block_in, L = p.lut_len;
    const int sbase = MAP ? 0 : p.stream0 + sg * nsw;
    const int lbase = MAP ? sg * nsw : sbase;              // list position of the warp's first stream, checked against stream_end
    int *sS = reinterpret_cast<int *>(sK + 16);
    auto srow = [&](int s) { return MAP ? sS[s] : s; };    // row of warp-local stream s, counted from stream sbase
    const int t_begin = span * p.tiles_per_span;
    const int t_end = (t_begin + p.tiles_per_span < p.n_tiles) ? t_begin + p.tiles_per_span : p.n_tiles;
    if (t_begin >= t_end) return;

    // ---- role B of this lane: row = lane = sB * nv + vB ----
    const int sB = lane / nv, vB = lane - sB * nv;
    const bool rowB = sB < nsw && (lbase + sB) < p.stream_end;
    const int SB = p.v[rowB ? vB : 0].S;
    if (MAP) {
        if (lane < nsw) sS[lane] = lbase + lane < p.stream_end ? p.map[lbase + lane] : p.map[lbase];
        env.sync();
    }
    float2 *outB = p.v[rowB ? vB : 0].out + (size_t)(sbase + srow(rowB ? sB : 0)) * (size_t)p.out_stride + p.v[rowB ? vB : 0].hist +
                   (size_t)b * (size_t)p.v[rowB ? vB : 0].block_out;
    K3Hist H;
#pragma unroll
    for (int i = 0; i < 11; ++i) {
        H.h2[i] = make_float2(0.f, 0.f); H.h3[i] = make_float2(0.f, 0.f);
        H.h4[i] = make_float2(0.f, 0.f); H.h5[i] = make_float2(0.f, 0.f);
    }
    const int SBw = rowB ? SB : 0;
    // per stream of the warp: table index of callback coordinate 0 and "this callback starts the stream" (oscillator.cpp:26-30)
    if (lane < nsw) {
        int kb = 0, zero = 0;
        if (lbase + lane < p.stream_end) {
            const long long blk = k3_ldg(p.blocks_done + sbase + srow(lane)) + b;
            kb = (int)((blk * (long long)B) % L);
            zero = blk == 0;
        }
        sK[lane] = make_int2(kb, zero);
    }
    env.sync();
    const float2 *lutB = p.v[rowB ? vB : 0].lut;
    const int kbB = sK[rowB ? sB : 0].x;
    auto wrapL = [L](int k) { if (k < 0) k += L; if (k >= L) k -= L; return k; };
    // the table entry of this row's (stream, VFO) at the first sample of a tile travels global -> shared one tile ahead
    // (sF is two buffers of 32 entries): no register holds it while the previous tile is being worked on
    k3_async_copy8(sF + lane, lutB + wrapL(kbB + (t_begin - K3_WARM) * K3_TILE));
    int fpar = 0;
    const float2 *in0 = p.in + (size_t)sbase * (size_t)p.in_stride + p.hist_in + (long long)b * B;         // sample 0 of stream sbase
    int n_str = 0;
    for (int s = 0; s < nsw && lbase + s < p.stream_end; ++s) n_str++;
    const float2 *in_pf = in0 + K3_TILE - 16 + 16 * lane;                                                  // this lane's line of the next tile
    const float2 *in_ln = in0 + 4 * lane;                                                                  // this lane's chunk of a tile
    // Output copy, common case (at most 32 sixteen-byte chunks per stream and tile): this lane's chunk is the same for every
    // tile and stream, so its source offset and destination are kept in registers instead of being looked up per tile.
    const bool cp_fast = n_slots <= 32;
    int cp_src = 0, cp_shift = 0;
    float2 *cp_dst = nullptr;
    if (cp_fast && lane < n_slots) {
        const unsigned e = stab[lane];
        const int v = (int)(e >> 8), ch = (int)(e & 0xffu);
        cp_src = v * K3_ROW + 2 * ch;
        cp_shift = p.v[v].S - 1;
        cp_dst = p.v[v].out + (size_t)sbase * (size_t)p.out_stride + p.v[v].hist + (size_t)b * (size_t)p.v[v].block_out + 2 * ch;
    }

    for (int t = t_begin - K3_WARM; t < t_end; ++t) {
        const int c0 = t * K3_TILE;                          // callback coordinate of the tile's first sample (may be negative)
        const float2 *sFt = sF + 32 * fpar;                  // this tile's anchors
        k3_async_wait();
        env.sync();
        fpar ^= 1;
        k3_async_copy8(sF + 32 * fpar + lane, lutB + wrapL(kbB + c0 + K3_TILE));
        // The coming tile's lines into L1 (10 x 128 bytes cover 128 + 14 samples). Measured and not kept (profiles/r02_experiments.md
        // section 1): a request per 32-byte sector, real "touch" loads instead of the prefetch instruction, the first stream's loads
        // hoisted above the barrier, staged input -- none of them moves the kernel's time.
        if (t + 1 < t_end && lane < 10) {
            const float2 *pf = in_pf + c0;
            if (MAP) {
                for (int s = 0; s < n_str; ++s) k3_prefetch_l1(pf + (size_t)sS[s] * (size_t)p.in_stride);
            } else {
                for (int s = 0; s < n_str; ++s, pf += p.in_stride) k3_prefetch_l1(pf);
            }
        }
        // =============================== role A ===============================
        for (int s0 = 0; s0 < nsw; s0 += 2) {
            const int strA = lbase + s0, strB = lbase + s0 + 1;
            const bool hasA = strA < p.stream_end, hasB = (s0 + 1 < nsw) && strB < p.stream_end;
            const int2 baseA = sK[s0], baseB = sK[hasB ? s0 + 1 : s0];
            const int kaA = wrapL(baseA.x + c0), kaB = wrapL(baseB.x + c0);      // table index of sample c0
            const bool fastA = c0 != 0 && kaA >= K3_LUT_STEADY + 16 && kaA + K3_TILE + 8 <= L;
            const bool fastB = c0 != 0 && kaB >= K3_LUT_STEADY + 16 && kaB + K3_TILE + 8 <= L;
            // sample c0 + 4l of the two streams
            const float2 *inA = in_ln + (size_t)srow(s0) * (size_t)p.in_stride + c0;
            const float2 *inB = in_ln + (size_t)srow(hasB ? s0 + 1 : s0) * (size_t)p.in_stride + c0;
            if (env.all(fastA && fastB)) {              // a vote: the compiler then knows the branch (and the VFO loop in it) is warp-uniform
                // ---- sums and differences, once for all VFOs ----
                // x[i] = sample c0 + 4l - 10 + i; outputs m' = 0, 1 have centres i = 5, 7
                float2 cen[2][2], sm[2][2][3], df[2][2][3];          // [stream][output][d]
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    float2 x[14];
                    const float4 *xp = reinterpret_cast<const float4 *>((q ? inB : inA) - 10);
                    const bool has = q ? hasB : hasA;
#pragma unroll
                    for (int i = 0; i < 7; ++i) {
                        const float4 v = has ? k3_ldg(xp + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                        x[2 * i] = make_float2(v.x, v.y);
                        x[2 * i + 1] = make_float2(v.z, v.w);
                    }
#pragma unroll
                    for (int m = 0; m < 2; ++m) {
                        const int ic = 5 + 2 * m;
                        cen[q][m] = x[ic];
#pragma unroll
                        for (int d = 0; d < 3; ++d) {
                            const int dd = 2 * d + 1;
                            sm[q][m][d] = k3_add(x[ic + dd], x[ic - dd]);
                            const float2 tt = k3_sub(x[ic + dd], x[ic - dd]);
                            df[q][m][d] = make_float2(tt.y, tt.x);          // swapped: (-b, b) * (t.y, t.x) = j b t
                        }
                    }
                }
                const bool sameK = env.all(kaA == kaB);
                // software pipeline: the rotation-table pair and the anchors of VFO v+1 are fetched while VFO v is computed
                float4 rr_n = *reinterpret_cast<const float4 *>(srrel + 2 * lane);
                float2 FA_n = sFt[s0 * nv], FB_n = sFt[(hasB ? s0 + 1 : s0) * nv];
#pragma unroll 4
                for (int v = 0; v < nv; ++v) {
                    const float4 rr = rr_n;
                    const float2 FA = FA_n, FB = FB_n;
                    if (v + 1 < nv) {
                        rr_n = *reinterpret_cast<const float4 *>(srrel + (v + 1) * K3_OUT1 + 2 * lane);
                        FA_n = sFt[s0 * nv + v + 1];
                        FB_n = sFt[(hasB ? s0 + 1 : s0) * nv + v + 1];
                    }
                    const float2 a1 = p.v[v].A[0], a3 = p.v[v].A[1], a5 = p.v[v].A[2];
                    const float2 b1 = p.v[v].Bc[0], b3 = p.v[v].Bc[1], b5 = p.v[v].Bc[2];
                    float2 G[2][2];                                      // [stream][output]
                    G[0][0] = k3_cmul(FA, make_float2(rr.x, rr.y));
                    G[0][1] = k3_cmul(FA, make_float2(rr.z, rr.w));
                    G[1][0] = G[0][0]; G[1][1] = G[0][1];
                    if (!sameK) { G[1][0] = k3_cmul(FB, make_float2(rr.x, rr.y)); G[1][1] = k3_cmul(FB, make_float2(rr.z, rr.w)); }
                    // the four outputs (2 streams x 2) advance together, tap by tap: four independent FFMA2 chains
                    float2 acc[2][2];
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int m = 0; m < 2; ++m) acc[q][m] = k3_fma(a1, sm[q][m][0], cen[q][m]);
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int m = 0; m < 2; ++m) acc[q][m] = k3_fma(b1, df[q][m][0], acc[q][m]);
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int m = 0; m < 2; ++m) acc[q][m] = k3_fma(a3, sm[q][m][1], acc[q][m]);
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int m = 0; m < 2; ++m) acc[q][m] = k3_fma(b3, df[q][m][1], acc[q][m]);
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int m = 0; m < 2; ++m) acc[q][m] = k3_fma(a5, sm[q][m][2], acc[q][m]);
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int m = 0; m < 2; ++m) acc[q][m] = k3_fma(b5, df[q][m][2], acc[q][m]);
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const float2 o0 = k3_cmul(G[q][0], acc[q][0]), o1 = k3_cmul(G[q][1], acc[q][1]);
                        if (q ? hasB : hasA)
                            *reinterpret_cast<float4 *>(ring + ((s0 + q) * nv + v) * K3_ROW + 2 * lane) = make_float4(o0.x, o0.y, o1.x, o1.y);
                    }
                }
            } else {
                // ---- exact path: every rotation from the Oscillator table (start-up, wrap, stream sample 0, callback head) ----
#pragma unroll 1
                for (int q = 0; q < 2; ++q) {
                    if (!(q ? hasB : hasA)) continue;
                    const int k0 = (q ? kaB : kaA) + 4 * lane;               // table index of sample c0 + 4l
                    const bool zero = (q ? baseB.y : baseA.y) != 0;          // this callback starts the stream
                    const float4 *xp = reinterpret_cast<const float4 *>((q ? inB : inA) - 12);
                    float2 xe[16];                                           // xe[i] = sample c0 + 4l - 12 + i
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 v = k3_ldg(xp + i);
                        xe[2 * i] = make_float2(v.x, v.y);
                        xe[2 * i + 1] = make_float2(v.z, v.w);
                    }
                    const bool head = c0 == 0;
#pragma unroll 1
                    for (int v = 0; v < nv; ++v) {
                        const float2 *lut = p.v[v].lut;
                        float2 u[13];
#pragma unroll
                        for (int i = 0; i < 13; ++i) {
                            const int c = c0 + 4 * lane - 10 + i;             // window slot coordinate
                            const int sh = (head && c < 0) ? 1 : 0;           // a slot at a negative coordinate holds sample c - 1
                            int k = wrapL(k0 - 10 + i - sh);
                            if (zero && c - sh == 0) k = L - 1;               // stream sample 0 uses the last entry (oscillator.cpp:26-30)
                            u[i] = k3_cmul(k3_ldg(lut + k), sh ? xe[1 + i] : xe[2 + i]);
                        }
                        const float sc = 1.0f / (float)(1 << p.v[v].S);
                        float2 o0 = k3_hb(u[0], u[2], u[4], u[5], u[6], u[8], u[10]);
                        float2 o1 = k3_hb(u[2], u[4], u[6], u[7], u[8], u[10], u[12]);
                        o0 = make_float2(o0.x * sc, o0.y * sc);
                        o1 = make_float2(o1.x * sc, o1.y * sc);
                        *reinterpret_cast<float4 *>(ring + ((s0 + q) * nv + v) * K3_ROW + 2 * lane) = make_float4(o0.x, o0.y, o1.x, o1.y);
                    }
                }
            }
        }
        env.sync();
        // =============================== role B ===============================
        // lanes without a row store nothing and read the (read-only, >= 64 entries) rotation table instead of somebody's row: a row is
        // rewritten in place by its owner while it is read, and a second reader would be a data race (compute-sanitizer racecheck)
        const float2 *myrow = rowB ? ring + lane * K3_ROW : srrel;
        if (c0 == 0) {
            k3_head_shift(H.h2);
            if (MAXS > 2) k3_head_shift(H.h3);
            if (MAXS > 3) k3_head_shift(H.h4);
            if (MAXS > 4) k3_head_shift(H.h5);
        }
#pragma unroll
        for (int sub = 0; sub < K3_OUT1 / 16; ++sub) {
            const float4 *rp = reinterpret_cast<const float4 *>(myrow + 16 * sub);
            float2 *wr = ring + (rowB ? lane : 0) * K3_ROW;  // outputs go to the front of the row (always behind the read position)
            if (MAXS >= 2) {
                // stage 2 in two halves of 8 inputs: only half of the 16 first-stage samples is in registers at any time
                float2 o2[8];
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    float2 in[8], oh[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 v = rp[4 * hf + i];
                        in[2 * i] = make_float2(v.x, v.y);
                        in[2 * i + 1] = make_float2(v.z, v.w);
                    }
                    k3_stage<8>(H.h2, in, oh);
#pragma unroll
                    for (int r = 0; r < 4; ++r) o2[4 * hf + r] = oh[r];
                }
                if (SBw == 2) {
#pragma unroll
                    for (int r = 0; r < 4; ++r)
                        *reinterpret_cast<float4 *>(wr + 8 * sub + 2 * r) = make_float4(o2[2 * r].x, o2[2 * r].y, o2[2 * r + 1].x, o2[2 * r + 1].y);
                }
                if (MAXS >= 3) {
                    float2 o3[4];
                    k3_stage<8>(H.h3, o2, o3);
                    if (SBw == 3) {
#pragma unroll
                        for (int r = 0; r < 2; ++r)
                            *reinterpret_cast<float4 *>(wr + 4 * sub + 2 * r) = make_float4(o3[2 * r].x, o3[2 * r].y, o3[2 * r + 1].x, o3[2 * r + 1].y);
                    }
                    if (MAXS >= 4) {
                        float2 o4[2];
                        k3_stage<4>(H.h4, o3, o4);
                        if (SBw == 4) *reinterpret_cast<float4 *>(wr + 2 * sub) = make_float4(o4[0].x, o4[0].y, o4[1].x, o4[1].y);
                        if (MAXS >= 5) {
                            float2 o5[1];
                            k3_stage<2>(H.h5, o4, o5);
                            if (SBw == 5) wr[sub] = o5[0];
                        }
                    }
                }
            }
            // S == 1: the first-stage outputs are the result and already sit where the copy expects them
        }
        if (t >= t_begin) {
            if (cp_fast) {
                env.sync();
                if (lane < n_slots) {
                    const long long adv = ((long long)t * K3_OUT1) >> cp_shift;      // out1 index 64 t -> index of the VFO's own output
                    for (int s = 0; s < nsw && lbase + s < p.stream_end; ++s) {
                        const float4 v = *reinterpret_cast<const float4 *>(ring + s * nv * K3_ROW + cp_src);
                        k3_store_global16(cp_dst + (size_t)srow(s) * (size_t)p.out_stride + adv, v);
                    }
                }
            } else {
                // where this row's outputs of the tile go: out1 index 64 t -> index (64 t) >> (S - 1) of the VFO's callback record
                sdst[lane] = outB + (((long long)t * K3_OUT1) >> (SB - 1));
                env.sync();
                // cooperative, coalesced copy: slot -> (VFO, 16-byte chunk); chunks of a row are consecutive slots
                // Four slots per lane and trip, in three phases (slot table, then chunk + destination, then the stores): the chain
                // slot -> row -> chunk -> store is three dependent shared loads long, and with one slot per trip it was a fifth of the
                // 2-stage kernel's time (profiles/r02_experiments.md section 1). The stores are st.global: a generic store would keep the
                // compiler from moving the next shared loads above it.
                for (int s = 0; s < nsw; ++s) {
                    if (lbase + s >= p.stream_end) break;
                    for (int slot0 = lane; slot0 < n_slots; slot0 += 128) {
                        int e[4];
                        float4 v[4];
                        float2 *d[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) e[u] = slot0 + 32 * u < n_slots ? (int)stab[slot0 + 32 * u] : -1;
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int r = s * nv + (e[u] >= 0 ? (e[u] >> 8) : 0), ch = e[u] >= 0 ? (e[u] & 0xff) : 0;
                            v[u] = *reinterpret_cast<const float4 *>(ring + r * K3_ROW + 2 * ch);
                            d[u] = sdst[r] + 2 * ch;
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (e[u] >= 0) k3_store_global16(d[u], v[u]);
                    }
                }
            }
        }
        env.sync();
    }
}

#ifdef __CUDACC__
struct K3DevEnv {
    int lane;
    __device__ __forceinline__ void sync() { __syncwarp(); }
    __device__ __forceinline__ bool all(bool v) { return __all_sync(0xffffffffu, v) != 0; }
};

constexpr int K3_WARPS = 2;                                 // default warps per CTA; the kernel works with any CTA size (independent warps that
                                                            // only share the read-only tables)

// grid: x = ceil(stream groups / warps per CTA), y = spans, z = callbacks. MAP: the stream groups are groups of consecutive entries
// of p.map (stream-list calls)
// Register cap: 168 for 2 and 3 stages (three warps per scheduler = 12 per SM). At 168 the 5-stage cascade spills a history array; at 200
// it holds two warps per scheduler = 8 per SM (the register file is per scheduler: 16384 registers), without spills.
template <int MAXS, bool MAP = false>
__global__ void __maxnreg__(MAXS == 5 ? 200 : 168) k2a_v3(const __grid_constant__ K3Params p) {
    extern __shared__ __align__(16) unsigned char k3_smem[];
    float2 *srrel = reinterpret_cast<float2 *>(k3_smem);
    unsigned short *stab = reinterpret_cast<unsigned short *>(srrel + p.count * K3_OUT1);
    unsigned char *wbase = reinterpret_cast<unsigned char *>(stab + K3_MAX_SLOTS);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int e = threadIdx.x; e < p.count * K3_OUT1; e += blockDim.x) srrel[e] = p.rrel[e];
    // slot table: VFO v contributes 32 >> (S - 1) chunks of 16 bytes per tile
    int n_slots = 0;
    for (int v = 0; v < p.count; ++v) {
        const int n = 32 >> (p.v[v].S - 1);
        for (int c = threadIdx.x; c < n; c += blockDim.x) stab[n_slots + c] = (unsigned short)((v << 8) | c);
        n_slots += n;
    }
    __syncthreads();
    const int rows = p.nsw * p.count;
    float2 *ring = reinterpret_cast<float2 *>(wbase + (size_t)warp * k3_warp_smem_bytes(rows));
    float2 **sdst = reinterpret_cast<float2 **>(ring + rows * K3_ROW);
    float2 *sF = reinterpret_cast<float2 *>(sdst + 32);
    int2 *sK = reinterpret_cast<int2 *>(sF + 64);
    const int sg = blockIdx.x * (int)(blockDim.x >> 5) + warp;
    if ((MAP ? 0 : p.stream0) + sg * p.nsw >= p.stream_end) return;
    K3DevEnv env{lane};
    k3_unit<MAXS, MAP>(env, p, sg, (int)blockIdx.y, p.b0 + (int)blockIdx.z, ring, sdst, sF, sK, srrel, stab, n_slots);
}
#endif


}  // namespace sdrb
