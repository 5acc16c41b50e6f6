// Per-class device primitives behind the C++ facades (Oscillator/vfo mix loop,
// HalfBandDecimator, FIR, FIRHilbert+DelayThing, FFTWrapper). One CTA row per channel;
// state is explicit (history arrays), exactly what the reference objects hold.
#pragma once
#include <cuda_runtime.h>
#include "kernels.cuh"

namespace sdrb {

// vfo::process mix loop (vfo.cpp:237-245) with Oscillator::tick indexing (oscillator.cpp:39-50)
__global__ void __launch_bounds__(256) prim_nco_mix(const float2 *__restrict__ table, int L, long long n0,
                                                     const float2 *__restrict__ in, float2 *__restrict__ out, int n) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const long long g = n0 + i;
    const int idx = (g == 0) ? L - 1 : (int)(g % L);
    const size_t at = (size_t)blockIdx.y * n + i;
    out[at] = cmul(__ldg(table + idx), in[at]);
}

// HalfBandDecimator::decimate, 11 taps (halfbanddecimator.cpp:43-72; dsp.cpp:96-148):
// queue = [hist(11) | block]; output m reads queue[2m+1 .. 2m+11].
__global__ void __launch_bounds__(256) prim_halfband11(const float2 *__restrict__ in, float2 *__restrict__ out,
                                                        const float2 *__restrict__ hist, int n) {
    const int m = blockIdx.x * 256 + threadIdx.x;
    if (m >= n / 2) return;
    const float2 *x = in + (size_t)blockIdx.y * n;
    const float2 *h = hist + (size_t)blockIdx.y * 11;
    auto q = [&](int j) -> float2 { return j < 11 ? h[j] : x[j - 11]; };
    const int t = 2 * m + 1;
    const float2 w0 = q(t), w2 = q(t + 2), w4 = q(t + 4), w5 = q(t + 5), w6 = q(t + 6), w8 = q(t + 8), w10 = q(t + 10);
    float2 y;
    y.x = HB_P0 * (w0.x + w10.x) + HB_P2 * (w2.x + w8.x) + HB_P4 * (w4.x + w6.x) + HB_P5 * w5.x;
    y.y = HB_P0 * (w0.y + w10.y) + HB_P2 * (w2.y + w8.y) + HB_P4 * (w4.y + w6.y) + HB_P5 * w5.y;
    out[(size_t)blockIdx.y * (n / 2) + m] = y;
}

// FIRQueueBackToFront (dsp.cpp:163-173): new head = queue[B-1 .. B+9] = block[B-12 .. B-2].
__global__ void prim_halfband11_carry(const float2 *__restrict__ in, float2 *__restrict__ hist, int n) {
    if (threadIdx.x < 11) hist[(size_t)blockIdx.x * 11 + threadIdx.x] = in[(size_t)blockIdx.x * n + (n - 12 + threadIdx.x)];
}

// HalfBandDecimator with the 23- and 51-tap tables (halfbanddecimator.h:28-63; dsp.cpp:106-136). vfo.cpp
// only ever builds the 11-tap one (vfo.cpp:130), these back the class facade. Same queue rule as the
// 11-tap stage for any length N: window slot t = 2m+1 in [hist(N) | block], history carried with the
// off-by-one of FIRQueueBackToFront. Other lengths (15, 21 have tables but no `case`): the reference's
// switch falls through and every output is 0 -- reproduced by NZ = 0.
__constant__ float c_hb23[7] = {-0.00014987651418332164f, 0.0014748633283609852f, -0.0074416944990005314f, 0.026163522731980929f,
                                -0.077593699116544707f, 0.30754683719791986f, 0.5f};
__constant__ float c_hb51[14] = {0.0010175926971811044f, -0.0013058886799502411f, 0.0020730260200910026f, -0.0034255790572079265f,
                                 0.005490505092950141f,  -0.008434405740804745f,  0.012502602797600649f,  -0.01810260996706492f,
                                 0.026000146160530365f,  -0.037851497102093665f,  0.05801218485928863f,   -0.1025751653146947f,
                                 0.31684426465520726f,   0.499509647157934f};

// coef: the even-indexed points 0, 2, .., N-3 followed by the centre point; NZ = (N+1)/4 + 1 of them, or 0
__global__ void __launch_bounds__(256) prim_halfband_n(const float2 *__restrict__ in, float2 *__restrict__ out,
                                                        const float2 *__restrict__ hist, int n, int N, const float *coef, int NZ) {
    const int m = blockIdx.x * 256 + threadIdx.x;
    if (m >= n / 2) return;
    const float2 *x = in + (size_t)blockIdx.y * n;
    const float2 *h = hist + (size_t)blockIdx.y * N;
    auto q = [&](int j) -> float2 { return j < N ? h[j] : x[j - N]; };
    const int t = 2 * m + 1;
    float2 y = make_float2(0.f, 0.f);
    for (int k = 0; k + 1 < NZ; ++k) {                       // points[2k]*(q[t+2k] + q[t+N-1-2k]), summed in the reference's order
        const float2 a = q(t + 2 * k), b = q(t + N - 1 - 2 * k);
        y.x = __fadd_rn(y.x, __fmul_rn(coef[k], __fadd_rn(a.x, b.x)));
        y.y = __fadd_rn(y.y, __fmul_rn(coef[k], __fadd_rn(a.y, b.y)));
    }
    if (NZ > 0) {
        const float2 c = q(t + (N - 1) / 2);
        y.x = __fadd_rn(y.x, __fmul_rn(coef[NZ - 1], c.x));
        y.y = __fadd_rn(y.y, __fmul_rn(coef[NZ - 1], c.y));
    }
    out[(size_t)blockIdx.y * (n / 2) + m] = y;
}

// FIRQueueBackToFront for any N and any even block length: new head = q[B-1 .. B+N-2] of q = [hist | block]
__global__ void prim_halfband_n_carry(const float2 *__restrict__ in, float2 *__restrict__ hist, int n, int N) {
    extern __shared__ float2 hstage[];
    const float2 *x = in + (size_t)blockIdx.x * n;
    float2 *h = hist + (size_t)blockIdx.x * N;
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const int c = n - 1 + j;
        hstage[j] = c < N ? h[c] : x[c - N];
    }
    __syncthreads();
    for (int j = threadIdx.x; j < N; j += blockDim.x) h[j] = hstage[j];
}

// FIR::FIRUpdateAndProcess (dsp.cpp:59-71): y[m] = sum_i taps[i] * x[decim*m - N + i]  (newest excluded),
// or with inc = 1 the FIRHilbert form (dsp.cpp:218-231): y[m] = sum_i taps[i] * x[decim*m - N + 1 + i].
__global__ void __launch_bounds__(256) prim_fir(const float *__restrict__ taps, int N, const float *__restrict__ in,
                                                 float *__restrict__ out, const float *__restrict__ hist, int n,
                                                 int decim, int n_out, int inc) {
    const int m = blockIdx.x * 256 + threadIdx.x;
    if (m >= n_out) return;
    const float *x = in + (size_t)blockIdx.y * n;
    const float *h = hist + (size_t)blockIdx.y * N;
    const int base = decim * m - N + inc;
    float acc = 0.f;
    for (int i = 0; i < N; ++i) {
        const int j = base + i;
        acc = fmaf(__ldg(taps + i), j < 0 ? h[N + j] : x[j], acc);
    }
    out[(size_t)blockIdx.y * n_out + m] = acc;
}

// History carry: the last `count` elements (of `width` floats) of [old history | block] become the
// new history; blocks shorter than the history are allowed (per-sample facade calls).
__global__ void prim_tail_carry(const float *__restrict__ in, float *__restrict__ hist, int n, int count, int width) {
    extern __shared__ float stage[];
    const float *x = in + (size_t)blockIdx.x * n * width;
    float *h = hist + (size_t)blockIdx.x * count * width;
    const int total = count * width;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
        const int c = n * width + e;                      // position in [old history | block]
        stage[e] = c < total ? h[c] : x[c - total];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < total; e += blockDim.x) h[e] = stage[e];
}

// usb = DelayThing(62)(re) - FIRHilbert125(im)  (vfo.cpp:316-324; dsp.cpp:218-231)
__global__ void __launch_bounds__(256) prim_usb(const float *__restrict__ pts, const float2 *__restrict__ in,
                                                 float *__restrict__ out, const float2 *__restrict__ hist, int n) {
    __shared__ float sp[125];
    if (threadIdx.x < 125) sp[threadIdx.x] = pts[threadIdx.x];
    __syncthreads();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const float2 *x = in + (size_t)blockIdx.y * n;
    const float2 *h = hist + (size_t)blockIdx.y * 124;
    auto at = [&](int j) -> float2 { return j < 0 ? h[124 + j] : x[j]; };
    float acc = 0.f;
    for (int k = 1; k < 125; k += 2) acc = fmaf(sp[k], at(i - 124 + k).y, acc);   // even points are exactly 0
    out[(size_t)blockIdx.y * n + i] = at(i - 62).x - acc;
}

// Spectrum path: Hann window (mainwindow.cpp:284-288, 416-423) and an 8192-point forward complex
// FFT, unscaled like kiss_fft (kiss_fft.c:339-388). One CTA per transform, whole transform in
// shared memory: bit-reversed load, then four radix-8 passes (three radix-2 stages each, on eight
// registers per group) and one radix-2 pass -- 5 barriers instead of 13 -- with twiddles read from a
// table the host builds like kiss_fft does (exp(-2 pi i k/N) in double, cast to float: kiss_fft.c:357-363)
// and the Hann window from a table built with the reference's own expression (mainwindow.cpp:287).
constexpr int FFT_N = 8192, FFT_LOGN = 13, FFT_THREADS = 512;

struct FftTables {
    const float2 *tw;            // [FFT_N / 2]: exp(-2 pi i m / N)
    const float *hann;           // [FFT_N]
};

__device__ __forceinline__ float2 fft_cmul(float2 a, float2 w) { return make_float2(a.x * w.x - a.y * w.y, a.x * w.y + a.y * w.x); }

// radix-2 stages st, st+1, st+2 on the eight elements base + j * 2^st of a group (decimation in time, natural order out)
__device__ __forceinline__ void fft_radix8_group(float2 *s, const float2 *__restrict__ tw, int st, int g) {
    const int span = 1 << st;
    const int k0 = g & (span - 1);
    const int base = ((g >> st) << (st + 3)) + k0;
    float2 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = s[base + j * span];
    // stage st: pairs (j, j+1), twiddle exponent k0 / 2^st half-turns
    {
        const float2 w = tw[k0 << (FFT_LOGN - 1 - st)];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            const float2 t = fft_cmul(v[j + 1], w);
            v[j + 1] = make_float2(v[j].x - t.x, v[j].y - t.y);
            v[j] = make_float2(v[j].x + t.x, v[j].y + t.y);
        }
    }
    // stage st+1: pairs (j, j+2), k = k0 + (j & 1) * 2^st
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const float2 w = tw[(k0 + q * span) << (FFT_LOGN - 2 - st)];
#pragma unroll
        for (int h = 0; h < 8; h += 4) {
            const int j = h + q;
            const float2 t = fft_cmul(v[j + 2], w);
            v[j + 2] = make_float2(v[j].x - t.x, v[j].y - t.y);
            v[j] = make_float2(v[j].x + t.x, v[j].y + t.y);
        }
    }
    // stage st+2: pairs (j, j+4), k = k0 + j * 2^st
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 w = tw[(k0 + j * span) << (FFT_LOGN - 3 - st)];
        const float2 t = fft_cmul(v[j + 4], w);
        v[j + 4] = make_float2(v[j].x - t.x, v[j].y - t.y);
        v[j] = make_float2(v[j].x + t.x, v[j].y + t.y);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) s[base + j * span] = v[j];
}

// s[] holds the input in bit-reversed order on entry (and a __syncthreads has been passed)
__device__ __forceinline__ void fft8192_stages(float2 *s, const float2 *__restrict__ tw) {
#pragma unroll 1
    for (int st = 0; st < 12; st += 3) {
        for (int g = threadIdx.x; g < FFT_N / 8; g += FFT_THREADS) fft_radix8_group(s, tw, st, g);
        __syncthreads();
    }
    // last stage (half = 4096)
    for (int k = threadIdx.x; k < FFT_N / 2; k += FFT_THREADS) {
        const float2 a = s[k], t = fft_cmul(s[k + FFT_N / 2], tw[k]);
        s[k] = make_float2(a.x + t.x, a.y + t.y);
        s[k + FFT_N / 2] = make_float2(a.x - t.x, a.y - t.y);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(FFT_THREADS) prim_fft8192(const float2 *__restrict__ in, float2 *__restrict__ out, int hann, FftTables T) {
    extern __shared__ float2 s[];
    const float2 *x = in + (size_t)blockIdx.x * FFT_N;
    for (int i = threadIdx.x; i < FFT_N; i += FFT_THREADS) {
        float2 v = x[i];
        if (hann) {
            const float w = T.hann[i];
            v.x *= w; v.y *= w;
        }
        s[__brev((unsigned)i) >> (32 - FFT_LOGN)] = v;
    }
    __syncthreads();
    fft8192_stages(s, T.tw);
    float2 *y = out + (size_t)blockIdx.x * FFT_N;
    for (int i = threadIdx.x; i < FFT_N; i += FFT_THREADS) y[i] = s[i];
}

// MainWindow::fftHandlerSlot (mainwindow.cpp:411-455) for a batch of independent spectrum displays,
// one CTA each. State per display in HBM: inr[N] (the windowed input; entries beyond `len` keep
// their previous content, mainwindow.cpp:418-425) and pwr[N] (double, the 0.95/0.05 dB average).
//   inr[a]  = data[a]*hann[a], a < min(N, len)
//   X       = FFT(inr)                                         (kiss_fft, unscaled)
//   pwr[b]  = pwr[b]*0.95 + 0.05*10*log10(max(1e5*|X[i]|/N, 1)),  b = (i + N/2) mod N
//   smooth[i] = (pwr[i] + ... + pwr[i+4])/5, i < N-10;  stats = {max(pwr) (at least avg+10), avg(pwr)}
// MAP: CTA i feeds display map[i] only (the streams of a stream-list call); the other displays are not touched.
template <bool MAP = false>
__global__ void __launch_bounds__(FFT_THREADS) k_spectrum_feed(const float2 *__restrict__ data, long long data_stride, int len,
                                                               float2 *__restrict__ inr, double *__restrict__ pwr,
                                                               double *__restrict__ smooth, double *__restrict__ stats,
                                                               float2 *__restrict__ fft_out, FftTables T,
                                                               const int *__restrict__ map = nullptr) {
    extern __shared__ float2 s[];
    __shared__ double red_max[FFT_THREADS / 32], red_sum[FFT_THREADS / 32];
    const int d = map_stream<MAP>(map, 0, blockIdx.x);
    const float2 *x = data + (size_t)d * data_stride;
    float2 *keep = inr + (size_t)d * FFT_N;
    double *P = pwr + (size_t)d * FFT_N;
    for (int i = threadIdx.x; i < FFT_N; i += FFT_THREADS) {
        float2 v;
        if (i < len) {
            const float w = T.hann[i];
            v = x[i];
            v.x *= w; v.y *= w;
            keep[i] = v;
        } else {
            v = keep[i];
        }
        s[__brev((unsigned)i) >> (32 - FFT_LOGN)] = v;
    }
    __syncthreads();
    fft8192_stages(s, T.tw);
    double mx = 0.0, sum = 0.0;
    for (int i = threadIdx.x; i < FFT_N; i += FFT_THREADS) {
        const float2 X = s[i];
        if (fft_out) fft_out[(size_t)d * FFT_N + i] = X;
        const int b = (i + FFT_N / 2) & (FFT_N - 1);
        const double val = (double)sqrtf(X.y * X.y + X.x * X.x);
        const double p = P[b] * 0.95 + 0.05 * 10 * log10(fmax(100000.0 * fabs((1.0 / FFT_N) * val), 1.0));
        P[b] = p;
        mx = fmax(mx, p);
        sum += p;
    }
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
    }
    if ((threadIdx.x & 31) == 0) { red_max[threadIdx.x >> 5] = mx; red_sum[threadIdx.x >> 5] = sum; }
    __syncthreads();                                           // also orders the pwr[] stores before the smoothing reads
    for (int i = threadIdx.x; i < FFT_N - 10; i += FFT_THREADS)
        smooth[(size_t)d * (FFT_N - 10) + i] = (P[i + 4] + P[i + 3] + P[i + 2] + P[i + 1] + P[i]) / 5;
    if (threadIdx.x == 0) {
        for (int w = 1; w < FFT_THREADS / 32; ++w) { mx = fmax(mx, red_max[w]); sum += red_sum[w]; }
        const double ave = sum / FFT_N;
        if (mx - ave < 10) mx = ave + 10.0;
        stats[2 * d] = mx;
        stats[2 * d + 1] = ave;
    }
}

}  // namespace sdrb
