// CPU execution of k2a_v3's warp body (kernels_v3.cuh: k3_unit is __host__ __device__): 32 host threads
// play the lanes of one warp, a std::barrier plays __syncwarp. The result is compared with a
// straightforward restatement of vfo::process's front (vfo.cpp:237-251): Oscillator table mix, then S
// HalfBandDecimator stages with FIRQueueBackToFront's shifted history (dsp.cpp:163-173), callback by
// callback. Built and run by tests/test_k3_sim.py (nvcc host compile; no GPU involved).
//
// k3_sim fs B n_streams nsw n_spans n_vfo [start0,start1,..]: the optional 7th argument gives each stream's callback count
// at the first call (default 0: every stream starts at sample 0). Checked per VFO: rel-L2 <= 2e-6 and worst |d| <= 9e-6 x
// the RMS of the reference output.
#include <barrier>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "../../sdrreceiver_b200/csrc/kernels_v3.cuh"
#include "../../sdrreceiver_b200/csrc/plan.hpp"

using namespace sdrb;

struct HostEnv {
    int lane;
    std::barrier<> *bar;
    void sync() { bar->arrive_and_wait(); }
    bool all(bool v) { return v; }                 // every lane evaluates the same warp-uniform condition
};

// ---- reference: one sub VFO front end over n_cb callbacks of B samples, state carried across ----
struct RefVfo {
    std::vector<cf32> lut;
    int S;
    long long n;                                // table position of the next sample: Oscillator::tick count mod L
    bool fresh;                                 // the next sample is stream sample 0 (oscillator.cpp:26-30)
    std::vector<std::vector<float2>> hist;      // per stage: 11 samples
    // a stream that has consumed `start` callbacks of B samples; its filter histories are those of all-zero input
    RefVfo(double fs, double f, int S_, long long start, int B)
        : lut(nco_table(fs, f)), S(S_), n((long long)((unsigned __int128)start * (unsigned)B % lut.size())), fresh(start == 0),
          hist((size_t)S_, std::vector<float2>(11, make_float2(0, 0))) {}
    void process(const float2 *x, int B, std::vector<float2> &out) {
        const int L = (int)lut.size();
        std::vector<float2> cur((size_t)B);
        for (int i = 0; i < B; ++i) {
            const long long a = (n + i) % L;
            const cf32 q = (fresh && i == 0) ? lut[(size_t)(L - 1)] : lut[(size_t)a];
            const float ac = q.re * x[i].x, bd = q.im * x[i].y, ad = q.re * x[i].y, bc = q.im * x[i].x;
            cur[(size_t)i] = make_float2(ac - bd, ad + bc);
        }
        n = (n + B) % L;
        fresh = false;
        int len = B;
        for (int s = 0; s < S; ++s) {
            std::vector<float2> q((size_t)(11 + len));
            for (int i = 0; i < 11; ++i) q[(size_t)i] = hist[(size_t)s][(size_t)i];
            for (int i = 0; i < len; ++i) q[(size_t)(11 + i)] = cur[(size_t)i];
            std::vector<float2> y((size_t)(len / 2));
            for (int i = 0; i < len; i += 2) {
                const int t = i + 1;
                auto tap = [&](int k) { return q[(size_t)(t + k)]; };
                float2 r;
                r.x = HB_P0 * (tap(0).x + tap(10).x) + HB_P2 * (tap(2).x + tap(8).x) + HB_P4 * (tap(4).x + tap(6).x) + HB_P5 * tap(5).x;
                r.y = HB_P0 * (tap(0).y + tap(10).y) + HB_P2 * (tap(2).y + tap(8).y) + HB_P4 * (tap(4).y + tap(6).y) + HB_P5 * tap(5).y;
                y[(size_t)(i / 2)] = r;
            }
            for (int i = 0; i < 11; ++i) hist[(size_t)s][(size_t)i] = q[(size_t)(len - 1 + i)];     // NOT len + i: dsp.cpp:169
            cur.swap(y);
            len /= 2;
        }
        out.insert(out.end(), cur.begin(), cur.begin() + len);
    }
};

static unsigned long long rng = 0x9E3779B97F4A7C15ull;
static float frand() {
    rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17;
    return (float)((double)(rng >> 11) / 9007199254740992.0 * 2.0 - 1.0);
}

template <int MAXS>
static void run_units(const K3Params &p, int n_cb, int n_spans) {
    const int n_groups = (p.stream_end - p.stream0 + p.nsw - 1) / p.nsw;
    // slot table and rrel as the kernel builds them
    std::vector<unsigned short> stab((size_t)K3_MAX_SLOTS);
    int n_slots = 0;
    for (int v = 0; v < p.count; ++v) {
        const int n = 32 >> (p.v[v].S - 1);
        for (int c = 0; c < n; ++c) stab[(size_t)(n_slots + c)] = (unsigned short)((v << 8) | c);
        n_slots += n;
    }
    for (int cb = 0; cb < n_cb; ++cb)
        for (int span = 0; span < n_spans; ++span)
            for (int sg = 0; sg < n_groups; ++sg) {
                std::vector<float2> ring((size_t)p.nsw * p.count * K3_ROW, make_float2(NAN, NAN));
                std::vector<float2 *> sdst(32, nullptr);
                std::vector<float2> sF(64, make_float2(NAN, NAN));
                std::vector<int2> sK(32, make_int2(0, 0));
                std::barrier<> bar(32);
                std::vector<std::thread> th;
                for (int lane = 0; lane < 32; ++lane)
                    th.emplace_back([&, lane]() {
                        HostEnv env{lane, &bar};
                        k3_unit<MAXS>(env, p, sg, span, p.b0 + cb, ring.data(), sdst.data(), sF.data(), sK.data(), p.rrel, stab.data(), n_slots);
                    });
                for (auto &t : th) t.join();
            }
}

int main(int argc, char **argv) {
    // geometry: parent rate fs, callbacks of B samples, table wrap every fs/B callbacks
    const int fs = argc > 1 ? atoi(argv[1]) : 30720, B = argc > 2 ? atoi(argv[2]) : 7680;
    const int n_streams = argc > 3 ? atoi(argv[3]) : 3, nsw = argc > 4 ? atoi(argv[4]) : 2;
    const int n_spans = argc > 5 ? atoi(argv[5]) : 4;
    const int calls = 3, cb_per_call = 2, HIST_IN = 512;
    const int S_of[16] = {5, 4, 3, 2, 1, 5, 5, 5, 2, 3, 4, 5, 1, 2, 5, 5};
    const double f_of[16] = {1234.0, -7321.0, 5000.5, -11000.0, 333.0, 9876.0, -2500.0, 14000.0, -13999.0, 0.0, 77.7, -4200.0, 6100.0, -900.0, 12000.0, -12500.0};
    const int nv = argc > 6 ? atoi(argv[6]) : 6;
    if (nsw * nv > 32) { printf("nsw*nv > 32\n"); return 2; }
    std::vector<long long> blocks_done((size_t)n_streams, 0);
    if (argc > 7) {
        const char *c = argv[7];
        for (int s = 0; s < n_streams; ++s) {
            char *e;
            blocks_done[(size_t)s] = strtoll(c, &e, 10);
            if (e == c || blocks_done[(size_t)s] < 0) { printf("bad start counts '%s'\n", argv[7]); return 2; }
            c = *e == ',' ? e + 1 : e;
        }
        if (*c) { printf("more start counts than streams in '%s'\n", argv[7]); return 2; }
    }

    const size_t in_stride = (size_t)HIST_IN + (size_t)cb_per_call * B;
    std::vector<float2> in((size_t)n_streams * in_stride, make_float2(0, 0));
    // outputs: per VFO a buffer [stream][hist + cb_per_call*block_out], hist = 64
    const int OHIST = 64;
    std::vector<std::vector<float2>> zbuf((size_t)nv);
    std::vector<float2> rrel((size_t)nv * K3_OUT1);
    std::vector<RefVfo> refs;
    K3Params p;
    memset(&p, 0, sizeof(p));
    std::vector<std::vector<cf32>> luts;
    size_t out_stride = 0;
    for (int v = 0; v < nv; ++v) out_stride = std::max(out_stride, (size_t)OHIST + (size_t)cb_per_call * (size_t)(B >> S_of[v]));
    for (int v = 0; v < nv; ++v) {
        luts.push_back(nco_table((double)fs, f_of[v]));
        zbuf[(size_t)v].assign((size_t)n_streams * out_stride, make_float2(NAN, NAN));
    }
    for (int v = 0; v < nv; ++v) {
        K3Vfo &V = p.v[v];
        k3_fill_vfo((double)fs, f_of[v], S_of[v], V, &rrel[(size_t)v * K3_OUT1]);
        V.lut = reinterpret_cast<const float2 *>(luts[(size_t)v].data());
        V.out = zbuf[(size_t)v].data();
        V.block_out = B >> S_of[v]; V.hist = OHIST;
    }
    p.rrel = rrel.data(); p.in = in.data(); p.blocks_done = blocks_done.data();
    p.in_stride = (long long)in_stride; p.out_stride = (long long)out_stride;
    p.hist_in = HIST_IN; p.count = nv; p.lut_len = fs; p.block_in = B; p.n_tiles = B / K3_TILE;
    p.tiles_per_span = (p.n_tiles + n_spans - 1) / n_spans;
    p.stream0 = 0; p.stream_end = n_streams; p.b0 = 0; p.nsw = nsw;

    std::vector<std::vector<RefVfo>> ref((size_t)n_streams);
    for (int s = 0; s < n_streams; ++s)
        for (int v = 0; v < nv; ++v) ref[(size_t)s].emplace_back((double)fs, f_of[v], S_of[v], blocks_done[(size_t)s], B);
    std::vector<std::vector<std::vector<float2>>> ref_out((size_t)n_streams, std::vector<std::vector<float2>>((size_t)nv));
    std::vector<std::vector<std::vector<float2>>> got((size_t)n_streams, std::vector<std::vector<float2>>((size_t)nv));

    for (int call = 0; call < calls; ++call) {
        for (int s = 0; s < n_streams; ++s) {
            float2 *body = in.data() + (size_t)s * in_stride + HIST_IN;
            for (int i = 0; i < cb_per_call * B; ++i) body[i] = make_float2(20.f * frand(), 20.f * frand());
            for (int cb = 0; cb < cb_per_call; ++cb)
                for (int v = 0; v < nv; ++v) ref[(size_t)s][(size_t)v].process(body + (size_t)cb * B, B, ref_out[(size_t)s][(size_t)v]);
        }
        run_units<5>(p, cb_per_call, n_spans);
        for (int s = 0; s < n_streams; ++s) {
            for (int v = 0; v < nv; ++v) {
                const float2 *z = zbuf[(size_t)v].data() + (size_t)s * out_stride + OHIST;
                got[(size_t)s][(size_t)v].insert(got[(size_t)s][(size_t)v].end(), z, z + (size_t)cb_per_call * (size_t)(B >> S_of[v]));
            }
            // carry: tail of the input becomes the history of the next call
            float2 *row = in.data() + (size_t)s * in_stride;
            memmove(row, row + (size_t)cb_per_call * B, (size_t)HIST_IN * sizeof(float2));
            blocks_done[(size_t)s] += cb_per_call;
        }
    }
    int bad = 0;
    for (int s = 0; s < n_streams; ++s)
        for (int v = 0; v < nv; ++v) {
            const auto &a = got[(size_t)s][(size_t)v];
            const auto &r = ref_out[(size_t)s][(size_t)v];
            if (a.size() != r.size()) { printf("size mismatch s%d v%d: %zu vs %zu\n", s, v, a.size(), r.size()); bad++; continue; }
            double num = 0, den = 0, worst = 0; size_t wi = 0;
            for (size_t i = 0; i < a.size(); ++i) {
                const double dx = (double)a[i].x - r[i].x, dy = (double)a[i].y - r[i].y;
                const double e = dx * dx + dy * dy;
                if (!(e <= worst)) { worst = e; wi = i; }
                num += e; den += (double)r[i].x * r[i].x + (double)r[i].y * r[i].y;
            }
            const double rel = sqrt(num / den), rms = sqrt(den / (double)a.size()), peak = sqrt(worst) / rms;
            printf("stream %d vfo %d (S=%d): rel-L2 %.3e  worst |d| %.3e = %.3e x RMS at %zu of %zu\n", s, v, S_of[v], rel,
                   sqrt(worst), peak, wi, a.size());
            if (!(rel <= 2e-6) || !(peak <= 9e-6)) bad++;
        }
    printf(bad ? "FAIL\n" : "OK\n");
    return bad ? 1 : 0;
}
