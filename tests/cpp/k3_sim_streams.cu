// CPU execution of k2a_v3's stream-list form (kernels_v3.cuh: k3_unit<MAXS, true>): warp-local stream s of stream group g is
// bank stream map[g*nsw + s], so a warp holds whichever streams a call lists, in list order. Every call processes the listed
// streams only; their outputs are compared with the same plain cascade and within the same bounds as k3_sim.cu (rel-L2 <= 2e-6
// and worst |d| <= 9e-6 x RMS per VFO), and the output rows of the streams the list leaves out must stay as they were created
// (NaN). Built and run by tests/test_k3_sim_streams.py (nvcc host compile; no GPU involved).
//
// k3_sim_streams fs B n_streams nsw n_spans n_vfo start0,start1,.. list0,list1,..
//   start: each stream's callback count at the first call; list: the distinct streams every call processes, in this order.

// The reference cascade, the host warp and the input generator are k3_sim.cu's; its own main is renamed out of the way.
#define main k3_sim_plain_main
#include "k3_sim.cu"
#undef main

static bool parse_list(const char *c, std::vector<long long> &out) {
    while (*c) {
        char *e;
        const long long v = strtoll(c, &e, 10);
        if (e == c || v < 0) return false;
        out.push_back(v);
        c = *e == ',' ? e + 1 : e;
    }
    return true;
}

template <int MAXS>
static void run_listed(const K3Params &p, int n_cb, int n_spans) {
    const int n_groups = (p.stream_end + p.nsw - 1) / p.nsw;
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
                        k3_unit<MAXS, true>(env, p, sg, span, p.b0 + cb, ring.data(), sdst.data(), sF.data(), sK.data(), p.rrel,
                                            stab.data(), n_slots);
                    });
                for (auto &t : th) t.join();
            }
}

int main(int argc, char **argv) {
    if (argc != 9) { printf("usage: k3_sim_streams fs B n_streams nsw n_spans n_vfo starts list\n"); return 2; }
    const int fs = atoi(argv[1]), B = atoi(argv[2]), n_streams = atoi(argv[3]), nsw = atoi(argv[4]), n_spans = atoi(argv[5]);
    const int nv = atoi(argv[6]);
    const int calls = 3, cb_per_call = 2, HIST_IN = 512, OHIST = 64;
    const int S_of[16] = {5, 4, 3, 2, 1, 5, 5, 5, 2, 3, 4, 5, 1, 2, 5, 5};
    const double f_of[16] = {1234.0, -7321.0, 5000.5, -11000.0, 333.0, 9876.0, -2500.0, 14000.0, -13999.0, 0.0, 77.7, -4200.0, 6100.0, -900.0, 12000.0, -12500.0};
    if (nsw * nv > 32) { printf("nsw*nv > 32\n"); return 2; }
    std::vector<long long> blocks_done, lst;
    if (!parse_list(argv[7], blocks_done) || (int)blocks_done.size() != n_streams) { printf("bad start counts '%s'\n", argv[7]); return 2; }
    std::vector<char> listed((size_t)n_streams, 0);
    std::vector<int> list;
    if (!parse_list(argv[8], lst) || lst.empty()) { printf("bad stream list '%s'\n", argv[8]); return 2; }
    for (long long s : lst) {
        if (s >= n_streams || listed[(size_t)s]) { printf("bad stream list '%s'\n", argv[8]); return 2; }
        listed[(size_t)s] = 1; list.push_back((int)s);
    }

    const size_t in_stride = (size_t)HIST_IN + (size_t)cb_per_call * B;
    std::vector<float2> in((size_t)n_streams * in_stride, make_float2(0, 0));
    std::vector<std::vector<float2>> zbuf((size_t)nv);
    std::vector<float2> rrel((size_t)nv * K3_OUT1);
    K3Params p;
    memset(&p, 0, sizeof(p));
    std::vector<std::vector<cf32>> luts;
    size_t out_stride = 0;
    for (int v = 0; v < nv; ++v) out_stride = std::max(out_stride, (size_t)OHIST + (size_t)cb_per_call * (size_t)(B >> S_of[v]));
    for (int v = 0; v < nv; ++v) {
        luts.push_back(nco_table((double)fs, f_of[v]));
        zbuf[(size_t)v].assign((size_t)n_streams * out_stride, make_float2(NAN, NAN));
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
    p.stream0 = 0; p.stream_end = (int)list.size(); p.b0 = 0; p.nsw = nsw; p.map = list.data();

    std::vector<std::vector<RefVfo>> ref((size_t)n_streams);
    for (int s = 0; s < n_streams; ++s)
        for (int v = 0; v < nv; ++v) ref[(size_t)s].emplace_back((double)fs, f_of[v], S_of[v], blocks_done[(size_t)s], B);
    std::vector<std::vector<std::vector<float2>>> ref_out((size_t)n_streams, std::vector<std::vector<float2>>((size_t)nv));
    std::vector<std::vector<std::vector<float2>>> got((size_t)n_streams, std::vector<std::vector<float2>>((size_t)nv));

    for (int call = 0; call < calls; ++call) {
        for (int s : list) {
            float2 *body = in.data() + (size_t)s * in_stride + HIST_IN;
            for (int i = 0; i < cb_per_call * B; ++i) body[i] = make_float2(20.f * frand(), 20.f * frand());
            for (int cb = 0; cb < cb_per_call; ++cb)
                for (int v = 0; v < nv; ++v) ref[(size_t)s][(size_t)v].process(body + (size_t)cb * B, B, ref_out[(size_t)s][(size_t)v]);
        }
        run_listed<5>(p, cb_per_call, n_spans);
        for (int s : list) {
            for (int v = 0; v < nv; ++v) {
                const float2 *z = zbuf[(size_t)v].data() + (size_t)s * out_stride + OHIST;
                got[(size_t)s][(size_t)v].insert(got[(size_t)s][(size_t)v].end(), z, z + (size_t)cb_per_call * (size_t)(B >> S_of[v]));
            }
            float2 *row = in.data() + (size_t)s * in_stride;
            memmove(row, row + (size_t)cb_per_call * B, (size_t)HIST_IN * sizeof(float2));
            blocks_done[(size_t)s] += cb_per_call;
        }
    }
    int bad = 0;
    for (int s = 0; s < n_streams; ++s)
        for (int v = 0; v < nv; ++v) {
            if (!listed[(size_t)s]) {
                const float2 *z = zbuf[(size_t)v].data() + (size_t)s * out_stride;
                for (size_t i = 0; i < out_stride; ++i)
                    if (!std::isnan(z[i].x) || !std::isnan(z[i].y)) { printf("unlisted stream %d vfo %d written at %zu\n", s, v, i); bad++; break; }
                continue;
            }
            const auto &a = got[(size_t)s][(size_t)v];
            const auto &r = ref_out[(size_t)s][(size_t)v];
            if (a.size() != r.size()) { printf("size mismatch s%d v%d: %zu vs %zu\n", s, v, a.size(), r.size()); bad++; continue; }
            double num = 0, den = 0, worst = 0;
            for (size_t i = 0; i < a.size(); ++i) {
                const double dx = (double)a[i].x - r[i].x, dy = (double)a[i].y - r[i].y;
                const double e = dx * dx + dy * dy;
                if (!(e <= worst)) worst = e;
                num += e; den += (double)r[i].x * r[i].x + (double)r[i].y * r[i].y;
            }
            const double rel = sqrt(num / den), rms = sqrt(den / (double)a.size()), peak = sqrt(worst) / rms;
            printf("stream %d vfo %d (S=%d): rel-L2 %.3e  worst |d| = %.3e x RMS\n", s, v, S_of[v], rel, peak);
            if (!(rel <= 2e-6) || !(peak <= 9e-6)) bad++;
        }
    printf(bad ? "FAIL\n" : "OK\n");
    return bad ? 1 : 0;
}
