// C ABI of libsdrb200.so (include/sdrb200.h): plan upload, receiver bank, launches.
// Host logic only; the kernels live in kernels.cuh / prims.cuh. No CPU compute path exists
// here: every process_* entry point fails with SDRB_E_CUDA when no device is usable.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "plan.hpp"
#include "kernels.cuh"
#include "kernels_v2.cuh"
#include "kernels_v3.cuh"
#include "prims.cuh"

namespace sdrb {
const char *last_error_cstr();
}
using namespace sdrb;

#define CU_TRY(expr)                                                                           \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(e_));                     \
            return SDRB_E_CUDA;                                                                \
        }                                                                                      \
    } while (0)

// ------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------
struct sdrb_plan {
    HostPlan h;
};

extern "C" int sdrb_plan_from_ini(const char *ini_path, sdrb_plan **out) {
    if (!out) { set_error("sdrb_plan_from_ini: out is NULL"); return SDRB_E_INVALID; }
    *out = nullptr;
    sdrb_plan *p = new (std::nothrow) sdrb_plan();
    if (!p) return SDRB_E_NOMEM;
    const int rc = plan_from_ini(ini_path, p->h);
    if (rc != SDRB_OK) { delete p; return rc; }
    *out = p;
    return SDRB_OK;
}

extern "C" int sdrb_plan_create(const sdrb_plan_desc *desc, sdrb_plan **out) {
    if (!desc || !out) { set_error("sdrb_plan_create: NULL argument"); return SDRB_E_INVALID; }
    *out = nullptr;
    sdrb_plan *p = new (std::nothrow) sdrb_plan();
    if (!p) return SDRB_E_NOMEM;
    const int rc = plan_from_desc(*desc, p->h);
    if (rc != SDRB_OK) { delete p; return rc; }
    *out = p;
    return SDRB_OK;
}

extern "C" void sdrb_plan_destroy(sdrb_plan *plan) { delete plan; }

extern "C" int sdrb_plan_get_info(const sdrb_plan *plan, sdrb_plan_info *info) {
    if (!plan || !info) { set_error("sdrb_plan_get_info: NULL argument"); return SDRB_E_INVALID; }
    const HostPlan &h = plan->h;
    memset(info, 0, sizeof(*info));
    info->sample_rate = h.fs; info->block = h.block; info->bufsplit = h.bufsplit;
    info->correct_dc = h.correct_dc; info->n_main = (int)h.mains.size(); info->n_sub = (int)h.subs.size();
    info->center_frequency = h.center; info->pcm_per_block = h.pcm_per_block;
    info->alg_bytes_per_sample = h.alg_bytes; info->alg_flops_per_sample = h.alg_flops;
    strncpy(info->zmq_address, h.zmq_address.c_str(), sizeof(info->zmq_address) - 1);
    return SDRB_OK;
}

extern "C" int sdrb_plan_get_main(const sdrb_plan *plan, int idx, sdrb_main_info *info) {
    if (!plan || !info || idx < 0 || idx >= (int)plan->h.mains.size()) {
        set_error("sdrb_plan_get_main: bad argument"); return SDRB_E_INVALID;
    }
    const MainVfo &m = plan->h.mains[(size_t)idx];
    info->mixer_hz = m.mixer; info->frequency = m.frequency; info->decim = m.decim;
    info->out_rate = m.out_rate; info->block_out = m.block_out;
    info->n_subs = m.n_subs; info->forward = (m.n_subs == 0 && !m.topic.empty()) ? 1 : 0;
    info->compress_scale = m.compress_scale; info->compress_style = m.compress_style;
    info->fwd_bytes_per_block = m.fwd_bytes;
    memset(info->topic, 0, sizeof(info->topic));
    strncpy(info->topic, m.topic.c_str(), sizeof(info->topic) - 1);
    memset(info->zmq_address, 0, sizeof(info->zmq_address));
    strncpy(info->zmq_address, m.zmq_address.c_str(), sizeof(info->zmq_address) - 1);
    return SDRB_OK;
}

extern "C" int sdrb_plan_get_sub(const sdrb_plan *plan, int idx, sdrb_sub_info *info) {
    if (!plan || !info || idx < 0 || idx >= (int)plan->h.subs.size()) {
        set_error("sdrb_plan_get_sub: bad argument"); return SDRB_E_INVALID;
    }
    const SubVfo &s = plan->h.subs[(size_t)idx];
    memset(info, 0, sizeof(*info));
    strncpy(info->topic, s.topic.c_str(), sizeof(info->topic) - 1);
    info->frequency = s.frequency; info->data_rate = s.data_rate; info->main_idx = s.main_idx;
    info->decim = s.decim; info->late = s.late; info->filter_bw = s.filter_bw; info->gain = s.gain;
    info->mixer_hz = s.mixer; info->in_rate = s.fs; info->out_rate = s.out_rate;
    info->samples_out = s.samples_out; info->pcm_offset = s.pcm_offset;
    info->n_dec_taps = (int)s.dec_taps.size(); info->n_lpf_taps = (int)s.lpf_taps.size();
    return SDRB_OK;
}

extern "C" int sdrb_plan_get_setting(const sdrb_plan *plan, const char *key, char *out, size_t out_len) {
    if (!plan || !key) { set_error("sdrb_plan_get_setting: NULL argument"); return SDRB_E_INVALID; }
    auto it = plan->h.settings.find(key);
    if (it == plan->h.settings.end()) return -1;
    if (out && out_len) {
        const size_t n = std::min(out_len - 1, it->second.size());
        memcpy(out, it->second.data(), n);
        out[n] = 0;
    }
    return (int)it->second.size();
}

extern "C" long sdrb_plan_copy_table(const sdrb_plan *plan, int kind, int idx, float *dst, long max_elems) {
    if (!plan) { set_error("sdrb_plan_copy_table: NULL plan"); return SDRB_E_INVALID; }
    const HostPlan &h = plan->h;
    const float *src = nullptr;
    long n = 0, width = 1;
    if (kind == 0 && idx >= 0 && idx < (int)h.mains.size()) {
        src = &h.mains[(size_t)idx].lut[0].re; n = (long)h.mains[(size_t)idx].lut.size(); width = 2;
    } else if (idx >= 0 && idx < (int)h.subs.size()) {
        const SubVfo &s = h.subs[(size_t)idx];
        if (kind == 1) { src = &s.lut[0].re; n = (long)s.lut.size(); width = 2; }
        else if (kind == 2) { src = s.dec_taps.data(); n = (long)s.dec_taps.size(); }
        else if (kind == 3) { src = s.lpf_taps.data(); n = (long)s.lpf_taps.size(); }
        else if (kind == 4) { src = s.hilbert.data(); n = (long)s.hilbert.size(); }
        else { set_error("sdrb_plan_copy_table: unknown kind"); return SDRB_E_INVALID; }
    } else { set_error("sdrb_plan_copy_table: index out of range"); return SDRB_E_INVALID; }
    if (dst && n > 0 && max_elems > 0) memcpy(dst, src, sizeof(float) * (size_t)(std::min(n, max_elems) * width));
    return n;
}

// FNV-1a over a canonical serialisation (little-endian 64-bit integers, IEEE bits of doubles and floats) of what can change
// an output sample. The NCO tables follow from (fs, mixer) and the Hilbert points from the rates; topics, addresses, the
// centre frequency and operational ini keys stay out, so renaming a topic keeps the fingerprint.
static uint64_t plan_fingerprint(const HostPlan &h) {
    uint64_t x = 0xcbf29ce484222325ull;
    auto bytes = [&](const void *p, size_t n) {
        for (size_t k = 0; k < n; k++) { x ^= ((const unsigned char *)p)[k]; x *= 0x100000001b3ull; }
    };
    auto i64 = [&](int64_t v) { uint64_t u = (uint64_t)v; unsigned char b[8]; for (int k = 0; k < 8; k++) b[k] = (unsigned char)(u >> (8 * k)); bytes(b, 8); };
    auto f64 = [&](double v) { int64_t u; memcpy(&u, &v, 8); i64(u); };
    auto f32 = [&](float v) { uint32_t u; memcpy(&u, &v, 4); i64(u); };
    bytes("sdrb-plan-1", 11);
    i64(h.fs); i64(h.block); i64(h.bufsplit); i64(h.correct_dc);
    i64((int64_t)h.mains.size());
    for (const MainVfo &m : h.mains) { f64(m.mixer); i64(m.decim); i64(m.compress_scale); i64(m.compress_style); }
    i64((int64_t)h.subs.size());
    for (const SubVfo &s : h.subs) {
        i64(s.main_idx); f64(s.mixer); i64(s.decim); i64(s.late); f32(s.gain);
        i64((int64_t)s.dec_taps.size());
        for (float v : s.dec_taps) f32(v);
        i64((int64_t)s.lpf_taps.size());
        for (float v : s.lpf_taps) f32(v);
    }
    return x;
}

extern "C" int sdrb_plan_fingerprint(const sdrb_plan *plan, uint64_t *out) {
    if (!plan || !out) { set_error("sdrb_plan_fingerprint: NULL argument"); return SDRB_E_INVALID; }
    *out = plan_fingerprint(plan->h);
    return SDRB_OK;
}

// ------------------------------------------------------------------------------------
// bank
// ------------------------------------------------------------------------------------
namespace {

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int alloc(size_t n) {
        bytes = n;
        cudaError_t e = cudaMalloc(&p, n ? n : 16);
        if (e != cudaSuccess) { set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); return SDRB_E_NOMEM; }
        return SDRB_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; }
};

// CTA size of a k1_v2 / k2a_v2 launch with `halo` halo threads per tile. Occupancy is 12 warps per SM
// at any size (168 registers); measured on B200, a 64-thread CTA runs ~10 % and a 96-thread CTA ~3 %
// faster per thread than a 128-thread one (shorter barrier domains), and (NT - halo)/NT of the
// threads do useful work. `env` (64, 96 or 128) overrides the choice for tuning runs.
static int v2_pick_threads(int halo, const char *env) {
    if (const char *e = getenv(env)) {
        const int v = atoi(e);
        if ((v == 64 || v == 96 || v == 128) && v > 2 * halo) return v;
    }
    static const int nt[3] = {64, 96, 128};
    static const double speed[3] = {1.10, 1.03, 1.00};
    int best = 128; double best_score = 0.0;
    for (int i = 0; i < 3; i++) {
        const double score = speed[i] * (double)(nt[i] - halo) / (double)nt[i];
        if (score > best_score) { best_score = score; best = nt[i]; }
    }
    return best;
}

template <int NT, bool MAP = false>
static void launch_k1_v2(const K1V2Params &q, bool dc, int ns, int block, cudaStream_t st, bool bulk = false) {
    const int tiles = (block + k1v2_adv<NT>() - 1) / k1v2_adv<NT>();
    const dim3 grid((unsigned)ns, (unsigned)((tiles + K1_TPC - 1) / K1_TPC), 1u);
    if (NT == 64 && bulk) {          // the bulk-copy (TMA) prefetch exists for the default CTA size; SDRB_K1_BULK=0 turns it off
        if (dc) k1_v2<true, 64, true, MAP><<<grid, 64, k1v2_smem_bulk<64>(), st>>>(q);
        else k1_v2<false, 64, true, MAP><<<grid, 64, k1v2_smem_bulk<64>(), st>>>(q);
        return;
    }
    if (dc) k1_v2<true, NT, false, MAP><<<grid, NT, k1v2_smem<NT>(), st>>>(q);
    else k1_v2<false, NT, false, MAP><<<grid, NT, k1v2_smem<NT>(), st>>>(q);
}

struct SubGroup {           // sub VFOs of one main VFO (at most V2_MAX_VFO) -> one k2a_v2 launch
    int main_idx;
    int tiles;              // tiles per callback
    int halo;               // halo threads in front of every tile
    int threads;            // CTA size of this group's launch (64, 96 or 128)
    int first, count;       // range in the device CascVfo / Rf arrays (sorted by group)
    int lut_len, block_in;  // Oscillator table length and callback size of the group's sub VFOs
    // k2a_v3 (kernels_v3.cuh): used when every sub VFO of the group has 1..5 half-band stages and the callback is a
    // whole number of 128-sample tiles; otherwise the group stays on k2a_v2
    bool v3 = false;
    int v3_maxs = 5, v3_nsw = 1;
    bool ragged = false;    // callback not a whole number of 32-sample chunks: k2a_v2's masked instantiation
};

// Rf[j] = (rot/|rot|)^j, j = -10..31 (index j + 10), rot = the float rotation the Oscillator table is
// built from (oscillator.cpp:9-14); see kernels_v2.cuh
void rf_table(double sample_rate, double frequency, float2 *dst);
// the kernel-parameter form: (c, c, -s, s) per rotation (kernels_v2.cuh: RfTab)
void rf_tab(double sample_rate, double frequency, RfTab *t) {
    float2 rf[RF_LEN];
    rf_table(sample_rate, frequency, rf);
    for (int i = 0; i < RF_LEN; i++) t->q[i] = make_float4(rf[i].x, rf[i].x, -rf[i].y, rf[i].y);
}
void rf_table(double sample_rate, double frequency, float2 *dst) {
    const double step = 2.0 * M_PI * frequency / sample_rate;
    const float rr = (float)cos(step), ri = (float)sin(step);
    const double w = atan2((double)ri, (double)rr);
    for (int i = 0; i < RF_LEN; i++) {
        const int j = i - 10;
        dst[i] = i < 42 ? make_float2((float)cos(w * j), (float)sin(w * j)) : make_float2(0.f, 0.f);
    }
}

inline size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

}  // namespace

struct sdrb_bank {
    const sdrb_plan *plan = nullptr;
    int device = 0, n_streams = 0, max_blocks = 0;
    int last_launches = 0;
    // tables
    DevBuf luts, taps;
    // state
    DevBuf blocks_done, dc_state, raw_tail, cf_tail;
    // work
    DevBuf dc_anchor, dc_stats, dc_table, dc_qtab, main_out, zbuf, dbuf;
    int dc_stride = 0;                      // DC blocks (of 32 samples) per stream in dc_stats; table has DC_HALO_BLKS more
    // dc_anchor and dc_table exist twice and alternate from call to call: the DC pre-pass of call
    // n+1 (side stream) may then run while the filters of call n still read call n's table.
    int dc_par = 0;                         // buffer the NEXT call writes
    cudaEvent_t ev_end[2] = {nullptr, nullptr};   // end of the last call that used buffer 0 / 1
    bool ev_end_valid[2] = {false, false};
    int *qtab_buf(int par) const { return (int *)dc_qtab.p + (size_t)par * 512 * (size_t)n_streams; }
    DcAnchor *anchor_buf(int par) const { return (DcAnchor *)dc_anchor.p + (size_t)par * 2 * (size_t)n_streams; }
    uint2 *table_buf(int par) const { return (uint2 *)dc_table.p + (size_t)par * 2 * (size_t)n_streams * (size_t)(dc_stride + DC_HALO_BLKS); }
    // stream-list calls: the device copy of the call's list, per call parity like the tables above -- the DC pre-pass of call n+1
    // reads its list while the filters of call n still read theirs
    DevBuf stream_list;
    int *list_buf(int par) const { return (int *)stream_list.p + (size_t)par * (size_t)n_streams; }
    // descriptors
    K1Params k1{};          // cf32-input variant (vfo::process entry)
    K1V2Params k1v2{};
    int k1_threads = 64;
    std::vector<K2V2Params> k2v2;                 // one prebuilt parameter block per sub-VFO group
    std::vector<int> k3_cw;                       // warps per CTA chosen for each group's k2a_v3 launches
    std::vector<int> k3_slots;                    // resident CTAs of each group's k2a_v3 instantiation (-1: not asked yet)
    std::vector<K3Params> k3;                     // ... and for the groups that run k2a_v3
    std::vector<bool> sub_fused;                  // NCO mix fused into the /late FIR kernel: z exists only on demand
    std::vector<CascVfo> sub_casc;
    std::vector<RfTab> sub_rf;
    DevBuf k3_rrel;
    bool per_cb = false;                          // SDRB_PER_CB=1: device-resident calls launch every kernel class per callback
    bool k1_bulk = true;                          // k1_v2 (64-thread CTAs) prefetches tiles with cp.async.bulk + mbarrier; SDRB_K1_BULK=0: per-thread cp.async records
    int dbg_only = 0;                             // SDRB_DEBUG_ONLY=dc|filters: profiling aid, device-resident calls skip the other half (results are then meaningless)
    DevBuf cascdev, rfdev, latedev, usbdev, carry;
    std::vector<SubGroup> groups;
    int n_late = 0, n_usb = 0, n_carry = 0;
    int max_usb_samples = 0, max_late_samples = 0;
    int late_taps_per_phase = 0;    // taps per polyphase branch if all late VFOs share it (10 or 13 select a compile-time instantiation), else -1
    int late_factor = 0;            // the plan's /late factor if all late VFOs share it and their taps fit k2_late_v2, else -1
    int uv_np_max = 0, uv_eo_rows = 0, uv_warp_floats = 0, uv_tiles = 0;   // k2b_v2 launch geometry
    std::vector<unsigned short> uv_vfo_tiles;                              // tiles per callback of each USB VFO
    std::vector<int> uv_vfo_out, uv_vfo_np;                                // samples per callback and padded low-pass length of each USB VFO
    size_t uv_smem = 0;
    std::vector<size_t> main_off;           // per main: offset (float2 units) inside main_out per stream
    size_t main_stride = 0;                 // float2 per stream
    size_t z_stride = 0;                    // float2 per stream in zbuf
    std::vector<size_t> sub_z_off;          // per sub VFO: offset of its slice inside a stream's zbuf row
    std::vector<int> sub_z_hist;            // ... and the history samples in front of the body
    // VFOs deeper than their mixing kernel's cascade (main VFOs with 4..8 stages, sub VFOs with 6..8): the mixing kernel writes
    // a staging slice (k1_v2 / k1_ingest_main: 3 stages, k2a_v3 / k2a_v2: 5) inside the same per-stream row as the real outputs
    // (main_out, zbuf), and k_hb_tail runs the remaining stages into the real output. Empty for plans without such VFOs.
    DevBuf main_tails, sub_tails;           // TailDev per deep main / sub VFO
    int n_main_tails = 0, n_sub_tails = 0, main_tail_tiles = 0, sub_tail_tiles = 0;   // channels and the longest channel's tiles
    // receiver state records (k_state_io): where each carry item sits in a record, the record's size and the header fields
    // of this bank; the stream list of a save / load, and the host variants' staging
    DevBuf state_items, state_streams, d_state;
    size_t state_bytes = 0;
    StateHeader state_hdr{};
    // end of the last save / load (recorded on the caller's stream): the next call's DC pre-pass waits for it, it may
    // otherwise run as soon as that call's input is ready
    cudaEvent_t ev_state = nullptr;
    bool state_pending = false;
    // what the last process call consumed (inspection entry points: spectrum of the raw input)
    const uint8_t *last_iq = nullptr; size_t last_iq_stride = 0;
    const float2 *last_cf = nullptr; size_t last_cf_stride = 0;
    int last_blocks = 0, last_par = 0;
    const int *last_map = nullptr; int last_n = 0;   // a stream-list call: its device list and length (inspection covers those streams)
    // host staging for process_host
    DevBuf d_iq, d_pcm, d_tap, d_cf, d_fwd;
    cudaStream_t s_copy_in = nullptr, s_compute = nullptr, s_copy_out = nullptr;
    std::vector<cudaEvent_t> ev_in, ev_done, ev_free, ev_out;   // per (group, callback) chunk of process_host
    bool host_inflight = false, host_inflight_tap = false;       // sdrb_bank_process_host_async calls not yet waited for
    int host_inflight_blocks = 0;
    std::deque<cudaEvent_t> host_calls;                          // one completion event per call in flight, oldest first
    // end of the last device-resident call (recorded on the caller's stream): a host call that follows waits for it,
    // its internal streams never see the caller's stream otherwise
    cudaEvent_t ev_device_tail = nullptr;
    bool device_tail_pending = false;
    std::vector<std::pair<int, int>> host_groups;      // (first stream, count) of each pipeline group of process_host
    // DC recursion runs on side streams, one callback ahead of the ingest kernel
    static constexpr int kSide = 8;
    cudaStream_t s_dc[kSide] = {nullptr};
    cudaEvent_t ev_entry[kSide] = {nullptr};
    std::vector<cudaEvent_t> ev_dc[kSide];
    // optional per-kernel timing (bench.py roofline): event pairs around each kernel class
    bool timing = false;
    std::vector<cudaEvent_t> tev;           // start/end pairs, recycled
    std::vector<int> tev_cls;               // class of each pair
    size_t tev_used = 0;
    double kernel_ms[SDRB_N_KERNEL_CLASSES] = {0};
    long kernel_calls[SDRB_N_KERNEL_CLASSES] = {0};
};

extern "C" void sdrb_bank_destroy(sdrb_bank *b) {
    if (!b) return;
    cudaSetDevice(b->device);
    cudaDeviceSynchronize();                                 // asynchronous host calls may still be in flight
    DevBuf *all[] = {&b->luts, &b->taps, &b->blocks_done, &b->dc_state, &b->raw_tail, &b->cf_tail, &b->dc_anchor, &b->dc_stats, &b->dc_table, &b->dc_qtab,
                     &b->main_out, &b->zbuf, &b->dbuf, &b->cascdev, &b->rfdev, &b->latedev, &b->usbdev, &b->carry,
                     &b->main_tails, &b->sub_tails, &b->state_items, &b->state_streams, &b->d_state, &b->stream_list,
                     &b->d_iq, &b->d_pcm, &b->d_tap, &b->d_cf, &b->d_fwd, &b->k3_rrel};
    for (DevBuf *d : all) d->release();
    if (b->ev_state) cudaEventDestroy(b->ev_state);
    for (cudaEvent_t e : b->ev_in) cudaEventDestroy(e);
    for (cudaEvent_t e : b->ev_free) cudaEventDestroy(e);
    for (cudaEvent_t e : b->ev_out) cudaEventDestroy(e);
    for (cudaEvent_t e : b->ev_done) cudaEventDestroy(e);
    for (cudaEvent_t e : b->tev) cudaEventDestroy(e);
    for (cudaEvent_t e : b->host_calls) cudaEventDestroy(e);
    if (b->ev_device_tail) cudaEventDestroy(b->ev_device_tail);
    for (int k = 0; k < sdrb_bank::kSide; k++) {
        if (b->s_dc[k]) cudaStreamDestroy(b->s_dc[k]);
        if (b->ev_entry[k]) cudaEventDestroy(b->ev_entry[k]);
        if (k < 2 && b->ev_end[k]) cudaEventDestroy(b->ev_end[k]);
        for (cudaEvent_t e : b->ev_dc[k]) cudaEventDestroy(e);
    }
    if (b->s_copy_in) cudaStreamDestroy(b->s_copy_in);
    if (b->s_compute) cudaStreamDestroy(b->s_compute);
    if (b->s_copy_out) cudaStreamDestroy(b->s_copy_out);
    delete b;
}

extern "C" int sdrb_bank_create(const sdrb_plan *plan, int device, int n_streams, int max_blocks, sdrb_bank **out) {
    if (!plan || !out || n_streams <= 0 || max_blocks <= 0) {
        set_error("sdrb_bank_create: bad argument"); return SDRB_E_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("sdrb_bank_create: no CUDA device (this library has no CPU path)");
        return SDRB_E_CUDA;
    }
    if (device < 0 || device >= ndev) { set_error("sdrb_bank_create: device index out of range"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(device));
    const HostPlan &h = plan->h;
    sdrb_bank *b = new (std::nothrow) sdrb_bank();
    if (!b) return SDRB_E_NOMEM;
    b->plan = plan; b->device = device; b->n_streams = n_streams; b->max_blocks = max_blocks;
    int rc = SDRB_OK;

#define BANK_TRY(x) do { rc = (x); if (rc != SDRB_OK) { sdrb_bank_destroy(b); return rc; } } while (0)
#define BANK_CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { set_error(std::string(#x) + ": " + cudaGetErrorString(e_)); sdrb_bank_destroy(b); return SDRB_E_CUDA; } } while (0)

    // ---- tables: all NCO tables in one buffer, all taps in another ----
    size_t lut_elems = 0;
    for (const MainVfo &m : h.mains) lut_elems += round_up(m.lut.size(), 2);
    for (const SubVfo &s : h.subs) lut_elems += round_up(s.lut.size(), 2);
    BANK_TRY(b->luts.alloc(lut_elems * sizeof(float2)));
    std::vector<size_t> main_lut_off, sub_lut_off;
    {
        size_t at = 0;
        for (const MainVfo &m : h.mains) {
            main_lut_off.push_back(at);
            BANK_CU(cudaMemcpy((float2 *)b->luts.p + at, m.lut.data(), m.lut.size() * sizeof(float2), cudaMemcpyHostToDevice));
            at += round_up(m.lut.size(), 2);
        }
        for (const SubVfo &s : h.subs) {
            sub_lut_off.push_back(at);
            BANK_CU(cudaMemcpy((float2 *)b->luts.p + at, s.lut.data(), s.lut.size() * sizeof(float2), cudaMemcpyHostToDevice));
            at += round_up(s.lut.size(), 2);
        }
    }
    // taps per sub: hil[64] | lpf[np] | dec[ntaps]  (16-byte aligned pieces)
    std::vector<float> taps_host;
    std::vector<size_t> hil_off, lpf_off, dec_off;
    std::vector<int> np_of;
    for (const SubVfo &s : h.subs) {
        hil_off.push_back(taps_host.size());
        taps_host.push_back(0.f); taps_host.push_back(0.f);
        for (int j = 0; j < 62; j++) taps_host.push_back(s.hilbert[(size_t)(2 * j + 1)]);
        const int n = (int)s.lpf_taps.size(), np = (int)round_up((size_t)n, 16);   // k2b_v2 works in blocks of 16 taps
        if (np > MAX_FIR_TAPS || (int)s.dec_taps.size() > MAX_FIR_TAPS) {
            set_error("bank: filter longer than 512 taps"); sdrb_bank_destroy(b); return SDRB_E_INVALID;
        }
        np_of.push_back(np);
        lpf_off.push_back(taps_host.size());
        for (int j = 0; j < np - n; j++) taps_host.push_back(0.f);
        for (int j = 0; j < n; j++) taps_host.push_back(s.lpf_taps[(size_t)j]);
        dec_off.push_back(taps_host.size());
        for (float v : s.dec_taps) taps_host.push_back(v);
        while (taps_host.size() % 4) taps_host.push_back(0.f);
    }
    BANK_TRY(b->taps.alloc(taps_host.size() * sizeof(float)));
    if (!taps_host.empty())
        BANK_CU(cudaMemcpy(b->taps.p, taps_host.data(), taps_host.size() * sizeof(float), cudaMemcpyHostToDevice));

    // ---- state ----
    BANK_TRY(b->blocks_done.alloc(sizeof(long long) * (size_t)n_streams));
    BANK_TRY(b->dc_state.alloc(sizeof(float2) * (size_t)n_streams));
    BANK_TRY(b->raw_tail.alloc((size_t)n_streams * 2 * RAW_TAIL));
    BANK_TRY(b->cf_tail.alloc((size_t)n_streams * RAW_TAIL * sizeof(float2)));

    // ---- work buffers ----
    b->dc_stride = max_blocks * (h.block / DC_BLK);
    BANK_TRY(b->dc_anchor.alloc(2 * sizeof(DcAnchor) * 2 * (size_t)n_streams));
    BANK_TRY(b->dc_qtab.alloc(2 * sizeof(int) * 512 * (size_t)n_streams));
    BANK_TRY(b->stream_list.alloc(2 * sizeof(int) * (size_t)n_streams));
    BANK_TRY(b->dc_stats.alloc(h.correct_dc ? sizeof(DcStats) * 2 * (size_t)n_streams * (size_t)b->dc_stride + 1024 : 16));
    BANK_TRY(b->dc_table.alloc(h.correct_dc ? 2 * sizeof(uint2) * 2 * (size_t)n_streams * (size_t)(b->dc_stride + DC_HALO_BLKS) : 64));
    // the halo entries a state record saves exist before any u8 call writes them (a bank fed only cf32 input): start them at zero
    BANK_CU(cudaMemset(b->dc_table.p, 0, b->dc_table.bytes));
    // staging slices of the deep VFOs: first stage count a mixing kernel runs, and the rest for k_hb_tail
    static_assert(TAIL_HIST == MAIN_HIST, "k1_ingest_main writes every main output, staged or not, behind MAIN_HIST samples");
    constexpr int kMainStaged = 3, kSubStaged = 5;
    std::vector<size_t> main_stage_off(h.mains.size(), 0), sub_stage_off(h.subs.size(), 0);
    {
        size_t at = 0;
        for (const MainVfo &m : h.mains) {
            b->main_off.push_back(at);
            at += round_up((size_t)MAIN_HIST + (size_t)max_blocks * m.block_out, 2);
        }
        for (size_t i = 0; i < h.mains.size(); i++)
            if (h.mains[i].decim > kMainStaged) {
                main_stage_off[i] = at;
                at += round_up((size_t)TAIL_HIST + (size_t)max_blocks * (h.block >> kMainStaged), 2);
            }
        b->main_stride = at;
    }
    BANK_TRY(b->main_out.alloc(sizeof(float2) * b->main_stride * (size_t)n_streams));

    // z / d buffers per sub
    std::vector<size_t> z_off, d_off;
    std::vector<int> z_hist, d_hist;
    size_t z_stride = 0, d_stride = 0;
    for (size_t i = 0; i < h.subs.size(); i++) {
        const SubVfo &s = h.subs[i];
        int zh, dh = 0;
        if (s.late > 0) { zh = (int)round_up(s.dec_taps.size(), 64); dh = (int)round_up((size_t)np_of[i] + 128, 64); }
        else zh = (int)round_up((size_t)np_of[i] + 128, 64);
        z_hist.push_back(zh); d_hist.push_back(dh);
        z_off.push_back(z_stride);
        z_stride += round_up((size_t)zh + (size_t)max_blocks * s.block_z, 2);
        d_off.push_back(d_stride);
        if (s.late > 0) d_stride += round_up((size_t)dh + (size_t)max_blocks * s.samples_out, 2);
    }
    for (size_t i = 0; i < h.subs.size(); i++)
        if (h.subs[i].decim > kSubStaged) {
            sub_stage_off[i] = z_stride;
            z_stride += round_up((size_t)TAIL_HIST + (size_t)max_blocks * (h.subs[i].block_in >> kSubStaged), 2);
        }
    BANK_TRY(b->zbuf.alloc(sizeof(float2) * z_stride * (size_t)n_streams));
    BANK_TRY(b->dbuf.alloc(sizeof(float2) * d_stride * (size_t)n_streams));

    // ---- descriptors ----
    K1Params &k1 = b->k1;
    k1.cf_in = nullptr; k1.cf_stride = 0; k1.cf_tail = (const float2 *)b->cf_tail.p;
    k1.blocks_done = (const long long *)b->blocks_done.p;
    k1.block = h.block; k1.n_main = (int)h.mains.size();
    for (size_t i = 0; i < h.mains.size(); i++) {
        MainDev &M = k1.mains[i];
        M.lut = (const float2 *)b->luts.p + main_lut_off[i];
        M.out = (float2 *)b->main_out.p + b->main_off[i];
        M.out_stride = (long long)b->main_stride;
        M.lut_len = (int)h.mains[i].lut.size(); M.decim = h.mains[i].decim; M.block_out = h.mains[i].block_out;
        if (h.mains[i].decim > kMainStaged) {
            M.out = (float2 *)b->main_out.p + main_stage_off[i];
            M.decim = kMainStaged; M.block_out = h.block >> kMainStaged;
        }
    }
    // sub VFOs grouped by parent main VFO: one k2a_v2 launch per group, the parent's output is
    // read once per thread and kept in registers for all sub VFOs of the group
    static const int kHalo[6] = {0, 0, 1, 2, 5, 11};    // halo chunks a cascade of S stages needs (+1 sample/stage at callback heads)
    // /late factor of the plan (k2_late_v2 handles one factor per launch) and the sub VFOs whose NCO mix is fused into that
    // kernel: no half-band stages and a /5 or /6 FIR behind -- their full-rate z is then never written nor read back
    for (const SubVfo &s : h.subs)
        if (s.late > 0) {
            const int lf = ((int)s.dec_taps.size() <= s.late * LV_AMAX) ? s.late : -1;
            b->late_factor = (b->late_factor == 0 || b->late_factor == lf) ? lf : -1;
            const int tpp = ((int)s.dec_taps.size() + s.late - 1) / s.late;
            b->late_taps_per_phase = (b->late_taps_per_phase == 0 || b->late_taps_per_phase == tpp) ? tpp : -1;
        }
    if (const char *e = getenv("SDRB_LATE_GENERIC")) { if (atoi(e) != 0) b->late_taps_per_phase = -1; }
    {
        const char *ef = getenv("SDRB_FUSE_LATE");
        const bool want = !(ef && atoi(ef) == 0) && (b->late_factor == 5 || b->late_factor == 6);
        for (const SubVfo &s : h.subs) b->sub_fused.push_back(want && s.late > 0 && s.decim == 0);
    }
    std::vector<int> order;
    for (size_t mi = 0; mi < h.mains.size(); mi++) {
        SubGroup g; g.main_idx = (int)mi; g.first = (int)order.size(); g.count = 0; g.tiles = 0; g.halo = 0;
        for (size_t i = 0; i < h.subs.size(); i++) {
            if (h.subs[i].main_idx != (int)mi || b->sub_fused[i]) continue;
            if (g.count == V2_MAX_VFO) { b->groups.push_back(g); g.first = (int)order.size(); g.count = 0; g.halo = 0; }
            order.push_back((int)i); g.count++;
            g.halo = std::max(g.halo, kHalo[std::min(h.subs[i].decim, kSubStaged)]);
        }
        if (g.count) b->groups.push_back(g);
    }
    for (SubGroup &g : b->groups) {
        g.threads = v2_pick_threads(g.halo, "SDRB_K2A_THREADS");
        const int adv = (g.threads - g.halo) * V2_CHUNK;
        const SubVfo &s0v = h.subs[(size_t)order[(size_t)g.first]];
        g.lut_len = (int)s0v.lut.size(); g.block_in = s0v.block_in;
        g.tiles = (g.block_in + adv - 1) / adv;
        g.ragged = g.block_in % V2_CHUNK != 0;
    }
    std::vector<CascVfo> cascdev;
    std::vector<float2> rfhost((h.mains.size() + h.subs.size()) * RF_LEN);
    std::vector<LateDev> latedev;
    std::vector<UsbDev> usbdev;
    std::vector<CarryItem> carry;
    // per carry item: 1 if a kernel reads its history in the next call. A state record holds the others as zeros: the z of a
    // sub VFO whose mix is fused into the /late FIR (that kernel reads the parent's output instead) and the output of a main
    // VFO without sub VFOs (the forwarder and copy_main read only the body)
    std::vector<int> carry_read;
    // the mixing cascade of sub VFO i: z itself, or the staging slice of a sub VFO with more than 5 stages
    auto sub_cascade = [&](size_t i) {
        const SubVfo &s = h.subs[i];
        CascVfo D;
        D.lut = (const float2 *)b->luts.p + sub_lut_off[i];
        D.out = (float2 *)b->zbuf.p + z_off[i];
        D.S = s.decim; D.block_out = s.block_z; D.hist = z_hist[i]; D.pad = 0;
        if (s.decim > kSubStaged) {
            D.out = (float2 *)b->zbuf.p + sub_stage_off[i];
            D.S = kSubStaged; D.block_out = s.block_in >> kSubStaged; D.hist = TAIL_HIST;
        }
        return D;
    };
    for (size_t i = 0; i < h.mains.size(); i++) rf_table((double)h.fs, h.mains[i].mixer, &rfhost[i * RF_LEN]);
    for (size_t k = 0; k < order.size(); k++) {
        const int i = order[k];
        const SubVfo &s = h.subs[(size_t)i];
        cascdev.push_back(sub_cascade((size_t)i));
        rf_table((double)s.fs, s.mixer, &rfhost[(h.mains.size() + k) * RF_LEN]);
    }
    b->z_stride = z_stride;
    b->sub_z_off = z_off; b->sub_z_hist = z_hist;
    // every sub VFO's own descriptor and rotation table: the inspection entry points produce the z of a fused VFO on demand
    b->sub_casc.resize(h.subs.size()); b->sub_rf.resize(h.subs.size());
    for (size_t i = 0; i < h.subs.size(); i++) {
        const SubVfo &s = h.subs[i];
        b->sub_casc[i] = sub_cascade(i);
        rf_tab((double)s.fs, s.mixer, &b->sub_rf[i]);
    }
    for (size_t i = 0; i < h.subs.size(); i++) {
        const SubVfo &s = h.subs[i];
        UsbDev U;
        if (s.late > 0) {
            LateDev L;
            L.z = (const float2 *)b->zbuf.p + z_off[i];
            L.d = (float2 *)b->dbuf.p + d_off[i];
            L.taps = (const float *)b->taps.p + dec_off[i];
            L.z_stride = (long long)z_stride; L.d_stride = (long long)d_stride;
            L.z_hist = z_hist[i]; L.d_hist = d_hist[i]; L.block_z = s.block_z; L.samples_out = s.samples_out;
            L.late = s.late; L.ntaps = (int)s.dec_taps.size();
            L.mix_lut = nullptr; L.blocks_done = (const long long *)b->blocks_done.p; L.lut_len = (int)s.lut.size(); L.pad = 0;
            if (b->sub_fused[i]) {
                L.z = (const float2 *)b->main_out.p + b->main_off[(size_t)s.main_idx];
                L.z_stride = (long long)b->main_stride; L.z_hist = MAIN_HIST;
                L.mix_lut = (const float2 *)b->luts.p + sub_lut_off[i];
            }
            latedev.push_back(L);
            b->max_late_samples = std::max(b->max_late_samples, s.samples_out);
            U.src = L.d; U.src_stride = L.d_stride; U.src_hist = L.d_hist;
            CarryItem c; c.base = L.d; c.stride = (long long)(d_stride * sizeof(float2));
            c.hist_bytes = L.d_hist * (int)sizeof(float2); c.block_bytes = s.samples_out * (int)sizeof(float2);
            carry.push_back(c); carry_read.push_back(1);
        } else {
            U.src = (const float2 *)b->zbuf.p + z_off[i]; U.src_stride = (long long)z_stride; U.src_hist = z_hist[i];
        }
        U.samples_out = s.samples_out; U.np = np_of[i]; U.pcm_offset = s.pcm_offset;
        U.hil = (const float *)b->taps.p + hil_off[i];
        U.lpf = (const float *)b->taps.p + lpf_off[i];
        U.gain = s.gain;
        usbdev.push_back(U);
        b->max_usb_samples = std::max(b->max_usb_samples, s.samples_out);
        b->uv_np_max = std::max(b->uv_np_max, U.np);
        b->uv_tiles = std::max(b->uv_tiles, (s.samples_out + (UV_USB - U.np) - 1) / (UV_USB - U.np));
        b->uv_vfo_tiles.push_back((unsigned short)((s.samples_out + (UV_USB - U.np) - 1) / (UV_USB - U.np)));
        b->uv_vfo_out.push_back(s.samples_out); b->uv_vfo_np.push_back(U.np);
        CarryItem c; c.base = (float2 *)b->zbuf.p + z_off[i]; c.stride = (long long)(z_stride * sizeof(float2));
        c.hist_bytes = z_hist[i] * (int)sizeof(float2); c.block_bytes = s.block_z * (int)sizeof(float2);
        carry.push_back(c); carry_read.push_back(b->sub_fused[i] ? 0 : 1);
    }
    for (size_t i = 0; i < h.mains.size(); i++) {
        CarryItem c; c.base = (float2 *)b->main_out.p + b->main_off[i];
        c.stride = (long long)(b->main_stride * sizeof(float2));
        c.hist_bytes = MAIN_HIST * (int)sizeof(float2); c.block_bytes = h.mains[i].block_out * (int)sizeof(float2);
        carry.push_back(c); carry_read.push_back(h.mains[i].n_subs > 0 ? 1 : 0);
    }
    // deep VFOs: the tail kernels' descriptors, and the staging slices' histories among the carry items
    std::vector<TailDev> main_tails, sub_tails;
    auto add_tail = [&](std::vector<TailDev> &list, float2 *in, float2 *out, size_t stride, int out_hist, int block_in, int S) {
        TailDev T;
        T.in = in; T.out = out; T.in_stride = T.out_stride = (long long)stride;
        T.in_hist = TAIL_HIST; T.out_hist = out_hist; T.block_in = block_in; T.S = S;
        T.HT = kHalo[S];
        T.tiles = (block_in + (TAIL_NT - T.HT) * V2_CHUNK - 1) / ((TAIL_NT - T.HT) * V2_CHUNK);
        list.push_back(T);
        CarryItem c; c.base = in; c.stride = (long long)(stride * sizeof(float2));
        c.hist_bytes = TAIL_HIST * (int)sizeof(float2); c.block_bytes = block_in * (int)sizeof(float2);
        carry.push_back(c); carry_read.push_back(1);
        return T.tiles;
    };
    for (size_t i = 0; i < h.mains.size(); i++)
        if (h.mains[i].decim > kMainStaged)
            b->main_tail_tiles = std::max(b->main_tail_tiles,
                                          add_tail(main_tails, (float2 *)b->main_out.p + main_stage_off[i], (float2 *)b->main_out.p + b->main_off[i],
                                                   b->main_stride, MAIN_HIST, h.block >> kMainStaged, h.mains[i].decim - kMainStaged));
    for (size_t i = 0; i < h.subs.size(); i++)
        if (h.subs[i].decim > kSubStaged)
            b->sub_tail_tiles = std::max(b->sub_tail_tiles,
                                         add_tail(sub_tails, (float2 *)b->zbuf.p + sub_stage_off[i], (float2 *)b->zbuf.p + z_off[i], z_stride,
                                                  z_hist[i], h.subs[i].block_in >> kSubStaged, h.subs[i].decim - kSubStaged));
    b->n_main_tails = (int)main_tails.size(); b->n_sub_tails = (int)sub_tails.size();
    BANK_TRY(b->main_tails.alloc(sizeof(TailDev) * std::max<size_t>(main_tails.size(), 1)));
    BANK_TRY(b->sub_tails.alloc(sizeof(TailDev) * std::max<size_t>(sub_tails.size(), 1)));
    if (!main_tails.empty()) BANK_CU(cudaMemcpy(b->main_tails.p, main_tails.data(), sizeof(TailDev) * main_tails.size(), cudaMemcpyHostToDevice));
    if (!sub_tails.empty()) BANK_CU(cudaMemcpy(b->sub_tails.p, sub_tails.data(), sizeof(TailDev) * sub_tails.size(), cudaMemcpyHostToDevice));
    b->n_late = (int)latedev.size(); b->n_usb = (int)usbdev.size(); b->n_carry = (int)carry.size();
    BANK_TRY(b->cascdev.alloc(sizeof(CascVfo) * std::max<size_t>(cascdev.size(), 1)));
    BANK_TRY(b->rfdev.alloc(sizeof(float2) * rfhost.size()));
    BANK_CU(cudaMemcpy(b->rfdev.p, rfhost.data(), sizeof(float2) * rfhost.size(), cudaMemcpyHostToDevice));
    BANK_TRY(b->latedev.alloc(sizeof(LateDev) * std::max<size_t>(latedev.size(), 1)));
    BANK_TRY(b->usbdev.alloc(sizeof(UsbDev) * std::max<size_t>(usbdev.size(), 1)));
    BANK_TRY(b->carry.alloc(sizeof(CarryItem) * std::max<size_t>(carry.size(), 1)));
    if (!cascdev.empty()) BANK_CU(cudaMemcpy(b->cascdev.p, cascdev.data(), sizeof(CascVfo) * cascdev.size(), cudaMemcpyHostToDevice));
    {
        K1V2Params &q = b->k1v2;
        q.tail = (const uint8_t *)b->raw_tail.p;
        q.dc_table = (const uint2 *)b->dc_table.p;
        q.dc_anchor = (const DcAnchor *)b->dc_anchor.p;
        q.blocks_done = (const long long *)b->blocks_done.p;
        for (size_t i = 0; i < h.mains.size(); i++) rf_tab((double)h.fs, h.mains[i].mixer, &q.rf[i]);
        q.out_stride = (long long)b->main_stride;
        q.dc_stride = b->dc_stride + DC_HALO_BLKS; q.block = h.block; q.lut_len = (int)h.mains[0].lut.size();
        q.n_main = (int)h.mains.size();
        for (size_t i = 0; i < h.mains.size(); i++) {
            CascVfo &M = q.vfos[i];
            M.lut = (const float2 *)b->luts.p + main_lut_off[i];
            M.out = (float2 *)b->main_out.p + b->main_off[i];
            M.S = h.mains[i].decim; M.block_out = h.mains[i].block_out; M.hist = MAIN_HIST; M.pad = 0;
            if (h.mains[i].decim > kMainStaged) {           // k1_v2 runs 3 stages (cascade_loop<3>); k_hb_tail the rest
                M.out = (float2 *)b->main_out.p + main_stage_off[i];
                M.S = kMainStaged; M.block_out = h.block >> kMainStaged; M.hist = TAIL_HIST;
            }
        }
    }
    b->k2v2.assign(b->groups.size(), K2V2Params{});
    for (size_t gi = 0; gi < b->groups.size(); gi++) {
        const SubGroup &g = b->groups[gi];
        K2V2Params &kp = b->k2v2[gi];
        for (int v = 0; v < g.count; v++) {
            kp.vfos[v] = cascdev[(size_t)(g.first + v)];
            kp.rf[v] = b->sub_rf[(size_t)order[(size_t)(g.first + v)]];
        }
        kp.in = (const float2 *)b->main_out.p + b->main_off[(size_t)g.main_idx];
        kp.blocks_done = (const long long *)b->blocks_done.p;
        kp.in_stride = (long long)b->main_stride; kp.out_stride = (long long)b->z_stride;
        kp.count = g.count; kp.lut_len = g.lut_len; kp.block_in = g.block_in; kp.HT = g.halo;
    }
    // k2a_v3 parameter blocks: folded taps and rotation tables per sub VFO (kernels_v3.cuh)
    static_assert(K3_MAX_VFO >= V2_MAX_VFO, "a sub-VFO group (at most V2_MAX_VFO) must fit K3Params::v");
    {
        const char *ev3 = getenv("SDRB_K2A_V3");
        const bool want_v3 = !(ev3 && atoi(ev3) == 0);
        b->per_cb = getenv("SDRB_PER_CB") && atoi(getenv("SDRB_PER_CB")) != 0;
        if (const char *e = getenv("SDRB_DEBUG_ONLY")) b->dbg_only = !strcmp(e, "dc") ? 1 : (!strcmp(e, "filters") ? 2 : 0);
        b->k3.assign(b->groups.size(), K3Params{});
        std::vector<float2> rrel(std::max<size_t>(cascdev.size(), 1) * K3_OUT1);
        BANK_TRY(b->k3_rrel.alloc(sizeof(float2) * rrel.size()));
        for (size_t gi = 0; gi < b->groups.size(); gi++) {
            SubGroup &g = b->groups[gi];
            K3Params &kp = b->k3[gi];
            bool ok = want_v3 && g.count <= K3_MAX_VFO && g.block_in % K3_TILE == 0 && g.block_in / K3_TILE >= 8 &&
                      g.lut_len >= 4 * K3_LUT_STEADY && MAIN_HIST >= (K3_WARM + 1) * K3_TILE;
            int maxs = 0;
            for (int v = 0; v < g.count; v++) {
                const SubVfo &sv = h.subs[(size_t)order[(size_t)(g.first + v)]];
                const int staged = cascdev[(size_t)(g.first + v)].S;   // a deep sub VFO's first 5 stages; its 2^-S factor is that of the 5
                if (staged < 1) ok = false;
                maxs = std::max(maxs, staged);
                K3Vfo &V = kp.v[v];
                k3_fill_vfo((double)sv.fs, sv.mixer, std::max(staged, 1), V, &rrel[(size_t)(g.first + v) * K3_OUT1]);
                V.lut = cascdev[(size_t)(g.first + v)].lut; V.out = cascdev[(size_t)(g.first + v)].out;
                V.block_out = cascdev[(size_t)(g.first + v)].block_out; V.hist = cascdev[(size_t)(g.first + v)].hist; V.pad = 0;
            }
            kp.rrel = (const float2 *)b->k3_rrel.p + (size_t)g.first * K3_OUT1;
            kp.in = (const float2 *)b->main_out.p + b->main_off[(size_t)g.main_idx];
            kp.blocks_done = (const long long *)b->blocks_done.p;
            kp.in_stride = (long long)b->main_stride; kp.out_stride = (long long)b->z_stride;
            kp.hist_in = MAIN_HIST; kp.count = g.count; kp.lut_len = g.lut_len; kp.block_in = g.block_in;
            kp.n_tiles = g.block_in / K3_TILE;
            g.v3 = ok;
            g.v3_maxs = maxs <= 2 ? 2 : (maxs == 3 ? 3 : 5);
            g.v3_nsw = std::max(1, std::min(8, (32 / std::max(g.count, 1)) & ~1));
            if (32 / std::max(g.count, 1) < 2) g.v3_nsw = 1;
            kp.nsw = g.v3_nsw;
        }
        BANK_CU(cudaMemcpy(b->k3_rrel.p, rrel.data(), sizeof(float2) * rrel.size(), cudaMemcpyHostToDevice));
        BANK_CU(cudaFuncSetAttribute(k2a_v3<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        BANK_CU(cudaFuncSetAttribute(k2a_v3<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        BANK_CU(cudaFuncSetAttribute(k2a_v3<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        BANK_CU((cudaFuncSetAttribute(k2a_v3<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)));
        BANK_CU((cudaFuncSetAttribute(k2a_v3<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)));
        BANK_CU((cudaFuncSetAttribute(k2a_v3<5, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)));
    }
    if (!latedev.empty()) BANK_CU(cudaMemcpy(b->latedev.p, latedev.data(), sizeof(LateDev) * latedev.size(), cudaMemcpyHostToDevice));
    if (!usbdev.empty()) BANK_CU(cudaMemcpy(b->usbdev.p, usbdev.data(), sizeof(UsbDev) * usbdev.size(), cudaMemcpyHostToDevice));
    BANK_CU(cudaMemcpy(b->carry.p, carry.data(), sizeof(CarryItem) * carry.size(), cudaMemcpyHostToDevice));
    {
        // receiver state records: the carry items' histories in bank order behind the fixed sections (kernels.cuh, k_state_io)
        std::vector<int2> rec(carry.size());
        size_t at = STATE_ITEMS_OFF;
        for (size_t k = 0; k < carry.size(); k++) {
            rec[k] = make_int2((int)at, carry_read[k]);
            at += (size_t)carry[k].hist_bytes;
        }
        b->state_bytes = at;
        BANK_TRY(b->state_items.alloc(sizeof(int2) * std::max<size_t>(rec.size(), 1)));
        if (!rec.empty()) BANK_CU(cudaMemcpy(b->state_items.p, rec.data(), sizeof(int2) * rec.size(), cudaMemcpyHostToDevice));
        BANK_TRY(b->state_streams.alloc(sizeof(int) * (size_t)n_streams));
        StateHeader &sh = b->state_hdr;
        sh.magic = STATE_MAGIC; sh.version = STATE_VERSION; sh.record_bytes = at; sh.fingerprint = plan_fingerprint(h);
        sh.flags = (h.correct_dc ? STATE_FLAG_DC : 0u) |
                   (std::find(b->sub_fused.begin(), b->sub_fused.end(), true) != b->sub_fused.end() ? STATE_FLAG_FUSED_LATE : 0u);
    }

    b->uv_eo_rows = 34 + b->uv_np_max / 32;
    b->uv_warp_floats = std::max(UV_IN_FLOATS, 2 * b->uv_eo_rows * UV_ROW);
    b->uv_smem = sizeof(float) * (2 * (size_t)(64 + b->uv_np_max) + (size_t)UV_WARPS * b->uv_warp_floats);
    BANK_CU(cudaFuncSetAttribute(k2b_v2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->uv_smem));
    BANK_CU(cudaFuncSetAttribute(k0_dc_walk<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DCW_SMEM));
    // the stream-list instantiations (MAP = true) of the kernels above and below
    BANK_CU(cudaFuncSetAttribute(k2b_v2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->uv_smem));
    BANK_CU(cudaFuncSetAttribute(k0_dc_walk<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DCW_SMEM));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<5, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<5>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<6, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<6>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<5, 10, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<5>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<6, 13, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<6>())));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<64, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<64>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<96, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<96>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<128, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<128>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<64, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<64>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<96, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<96>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<128, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<128>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 64, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<64>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 64, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<64>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 96, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<96>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 96, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<96>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 128, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<128>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 128, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<128>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 64, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem_bulk<64>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 64, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem_bulk<64>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<5, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<5>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<6, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<6>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<5, 10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<5>())));
    BANK_CU((cudaFuncSetAttribute(k2_late_v2<6, 13>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv_smem<6>())));
    BANK_CU(cudaFuncSetAttribute(k2a_v2<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<64>::SMEM));
    BANK_CU(cudaFuncSetAttribute(k2a_v2<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<96>::SMEM));
    BANK_CU(cudaFuncSetAttribute(k2a_v2<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<128>::SMEM));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<64>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<96, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<96>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k2a_v2<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)V2L<128>::SMEM)));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<64>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<64>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 96>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<96>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 96>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<96>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<128>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem<128>())));
    b->k1_threads = v2_pick_threads(K1V2_HT, "SDRB_K1_THREADS");
    b->k1_bulk = !(getenv("SDRB_K1_BULK") && atoi(getenv("SDRB_K1_BULK")) == 0);   // default on: 0.59 -> 0.535 ms per step (profiles/r02_experiments.md)
    BANK_CU((cudaFuncSetAttribute(k1_v2<true, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem_bulk<64>())));
    BANK_CU((cudaFuncSetAttribute(k1_v2<false, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1v2_smem_bulk<64>())));
    BANK_CU(cudaStreamCreateWithFlags(&b->s_copy_in, cudaStreamNonBlocking));
    BANK_CU(cudaStreamCreateWithFlags(&b->s_compute, cudaStreamNonBlocking));
    BANK_CU(cudaStreamCreateWithFlags(&b->s_copy_out, cudaStreamNonBlocking));
    if (h.correct_dc) {
        // The DC walk is a long dependent chain on few warps: give its side streams the highest priority so its
        // CTAs take the first registers/shared memory the filter kernels free instead of queueing behind their grids.
        int prio_least = 0, prio_greatest = 0;
        BANK_CU(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
        for (int k = 0; k < sdrb_bank::kSide; k++) {
            BANK_CU(cudaStreamCreateWithPriority(&b->s_dc[k], cudaStreamNonBlocking, prio_greatest));
            BANK_CU(cudaEventCreateWithFlags(&b->ev_entry[k], cudaEventDisableTiming));
            if (k < 2) BANK_CU(cudaEventCreateWithFlags(&b->ev_end[k], cudaEventDisableTiming));
            for (int j = 0; j < max_blocks; j++) {
                cudaEvent_t e;
                BANK_CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                b->ev_dc[k].push_back(e);
            }
        }
    }
#undef BANK_TRY
#undef BANK_CU
    rc = sdrb_bank_reset(b, -1);
    if (rc != SDRB_OK) { sdrb_bank_destroy(b); return rc; }
    *out = b;
    return SDRB_OK;
}

extern "C" int sdrb_bank_reset(sdrb_bank *b, int stream) {
    if (!b || stream < -1 || stream >= b->n_streams) { set_error("sdrb_bank_reset: bad argument"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(b->device));
    const int s0 = stream < 0 ? 0 : stream, ns = stream < 0 ? b->n_streams : 1;
    CU_TRY(cudaDeviceSynchronize());                     // nothing of an earlier call may still be in flight
    CU_TRY(cudaMemset((long long *)b->blocks_done.p + s0, 0, sizeof(long long) * (size_t)ns));
    CU_TRY(cudaMemset((float2 *)b->dc_state.p + (size_t)s0, 0, sizeof(float2) * (size_t)ns));
    CU_TRY(cudaMemset((uint8_t *)b->raw_tail.p + (size_t)s0 * 2 * RAW_TAIL, 0, (size_t)ns * 2 * RAW_TAIL));
    CU_TRY(cudaMemset((float2 *)b->cf_tail.p + (size_t)s0 * RAW_TAIL, 0, (size_t)ns * RAW_TAIL * sizeof(float2)));
    // history regions: zero whole per-stream slices (cheap, and only done on reset)
    const size_t ms = b->main_stride * sizeof(float2);
    CU_TRY(cudaMemset((char *)b->main_out.p + ms * (size_t)s0, 0, ms * (size_t)ns));
    const size_t zs = b->zbuf.bytes / (size_t)b->n_streams, ds = b->dbuf.bytes / (size_t)b->n_streams;
    if (zs) CU_TRY(cudaMemset((char *)b->zbuf.p + zs * (size_t)s0, 0, zs * (size_t)ns));
    if (ds) CU_TRY(cudaMemset((char *)b->dbuf.p + ds * (size_t)s0, 0, ds * (size_t)ns));
    CU_TRY(cudaDeviceSynchronize());
    return SDRB_OK;
}

extern "C" int sdrb_bank_blocks_done(sdrb_bank *b, int stream, int64_t *blocks) {
    if (!b || !blocks || stream < 0 || stream >= b->n_streams) { set_error("sdrb_bank_blocks_done: bad argument"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(b->device));
    long long v = 0;
    CU_TRY(cudaMemcpy(&v, (long long *)b->blocks_done.p + stream, sizeof(v), cudaMemcpyDeviceToHost));
    *blocks = v;
    return SDRB_OK;
}

static int host_drain(sdrb_bank *b);   // waits for asynchronous host calls still in flight (defined with process_host)

// Per-kernel timing (bench.py roofline): when enabled, a cudaEvent pair brackets every launch
// on its own stream; sdrb_bank_kernel_times() folds them into per-class totals after a
// synchronize. Classes: 0 DC recursion, 1 ingest+main VFOs, 2 sub-VFO cascades, 3 /late FIR,
// 4 USB audio, 5 carry.
struct TimedScope {
    sdrb_bank *b; cudaStream_t st; int cls; bool on;
    TimedScope(sdrb_bank *b_, cudaStream_t st_, int cls_);
    ~TimedScope();
};

// One process call, as seen by the launch helpers.
struct CallCtx {
    const uint8_t *d_iq = nullptr; size_t iq_stride = 0;
    const float2 *d_cf = nullptr; size_t cf_stride = 0;    // cf32 input variant (no DC stage)
    int n_blocks = 0;
    int16_t *d_pcm = nullptr; float *d_tap = nullptr;
    int par = 0;                                            // which dc_anchor / dc_table buffer this call owns
    // stream-list calls: the caller's list (host) and its device copy; the launch helpers then get s0 = 0 and ns = its length
    const int32_t *h_map = nullptr; int n_map = 0;
    const int *map = nullptr;
};

// DC recursion of callback cb for streams [s0, s0+ns) on the side stream `sd`: (anchor once per
// call,) parallel block statistics, sequential walk. `ready` (optional) = the input of this
// callback has landed; `done` is recorded when the table of this callback is complete.
static int enqueue_dc_cb(sdrb_bank *b, const CallCtx &c, int s0, int ns, cudaStream_t sd, int cb, cudaEvent_t ready,
                         cudaEvent_t done, int *nl) {
    const HostPlan &h = b->plan->h;
    const int per_cb = h.block / DC_BLK;
    if (ready) CU_TRY(cudaStreamWaitEvent(sd, ready, 0));
    if (cb == 0) {
        TimedScope t(b, sd, 0);
        const dim3 ga((unsigned)((2 * ns + 127) / 128));
        if (c.map) {
            k0_dc_anchor<true><<<ga, 128, 0, sd>>>((const float2 *)b->dc_state.p, b->anchor_buf(c.par), ns, s0, c.map);
            k0_dc_qtab<true><<<(unsigned)(2 * ns), 256, 0, sd>>>(b->anchor_buf(c.par), b->qtab_buf(c.par), s0, c.map);
        } else {
            k0_dc_anchor<<<ga, 128, 0, sd>>>((const float2 *)b->dc_state.p, b->anchor_buf(c.par), ns, s0);
            k0_dc_qtab<<<(unsigned)(2 * ns), 256, 0, sd>>>(b->anchor_buf(c.par), b->qtab_buf(c.par), s0);
        }
        (*nl) += 2;
    }
    {
        TimedScope t(b, sd, 0);
        const dim3 gb((unsigned)((per_cb + 127) / 128), (unsigned)ns);
        if (c.map)
            k0_dc_blocks<true><<<gb, 128, 0, sd>>>(c.d_iq, c.iq_stride, b->anchor_buf(c.par), b->qtab_buf(c.par), (DcStats *)b->dc_stats.p,
                                                   b->dc_stride, cb * per_cb, per_cb, s0, c.map);
        else
            k0_dc_blocks<<<gb, 128, 0, sd>>>(c.d_iq, c.iq_stride, b->anchor_buf(c.par), b->qtab_buf(c.par), (DcStats *)b->dc_stats.p,
                                             b->dc_stride, cb * per_cb, per_cb, s0);
    }
    {
        TimedScope t(b, sd, 0);
        if (c.map)
            k0_dc_walk<true><<<(unsigned)ns, 64, DCW_SMEM, sd>>>(c.d_iq, c.iq_stride, (const DcStats *)b->dc_stats.p, b->dc_stride,
                                                                b->anchor_buf(c.par), b->qtab_buf(c.par), (float2 *)b->dc_state.p,
                                                                b->table_buf(c.par), b->dc_stride + DC_HALO_BLKS, cb * per_cb, per_cb, s0,
                                                                c.map);
        else
            k0_dc_walk<<<(unsigned)ns, 64, DCW_SMEM, sd>>>(c.d_iq, c.iq_stride, (const DcStats *)b->dc_stats.p, b->dc_stride,
                                                          b->anchor_buf(c.par), b->qtab_buf(c.par), (float2 *)b->dc_state.p, b->table_buf(c.par),
                                                          b->dc_stride + DC_HALO_BLKS, cb * per_cb, per_cb, s0);
    }
    (*nl) += 2;
    CU_TRY(cudaEventRecord(done, sd));
    return SDRB_OK;
}

// Ingest + main VFOs of callback cb. `wait` (optional) gates the kernel.
static int enqueue_ingest_cb(sdrb_bank *b, const CallCtx &c, int s0, int ns, cudaStream_t st, int cb, cudaEvent_t wait, int *nl) {
    const HostPlan &h = b->plan->h;
    if (wait) CU_TRY(cudaStreamWaitEvent(st, wait, 0));
    K1Params k1 = b->k1;
    k1.stream0 = s0; k1.b0 = cb;
    k1.cf_in = c.d_cf; k1.cf_stride = c.cf_stride;
    if (c.d_cf) {
        const int k1_tiles = (h.block + K1_TILE - 1) / K1_TILE;
        TimedScope t(b, st, 1);
        k1_ingest_main<<<dim3((unsigned)ns, (unsigned)k1_tiles, 1u), K1_THREADS, 0, st>>>(k1);
    } else {
        K1V2Params q = b->k1v2;
        q.iq = c.d_iq; q.iq_stride = c.iq_stride; q.stream0 = s0; q.b0 = cb;
        q.dc_table = b->table_buf(c.par); q.dc_anchor = b->anchor_buf(c.par);
        q.map = c.map;
        TimedScope t(b, st, 1);
        if (c.map) {
            if (b->k1_threads == 64) launch_k1_v2<64, true>(q, h.correct_dc, ns, h.block, st, b->k1_bulk);
            else if (b->k1_threads == 96) launch_k1_v2<96, true>(q, h.correct_dc, ns, h.block, st);
            else launch_k1_v2<128, true>(q, h.correct_dc, ns, h.block, st);
        } else if (b->k1_threads == 64) launch_k1_v2<64>(q, h.correct_dc, ns, h.block, st, b->k1_bulk);
        else if (b->k1_threads == 96) launch_k1_v2<96>(q, h.correct_dc, ns, h.block, st);
        else launch_k1_v2<128>(q, h.correct_dc, ns, h.block, st);
    }
    (*nl)++;
    return SDRB_OK;
}

// k2a_v3 launch geometry: one warp per (stream group, span, callback). `slots` = CTAs of this kernel the device holds at once
// (occupancy x SM count): the spans are chosen so that the grid is just under two full waves of it -- the
// 5-stage kernel holds 4 CTAs per SM (two 200-register warps per scheduler), and a grid of 2.4 waves left the last third of its run
// 60 % empty (profiles/r02_experiments.md section 1). Never shorter than 16 tiles: 3 warm-up tiles are recomputed per span.
static void k3_geometry(const SubGroup &g, K3Params &kp, int ns, int ncb, int cta_warps, int slots, dim3 *grid) {
    const int sgroups = (ns + g.v3_nsw - 1) / g.v3_nsw;
    const int ctas_x = (sgroups + cta_warps - 1) / cta_warps;
    const int target_ctas = slots > 0 ? 2 * slots : 148 * 10;
    int spans = std::max(1, target_ctas / std::max(1, ctas_x * ncb));
    int tps = std::max(16, (kp.n_tiles + spans - 1) / spans);
    tps = std::min(tps, kp.n_tiles);
    spans = (kp.n_tiles + tps - 1) / tps;
    kp.tiles_per_span = tps;
    *grid = dim3((unsigned)ctas_x, (unsigned)spans, (unsigned)ncb);
}

template <class K>
static int k3_slots(K kernel, int threads, size_t smem) {
    int per_sm = 0, dev = 0, sms = 148;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess) return 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return per_sm * sms;
}

// One k2a_v3 launch for sub-VFO group gi. First launch of the group: CTA size and resident CTAs. The 5-stage kernel holds two warps
// per scheduler whatever the CTA size (registers); the shorter cascades fit three, and how many CTAs fit is a matter of shared memory
// (the rotation table is per CTA, a ring per warp): take the CTA size with the most resident warps (25E's 15 two-stage VFOs: 6 warps,
// 12 per SM).
template <int MAXS>
static void launch_k3(sdrb_bank *b, size_t gi, int ns, int ncb, cudaStream_t st, bool map) {
    const SubGroup &g = b->groups[gi];
    K3Params &kp = b->k3[gi];
    int &slots = b->k3_slots[gi], &cw = b->k3_cw[gi];
    const int rows = g.v3_nsw * g.count;
    if (slots < 0) {
        cw = K3_WARPS;
        if (MAXS <= 3) {
            int best = 0;
            for (int c : {2, 3, 4, 6}) {
                const int w = c * k3_slots(k2a_v3<MAXS>, c * 32, k3_cta_smem_bytes(g.count, c, rows));
                if (w > best) { best = w; cw = c; }
            }
        }
        slots = k3_slots(k2a_v3<MAXS>, cw * 32, k3_cta_smem_bytes(g.count, cw, rows));
    }
    dim3 grid;
    k3_geometry(g, kp, ns, ncb, cw, slots, &grid);
    TimedScope t(b, st, 2);
    if (map) k2a_v3<MAXS, true><<<grid, cw * 32, k3_cta_smem_bytes(g.count, cw, rows), st>>>(kp);
    else k2a_v3<MAXS><<<grid, cw * 32, k3_cta_smem_bytes(g.count, cw, rows), st>>>(kp);
}

// The half-band stages of the deep main VFOs (subs = false, timed with the ingest class) or sub VFOs (timed with the cascades)
// that their mixing kernel does not run, for callbacks cb0 .. cb0+ncb-1: one k_hb_tail launch, nothing for a plan without them.
static int enqueue_tails(sdrb_bank *b, const CallCtx &c, bool subs, int s0, int ns, cudaStream_t st, int cb0, int ncb, int *nl) {
    const int n = subs ? b->n_sub_tails : b->n_main_tails, tiles = subs ? b->sub_tail_tiles : b->main_tail_tiles;
    if (n == 0) return SDRB_OK;
    TimedScope t(b, st, subs ? 2 : 1);
    const dim3 grid((unsigned)ns, (unsigned)(n * tiles), (unsigned)ncb);
    const TailDev *devs = (const TailDev *)(subs ? b->sub_tails.p : b->main_tails.p);
    if (c.map) k_hb_tail<true><<<grid, TAIL_NT, V2L<TAIL_NT>::SMEM, st>>>(devs, tiles, s0, cb0, c.map);
    else k_hb_tail<<<grid, TAIL_NT, V2L<TAIL_NT>::SMEM, st>>>(devs, tiles, s0, cb0);
    (*nl)++;
    return SDRB_OK;
}

// Sub-VFO cascades of callbacks cb0 .. cb0+ncb-1 (and the tails of the deep ones).
static int enqueue_subs(sdrb_bank *b, const CallCtx &c, int s0, int ns, cudaStream_t st, int cb0, int ncb, int *nl) {
    for (const SubGroup &g : b->groups) {
        const size_t gi = (size_t)(&g - b->groups.data());
        if (g.v3) {
            K3Params &kp = b->k3[gi];
            kp.stream0 = s0; kp.stream_end = s0 + ns; kp.b0 = cb0; kp.map = c.map;
            if (b->k3_slots.size() <= gi) { b->k3_slots.resize(gi + 1, -1); b->k3_cw.resize(gi + 1, 0); }
            if (g.v3_maxs == 2) launch_k3<2>(b, gi, ns, ncb, st, c.map != nullptr);
            else if (g.v3_maxs == 3) launch_k3<3>(b, gi, ns, ncb, st, c.map != nullptr);
            else launch_k3<5>(b, gi, ns, ncb, st, c.map != nullptr);
            (*nl)++;
            continue;
        }
        K2V2Params &kp = b->k2v2[gi];
        kp.stream0 = s0; kp.b0 = cb0; kp.map = c.map;
        TimedScope t(b, st, 2);
        const dim3 grid((unsigned)ns, (unsigned)g.tiles, (unsigned)ncb);
        if (c.map) {
            if (g.ragged) {
                if (g.threads == 64) k2a_v2<64, true, true><<<grid, 64, V2L<64>::SMEM, st>>>(kp);
                else if (g.threads == 96) k2a_v2<96, true, true><<<grid, 96, V2L<96>::SMEM, st>>>(kp);
                else k2a_v2<128, true, true><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
            } else if (g.threads == 64) k2a_v2<64, false, true><<<grid, 64, V2L<64>::SMEM, st>>>(kp);
            else if (g.threads == 96) k2a_v2<96, false, true><<<grid, 96, V2L<96>::SMEM, st>>>(kp);
            else k2a_v2<128, false, true><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
        } else if (g.ragged) {
            if (g.threads == 64) k2a_v2<64, true><<<grid, 64, V2L<64>::SMEM, st>>>(kp);
            else if (g.threads == 96) k2a_v2<96, true><<<grid, 96, V2L<96>::SMEM, st>>>(kp);
            else k2a_v2<128, true><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
        } else if (g.threads == 64) k2a_v2<64><<<grid, 64, V2L<64>::SMEM, st>>>(kp);
        else if (g.threads == 96) k2a_v2<96><<<grid, 96, V2L<96>::SMEM, st>>>(kp);
        else k2a_v2<128><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
        (*nl)++;
    }
    return enqueue_tails(b, c, true, s0, ns, st, cb0, ncb, nl);
}

// /late FIR and USB audio of callbacks cb0 .. cb0+ncb-1. `out_done` (optional) is recorded at the end.
static int enqueue_audio(sdrb_bank *b, const CallCtx &c, int s0, int ns, cudaStream_t st, int cb0, int ncb, cudaEvent_t out_done,
                         int *nl) {
    const HostPlan &h = b->plan->h;
    if (b->n_late) {
        TimedScope t(b, st, 3);
        if (b->late_factor == 5 || b->late_factor == 6) {           // every late VFO of the plan divides by the same 5 or 6
            const dim3 grid((unsigned)ns, (unsigned)b->n_late, (unsigned)((ncb * b->max_late_samples + LV_TILE - 1) / LV_TILE));
            // late_taps_per_phase: the reference's 49-tap /5 and 73-tap /6 filters get their tap loops at compile time
            const LateDev *ld = (const LateDev *)b->latedev.p;
            if (c.map) {
                if (b->late_factor == 5 && b->late_taps_per_phase == 10) k2_late_v2<5, 10, true><<<grid, LV_THREADS, lv_smem<5>(), st>>>(ld, cb0, ncb, s0, c.map);
                else if (b->late_factor == 5) k2_late_v2<5, 0, true><<<grid, LV_THREADS, lv_smem<5>(), st>>>(ld, cb0, ncb, s0, c.map);
                else if (b->late_taps_per_phase == 13) k2_late_v2<6, 13, true><<<grid, LV_THREADS, lv_smem<6>(), st>>>(ld, cb0, ncb, s0, c.map);
                else k2_late_v2<6, 0, true><<<grid, LV_THREADS, lv_smem<6>(), st>>>(ld, cb0, ncb, s0, c.map);
            } else if (b->late_factor == 5 && b->late_taps_per_phase == 10) k2_late_v2<5, 10><<<grid, LV_THREADS, lv_smem<5>(), st>>>(ld, cb0, ncb, s0);
            else if (b->late_factor == 5) k2_late_v2<5, 0><<<grid, LV_THREADS, lv_smem<5>(), st>>>(ld, cb0, ncb, s0);
            else if (b->late_taps_per_phase == 13) k2_late_v2<6, 13><<<grid, LV_THREADS, lv_smem<6>(), st>>>(ld, cb0, ncb, s0);
            else k2_late_v2<6, 0><<<grid, LV_THREADS, lv_smem<6>(), st>>>(ld, cb0, ncb, s0);
        } else {
            const int tiles = (ncb * b->max_late_samples + LATE_TILE - 1) / LATE_TILE;
            const dim3 grid((unsigned)ns, (unsigned)b->n_late, (unsigned)tiles);
            if (c.map) k2_late_fir<true><<<grid, LATE_TILE, 0, st>>>((const LateDev *)b->latedev.p, cb0, ncb, s0, c.map);
            else k2_late_fir<<<grid, LATE_TILE, 0, st>>>((const LateDev *)b->latedev.p, cb0, ncb, s0);
        }
        (*nl)++;
    }
    if (b->n_usb) {
        K2bV2Params up;
        up.devs = (const UsbDev *)b->usbdev.p; up.pcm = c.d_pcm; up.tap = c.d_tap;
        up.n_blocks = c.n_blocks; up.cb0 = cb0; up.ncb = ncb; up.stream0 = s0; up.stream_end = s0 + ns;
        up.pcm_per_block = h.pcm_per_block; up.warp_floats = b->uv_warp_floats; up.eo_rows = b->uv_eo_rows;
        up.np_max = b->uv_np_max; up.map = c.map;
        int max_tiles = 0;
        for (size_t k = 0; k < b->uv_vfo_out.size() && k < (size_t)SDRB_MAX_SUB; k++) {
            const int tile_out = UV_USB - b->uv_vfo_np[k];
            const int tiles = (ncb * b->uv_vfo_out[k] + tile_out - 1) / tile_out;
            up.tiles[k] = (unsigned short)tiles;
            max_tiles = std::max(max_tiles, tiles);
        }
        TimedScope t(b, st, 4);
        const dim3 grid((unsigned)((ns + UV_WARPS - 1) / UV_WARPS), (unsigned)b->n_usb, (unsigned)max_tiles);
        if (c.map) k2b_v2<true><<<grid, UV_WARPS * 32, b->uv_smem, st>>>(up);
        else k2b_v2<<<grid, UV_WARPS * 32, b->uv_smem, st>>>(up);
        (*nl)++;
    }
    if (out_done) CU_TRY(cudaEventRecord(out_done, st));
    return SDRB_OK;
}

// Everything after the DC stage for callback cb: ingest + main VFOs, sub-VFO cascades, /late FIR,
// USB audio. `wait` (optional) gates the first kernel; `out_done` (optional) is recorded at the end.
static int enqueue_main_cb(sdrb_bank *b, const CallCtx &c, int s0, int ns, cudaStream_t st, int cb, cudaEvent_t wait,
                           cudaEvent_t out_done, int *nl) {
    int rc;
    if ((rc = enqueue_ingest_cb(b, c, s0, ns, st, cb, wait, nl)) != SDRB_OK) return rc;
    if ((rc = enqueue_tails(b, c, false, s0, ns, st, cb, 1, nl)) != SDRB_OK) return rc;
    if ((rc = enqueue_subs(b, c, s0, ns, st, cb, 1, nl)) != SDRB_OK) return rc;
    return enqueue_audio(b, c, s0, ns, st, cb, 1, out_done, nl);
}

// End of a call: filter tails, raw tail and callback counters for the next call.
static int enqueue_carry(sdrb_bank *b, const CallCtx &c, int s0, int ns, cudaStream_t st, int *nl) {
    const HostPlan &h = b->plan->h;
    const bool dc = h.correct_dc && !c.d_cf;
    if (dc && c.map) {
        // Every stream's DC halo moves from the buffer this call read (par) to the one the next call reads (par ^ 1); k3_carry then
        // overwrites it for the listed streams. Without this an unlisted stream would find in its next call the halo of the call
        // before its last one. Entries 0 .. DC_HALO_BLKS-1 of a stream are never written by the DC walk, so this does not race with
        // a next call's DC pre-pass that already runs on table_buf(par ^ 1).
        const size_t pitch = (size_t)(b->dc_stride + DC_HALO_BLKS) * 2 * sizeof(uint2);
        CU_TRY(cudaMemcpy2DAsync(b->table_buf(c.par ^ 1), pitch, b->table_buf(c.par), pitch, 2 * DC_HALO_BLKS * sizeof(uint2),
                                 (size_t)b->n_streams, cudaMemcpyDeviceToDevice, st));
    }
    TimedScope t(b, st, 5);
    const dim3 grid((unsigned)ns, (unsigned)(b->n_carry + 1));
    if (c.map)
        k3_carry<true><<<grid, 128, 0, st>>>(
            (const CarryItem *)b->carry.p, b->n_carry, c.n_blocks, c.d_iq, c.iq_stride, h.block, (uint8_t *)b->raw_tail.p,
            (long long *)b->blocks_done.p, dc ? b->table_buf(c.par) : nullptr, b->table_buf(c.par ^ 1), b->anchor_buf(c.par),
            b->dc_stride + DC_HALO_BLKS, c.n_blocks * (h.block / DC_BLK), s0, c.d_cf, c.cf_stride, (float2 *)b->cf_tail.p, c.map);
    else
        k3_carry<<<grid, 128, 0, st>>>(
            (const CarryItem *)b->carry.p, b->n_carry, c.n_blocks, c.d_iq, c.iq_stride, h.block, (uint8_t *)b->raw_tail.p,
            (long long *)b->blocks_done.p, dc ? b->table_buf(c.par) : nullptr, b->table_buf(c.par ^ 1), b->anchor_buf(c.par),
            b->dc_stride + DC_HALO_BLKS, c.n_blocks * (h.block / DC_BLK), s0, c.d_cf, c.cf_stride, (float2 *)b->cf_tail.p);
    (*nl)++;
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

// Whole call for all streams of the bank, or for the streams c.h_map lists, on one stream (device-resident entry points): the DC
// walk of callback cb+1 runs on the side stream while callback cb is filtered.
// `input_ready` (optional cudaEvent_t): the input of this call is valid once that event has fired.
// The DC pre-pass then waits only for it (and for the call before the previous one, whose table
// buffer it reuses) instead of for everything queued on `st` -- it overlaps the previous call.
static int enqueue_all(sdrb_bank *b, CallCtx &c, cudaStream_t st, int *launches, cudaEvent_t input_ready = nullptr) {
    const HostPlan &h = b->plan->h;
    const bool dc = h.correct_dc && !c.d_cf;
    const int ns = c.h_map ? c.n_map : b->n_streams;
    int rc;
    c.par = b->dc_par;
    b->last_iq = c.d_iq; b->last_iq_stride = c.iq_stride; b->last_cf = c.d_cf; b->last_cf_stride = c.cf_stride;
    b->last_blocks = c.n_blocks; b->last_par = c.par;
    b->last_map = c.h_map ? b->list_buf(c.par) : nullptr; b->last_n = ns;
    if (b->state_pending) {             // a save or load since the last call: the DC pre-pass and the filters come after it
        CU_TRY(cudaStreamWaitEvent(st, b->ev_state, 0));
        if (dc) CU_TRY(cudaStreamWaitEvent(b->s_dc[0], b->ev_state, 0));
        b->state_pending = false;
    }
    if (c.h_map) {
        // the list goes where the call's first kernel runs; the call two before this one, which read the same buffer, must be over
        cudaStream_t first = dc ? b->s_dc[0] : st;
        if (dc && b->ev_end_valid[c.par]) CU_TRY(cudaStreamWaitEvent(first, b->ev_end[c.par], 0));
        // without a DC pre-pass the first kernel reads d_iq on `st`: it waits for input_ready there (a DC plan's side stream does below)
        if (!dc && input_ready) CU_TRY(cudaStreamWaitEvent(st, input_ready, 0));
        const std::vector<int> list(c.h_map, c.h_map + ns);  // pageable: staged before cudaMemcpyAsync returns, the caller may reuse it
        CU_TRY(cudaMemcpyAsync(b->list_buf(c.par), list.data(), sizeof(int) * (size_t)ns, cudaMemcpyHostToDevice, first));
        c.map = b->list_buf(c.par);
        if (dc) {                       // the filters on `st` read the list too
            CU_TRY(cudaEventRecord(b->ev_entry[1], first));
            CU_TRY(cudaStreamWaitEvent(st, b->ev_entry[1], 0));
        }
    }
    if (dc) {
        cudaStream_t sd = b->s_dc[0];
        if (input_ready) {
            CU_TRY(cudaStreamWaitEvent(sd, input_ready, 0));
            if (b->ev_end_valid[c.par]) CU_TRY(cudaStreamWaitEvent(sd, b->ev_end[c.par], 0));
        } else {
            CU_TRY(cudaEventRecord(b->ev_entry[0], st));         // everything queued before this call
            CU_TRY(cudaStreamWaitEvent(sd, b->ev_entry[0], 0));
        }
        for (int cb = 0; cb < c.n_blocks; cb++) {
            if (b->dbg_only == 2 && b->ev_end_valid[0] && b->ev_end_valid[1]) {      // filters only: reuse the tables of the first two calls
                CU_TRY(cudaEventRecord(b->ev_dc[0][(size_t)cb], sd));
                continue;
            }
            if ((rc = enqueue_dc_cb(b, c, 0, ns, sd, cb, nullptr, b->ev_dc[0][(size_t)cb], launches)) != SDRB_OK) return rc;
        }
    }
    if (b->dbg_only == 1) {
        for (int cb = 0; cb < c.n_blocks; cb++) CU_TRY(cudaStreamWaitEvent(st, b->ev_dc[0][(size_t)cb], 0));
    } else if (b->per_cb) {
        for (int cb = 0; cb < c.n_blocks; cb++)
            if ((rc = enqueue_main_cb(b, c, 0, ns, st, cb, dc ? b->ev_dc[0][(size_t)cb] : nullptr, nullptr, launches)) != SDRB_OK)
                return rc;
    } else {
        // kernel class by kernel class over all callbacks of the call: the sub-VFO warps of k2a_v3 walk long spans
        // (their warm-up tiles amortise), and the DC walk of the next call has the whole cascade/audio phase to hide in
        for (int cb = 0; cb < c.n_blocks; cb++)
            if ((rc = enqueue_ingest_cb(b, c, 0, ns, st, cb, dc ? b->ev_dc[0][(size_t)cb] : nullptr, launches)) != SDRB_OK) return rc;
        if ((rc = enqueue_tails(b, c, false, 0, ns, st, 0, c.n_blocks, launches)) != SDRB_OK) return rc;
        if ((rc = enqueue_subs(b, c, 0, ns, st, 0, c.n_blocks, launches)) != SDRB_OK) return rc;
        if ((rc = enqueue_audio(b, c, 0, ns, st, 0, c.n_blocks, nullptr, launches)) != SDRB_OK) return rc;
    }
    if ((rc = enqueue_carry(b, c, 0, ns, st, launches)) != SDRB_OK) return rc;
    if (dc) {
        CU_TRY(cudaEventRecord(b->ev_end[c.par], st));
        b->ev_end_valid[c.par] = true;
    }
    b->dc_par ^= 1;
    if (!b->ev_device_tail) CU_TRY(cudaEventCreateWithFlags(&b->ev_device_tail, cudaEventDisableTiming));
    CU_TRY(cudaEventRecord(b->ev_device_tail, st));
    b->device_tail_pending = true;
    return SDRB_OK;
}

TimedScope::TimedScope(sdrb_bank *b_, cudaStream_t st_, int cls_) : b(b_), st(st_), cls(cls_), on(b_->timing) {
    if (!on) return;
    if (b->tev_used + 2 > b->tev.size()) {
        for (int k = 0; k < 2; k++) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) { on = false; return; }
            b->tev.push_back(e);
        }
        b->tev_cls.resize(b->tev.size() / 2);
    }
    b->tev_cls[b->tev_used / 2] = cls;
    cudaEventRecord(b->tev[b->tev_used], st);
}
TimedScope::~TimedScope() {
    if (!on) return;
    cudaEventRecord(b->tev[b->tev_used + 1], st);
    b->tev_used += 2;
}

extern "C" int sdrb_bank_set_timing(sdrb_bank *b, int on) {
    if (!b) { set_error("sdrb_bank_set_timing: NULL bank"); return SDRB_E_INVALID; }
    b->timing = on != 0;
    b->tev_used = 0;
    for (int k = 0; k < SDRB_N_KERNEL_CLASSES; k++) { b->kernel_ms[k] = 0; b->kernel_calls[k] = 0; }
    return SDRB_OK;
}

extern "C" int sdrb_bank_kernel_times(sdrb_bank *b, double *ms, long *calls) {
    if (!b || !ms) { set_error("sdrb_bank_kernel_times: NULL argument"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(b->device));
    CU_TRY(cudaDeviceSynchronize());
    for (size_t c = 0; c + 2 <= b->tev_used; c += 2) {
        float t = 0.f;
        const int k = b->tev_cls[c / 2];
        if (cudaEventElapsedTime(&t, b->tev[c], b->tev[c + 1]) == cudaSuccess) {
            b->kernel_ms[k] += t;
            b->kernel_calls[k] += 1;
        }
    }
    b->tev_used = 0;
    for (int k = 0; k < SDRB_N_KERNEL_CLASSES; k++) { ms[k] = b->kernel_ms[k]; if (calls) calls[k] = b->kernel_calls[k]; }
    return SDRB_OK;
}

static int check_process_args(sdrb_bank *b, const void *iq, size_t iq_stride, int n_blocks, const void *pcm) {
    if (!b || !iq || !pcm) { set_error("process: NULL argument"); return SDRB_E_INVALID; }
    if (n_blocks <= 0 || n_blocks > b->max_blocks) { set_error("process: n_blocks outside 1..max_blocks"); return SDRB_E_INVALID; }
    const size_t need = (size_t)n_blocks * (size_t)b->plan->h.block * 2;
    if (iq_stride < need || iq_stride % 16 != 0 || ((uintptr_t)iq) % 16 != 0) {
        set_error("process: iq_stride must be >= n_blocks*block*2 and, like the base pointer, 16-byte aligned");
        return SDRB_E_INVALID;
    }
    return SDRB_OK;
}

// A list of n distinct streams of the bank (state records, stream-list calls) and the buffer that goes with it.
static int check_stream_list(const sdrb_bank *b, const int32_t *streams, int n, const void *data, const char *who) {
    if (!b || !streams || !data) { set_error(std::string(who) + ": NULL argument"); return SDRB_E_INVALID; }
    if (n <= 0 || n > b->n_streams) { set_error(std::string(who) + ": n must be 1..n_streams"); return SDRB_E_INVALID; }
    std::vector<char> seen((size_t)b->n_streams, 0);
    for (int k = 0; k < n; k++) {
        const int s = streams[k];
        const char *bad = (s < 0 || s >= b->n_streams) ? "is outside 0..n_streams-1" : (seen[(size_t)s] ? "is listed twice" : nullptr);
        if (bad) { set_error(std::string(who) + ": streams[" + std::to_string(k) + "] = " + std::to_string(s) + " " + bad); return SDRB_E_INVALID; }
        seen[(size_t)s] = 1;
    }
    return SDRB_OK;
}

extern "C" int sdrb_bank_process_device_ex(sdrb_bank *b, const uint8_t *d_iq, size_t iq_stride, int n_blocks,
                                           int16_t *d_pcm, float *d_tap, void *cuda_stream, void *input_ready_event) {
    int rc = check_process_args(b, d_iq, iq_stride, n_blocks, d_pcm);
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    b->last_launches = 0;
    CallCtx c;
    c.d_iq = d_iq; c.iq_stride = iq_stride; c.n_blocks = n_blocks; c.d_pcm = d_pcm; c.d_tap = d_tap;
    return enqueue_all(b, c, (cudaStream_t)cuda_stream, &b->last_launches, (cudaEvent_t)input_ready_event);
}

extern "C" int sdrb_bank_process_device(sdrb_bank *b, const uint8_t *d_iq, size_t iq_stride, int n_blocks,
                                        int16_t *d_pcm, float *d_tap, void *cuda_stream) {
    return sdrb_bank_process_device_ex(b, d_iq, iq_stride, n_blocks, d_pcm, d_tap, cuda_stream, nullptr);
}

extern "C" int sdrb_bank_process_streams_device(sdrb_bank *b, const int32_t *streams, int n, const uint8_t *d_iq, size_t iq_stride,
                                                int n_blocks, int16_t *d_pcm, float *d_tap, void *cuda_stream, void *input_ready_event) {
    int rc = check_stream_list(b, streams, n, d_iq, "sdrb_bank_process_streams_device");
    if (rc != SDRB_OK || (rc = check_process_args(b, d_iq, iq_stride, n_blocks, d_pcm)) != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    if ((rc = host_drain(b)) != SDRB_OK) return rc;
    b->last_launches = 0;
    CallCtx c;
    c.d_iq = d_iq; c.iq_stride = iq_stride; c.n_blocks = n_blocks; c.d_pcm = d_pcm; c.d_tap = d_tap;
    c.h_map = streams; c.n_map = n;
    return enqueue_all(b, c, (cudaStream_t)cuda_stream, &b->last_launches, (cudaEvent_t)input_ready_event);
}

extern "C" int sdrb_bank_copy_main(sdrb_bank *b, int main_idx, int n_blocks, float *d_out, void *cuda_stream) {
    if (!b || !d_out || main_idx < 0 || main_idx >= (int)b->plan->h.mains.size() || n_blocks <= 0 || n_blocks > b->max_blocks) {
        set_error("sdrb_bank_copy_main: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const MainVfo &m = b->plan->h.mains[(size_t)main_idx];
    // The carry kernel has already moved the tail to the front, but the body is intact.
    const size_t row = (size_t)n_blocks * m.block_out * sizeof(float2);
    CU_TRY(cudaMemcpy2DAsync(d_out, row, (float2 *)b->main_out.p + b->main_off[(size_t)main_idx] + MAIN_HIST,
                             b->main_stride * sizeof(float2), row, (size_t)b->n_streams, cudaMemcpyDeviceToDevice,
                             (cudaStream_t)cuda_stream));
    return SDRB_OK;
}

// vfo::compress (vfo.cpp:389-424) of a main VFO's output of the last call, straight from main_out.
static int forward_launch(sdrb_bank *b, int main_idx, int n_blocks, uint8_t *d_out, cudaStream_t st) {
    const MainVfo &m = b->plan->h.mains[(size_t)main_idx];
    const int n = n_blocks * m.block_out;
    const int per = m.compress_style == 1 ? 1 : 2;
    k_compress<<<dim3((unsigned)(((n + 3) / 4 + 255) / 256), (unsigned)b->n_streams), 256, 0, st>>>(
        (const float2 *)b->main_out.p + b->main_off[(size_t)main_idx] + MAIN_HIST, (long long)b->main_stride, d_out,
        (long long)n * per, n, (float)m.compress_scale, m.compress_style);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

extern "C" int sdrb_bank_copy_forward(sdrb_bank *b, int main_idx, int n_blocks, uint8_t *d_out, void *cuda_stream) {
    if (!b || !d_out || main_idx < 0 || main_idx >= (int)b->plan->h.mains.size() || n_blocks <= 0 || n_blocks > b->max_blocks) {
        set_error("sdrb_bank_copy_forward: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    return forward_launch(b, main_idx, n_blocks, d_out, (cudaStream_t)cuda_stream);
}

extern "C" int sdrb_bank_read_forward(sdrb_bank *b, int main_idx, int n_blocks, uint8_t *h_out) {
    if (!b || !h_out || main_idx < 0 || main_idx >= (int)b->plan->h.mains.size() || n_blocks <= 0 || n_blocks > b->max_blocks) {
        set_error("sdrb_bank_read_forward: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const MainVfo &m = b->plan->h.mains[(size_t)main_idx];
    const size_t bytes = (size_t)b->n_streams * (size_t)n_blocks * (size_t)m.fwd_bytes;
    if (b->d_fwd.bytes < bytes) {
        b->d_fwd.release(); b->d_fwd.bytes = 0;
        int rc = b->d_fwd.alloc((size_t)b->n_streams * (size_t)b->max_blocks * (size_t)m.fwd_bytes); if (rc) return rc;
    }
    cudaStream_t st = b->s_compute;
    int rc = forward_launch(b, main_idx, n_blocks, (uint8_t *)b->d_fwd.p, st);
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaMemcpyAsync(h_out, b->d_fwd.p, bytes, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return SDRB_OK;
}

extern "C" int sdrb_compress_iq(const float *d_in, uint8_t *d_out, int n_ch, int n, int scale, int style, void *cuda_stream) {
    if (!d_in || !d_out || n_ch <= 0 || n <= 0) { set_error("sdrb_compress_iq: bad argument"); return SDRB_E_INVALID; }
    if (scale <= 0) scale = 1;
    const int per = style == 1 ? 1 : 2;
    k_compress<<<dim3((unsigned)(((n + 3) / 4 + 255) / 256), (unsigned)n_ch), 256, 0, (cudaStream_t)cuda_stream>>>(
        (const float2 *)d_in, (long long)n, d_out, (long long)n * per, n, (float)scale, style);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

// sdrj::demodData's `samples` (sdrj.cpp:271-294) of callback cb of the last call, first n samples.
static int input_launch(sdrb_bank *b, int cb, int n, float2 *d_out, cudaStream_t st) {
    const HostPlan &h = b->plan->h;
    if (b->last_cf) {
        CU_TRY(cudaMemcpy2DAsync(d_out, (size_t)n * sizeof(float2), b->last_cf + (size_t)cb * h.block, b->last_cf_stride * sizeof(float2),
                                 (size_t)n * sizeof(float2), (size_t)b->n_streams, cudaMemcpyDeviceToDevice, st));
        return SDRB_OK;
    }
    const bool dc = h.correct_dc != 0;
    const dim3 grid((unsigned)((n / DC_BLK + 63) / 64), (unsigned)(b->last_map ? b->last_n : b->n_streams));
    if (b->last_map)                    // a stream-list call: the rows of its streams
        k_input_samples<true><<<grid, 64, 0, st>>>(b->last_iq, b->last_iq_stride, (size_t)cb * h.block, n,
                                                   dc ? b->table_buf(b->last_par) : nullptr, b->anchor_buf(b->last_par),
                                                   b->dc_stride + DC_HALO_BLKS, cb * (h.block / DC_BLK), d_out, b->last_map);
    else
        k_input_samples<<<grid, 64, 0, st>>>(b->last_iq, b->last_iq_stride, (size_t)cb * h.block, n, dc ? b->table_buf(b->last_par) : nullptr,
                                             b->anchor_buf(b->last_par), b->dc_stride + DC_HALO_BLKS, cb * (h.block / DC_BLK), d_out);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

static int check_input_args(sdrb_bank *b, int cb, int n, const void *out, const char *who) {
    if (!b || !out || !(b->last_iq || b->last_cf) || cb < 0 || cb >= b->last_blocks || n <= 0 || n > b->plan->h.block || n % DC_BLK != 0) {
        set_error(std::string(who) + ": needs a previous process call, 0 <= cb < its n_blocks and n a multiple of 128 up to the callback size");
        return SDRB_E_INVALID;
    }
    return SDRB_OK;
}

extern "C" int sdrb_bank_copy_input(sdrb_bank *b, int cb, int n, float *d_out, void *cuda_stream) {
    int rc = check_input_args(b, cb, n, d_out, "sdrb_bank_copy_input");
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    return input_launch(b, cb, n, (float2 *)d_out, (cudaStream_t)cuda_stream);
}

// z (decimate[decimateCount], vfo.cpp:290-293) of a sub VFO whose mix is fused into the /late kernel: produced here, on demand,
// for the callbacks of the last call -- the parent's output of that call is still in place, the callback counters have moved on.
static int ensure_sub_z(sdrb_bank *b, int sub_idx, cudaStream_t st) {
    if (!b->sub_fused[(size_t)sub_idx] || b->last_blocks <= 0) return SDRB_OK;
    const SubVfo &s = b->plan->h.subs[(size_t)sub_idx];
    K2V2Params kp{};
    kp.vfos[0] = b->sub_casc[(size_t)sub_idx];
    kp.rf[0] = b->sub_rf[(size_t)sub_idx];
    kp.in = (const float2 *)b->main_out.p + b->main_off[(size_t)s.main_idx];
    kp.blocks_done = (const long long *)b->blocks_done.p;
    kp.in_stride = (long long)b->main_stride; kp.out_stride = (long long)b->z_stride;
    kp.count = 1; kp.lut_len = (int)s.lut.size(); kp.block_in = s.block_in; kp.HT = 0; kp.stream0 = 0; kp.b0 = 0;
    kp.blk_off = -b->last_blocks;
    kp.map = b->last_map;
    const int tiles = (s.block_in + 128 * V2_CHUNK - 1) / (128 * V2_CHUNK);
    const dim3 grid((unsigned)(b->last_map ? b->last_n : b->n_streams), (unsigned)tiles, (unsigned)b->last_blocks);
    if (b->last_map) {                  // after a stream-list call only its streams have the counters the replay subtracts from
        if (s.block_in % V2_CHUNK != 0) k2a_v2<128, true, true><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
        else k2a_v2<128, false, true><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
    } else if (s.block_in % V2_CHUNK != 0) k2a_v2<128, true><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
    else k2a_v2<128><<<grid, 128, V2L<128>::SMEM, st>>>(kp);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

extern "C" int sdrb_bank_copy_sub(sdrb_bank *b, int sub_idx, int n_blocks, float *d_out, void *cuda_stream) {
    if (!b || !d_out || sub_idx < 0 || sub_idx >= (int)b->plan->h.subs.size() || n_blocks <= 0 || n_blocks > b->max_blocks) {
        set_error("sdrb_bank_copy_sub: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const SubVfo &s = b->plan->h.subs[(size_t)sub_idx];
    const size_t row = (size_t)n_blocks * s.block_z * sizeof(float2);
    { const int zrc = ensure_sub_z(b, sub_idx, (cudaStream_t)cuda_stream); if (zrc != SDRB_OK) return zrc; }
    CU_TRY(cudaMemcpy2DAsync(d_out, row, (float2 *)b->zbuf.p + b->sub_z_off[(size_t)sub_idx] + b->sub_z_hist[(size_t)sub_idx],
                             b->z_stride * sizeof(float2), row, (size_t)b->n_streams, cudaMemcpyDeviceToDevice,
                             (cudaStream_t)cuda_stream));
    return SDRB_OK;
}

// Host variants for the C++ facades: device scratch, copy, synchronise.
static int read_back(sdrb_bank *b, size_t bytes, void *h_out, const std::function<int(void *, cudaStream_t)> &fill) {
    void *tmp = nullptr;
    CU_TRY(cudaMalloc(&tmp, bytes ? bytes : 16));
    int rc = fill(tmp, b->s_compute);
    cudaError_t e = cudaSuccess;
    if (rc == SDRB_OK) e = cudaMemcpyAsync(h_out, tmp, bytes, cudaMemcpyDeviceToHost, b->s_compute);
    cudaStreamSynchronize(b->s_compute);
    cudaFree(tmp);
    if (rc == SDRB_OK && e != cudaSuccess) { set_error(std::string("read back: ") + cudaGetErrorString(e)); rc = SDRB_E_CUDA; }
    return rc;
}

extern "C" int sdrb_bank_read_input(sdrb_bank *b, int cb, int n, float *h_out) {
    int rc = check_input_args(b, cb, n, h_out, "sdrb_bank_read_input");
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    return read_back(b, (size_t)b->n_streams * (size_t)n * sizeof(float2), h_out,
                     [&](void *d, cudaStream_t st) { return input_launch(b, cb, n, (float2 *)d, st); });
}

extern "C" int sdrb_bank_read_sub(sdrb_bank *b, int sub_idx, int n_blocks, float *h_out) {
    if (!b || !h_out || sub_idx < 0 || sub_idx >= (int)b->plan->h.subs.size() || n_blocks <= 0 || n_blocks > b->max_blocks) {
        set_error("sdrb_bank_read_sub: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const size_t bytes = (size_t)b->n_streams * (size_t)n_blocks * (size_t)b->plan->h.subs[(size_t)sub_idx].block_z * sizeof(float2);
    return read_back(b, bytes, h_out, [&](void *d, cudaStream_t st) { return sdrb_bank_copy_sub(b, sub_idx, n_blocks, (float *)d, st); });
}

extern "C" int sdrb_bank_copy_dc_trace(sdrb_bank *b, int n_blocks, float *d_out, uint8_t *d_modes, void *cuda_stream) {
    if (!b || !d_out || n_blocks <= 0 || n_blocks > b->max_blocks || !b->plan->h.correct_dc) {
        set_error("sdrb_bank_copy_dc_trace: bad argument or plan without correct_dc_bias"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const int n = n_blocks * (b->plan->h.block / DC_BLK);
    dc_trace_gather<<<dim3((unsigned)((n + 255) / 256), (unsigned)b->n_streams), 256, 0, (cudaStream_t)cuda_stream>>>(
        b->table_buf(b->dc_par ^ 1), b->anchor_buf(b->dc_par ^ 1), b->dc_stride + DC_HALO_BLKS, n, (float2 *)d_out,
        d_modes);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

// Waits for every sdrb_bank_process_host_async call still in flight.
static int host_drain(sdrb_bank *b) {
    if (!b->host_inflight) return SDRB_OK;
    CU_TRY(cudaStreamSynchronize(b->s_copy_out));
    CU_TRY(cudaStreamSynchronize(b->s_compute));
    for (cudaEvent_t e : b->host_calls) cudaEventDestroy(e);
    b->host_calls.clear();
    b->host_inflight = false;
    return SDRB_OK;
}

extern "C" int sdrb_bank_host_wait(sdrb_bank *b) {
    if (!b) { set_error("sdrb_bank_host_wait: NULL bank"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(b->device));
    return host_drain(b);
}

// Waits until at most max_in_flight asynchronous host calls are unfinished (oldest first): their
// h_pcm / h_tap are complete and their host buffers may be reused.
extern "C" int sdrb_bank_host_wait_until(sdrb_bank *b, int max_in_flight) {
    if (!b || max_in_flight < 0) { set_error("sdrb_bank_host_wait_until: bad argument"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(b->device));
    if (max_in_flight == 0) return host_drain(b);
    while ((int)b->host_calls.size() > max_in_flight) {
        CU_TRY(cudaEventSynchronize(b->host_calls.front()));
        cudaEventDestroy(b->host_calls.front());
        b->host_calls.pop_front();
    }
    return SDRB_OK;
}

// Device staging of the host entry points: one input row of max_blocks callbacks and one PCM (and tap) record per stream.
static int host_staging(sdrb_bank *b, bool tap) {
    const HostPlan &h = b->plan->h;
    int rc;
    if (!b->d_iq.p) {
        rc = b->d_iq.alloc((size_t)b->max_blocks * h.block * 2 * (size_t)b->n_streams); if (rc) return rc;
        rc = b->d_pcm.alloc((size_t)b->max_blocks * h.pcm_per_block * sizeof(int16_t) * (size_t)b->n_streams); if (rc) return rc;
    }
    if (tap && !b->d_tap.p) {
        rc = b->d_tap.alloc((size_t)b->max_blocks * h.pcm_per_block * sizeof(float) * (size_t)b->n_streams); if (rc) return rc;
    }
    return SDRB_OK;
}

// Enqueues one host call. Consecutive calls may be in flight together (the staging buffers are shared,
// so per chunk: the copy-in of call n+1 waits until call n no longer reads that region, the filters of
// call n+1 wait until call n's copy-out of that region is done).
static int host_enqueue(sdrb_bank *b, const uint8_t *h_iq, size_t iq_stride, int n_blocks, int16_t *h_pcm, float *h_tap) {
    int rc = check_process_args(b, h_iq, iq_stride, n_blocks, h_pcm);
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    if (b->host_inflight && (n_blocks != b->host_inflight_blocks || (h_tap != nullptr) != b->host_inflight_tap)) {
        rc = host_drain(b);                                  // a different chunk layout: do not overlap with it
        if (rc != SDRB_OK) return rc;
    }
    const HostPlan &h = b->plan->h;
    const size_t in_row = (size_t)n_blocks * h.block * 2;
    const size_t rec = (size_t)n_blocks * h.pcm_per_block;
    const size_t in_max = (size_t)b->max_blocks * h.block * 2;
    if ((rc = host_staging(b, h_tap != nullptr)) != SDRB_OK) return rc;
    // Chunks = (callback, stream group), callback-major: copy-in, kernels and copy-out of different
    // chunks overlap on three streams (+ one DC side stream per group); a chunk's kernels start when
    // its copy has landed. Callback-major order gives every group's sequential DC walk the time of
    // the other groups' copies before its next callback arrives.
    // Stream groups: four equal shares by default; SDRB_HOST_GROUPS="w0,w1,.." (at most 8 weights) sets relative sizes,
    // e.g. a small last group shortens the un-overlapped tail (DC walk + filters + copy-out of the final chunk).
    if (b->host_groups.empty()) {
        std::vector<double> w;
        if (const char *e = getenv("SDRB_HOST_GROUPS")) {
            for (const char *p = e; *p && (int)w.size() < sdrb_bank::kSide;) {
                char *end = nullptr;
                const double v = strtod(p, &end);
                if (end == p) break;
                if (v > 0) w.push_back(v);
                p = *end ? end + 1 : end;
            }
        }
        // four equal groups measured best on B200/PCIe Gen5 (tools/host_groups_sweep.py: 8.38 ms per step vs 8.56
        // with eight and 9.07 with two, 128 receivers x 4 callbacks): fewer, larger copies, still a short tail
        if (w.empty()) w.assign((size_t)std::min(b->n_streams, 4), 1.0);
        double tot = 0, acc = 0;
        for (double v : w) tot += v;
        int s0 = 0;
        for (size_t g = 0; g < w.size() && s0 < b->n_streams; g++) {
            acc += w[g];
            int s1 = g + 1 == w.size() ? b->n_streams : (int)llround(acc / tot * b->n_streams);
            s1 = std::min(std::max(s1, s0 + 1), b->n_streams);
            b->host_groups.push_back({s0, s1 - s0});
            s0 = s1;
        }
        if (s0 < b->n_streams) b->host_groups.back().second += b->n_streams - s0;
    }
    const int n_groups = (int)b->host_groups.size();
    const size_t need_ev = (size_t)n_groups * (size_t)b->max_blocks;
    while (b->ev_in.size() < need_ev) {
        cudaEvent_t e1, e2, e3, e4;
        CU_TRY(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&e3, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&e4, cudaEventDisableTiming));
        b->ev_in.push_back(e1); b->ev_done.push_back(e2); b->ev_free.push_back(e3); b->ev_out.push_back(e4);
    }
    const bool chained = b->host_inflight;                  // an earlier call may still be running: honour its events
    if (b->device_tail_pending) {
        // a device-resident call on a caller's stream came before this one: its state updates (carry, counters, DC state)
        // must be complete before any of our internal streams touches the bank
        CU_TRY(cudaStreamWaitEvent(b->s_copy_in, b->ev_device_tail, 0));
        CU_TRY(cudaStreamWaitEvent(b->s_compute, b->ev_device_tail, 0));
        for (int k = 0; k < sdrb_bank::kSide; k++)
            if (b->s_dc[k]) CU_TRY(cudaStreamWaitEvent(b->s_dc[k], b->ev_device_tail, 0));
        b->device_tail_pending = false;
    }
    b->last_launches = 0;
    const size_t cb_in = (size_t)h.block * 2, cb_out = (size_t)h.pcm_per_block;
    const bool dc = h.correct_dc != 0;
    CallCtx c;
    c.d_iq = (const uint8_t *)b->d_iq.p; c.iq_stride = in_max; c.n_blocks = n_blocks;   // kernels index streams absolutely
    c.d_pcm = (int16_t *)b->d_pcm.p; c.d_tap = h_tap ? (float *)b->d_tap.p : nullptr;
    c.par = b->dc_par;
    b->last_iq = c.d_iq; b->last_iq_stride = c.iq_stride; b->last_cf = nullptr; b->last_cf_stride = 0;
    b->last_blocks = n_blocks; b->last_par = c.par; b->last_map = nullptr;
    b->dc_par ^= 1;                                       // host calls order themselves with per-chunk events
    b->ev_end_valid[0] = b->ev_end_valid[1] = false;
    for (int cb = 0; cb < n_blocks; cb++)
        for (int g = 0; g < n_groups; g++) {
            const int s0 = b->host_groups[(size_t)g].first, ns = b->host_groups[(size_t)g].second;
            if (ns <= 0) break;
            // the previous call reads this input region until the filters of the NEXT callback (halo) resp. the carry are done
            if (chained) CU_TRY(cudaStreamWaitEvent(b->s_copy_in, b->ev_free[(size_t)g * b->max_blocks + cb], 0));
            CU_TRY(cudaMemcpy2DAsync((uint8_t *)b->d_iq.p + (size_t)s0 * in_max + (size_t)cb * cb_in, in_max,
                                     h_iq + (size_t)s0 * iq_stride + (size_t)cb * cb_in, iq_stride, cb_in, (size_t)ns,
                                     cudaMemcpyHostToDevice, b->s_copy_in));
            CU_TRY(cudaEventRecord(b->ev_in[(size_t)g * b->max_blocks + cb], b->s_copy_in));
        }
    for (int cb = 0; cb < n_blocks; cb++)
        for (int g = 0; g < n_groups; g++) {
            const int s0 = b->host_groups[(size_t)g].first, ns = b->host_groups[(size_t)g].second;
            if (ns <= 0) break;
            cudaEvent_t ein = b->ev_in[(size_t)g * b->max_blocks + cb], eout = b->ev_done[(size_t)g * b->max_blocks + cb];
            // the previous call's copy-out of this output region must be over before it is rewritten
            if (chained) CU_TRY(cudaStreamWaitEvent(b->s_compute, b->ev_out[(size_t)g * b->max_blocks + cb], 0));
            if (dc && (rc = enqueue_dc_cb(b, c, s0, ns, b->s_dc[g], cb, ein, b->ev_dc[g][(size_t)cb], &b->last_launches)) != SDRB_OK)
                return rc;
            if ((rc = enqueue_main_cb(b, c, s0, ns, b->s_compute, cb, dc ? b->ev_dc[g][(size_t)cb] : ein, eout,
                                      &b->last_launches)) != SDRB_OK)
                return rc;
            if (cb == n_blocks - 1 && (rc = enqueue_carry(b, c, s0, ns, b->s_compute, &b->last_launches)) != SDRB_OK) return rc;
            // input region (cb-1, g) is free once this chunk's filters have run (they read its last samples as halo);
            // region (last, g) once the carry has saved the tail
            if (cb > 0) CU_TRY(cudaEventRecord(b->ev_free[(size_t)g * b->max_blocks + cb - 1], b->s_compute));
            if (cb == n_blocks - 1) CU_TRY(cudaEventRecord(b->ev_free[(size_t)g * b->max_blocks + cb], b->s_compute));
            CU_TRY(cudaStreamWaitEvent(b->s_copy_out, eout, 0));
            const size_t off = (size_t)s0 * rec + (size_t)cb * cb_out;
            CU_TRY(cudaMemcpy2DAsync(h_pcm + off, rec * sizeof(int16_t), (int16_t *)b->d_pcm.p + off, rec * sizeof(int16_t),
                                     cb_out * sizeof(int16_t), (size_t)ns, cudaMemcpyDeviceToHost, b->s_copy_out));
            if (h_tap)
                CU_TRY(cudaMemcpy2DAsync(h_tap + off, rec * sizeof(float), (float *)b->d_tap.p + off, rec * sizeof(float),
                                         cb_out * sizeof(float), (size_t)ns, cudaMemcpyDeviceToHost, b->s_copy_out));
            CU_TRY(cudaEventRecord(b->ev_out[(size_t)g * b->max_blocks + cb], b->s_copy_out));
        }
    {
        cudaEvent_t done;                                    // the copy-out stream is FIFO: this marks the call's last result
        CU_TRY(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
        CU_TRY(cudaEventRecord(done, b->s_copy_out));
        b->host_calls.push_back(done);
    }
    b->host_inflight = true;
    b->host_inflight_blocks = n_blocks;
    b->host_inflight_tap = h_tap != nullptr;
    return SDRB_OK;
}

extern "C" int sdrb_bank_process_host_async(sdrb_bank *b, const uint8_t *h_iq, size_t iq_stride, int n_blocks,
                                            int16_t *h_pcm, float *h_tap) {
    return host_enqueue(b, h_iq, iq_stride, n_blocks, h_pcm, h_tap);
}

extern "C" int sdrb_bank_process_host(sdrb_bank *b, const uint8_t *h_iq, size_t iq_stride, int n_blocks,
                                      int16_t *h_pcm, float *h_tap) {
    int rc = host_enqueue(b, h_iq, iq_stride, n_blocks, h_pcm, h_tap);
    if (rc != SDRB_OK) return rc;
    return host_drain(b);
}

// The stream-list call from host memory: each listed row into the staging row of its stream, the device-resident call on the
// compute stream, each record back into its compact place. Synchronous.
extern "C" int sdrb_bank_process_streams_host(sdrb_bank *b, const int32_t *streams, int n, const uint8_t *const *h_iq, int n_blocks,
                                              int16_t *h_pcm, float *h_tap) {
    static const char *who = "sdrb_bank_process_streams_host";
    int rc = check_stream_list(b, streams, n, h_iq, who);
    if (rc != SDRB_OK) return rc;
    if (!h_pcm) { set_error(std::string(who) + ": NULL argument"); return SDRB_E_INVALID; }
    if (n_blocks <= 0 || n_blocks > b->max_blocks) { set_error(std::string(who) + ": n_blocks outside 1..max_blocks"); return SDRB_E_INVALID; }
    for (int k = 0; k < n; k++)
        if (!h_iq[k]) { set_error(std::string(who) + ": h_iq[" + std::to_string(k) + "] is NULL"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(b->device));
    if ((rc = host_drain(b)) != SDRB_OK || (rc = host_staging(b, h_tap != nullptr)) != SDRB_OK) return rc;
    const HostPlan &h = b->plan->h;
    const size_t in_max = (size_t)b->max_blocks * h.block * 2, row = (size_t)n_blocks * h.block * 2;
    const size_t rec = (size_t)n_blocks * h.pcm_per_block;
    cudaStream_t st = b->s_compute;
    if (b->device_tail_pending) CU_TRY(cudaStreamWaitEvent(st, b->ev_device_tail, 0));   // the staging rows and the state it updates
    for (int k = 0; k < n; k++)
        CU_TRY(cudaMemcpyAsync((uint8_t *)b->d_iq.p + (size_t)streams[k] * in_max, h_iq[k], row, cudaMemcpyHostToDevice, st));
    b->last_launches = 0;
    CallCtx c;
    c.d_iq = (const uint8_t *)b->d_iq.p; c.iq_stride = in_max; c.n_blocks = n_blocks;
    c.d_pcm = (int16_t *)b->d_pcm.p; c.d_tap = h_tap ? (float *)b->d_tap.p : nullptr;
    c.h_map = streams; c.n_map = n;
    if ((rc = enqueue_all(b, c, st, &b->last_launches)) != SDRB_OK) return rc;
    for (int k = 0; k < n; k++) {
        const size_t at = (size_t)streams[k] * rec;
        CU_TRY(cudaMemcpyAsync(h_pcm + (size_t)k * rec, (int16_t *)b->d_pcm.p + at, rec * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
        if (h_tap) CU_TRY(cudaMemcpyAsync(h_tap + (size_t)k * rec, (float *)b->d_tap.p + at, rec * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    CU_TRY(cudaStreamSynchronize(st));
    return SDRB_OK;
}

extern "C" int sdrb_bank_process_cf32_host(sdrb_bank *b, const float *h_in, size_t stride_samples, int n_blocks,
                                           int16_t *h_pcm, float *h_tap) {
    if (!b || !h_in || !h_pcm || n_blocks <= 0 || n_blocks > b->max_blocks ||
        stride_samples < (size_t)n_blocks * (size_t)b->plan->h.block) {
        set_error("sdrb_bank_process_cf32_host: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const HostPlan &h = b->plan->h;
    const size_t row = (size_t)n_blocks * h.block, rec = (size_t)n_blocks * h.pcm_per_block;
    const size_t cap = (size_t)b->max_blocks * h.block;
    int rc;
    if (!b->d_cf.p) { rc = b->d_cf.alloc(cap * sizeof(float2) * (size_t)b->n_streams); if (rc) return rc; }
    if (!b->d_pcm.p) {
        rc = b->d_pcm.alloc((size_t)b->max_blocks * h.pcm_per_block * sizeof(int16_t) * (size_t)b->n_streams); if (rc) return rc;
    }
    if (h_tap && !b->d_tap.p) {
        rc = b->d_tap.alloc((size_t)b->max_blocks * h.pcm_per_block * sizeof(float) * (size_t)b->n_streams); if (rc) return rc;
    }
    cudaStream_t st = b->s_compute;
    CU_TRY(cudaMemcpy2DAsync(b->d_cf.p, cap * sizeof(float2), h_in, stride_samples * sizeof(float2), row * sizeof(float2),
                             (size_t)b->n_streams, cudaMemcpyHostToDevice, st));
    b->last_launches = 0;
    CallCtx c;
    c.d_cf = (const float2 *)b->d_cf.p; c.cf_stride = cap; c.n_blocks = n_blocks;
    c.d_pcm = (int16_t *)b->d_pcm.p; c.d_tap = h_tap ? (float *)b->d_tap.p : nullptr;
    rc = enqueue_all(b, c, st, &b->last_launches);
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaMemcpyAsync(h_pcm, b->d_pcm.p, rec * sizeof(int16_t) * (size_t)b->n_streams, cudaMemcpyDeviceToHost, st));
    if (h_tap) CU_TRY(cudaMemcpyAsync(h_tap, b->d_tap.p, rec * sizeof(float) * (size_t)b->n_streams, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return SDRB_OK;
}

extern "C" int sdrb_bank_read_main(sdrb_bank *b, int main_idx, int n_blocks, float *h_out) {
    if (!b || !h_out || main_idx < 0 || main_idx >= (int)b->plan->h.mains.size() || n_blocks <= 0 || n_blocks > b->max_blocks) {
        set_error("sdrb_bank_read_main: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    const MainVfo &m = b->plan->h.mains[(size_t)main_idx];
    const size_t row = (size_t)n_blocks * m.block_out * sizeof(float2);
    CU_TRY(cudaMemcpy2D(h_out, row, (float2 *)b->main_out.p + b->main_off[(size_t)main_idx] + MAIN_HIST,
                        b->main_stride * sizeof(float2), row, (size_t)b->n_streams, cudaMemcpyDeviceToHost));
    return SDRB_OK;
}

extern "C" int sdrb_bank_last_launches(const sdrb_bank *b) { return b ? b->last_launches : 0; }

// ---- receiver state records (layout: include/sdrb200.h, kernels.cuh k_state_io) ----
extern "C" size_t sdrb_bank_state_bytes(const sdrb_bank *b) { return b ? b->state_bytes : 0; }

// Every header of a batch against this bank, before anything is written: a load is all or nothing.
static int check_state_headers(const sdrb_bank *b, const int32_t *streams, int n, const unsigned char *h, size_t pitch, const char *who) {
    const StateHeader &w = b->state_hdr;
    for (int k = 0; k < n; k++) {
        StateHeader r;
        memcpy(&r, h + (size_t)k * pitch, sizeof(r));
        const char *field = nullptr;
        unsigned long long got = 0, want = 0;
        if (r.magic != w.magic) { field = "magic"; got = r.magic; want = w.magic; }
        else if (r.version != w.version) { field = "version"; got = r.version; want = w.version; }
        else if (r.record_bytes != w.record_bytes) { field = "record_bytes"; got = r.record_bytes; want = w.record_bytes; }
        else if (r.fingerprint != w.fingerprint) { field = "plan fingerprint"; got = r.fingerprint; want = w.fingerprint; }
        else if (r.flags != w.flags) { field = "flags (correct_dc, fused /late VFOs)"; got = r.flags; want = w.flags; }
        char msg[320];
        if (field) {
            snprintf(msg, sizeof(msg), "%s: record %d (for stream %d): %s is 0x%llx, this bank needs 0x%llx; nothing was loaded", who, k,
                     (int)streams[k], field, got, want);
            set_error(msg);
            return SDRB_E_INVALID;
        }
        // the two scalars every later call computes from: table indices (blocks_done * block) and the DC recursion
        const long long max_done = SDRB_STATE_MAX_BLOCKS_DONE(b->plan->h.block);
        if (r.blocks_done < 0 || r.blocks_done > max_done) {
            snprintf(msg, sizeof(msg), "%s: record %d (for stream %d): blocks_done is %lld, this bank needs 0..%lld; nothing was loaded",
                     who, k, (int)streams[k], r.blocks_done, max_done);
            set_error(msg);
            return SDRB_E_INVALID;
        }
        const float dc[2] = {r.dc_state.x, r.dc_state.y};
        for (int a = 0; a < 2; a++)
            if (!(fabsf(dc[a]) <= SDRB_STATE_MAX_DC)) {           // also refuses NaN
                snprintf(msg, sizeof(msg), "%s: record %d (for stream %d): dc_state %c is %.9g, this bank needs a finite value in "
                         "[-%g, %g]; nothing was loaded", who, k, (int)streams[k], a ? 'Q' : 'I', (double)dc[a],
                         (double)SDRB_STATE_MAX_DC, (double)SDRB_STATE_MAX_DC);
                set_error(msg);
                return SDRB_E_INVALID;
            }
    }
    return SDRB_OK;
}

// One k_state_io launch on `st` between records at d_records and the listed streams. Ordered after the last device-resident call
// and the last save / load, whatever stream those ran on; the next process call waits for it (ev_state, ev_device_tail).
static int state_enqueue(sdrb_bank *b, const int32_t *streams, int n, void *d_records, cudaStream_t st, bool save) {
    if (b->device_tail_pending) CU_TRY(cudaStreamWaitEvent(st, b->ev_device_tail, 0));
    if (b->state_pending) CU_TRY(cudaStreamWaitEvent(st, b->ev_state, 0));          // the last save / load still reads state_streams
    const std::vector<int> list(streams, streams + n);      // pageable: staged before cudaMemcpyAsync returns, the caller may reuse `streams`
    CU_TRY(cudaMemcpyAsync(b->state_streams.p, list.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
    StateIoParams p;
    p.items = (const CarryItem *)b->carry.p; p.item_rec = (const int2 *)b->state_items.p; p.n_items = b->n_carry;
    p.streams = (const int *)b->state_streams.p; p.rec = (unsigned char *)d_records; p.rec_bytes = b->state_bytes;
    p.blocks_done = (long long *)b->blocks_done.p; p.dc_state = (float2 *)b->dc_state.p;
    p.raw_tail = (uint8_t *)b->raw_tail.p; p.cf_tail = (float2 *)b->cf_tail.p;
    p.dc_table = b->plan->h.correct_dc ? b->table_buf(b->dc_par) : nullptr;   // the buffer the next call reads its halo from
    p.dc_table_stride = b->dc_stride + DC_HALO_BLKS;
    p.hdr = b->state_hdr;
    const dim3 grid((unsigned)n, (unsigned)(b->n_carry + 1));
    if (save) k_state_io<true><<<grid, 128, 0, st>>>(p);
    else k_state_io<false><<<grid, 128, 0, st>>>(p);
    CU_TRY(cudaGetLastError());
    if (!b->ev_state) CU_TRY(cudaEventCreateWithFlags(&b->ev_state, cudaEventDisableTiming));
    CU_TRY(cudaEventRecord(b->ev_state, st));
    b->state_pending = true;
    if (!b->ev_device_tail) CU_TRY(cudaEventCreateWithFlags(&b->ev_device_tail, cudaEventDisableTiming));
    CU_TRY(cudaEventRecord(b->ev_device_tail, st));       // a following host call waits for it like for a device call
    b->device_tail_pending = true;
    return SDRB_OK;
}

extern "C" int sdrb_bank_save_state(sdrb_bank *b, const int32_t *streams, int n, void *d_records, void *cuda_stream) {
    int rc = check_stream_list(b, streams, n, d_records, "sdrb_bank_save_state");
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    if ((rc = host_drain(b)) != SDRB_OK) return rc;
    return state_enqueue(b, streams, n, d_records, (cudaStream_t)cuda_stream, true);
}

extern "C" int sdrb_bank_load_state(sdrb_bank *b, const int32_t *streams, int n, const void *d_records, void *cuda_stream) {
    int rc = check_stream_list(b, streams, n, d_records, "sdrb_bank_load_state");
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    if ((rc = host_drain(b)) != SDRB_OK) return rc;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    std::vector<unsigned char> hdr((size_t)n * sizeof(StateHeader));
    CU_TRY(cudaMemcpy2DAsync(hdr.data(), sizeof(StateHeader), d_records, b->state_bytes, sizeof(StateHeader), (size_t)n,
                             cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if ((rc = check_state_headers(b, streams, n, hdr.data(), sizeof(StateHeader), "sdrb_bank_load_state")) != SDRB_OK) return rc;
    return state_enqueue(b, streams, n, const_cast<void *>(d_records), st, false);
}

static int state_staging(sdrb_bank *b, int n) {
    const size_t need = (size_t)n * b->state_bytes;
    if (b->d_state.bytes >= need && b->d_state.p) return SDRB_OK;
    b->d_state.release();
    return b->d_state.alloc((size_t)b->n_streams * b->state_bytes);
}

extern "C" int sdrb_bank_read_state(sdrb_bank *b, const int32_t *streams, int n, void *h_records) {
    int rc = check_stream_list(b, streams, n, h_records, "sdrb_bank_read_state");
    if (rc != SDRB_OK) return rc;
    CU_TRY(cudaSetDevice(b->device));
    if ((rc = host_drain(b)) != SDRB_OK || (rc = state_staging(b, n)) != SDRB_OK) return rc;
    cudaStream_t st = b->s_compute;
    if ((rc = state_enqueue(b, streams, n, b->d_state.p, st, true)) != SDRB_OK) return rc;
    CU_TRY(cudaMemcpyAsync(h_records, b->d_state.p, (size_t)n * b->state_bytes, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return SDRB_OK;
}

extern "C" int sdrb_bank_write_state(sdrb_bank *b, const int32_t *streams, int n, const void *h_records) {
    int rc = check_stream_list(b, streams, n, h_records, "sdrb_bank_write_state");
    if (rc != SDRB_OK) return rc;
    if ((rc = check_state_headers(b, streams, n, (const unsigned char *)h_records, b->state_bytes, "sdrb_bank_write_state")) != SDRB_OK)
        return rc;
    CU_TRY(cudaSetDevice(b->device));
    if ((rc = host_drain(b)) != SDRB_OK || (rc = state_staging(b, n)) != SDRB_OK) return rc;
    cudaStream_t st = b->s_compute;
    CU_TRY(cudaMemcpyAsync(b->d_state.p, h_records, (size_t)n * b->state_bytes, cudaMemcpyHostToDevice, st));
    if ((rc = state_enqueue(b, streams, n, b->d_state.p, st, false)) != SDRB_OK) return rc;
    CU_TRY(cudaStreamSynchronize(st));
    return SDRB_OK;
}

// ---- FP32 peak probe ----
namespace sdrb {
template <bool PACKED>
__global__ void __launch_bounds__(256) k_probe_fma(float *sink, int iters, float a, float b) {
    // 8 independent chains per thread; operands from registers only
    if constexpr (PACKED) {
        float2 c[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) c[k] = make_float2((float)(threadIdx.x + k), (float)k);
        const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
#pragma unroll
                for (int k = 0; k < 8; ++k) c[k] = fma2(c[k], a2, b2);
            }
        }
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) acc += c[k].x + c[k].y;
        if (acc == 123.456f) sink[0] = acc;
    } else {
        float c[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) c[k] = (float)(threadIdx.x + k);
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
#pragma unroll
                for (int k = 0; k < 16; ++k) c[k] = fmaf(c[k], a, b);
            }
        }
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < 16; ++k) acc += c[k];
        if (acc == 123.456f) sink[0] = acc;
    }
}
}  // namespace sdrb

extern "C" int sdrb_probe_fp32_tflops(int packed, int reps, double *tflops) {
    if (!tflops || reps < 1) { set_error("sdrb_probe_fp32_tflops: bad arguments"); return SDRB_E_INVALID; }
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        set_error("sdrb_probe_fp32_tflops: no CUDA device"); return SDRB_E_CUDA;
    }
    float *sink = nullptr;
    cudaEvent_t e0, e1;
    if (cudaMalloc(&sink, 4) != cudaSuccess) { set_error("sdrb_probe_fp32_tflops: cudaMalloc failed"); return SDRB_E_CUDA; }
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const int iters = 4096, ctas = sms * 8, threads = 256;
    const double flop = (double)ctas * threads * (double)iters * 8.0 * 16.0 * 2.0;      // 16 FMA lanes per inner step, either form
    double best = 0.0;
    for (int r = 0; r < reps + 1; ++r) {                     // first pass warms up
        cudaEventRecord(e0);
        if (packed) sdrb::k_probe_fma<true><<<ctas, threads>>>(sink, iters, 0.999f, 0.001f);
        else sdrb::k_probe_fma<false><<<ctas, threads>>>(sink, iters, 0.999f, 0.001f);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (r > 0 && ms > 0.f) best = std::max(best, flop / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || best <= 0.0) { set_error(std::string("sdrb_probe_fp32_tflops: ") + cudaGetErrorString(e)); return SDRB_E_CUDA; }
    *tflops = best;
    return SDRB_OK;
}

extern "C" void *sdrb_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
        set_error("sdrb_host_alloc: cudaHostAlloc failed");
        return nullptr;
    }
    return p;
}

extern "C" void sdrb_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" const char *sdrb_last_error(void) { return last_error_cstr(); }
extern "C" const char *sdrb_version(void) { return "sdrb200 0.1 (sm_100a)"; }

// ------------------------------------------------------------------------------------
// host-only table builders
// ------------------------------------------------------------------------------------
extern "C" long sdrb_nco_table(double sample_rate, double frequency, float *dst, long max_entries) {
    if (sample_rate < 1.0) { set_error("sdrb_nco_table: sample_rate < 1"); return SDRB_E_INVALID; }
    const std::vector<cf32> q = nco_table(sample_rate, frequency);
    if (dst && max_entries > 0) memcpy(dst, q.data(), sizeof(cf32) * (size_t)std::min<long>((long)q.size(), max_entries));
    return (long)q.size();
}

extern "C" int sdrb_low_pass(double gain, double fs, double cutoff, double tw, float *taps, int max_taps) {
    std::vector<float> t;
    const int n = low_pass_hamming(gain, fs, cutoff, tw, t);
    if (n < 0) return n;
    if (taps && max_taps > 0) memcpy(taps, t.data(), sizeof(float) * (size_t)std::min(n, max_taps));
    return n;
}

extern "C" int sdrb_hilbert_points(int len, int fs, float *points) {
    if (len <= 0 || !points) { set_error("sdrb_hilbert_points: bad argument"); return SDRB_E_INVALID; }
    std::vector<float> p;
    hilbert_points(len, fs, p);
    memcpy(points, p.data(), sizeof(float) * (size_t)len);
    return SDRB_OK;
}

// ------------------------------------------------------------------------------------
// per-class primitives (prims.cuh)
// ------------------------------------------------------------------------------------
extern "C" int sdrb_nco_mix(const float *d_table, int table_len, int64_t n0, const float *d_in, float *d_out,
                            int n_ch, int n, void *cuda_stream) {
    if (!d_table || !d_in || !d_out || table_len <= 0 || n_ch <= 0 || n <= 0 || n0 < 0) {
        set_error("sdrb_nco_mix: bad argument"); return SDRB_E_INVALID;
    }
    prim_nco_mix<<<dim3((unsigned)((n + 255) / 256), (unsigned)n_ch), 256, 0, (cudaStream_t)cuda_stream>>>(
        (const float2 *)d_table, table_len, (long long)n0, (const float2 *)d_in, (float2 *)d_out, n);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

extern "C" int sdrb_halfband11(const float *d_in, float *d_out, float *d_hist, int n_ch, int n, void *cuda_stream) {
    if (!d_in || !d_out || !d_hist || n_ch <= 0 || n < 12 || (n & 1)) {
        set_error("sdrb_halfband11: needs an even block of at least 12 samples"); return SDRB_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    prim_halfband11<<<dim3((unsigned)((n / 2 + 255) / 256), (unsigned)n_ch), 256, 0, st>>>(
        (const float2 *)d_in, (float2 *)d_out, (const float2 *)d_hist, n);
    prim_halfband11_carry<<<(unsigned)n_ch, 32, 0, st>>>((const float2 *)d_in, (float2 *)d_hist, n);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

extern "C" int sdrb_halfband(int taps, const float *d_in, float *d_out, float *d_hist, int n_ch, int n, void *cuda_stream) {
    if (taps == 11 && n >= 12) return sdrb_halfband11(d_in, d_out, d_hist, n_ch, n, cuda_stream);
    if (!d_in || !d_out || !d_hist || n_ch <= 0 || n < 2 || (n & 1) || taps < 3 || taps > 255 || !(taps & 1)) {
        set_error("sdrb_halfband: needs an odd filter length 3..255 and an even block"); return SDRB_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const float *coef = nullptr;
    int nz = 0;                                               // lengths without a `case` in dsp.cpp:106-136 output zeros
    static const float hb11_host[4] = {HB_P0, HB_P2, HB_P4, HB_P5};
    float *d_c11 = nullptr;
    if (taps == 23) { CU_TRY(cudaGetSymbolAddress((void **)&coef, c_hb23)); nz = 7; }
    else if (taps == 51) { CU_TRY(cudaGetSymbolAddress((void **)&coef, c_hb51)); nz = 14; }
    else if (taps == 11) {                                    // blocks shorter than 12 samples (per-sample facade use)
        CU_TRY(cudaMalloc(&d_c11, sizeof(hb11_host)));
        CU_TRY(cudaMemcpyAsync(d_c11, hb11_host, sizeof(hb11_host), cudaMemcpyHostToDevice, st));
        coef = d_c11; nz = 4;
    }
    prim_halfband_n<<<dim3((unsigned)((n / 2 + 255) / 256), (unsigned)n_ch), 256, 0, st>>>(
        (const float2 *)d_in, (float2 *)d_out, (const float2 *)d_hist, n, taps, coef, nz);
    prim_halfband_n_carry<<<(unsigned)n_ch, 64, sizeof(float2) * (size_t)taps, st>>>((const float2 *)d_in, (float2 *)d_hist, n, taps);
    cudaError_t e = cudaGetLastError();
    if (d_c11) { cudaStreamSynchronize(st); cudaFree(d_c11); }
    if (e != cudaSuccess) { set_error(std::string("sdrb_halfband: ") + cudaGetErrorString(e)); return SDRB_E_CUDA; }
    return SDRB_OK;
}

extern "C" int sdrb_fir_ex(const float *d_taps, int ntaps, const float *d_in, float *d_out, float *d_hist, int n_ch,
                           int n, int decim, int include_newest, void *cuda_stream) {
    if (!d_taps || !d_in || !d_out || !d_hist || ntaps <= 0 || ntaps > 4096 || n_ch <= 0 || n <= 0 || decim < 1) {
        set_error("sdrb_fir: bad argument"); return SDRB_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int n_out = (n + decim - 1) / decim;
    prim_fir<<<dim3((unsigned)((n_out + 255) / 256), (unsigned)n_ch), 256, 0, st>>>(d_taps, ntaps, d_in, d_out, d_hist, n,
                                                                                 decim, n_out, include_newest ? 1 : 0);
    prim_tail_carry<<<(unsigned)n_ch, 128, sizeof(float) * (size_t)ntaps, st>>>(d_in, d_hist, n, ntaps, 1);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

extern "C" int sdrb_fir(const float *d_taps, int ntaps, const float *d_in, float *d_out, float *d_hist, int n_ch,
                        int n, int decim, void *cuda_stream) {
    return sdrb_fir_ex(d_taps, ntaps, d_in, d_out, d_hist, n_ch, n, decim, 0, cuda_stream);
}

extern "C" int sdrb_usb_demod(const float *d_points, const float *d_in, float *d_out, float *d_hist, int n_ch, int n,
                              void *cuda_stream) {
    if (!d_points || !d_in || !d_out || !d_hist || n_ch <= 0 || n <= 0) {
        set_error("sdrb_usb_demod: bad argument"); return SDRB_E_INVALID;
    }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    prim_usb<<<dim3((unsigned)((n + 255) / 256), (unsigned)n_ch), 256, 0, st>>>(
        d_points, (const float2 *)d_in, d_out, (const float2 *)d_hist, n);
    prim_tail_carry<<<(unsigned)n_ch, 128, sizeof(float) * 248, st>>>(d_in, d_hist, n, 124, 2);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

// Twiddle and window tables of the 8192-point transform, one copy per device, built on the host with the reference's own
// expressions: exp(-2 pi i k/N) in double cast to float (kiss_fft.c:357-363), hann[i] = 0.5*(1 - cos(2 pi float(i)/(N-1)))
// cast to float (mainwindow.cpp:284-288).
static int fft_tables(int device, FftTables *out) {
    static FftTables tabs[64] = {};
    if (device < 0 || device >= 64) { set_error("fft_tables: device index out of range"); return SDRB_E_INVALID; }
    if (!tabs[device].tw) {
        std::vector<float2> tw((size_t)FFT_N / 2);
        std::vector<float> hann((size_t)FFT_N);
        const double pi = 3.14159265358979323846264338327950288;
        for (int m = 0; m < FFT_N / 2; m++) {
            const double phase = -2.0 * pi * (double)m / (double)FFT_N;
            tw[(size_t)m] = make_float2((float)cos(phase), (float)sin(phase));
        }
        for (int i = 0; i < FFT_N; i++) hann[(size_t)i] = (float)(0.5 * (1.0 - cos(2.0 * M_PI * (double)(float)i / (FFT_N - 1.0))));
        float2 *dtw = nullptr; float *dh = nullptr;
        CU_TRY(cudaMalloc(&dtw, tw.size() * sizeof(float2)));
        CU_TRY(cudaMalloc(&dh, hann.size() * sizeof(float)));
        CU_TRY(cudaMemcpy(dtw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(dh, hann.data(), hann.size() * sizeof(float), cudaMemcpyHostToDevice));
        tabs[device].tw = dtw; tabs[device].hann = dh;
    }
    *out = tabs[device];
    return SDRB_OK;
}

extern "C" int sdrb_spectrum_fft(const float *d_in, float *d_out, int n_batch, int nfft, int apply_hann, void *cuda_stream) {
    if (!d_in || !d_out || n_batch <= 0 || nfft != 8192) {
        set_error("sdrb_spectrum_fft: nfft must be 8192 (mainwindow.cpp:241)"); return SDRB_E_INVALID;
    }
    static bool attr = false;
    if (!attr) {
        CU_TRY(cudaFuncSetAttribute(prim_fft8192, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * (int)sizeof(float2)));
        attr = true;
    }
    FftTables T;
    { int dev = 0; CU_TRY(cudaGetDevice(&dev)); const int trc = fft_tables(dev, &T); if (trc != SDRB_OK) return trc; }
    prim_fft8192<<<(unsigned)n_batch, 512, 8192 * sizeof(float2), (cudaStream_t)cuda_stream>>>(
        (const float2 *)d_in, (float2 *)d_out, apply_hann, T);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

// ---- spectrum display state (MainWindow::fftHandlerSlot, mainwindow.cpp:411-455) ----
struct sdrb_spectrum {
    int device = 0, n = 0;
    DevBuf inr, pwr, smooth, stats, scratch;
};

extern "C" void sdrb_spectrum_destroy(sdrb_spectrum *sp) {
    if (!sp) return;
    cudaSetDevice(sp->device);
    sp->inr.release(); sp->pwr.release(); sp->smooth.release(); sp->stats.release(); sp->scratch.release();
    delete sp;
}

extern "C" int sdrb_spectrum_reset(sdrb_spectrum *sp, int display) {
    if (!sp || display < -1 || display >= sp->n) { set_error("sdrb_spectrum_reset: bad argument"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(sp->device));
    const size_t d0 = display < 0 ? 0 : (size_t)display, nd = display < 0 ? (size_t)sp->n : 1;
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemset((float2 *)sp->inr.p + d0 * FFT_N, 0, nd * FFT_N * sizeof(float2)));     // mainwindow.cpp:547-550
    CU_TRY(cudaMemset((double *)sp->pwr.p + d0 * FFT_N, 0, nd * FFT_N * sizeof(double)));     // mainwindow.cpp:542-545
    CU_TRY(cudaMemset((double *)sp->smooth.p + d0 * (FFT_N - 10), 0, nd * (FFT_N - 10) * sizeof(double)));
    CU_TRY(cudaMemset((double *)sp->stats.p + d0 * 2, 0, nd * 2 * sizeof(double)));
    CU_TRY(cudaDeviceSynchronize());
    return SDRB_OK;
}

extern "C" int sdrb_spectrum_create(int device, int n_displays, int nfft, sdrb_spectrum **out) {
    if (!out || n_displays <= 0 || nfft != FFT_N) {
        set_error("sdrb_spectrum_create: nfft must be 8192 (mainwindow.cpp:243)"); return SDRB_E_INVALID;
    }
    *out = nullptr;
    CU_TRY(cudaSetDevice(device));
    sdrb_spectrum *sp = new (std::nothrow) sdrb_spectrum();
    if (!sp) { set_error("out of memory"); return SDRB_E_NOMEM; }
    sp->device = device; sp->n = n_displays;
    int rc;
    if ((rc = sp->inr.alloc((size_t)n_displays * FFT_N * sizeof(float2))) || (rc = sp->pwr.alloc((size_t)n_displays * FFT_N * sizeof(double))) ||
        (rc = sp->smooth.alloc((size_t)n_displays * (FFT_N - 10) * sizeof(double))) || (rc = sp->stats.alloc((size_t)n_displays * 2 * sizeof(double)))) {
        sdrb_spectrum_destroy(sp); return rc;
    }
    if (cudaFuncSetAttribute(k_spectrum_feed<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FFT_N * (int)sizeof(float2)) != cudaSuccess ||
        cudaFuncSetAttribute(k_spectrum_feed<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FFT_N * (int)sizeof(float2)) != cudaSuccess) {
        set_error("sdrb_spectrum_create: cannot reserve 64 KB of shared memory"); sdrb_spectrum_destroy(sp); return SDRB_E_CUDA;
    }
    rc = sdrb_spectrum_reset(sp, -1);
    if (rc != SDRB_OK) { sdrb_spectrum_destroy(sp); return rc; }
    *out = sp;
    return SDRB_OK;
}

// k_spectrum_feed for every display, or (map != nullptr) for the n displays a device list names
static int spectrum_feed_launch(sdrb_spectrum *sp, const float *d_in, size_t in_stride, int len, float *d_fft_out, cudaStream_t st,
                                const int *map, int n) {
    FftTables T;
    { const int trc = fft_tables(sp->device, &T); if (trc != SDRB_OK) return trc; }
    if (map)
        k_spectrum_feed<true><<<(unsigned)n, FFT_THREADS, FFT_N * sizeof(float2), st>>>(
            (const float2 *)d_in, (long long)in_stride, len, (float2 *)sp->inr.p, (double *)sp->pwr.p, (double *)sp->smooth.p,
            (double *)sp->stats.p, (float2 *)d_fft_out, T, map);
    else
        k_spectrum_feed<<<(unsigned)sp->n, FFT_THREADS, FFT_N * sizeof(float2), st>>>(
            (const float2 *)d_in, (long long)in_stride, len, (float2 *)sp->inr.p, (double *)sp->pwr.p, (double *)sp->smooth.p,
            (double *)sp->stats.p, (float2 *)d_fft_out, T);
    CU_TRY(cudaGetLastError());
    return SDRB_OK;
}

extern "C" int sdrb_spectrum_feed_device(sdrb_spectrum *sp, const float *d_in, size_t in_stride, int len, float *d_fft_out,
                                         void *cuda_stream) {
    if (!sp || !d_in || len < 0 || (sp->n > 1 && in_stride < (size_t)std::min(len, FFT_N))) {
        set_error("sdrb_spectrum_feed_device: bad argument"); return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(sp->device));
    return spectrum_feed_launch(sp, d_in, in_stride, len, d_fft_out, (cudaStream_t)cuda_stream, nullptr, 0);
}

// fftHandlerSlot for every receiver of a bank at once, straight from the bank's device buffers:
// source -1 = "Main" (sdrj.cpp:296-303: the DC-corrected input samples), k >= 0 = sub VFO k
// (vfo.cpp:290-293: its decimate[decimateCount]); callback cb of the last process call.
extern "C" int sdrb_bank_spectrum_feed(sdrb_bank *b, sdrb_spectrum *sp, int source, int cb, float *d_fft_out, void *cuda_stream) {
    if (!b || !sp || sp->n != b->n_streams || sp->device != b->device || source < -1 || source >= (int)b->plan->h.subs.size() ||
        cb < 0 || cb >= b->last_blocks) {
        set_error("sdrb_bank_spectrum_feed: needs one display per stream of the bank, a valid source and a callback of the last call");
        return SDRB_E_INVALID;
    }
    CU_TRY(cudaSetDevice(b->device));
    { const int drc = host_drain(b); if (drc != SDRB_OK) return drc; }
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (source < 0) {
        const int n = std::min(b->plan->h.block, FFT_N) / DC_BLK * DC_BLK;
        if (!sp->scratch.p) { int rc = sp->scratch.alloc((size_t)sp->n * FFT_N * sizeof(float2)); if (rc) return rc; }
        int rc = input_launch(b, cb, n, (float2 *)sp->scratch.p, st);
        if (rc != SDRB_OK) return rc;
        // a callback shorter than the FFT (none of the supported rates) would leave the tail stale, like the reference
        return spectrum_feed_launch(sp, (const float *)sp->scratch.p, (size_t)n, n, (float *)d_fft_out, st, b->last_map, b->last_n);
    }
    const SubVfo &s = b->plan->h.subs[(size_t)source];
    { const int zrc = ensure_sub_z(b, source, st); if (zrc != SDRB_OK) return zrc; }
    const float2 *z = (const float2 *)b->zbuf.p + b->sub_z_off[(size_t)source] + b->sub_z_hist[(size_t)source] + (size_t)cb * s.block_z;
    // after a stream-list call the displays of its streams only: the others keep pwr, inr and stats
    return spectrum_feed_launch(sp, (const float *)z, b->z_stride, s.block_z, (float *)d_fft_out, st, b->last_map, b->last_n);
}

extern "C" int sdrb_spectrum_feed_host(sdrb_spectrum *sp, const float *h_in, size_t in_stride, int len) {
    if (!sp || !h_in || len < 0) { set_error("sdrb_spectrum_feed_host: bad argument"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(sp->device));
    const int use = std::min(len, FFT_N);                       // only the first nFFT samples are looked at
    float2 *stage = nullptr;
    CU_TRY(cudaMalloc(&stage, (size_t)sp->n * FFT_N * sizeof(float2)));
    cudaError_t e = cudaSuccess;
    if (use > 0)
        e = cudaMemcpy2D(stage, FFT_N * sizeof(float2), h_in, in_stride * sizeof(float2), (size_t)use * sizeof(float2), (size_t)sp->n,
                         cudaMemcpyHostToDevice);
    int rc = SDRB_OK;
    if (e != cudaSuccess) { set_error(std::string("sdrb_spectrum_feed_host: ") + cudaGetErrorString(e)); rc = SDRB_E_CUDA; }
    if (rc == SDRB_OK) rc = sdrb_spectrum_feed_device(sp, (const float *)stage, FFT_N, len, nullptr, nullptr);
    cudaDeviceSynchronize();
    cudaFree(stage);
    return rc;
}

extern "C" int sdrb_spectrum_read(sdrb_spectrum *sp, double *h_smooth, double *h_pwr, double *h_stats) {
    if (!sp) { set_error("sdrb_spectrum_read: NULL"); return SDRB_E_INVALID; }
    CU_TRY(cudaSetDevice(sp->device));
    CU_TRY(cudaDeviceSynchronize());
    if (h_smooth) CU_TRY(cudaMemcpy(h_smooth, sp->smooth.p, (size_t)sp->n * (FFT_N - 10) * sizeof(double), cudaMemcpyDeviceToHost));
    if (h_pwr) CU_TRY(cudaMemcpy(h_pwr, sp->pwr.p, (size_t)sp->n * FFT_N * sizeof(double), cudaMemcpyDeviceToHost));
    if (h_stats) CU_TRY(cudaMemcpy(h_stats, sp->stats.p, (size_t)sp->n * 2 * sizeof(double), cudaMemcpyDeviceToHost));
    return SDRB_OK;
}
