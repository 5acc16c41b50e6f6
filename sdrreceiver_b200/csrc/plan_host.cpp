// Host-side plan compiler: ini -> flat VFO plan with every init-time table the reference
// builds in vfo::init. Qt-free restatement of
//   mainwindow.cpp:27-235   (QSettings ini reading, callback size, VFO tree arithmetic)
//   oscillator.cpp:4-32     (NCO lookup table recursion)
//   gnuradio/firfilter.cpp:64-121,212-220 (firdes low_pass with a Hamming window)
//   jonti/dsp.cpp:184-216   (Hilbert coefficients)
// This translation unit is compiled with g++ -O2 -ffp-contract=off (no FMA contraction):
// the NCO recursion is chaotic enough that a fused multiply-add moves the final audio by
// ~1e-4 rel-L2 (SURVEY.md section 0.3), so tables are built here and uploaded, never
// regenerated on the GPU.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>

#include "plan.hpp"

#ifndef M_PI
#define M_PI 3.14159265358979323846264338327950288
#endif

namespace sdrb {

static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }
const char *last_error_cstr() { return g_error.c_str(); }

// ---- Oscillator table (oscillator.cpp:9-28) ----
std::vector<cf32> nco_table(double sample_rate, double frequency) {
    const double step = 2.0 * M_PI * frequency / sample_rate;
    const float rr = (float)cos(step), ri = (float)sin(step);
    float vr = 1.0f, vi = 0.0f;
    const int len = (int)sample_rate;
    std::vector<cf32> q((size_t)(len > 0 ? len : 0));
    for (int k = 0; k < len; k++) {
        // complex<float> *= complex<float>: four rounded products, two rounded sums
        const float pr = vr * rr, qi = vi * ri, pi = vr * ri, qr = vi * rr;
        const float nr = pr - qi, ni = pi + qr;
        const float shrink = 1.95f - (nr * nr + ni * ni);
        vr = nr * shrink;
        vi = ni * shrink;
        q[(size_t)k].re = vr;
        q[(size_t)k].im = vi;
    }
    return q;
}

// ---- firdes::low_pass, WIN_HAMMING (firfilter.cpp:64-108) ----
int low_pass_hamming(double gain, double fs, double cutoff, double tw, std::vector<float> &taps) {
    if (fs <= 0.0 || cutoff <= 0.0 || cutoff > fs / 2 || tw <= 0) {     // sanity_check_1f
        set_error("low_pass: arguments fail the firdes sanity check");
        return SDRB_E_INVALID;
    }
    int ntaps = (int)(53 * fs / (22.0 * tw));                            // compute_ntaps
    if ((ntaps & 1) == 0) ntaps++;
    taps.assign((size_t)ntaps, 0.0f);
    std::vector<float> win((size_t)ntaps);
    const float span = (float)(ntaps - 1);
    for (int n = 0; n < ntaps; n++) win[(size_t)n] = 0.54 - 0.46 * cos((2 * M_PI * n) / span);
    const int half = (ntaps - 1) / 2;
    const double w0 = 2 * M_PI * cutoff / fs;
    for (int n = -half; n <= half; n++) {
        const size_t j = (size_t)(n + half);
        if (n == 0) taps[j] = w0 / M_PI * win[j];
        else taps[j] = sin(n * w0) / (n * M_PI) * win[j];
    }
    double dc = taps[(size_t)half];
    for (int n = 1; n <= half; n++) dc += 2 * taps[(size_t)(n + half)];
    const double scale = gain / dc;
    for (int n = 0; n < ntaps; n++) taps[(size_t)n] *= scale;
    return ntaps;
}

// ---- FIRHilbert::FIRHilbert (dsp.cpp:198-216) ----
void hilbert_points(int len, int fs, std::vector<float> &pts) {
    std::vector<float> c((size_t)len);
    float energy = 0;
    for (int n = 0; n < len; n++) {
        const int k = n - len / 2;
        if (k == 0) c[(size_t)n] = 0;
        else c[(size_t)n] = fs / (M_PI * k) * (1 - cos(M_PI * k));
        energy += c[(size_t)n] * c[(size_t)n];
    }
    const double norm = sqrtf(energy);       // sqrt(float) picks the float overload in the reference
    pts.resize((size_t)len);
    for (int i = 0; i < len; i++) pts[(size_t)i] = c[(size_t)(len - i - 1)] / norm;
}

// ---- QSettings(IniFormat) subset ----
static std::string trim(const std::string &s) {
    const size_t a = s.find_first_not_of(" \t\r\n");
    if (a == std::string::npos) return "";
    const size_t b = s.find_last_not_of(" \t\r\n");
    return s.substr(a, b - a + 1);
}

struct IniFile {
    std::map<std::string, std::string> kv;
    bool load(const char *path) {
        std::ifstream f(path);
        if (!f) return false;
        std::string line, group;
        while (std::getline(f, line)) {
            line = trim(line);
            if (line.empty() || line[0] == ';') continue;   // '#' lines are keys, not comments
            if (line[0] == '[') {
                const size_t e = line.find(']');
                group = trim(line.substr(1, e == std::string::npos ? std::string::npos : e - 1));
                if (group == "General") group.clear();
                continue;
            }
            const size_t eq = line.find('=');
            if (eq == std::string::npos) continue;
            std::string k = trim(line.substr(0, eq)), v = trim(line.substr(eq + 1));
            for (char &c : k) if (c == '\\') c = '/';
            if (v.size() >= 2 && v.front() == '"' && v.back() == '"') v = v.substr(1, v.size() - 2);
            kv[group.empty() ? k : group + "/" + k] = v;
        }
        return true;
    }
    std::string str(const std::string &k) const {
        auto it = kv.find(k);
        return it == kv.end() ? std::string() : it->second;
    }
    int num(const std::string &k) const {       // QVariant::toInt(): 0 unless a clean int32
        const std::string s = str(k);
        if (s.empty()) return 0;
        char *end = 0;
        const long long v = strtoll(s.c_str(), &end, 10);
        if (*end != 0 || v < INT32_MIN || v > INT32_MAX) return 0;
        return (int)v;
    }
    float real(const std::string &k) const { return strtof(str(k).c_str(), 0); }
};

static int ilog2_floor_of_ratio(int num, int den) {
    // int(log2(num/den)) with integer division first, as written in the reference
    if (den <= 0 || num / den <= 0) return -1;
    return (int)std::log2((double)(num / den));
}

static std::string vfo_name(const char *kind, int idx, const std::string &topic) {
    std::string n = std::string(kind) + " " + std::to_string(idx + 1);
    if (!topic.empty()) n += " ('" + topic + "')";
    return n;
}

// A half-band stage writes in.size()/2 outputs and needs an even input (HalfBandDecimator::decimate; the reference is undefined
// otherwise), and every length the library stores per callback is moved in 16-byte pieces (k3_carry, float4 loads and stores),
// so it must be even too: the n per-callback lengths len, len/2, .., len/2^stages must all be even.
static bool even_cascade(int len, int stages, const std::string &name) {
    for (int a = 0; a < stages; a++, len /= 2)
        if (len % 2 != 0) {
            set_error("plan: " + name + ": half-band stage " + std::to_string(a + 1) + " would get " + std::to_string(len) +
                      " samples per callback, an odd count");
            return false;
        }
    if (len % 2 != 0) {
        set_error("plan: " + name + " would store " + std::to_string(len) + " samples per callback; stored lengths must be even");
        return false;
    }
    return true;
}

// Shared tail of both constructors: derive rates/sizes, build tables, validate.
static int finish_plan(HostPlan &p) {
    if (p.fs <= 0 || p.block <= 0 || p.mains.empty()) {
        set_error("plan: needs a sample rate, a callback size and at least one main VFO");
        return SDRB_E_INVALID;
    }
    if (p.mains.size() > SDRB_MAX_MAIN || p.subs.size() > SDRB_MAX_SUB) {
        set_error("plan: too many VFOs");
        return SDRB_E_INVALID;
    }
    if (p.block % 256 != 0) {
        set_error("plan: callback size must be a multiple of 256 complex samples");
        return SDRB_E_INVALID;
    }
    for (MainVfo &m : p.mains) {
        const std::string name = vfo_name("main VFO", (int)(&m - p.mains.data()), m.topic);
        if (m.decim < 0 || m.decim > MAX_DECIM) {                  // vfo::decimate[9] (vfo.h:39)
            set_error("plan: " + name + " needs 0..8 half-band stages (out_rate >= sample_rate/256), not " +
                      std::to_string(m.decim));
            return SDRB_E_INVALID;
        }
        if (!even_cascade(p.block, m.decim, name)) return SDRB_E_INVALID;
        // stages 4.. run on k1_v2's third-stage output; its tail kernel reaches up to 364 staged samples back, which must lie in the
        // previous callback's body, not across that callback's own head
        if (m.decim > 3 && (p.block >> 3) < MAIN_STAGE_MIN) {
            set_error("plan: " + name + " with more than 3 half-band stages needs at least " + std::to_string(MAIN_STAGE_MIN * 8) +
                      " samples per callback");
            return SDRB_E_INVALID;
        }
        m.out_rate = (int)(p.fs / std::pow(2, m.decim));               // vfo::getOutRate
        m.block_out = p.block >> m.decim;
        m.lut = nco_table(p.fs, m.mixer);
        if (m.compress_scale <= 0) m.compress_scale = 1;
        if (m.compress_style == 0) m.compress_style = 1;
        m.fwd_bytes = m.compress_style == 1 ? m.block_out : 2 * m.block_out;   // vfo.cpp:143-150
        m.n_subs = 0;
    }
    int off = 0;
    double out_rates = 0, flops = 0;
    for (SubVfo &s : p.subs) {
        if (s.main_idx < 0 || s.main_idx >= (int)p.mains.size()) {
            set_error("plan: sub VFO refers to a main VFO that does not exist");
            return SDRB_E_INVALID;
        }
        MainVfo &m = p.mains[(size_t)s.main_idx];
        m.n_subs++;
        s.fs = m.out_rate;
        s.block_in = m.out_rate / p.bufsplit;                           // mainwindow.cpp:223
        // the parent writes block >> decim samples per callback and the sub VFO reads out_rate / bufsplit: the two agree
        // only if block * bufsplit == sample_rate (true for every ini plan by construction, mainwindow.cpp:67-80)
        if (s.block_in != m.block_out) {
            set_error("plan: block * bufsplit must equal sample_rate (sub VFO '" + s.topic + "' would read " +
                      std::to_string(s.block_in) + " samples per callback, its main VFO writes " + std::to_string(m.block_out) + ")");
            return SDRB_E_INVALID;
        }
        if (s.decim < 0 || s.decim > MAX_DECIM || (s.late != 0 && s.late != 5 && s.late != 6)) {
            set_error("plan: sub VFO '" + s.topic + "' needs 0..8 half-band stages and late in {0,5,6} (it has " +
                      std::to_string(s.decim) + " stages, late " + std::to_string(s.late) + ")");
            return SDRB_E_INVALID;
        }
        if (!even_cascade(s.block_in, s.decim, "sub VFO '" + s.topic + "'")) return SDRB_E_INVALID;
        int rate = (int)(s.fs / std::pow(2, s.decim));                  // vfo.cpp:65-66
        s.block_z = (int)(s.block_in / std::pow(2, s.decim));
        s.samples_out = s.block_z;
        if (s.late > 0) {                                               // vfo.cpp:69-100
            rate = rate / s.late;
            if (s.block_z % s.late != 0) {
                set_error("plan: callback size not divisible by the late decimation");
                return SDRB_E_INVALID;
            }
            s.samples_out = s.block_z / s.late;
            if (s.samples_out % 2 != 0) {
                set_error("plan: sub VFO '" + s.topic + "' would store " + std::to_string(s.samples_out) +
                          " samples per callback after its /late FIR; stored lengths must be even");
                return SDRB_E_INVALID;
            }
            const int rc = low_pass_hamming(2, rate * s.late, rate / 2, (double)rate / (s.late - 1), s.dec_taps);
            if (rc < 0) return rc;
        }
        s.out_rate = rate;
        if (s.filter_bw > 0) {                                          // vfo.cpp:106-124
            const int rc = low_pass_hamming(2, rate, s.filter_bw, (double)s.filter_bw / 4, s.lpf_taps);
            if (rc < 0) return rc;
        }
        if ((int)(s.lpf_taps.size() + s.dec_taps.size()) + 124 >= s.samples_out) {
            set_error("plan: filters longer than one callback are not supported");
            return SDRB_E_INVALID;
        }
        s.lut = nco_table(s.fs, s.mixer);
        hilbert_points(125, s.samples_out, s.hilbert);                  // vfo.cpp:137
        s.pcm_offset = off;
        off += s.samples_out;
        out_rates += s.out_rate;
        // flop counting rule of SURVEY.md 8(d), per second of signal
        double f = 6.0 * s.fs;
        for (int a = 1; a <= s.decim; a++) f += 20.0 * s.fs / std::pow(2, a);
        if (s.late > 0) f += 2.0 * 2.0 * s.dec_taps.size() * s.out_rate;
        f += (2.0 * 62 + 1) * s.out_rate + 2.0 * s.lpf_taps.size() * s.out_rate + 2.0 * s.out_rate;
        flops += f;
    }
    p.pcm_per_block = off;
    double mf = 10.0 * p.fs;
    for (const MainVfo &m : p.mains) {
        mf += 6.0 * p.fs;
        for (int a = 1; a <= m.decim; a++) mf += 20.0 * p.fs / std::pow(2, a);
    }
    p.alg_bytes = 2.0 + 2.0 * out_rates / p.fs;
    p.alg_flops = (mf + flops) / p.fs;
    return SDRB_OK;
}

int plan_from_ini(const char *path, HostPlan &p) {
    IniFile ini;
    if (!path || !ini.load(path)) {
        set_error(std::string("cannot read ini file ") + (path ? path : "(null)"));
        return SDRB_E_IO;
    }
    p = HostPlan();
    p.settings = ini.kv;
    p.fs = ini.num("sample_rate");
    if (p.fs != 288000 && p.fs != 1536000 && p.fs != 1920000) {       // mainwindow.cpp:31-47
        set_error("sample_rate setting not supported, only 288000, 1536000, 1920000 are");
        return SDRB_E_INVALID;
    }
    p.center = ini.num("center_frequency");
    const int mix_offset = ini.num("mix_offset");
    int buflen;                                                         // mainwindow.cpp:67-80
    if (double((int((2 * p.fs) / 4)) % 512) > 0) { buflen = int((2 * p.fs) / 5); p.bufsplit = 5; }
    else { buflen = int((2 * p.fs) / 4); p.bufsplit = 4; }
    p.block = buflen / 2;
    p.zmq_address = ini.str("zmq_address");
    p.correct_dc = ini.str("correct_dc_bias") == "1" ? 1 : 0;

    const int n_main = ini.num("main_vfos/size");                       // mainwindow.cpp:98-140
    for (int i = 0; i < n_main; i++) {
        const std::string k = "main_vfos/" + std::to_string(i + 1) + "/";
        MainVfo m;
        m.frequency = ini.num(k + "frequency");
        const int want = ini.num(k + "out_rate");
        if (want <= 0) { set_error("main VFO without out_rate"); return SDRB_E_INVALID; }
        m.decim = (p.fs / want == 1) ? 0 : ilog2_floor_of_ratio(p.fs, want);
        m.mixer = p.center - m.frequency;
        m.out_rate = (int)(p.fs / std::pow(2, m.decim));
        const int compscale = ini.num(k + "compress_scale");            // mainwindow.cpp:112-118
        if (compscale > 0) m.compress_scale = compscale;
        const std::string addr = ini.str(k + "zmq_address"), topic = ini.str(k + "zmq_topic");
        if (!addr.empty() && !topic.empty()) { m.zmq_address = addr; m.topic = topic; }   // mainwindow.cpp:120-126
        p.mains.push_back(m);
    }
    const int n_sub = ini.num("vfos/size");                             // mainwindow.cpp:141-235
    for (int i = 0; i < n_sub; i++) {
        const std::string k = "vfos/" + std::to_string(i + 1) + "/";
        SubVfo s;
        s.frequency = ini.num(k + "frequency") + mix_offset;
        s.data_rate = ini.num(k + "data_rate");
        int out_rate = ini.num(k + "out_rate");
        if (out_rate == 0 && s.data_rate > 0)
            out_rate = s.data_rate == 600 ? 12000 : s.data_rate == 1200 ? 24000 : 48000;
        if (out_rate <= 0) { set_error("sub VFO without data_rate/out_rate"); return SDRB_E_INVALID; }
        s.filter_bw = ini.num(k + "filter_bandwidth");
        int parent_mix = 0, parent_rate = p.fs;
        s.main_idx = -1;
        for (size_t a = 0; a < p.mains.size(); a++) {
            const int diff = std::abs((p.center - p.mains[a].mixer) - s.frequency);
            if (diff < p.mains[a].out_rate) {
                s.main_idx = (int)a;
                parent_mix = (int)p.mains[a].mixer;
                parent_rate = p.mains[a].out_rate;
                break;
            }
        }
        if (s.main_idx < 0) {
            // Reference quirk (mainwindow.cpp:174-191): a sub VFO that matches no main keeps
            // Fs = sample_rate but is fed main 0's decimated buffer and indexes past its end
            // (vfo.cpp:244) -- undefined behaviour there, rejected here.
            set_error("plan: sub VFO '" + ini.str(k + "topic") + "' is outside every main VFO's passband");
            return SDRB_E_INVALID;
        }
        if (parent_rate / 48000 == 5) {
            s.decim = ilog2_floor_of_ratio(parent_rate, 5 * out_rate);
            s.late = 5;
        } else if (parent_rate / 48000 == 6) {
            s.decim = ilog2_floor_of_ratio(parent_rate, 6 * out_rate);
            s.late = 6;
        } else {
            s.decim = ilog2_floor_of_ratio(p.fs, out_rate) - ilog2_floor_of_ratio(p.fs, parent_rate);
        }
        s.gain = (float)ini.real(k + "gain") / 100;
        s.mixer = (p.center - parent_mix) - s.frequency;
        s.topic = ini.str(k + "topic");
        p.subs.push_back(s);
    }
    return finish_plan(p);
}

int plan_from_desc(const sdrb_plan_desc &d, HostPlan &p) {
    p = HostPlan();
    p.fs = d.sample_rate;
    p.block = d.block;
    p.bufsplit = d.bufsplit;
    p.correct_dc = d.correct_dc ? 1 : 0;
    if (d.n_main < 0 || d.n_main > SDRB_MAX_MAIN || d.n_sub < 0 || d.n_sub > SDRB_MAX_SUB || d.bufsplit <= 0) {
        set_error("plan: VFO counts out of range");
        return SDRB_E_INVALID;
    }
    for (int i = 0; i < d.n_main; i++) {
        MainVfo m;
        m.mixer = d.mains[i].mixer_hz;
        m.decim = d.mains[i].decim;
        m.topic.assign(d.mains[i].topic, strnlen(d.mains[i].topic, sizeof(d.mains[i].topic)));
        m.compress_scale = d.mains[i].compress_scale;
        m.compress_style = d.mains[i].compress_style;
        p.mains.push_back(m);
    }
    for (int i = 0; i < d.n_sub; i++) {
        SubVfo s;
        s.topic.assign(d.subs[i].topic, strnlen(d.subs[i].topic, sizeof(d.subs[i].topic)));
        s.main_idx = d.subs[i].main_idx;
        s.mixer = d.subs[i].mixer_hz;
        s.decim = d.subs[i].decim;
        s.late = d.subs[i].late;
        s.filter_bw = d.subs[i].filter_bw;
        s.gain = d.subs[i].gain;
        p.subs.push_back(s);
    }
    return finish_plan(p);
}

}  // namespace sdrb
