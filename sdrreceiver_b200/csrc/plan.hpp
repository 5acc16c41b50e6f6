// Internal host-side plan representation shared by plan_host.cpp (pure C++, compiled
// with -ffp-contract=off so the NCO tables match the reference bit for bit) and
// api.cu (device upload, launches).
#pragma once
#include <cstdint>
#include <map>
#include <string>
#include <vector>
#include "../../include/sdrb200.h"

namespace sdrb {

struct cf32 { float re, im; };

constexpr int MAX_DECIM = 8;            // half-band stages of a VFO: vfo::decimate is decimate[9] (vfo.h:39)
constexpr int MAIN_STAGE_MIN = 512;     // samples per callback after the third stage of a main VFO with more than 3 stages

struct MainVfo {
    int frequency = 0;
    double mixer = 0;
    int decim = 0;
    int out_rate = 0;
    int block_out = 0;          // samples per callback after the cascade
    std::vector<cf32> lut;      // Oscillator table, (int)Fs entries
    // IQ forwarder (vfo::compress): ini keys zmq_address / zmq_topic / compress_scale of [main_vfos]
    std::string topic, zmq_address;
    int compress_scale = 1;     // vfo::scalecomp, 1 unless compress_scale > 0 (vfo.cpp:24, mainwindow.cpp:112-118)
    int compress_style = 1;     // vfo::cstyle as MainWindow sets it (mainwindow.cpp:133)
    int n_subs = 0;
    int fwd_bytes = 0;          // payload bytes per callback
};

struct SubVfo {
    std::string topic;
    int frequency = 0, data_rate = 0;
    int main_idx = 0;
    int fs = 0;                 // parent's output rate
    double mixer = 0;
    int decim = 0, late = 0, filter_bw = 0;
    float gain = 0.01f;         // vfo::vfo default (vfo.cpp:9)
    int block_in = 0;           // samplesPerBuffer given to vfo::init (mainwindow.cpp:223)
    int block_z = 0;            // samples per callback after the half-band cascade
    int out_rate = 0;
    int samples_out = 0;        // per callback, after the optional /late
    int pcm_offset = 0;
    std::vector<cf32> lut;
    std::vector<float> dec_taps, lpf_taps;
    std::vector<float> hilbert;     // 125 points, FIRHilbert(125, samples_out) (vfo.cpp:137)
};

struct HostPlan {
    int fs = 0, block = 0, bufsplit = 4, correct_dc = 0, center = 0;
    std::string zmq_address;
    std::vector<MainVfo> mains;
    std::vector<SubVfo> subs;
    int pcm_per_block = 0;
    double alg_bytes = 0, alg_flops = 0;
    // every key of the ini file as QSettings would name it ("group/key", arrays "vfos/3/gain"): the keys the
    // hot path does not use (tuner_gain, remote_rtl, auto_start*, disable_fft, ... mainwindow.cpp:51-96) stay
    // readable through sdrb_plan_get_setting for the application that owns the device and the GUI
    std::map<std::string, std::string> settings;
};

void set_error(const std::string &msg);

// restatements of the reference's init-time table builders (plain float ops, no FMA)
std::vector<cf32> nco_table(double sample_rate, double frequency);
int low_pass_hamming(double gain, double fs, double cutoff, double tw, std::vector<float> &taps);
void hilbert_points(int len, int fs, std::vector<float> &pts);

int plan_from_ini(const char *path, HostPlan &plan);
int plan_from_desc(const sdrb_plan_desc &d, HostPlan &plan);

}  // namespace sdrb
