/*
 * sdrb200.h -- C ABI of libsdrb200.so, the B200 (sm_100a) channelizer that replaces the
 * CPU hot path of jeroenbeijer/SDRReceiver:
 *
 *   uint8 IQ -> (x-127) -> DC removal -> per main VFO: NCO mix + 11-tap half-band cascade
 *            -> per sub VFO: NCO mix + half-band cascade [+ /5 or /6 FIR] -> USB demod
 *               (delay62 - Hilbert125) [-> filter_bandwidth low-pass] -> gain -> int16
 *
 * The reference has no FFI layer; its boundary is the C++ class surface (SURVEY.md 8(b)).
 * Each entry point below names the reference code it stands in for (paths relative to the
 * SDRReceiver source tree). The header-compatible C++ facades (sdrreceiver_b200/host/) and
 * the Python binding (sdrreceiver_b200/binding.py) are thin layers over exactly this ABI.
 *
 * Conventions: plain C, caller-owned buffers, every function returns 0 on success or a
 * negative SDRB_E_* code and never throws; sdrb_last_error() gives the message of the last
 * failure on the calling thread. There is no CPU fallback: without a CUDA device the
 * compute entry points fail with SDRB_E_CUDA.
 */
#ifndef SDRB200_H
#define SDRB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDRB_OK 0
#define SDRB_E_INVALID (-1)     /* bad argument / unsupported plan */
#define SDRB_E_IO (-2)          /* ini file unreadable */
#define SDRB_E_CUDA (-3)        /* CUDA runtime error or no device */
#define SDRB_E_NOMEM (-4)
#define SDRB_E_ZMQ (-5)         /* libzmq not loadable / socket error */

#define SDRB_MAX_MAIN 8         /* the reference caps main VFOs at 3 (mainwindow.h:82) */
#define SDRB_MAX_SUB 256
#define SDRB_TOPIC_LEN 5        /* ZMQ topic frame is exactly 5 bytes (zmqpublisher.cpp:91) */

typedef struct sdrb_plan sdrb_plan;   /* immutable VFO plan: rates, tree, NCO tables, taps */
typedef struct sdrb_bank sdrb_bank;   /* n_streams receivers of one plan on one GPU: carry
                                         state (DC, sample counters, filter tails) + work buffers */

/* ---- plan description (what MainWindow::MainWindow computes, mainwindow.cpp:29-235) ---- */
typedef struct {
    double mixer_hz;        /* center_frequency - frequency          (mainwindow.cpp:131) */
    int32_t decim;          /* half-band stages, 0..8                (mainwindow.cpp:130, vfo.h:39) */
    /* IQ forwarder (vfo::compress, vfo.cpp:389-424): a main VFO WITHOUT sub VFOs re-publishes its
     * decimated IQ as bytes when it has a topic (mainwindow.cpp:109-126). */
    char topic[8];          /* zmq_topic, "" = nothing is published  (mainwindow.cpp:110) */
    int32_t compress_scale; /* compress_scale, <= 0 means 1          (mainwindow.cpp:112-118, vfo.cpp:24) */
    int32_t compress_style; /* vfo::cstyle: 1 = two 4-bit arms per byte (what MainWindow always sets,
                               mainwindow.cpp:133), anything else = int8 I,Q pairs; 0 here means 1 */
} sdrb_main_desc;

typedef struct {
    char topic[8];          /* zmq topic, first 5 bytes are sent     (mainwindow.cpp:193) */
    int32_t main_idx;       /* parent main VFO                       (mainwindow.cpp:178-191) */
    double mixer_hz;        /* main_freq - (frequency + mix_offset)  (mainwindow.cpp:220) */
    int32_t decim;          /* half-band stages, 0..8                (mainwindow.cpp:197-216, vfo.h:39) */
    int32_t late;           /* 0, or the /5 or /6 FIR decimation     (mainwindow.cpp:197-210) */
    int32_t filter_bw;      /* filter_bandwidth Hz, 0 = off          (mainwindow.cpp:218) */
    float gain;             /* ini gain / 100                        (mainwindow.cpp:219) */
} sdrb_sub_desc;

typedef struct {
    int32_t sample_rate;    /* 288000 | 1536000 | 1920000            (mainwindow.h:29) */
    int32_t block;          /* complex samples per callback = buflen/2 (mainwindow.cpp:67-80) */
    int32_t bufsplit;       /* callbacks per second, 4 or 5 */
    int32_t correct_dc;     /* correct_dc_bias                       (mainwindow.cpp:96) */
    int32_t n_main, n_sub;
    sdrb_main_desc mains[SDRB_MAX_MAIN];
    sdrb_sub_desc subs[SDRB_MAX_SUB];
} sdrb_plan_desc;

typedef struct {
    int32_t sample_rate, block, bufsplit, correct_dc, n_main, n_sub;
    int32_t center_frequency;     /* 0 when the plan was not built from an ini */
    int32_t pcm_per_block;        /* int16 samples per stream per callback, all sub VFOs */
    double alg_bytes_per_sample;  /* 2 + 2*sum(out_rate)/Fs            (SURVEY.md 8(d)) */
    double alg_flops_per_sample;  /* SURVEY.md 8(d) counting rule */
    char zmq_address[128];
} sdrb_plan_info;

typedef struct {
    double mixer_hz;
    int32_t frequency;            /* absolute Hz (ini plans), else 0 */
    int32_t decim, out_rate, block_out;   /* block_out = block >> decim */
    int32_t n_subs;               /* sub VFOs fed by this main VFO */
    int32_t forward;              /* 1: no sub VFOs and a topic -> publishes compressed IQ */
    int32_t compress_scale, compress_style;
    int32_t fwd_bytes_per_block;  /* ZMQ payload of one callback: block_out (style 1) or 2*block_out */
    char topic[8];
    char zmq_address[128];        /* the address this main VFO connects to (mainwindow.cpp:109) */
} sdrb_main_info;

typedef struct {
    char topic[8];
    int32_t frequency, data_rate; /* ini values (0 when built from a desc) */
    int32_t main_idx, decim, late, filter_bw;
    float gain;
    double mixer_hz;
    int32_t in_rate;              /* parent's output rate = this VFO's Fs */
    int32_t out_rate;             /* audio rate sent as ZMQ frame 2 */
    int32_t samples_out;          /* int16 samples per callback = ZMQ frame 3 / 2 */
    int32_t pcm_offset;           /* offset of this VFO inside one stream-callback record */
    int32_t n_dec_taps, n_lpf_taps;
} sdrb_sub_info;

/* Plan compiler: QSettings ini grammar + mainwindow.cpp:29-235, Qt-free. */
int sdrb_plan_from_ini(const char *ini_path, sdrb_plan **out);
/* Same plan from explicit numbers (what the vfo setters carry, vfo.cpp:177-233). */
int sdrb_plan_create(const sdrb_plan_desc *desc, sdrb_plan **out);
void sdrb_plan_destroy(sdrb_plan *plan);
int sdrb_plan_get_info(const sdrb_plan *plan, sdrb_plan_info *info);
int sdrb_plan_get_main(const sdrb_plan *plan, int idx, sdrb_main_info *info);
int sdrb_plan_get_sub(const sdrb_plan *plan, int idx, sdrb_sub_info *info);
/* Any key of the ini file the plan was compiled from, named as QSettings names it ("tuner_gain",
 * "remote_rtl", "auto_start", "disable_fft", "main_vfos/2/zmq_topic", "vfos/3/gain", ...): the
 * operational keys MainWindow reads for the device and the GUI (mainwindow.cpp:51-96) are not used by
 * the hot path but stay available to the application through the same parser. Returns the value's
 * length (copied, truncated to out_len-1, NUL-terminated) or -1 if the key is absent / the plan was
 * built from a description. */
int sdrb_plan_get_setting(const sdrb_plan *plan, const char *key, char *out, size_t out_len);
/* Host copies of the tables vfo::init builds (vfo.cpp:60-137), for inspection/tests:
 * kind 0 = main NCO table (cf32, (int)Fs entries), 1 = sub NCO table, 2 = sub /late FIR
 * taps, 3 = sub low-pass taps, 4 = Hilbert points (125). Returns the element count
 * (complex entries for 0/1, floats otherwise); copies at most max_elems. */
long sdrb_plan_copy_table(const sdrb_plan *plan, int kind, int idx, float *dst, long max_elems);

/* ---- receiver bank: replaces sdrj + the vfo tree for n_streams independent dongles ---- */
int sdrb_bank_create(const sdrb_plan *plan, int device, int n_streams, int max_blocks, sdrb_bank **out);
void sdrb_bank_destroy(sdrb_bank *bank);
/* Fresh filter/NCO/DC state, as after constructing the reference objects. stream = -1: all. */
int sdrb_bank_reset(sdrb_bank *bank, int stream);
/* Per-stream blocks consumed so far (sample counter / block). */
int sdrb_bank_blocks_done(sdrb_bank *bank, int stream, int64_t *blocks);

/*
 * n_blocks callbacks for every stream of the bank, everything resident on the device.
 * Stands in for n_blocks x { sdr::rtlsdr_callback (jonti/sdr.cpp:100-145) -> sdrj::demodData
 * (sdrj.cpp:266-305) -> vfo::process tree (vfo.cpp:235-296) } per stream.
 *   d_iq   device, stream s at d_iq + s*iq_stride, n_blocks*block*2 bytes of uint8 I,Q
 *   d_pcm  device int16 [n_streams][n_blocks][pcm_per_block]; VFO v of callback b of stream s
 *          starts at ((s*n_blocks + b)*pcm_per_block + pcm_offset[v]) -- each slice is one
 *          ready-made ZMQ payload (vfo::transmitData, vfo.cpp:426-453)
 *   d_tap  optional (NULL = off) float32, same layout: usb*gain*32768 before conversion
 *   stream cudaStream_t (NULL = default stream); the call only enqueues work
 */
int sdrb_bank_process_device(sdrb_bank *bank, const uint8_t *d_iq, size_t iq_stride, int n_blocks,
                             int16_t *d_pcm, float *d_tap, void *cuda_stream);
/* Same call for a streaming caller that double-buffers its input: `input_ready_event` is a
 * cudaEvent_t (NULL = behave like sdrb_bank_process_device) that fires when d_iq is valid. The
 * DC-removal pre-pass (a sequential recursion, sdrj.cpp:277-283, run on an internal side stream)
 * then waits only for that event, not for the work queued on `stream` before this call, and
 * overlaps the filters of the previous call. Everything the caller observes (d_pcm, d_tap, state)
 * is still ordered on `stream`. */
int sdrb_bank_process_device_ex(sdrb_bank *bank, const uint8_t *d_iq, size_t iq_stride, int n_blocks,
                                int16_t *d_pcm, float *d_tap, void *cuda_stream, void *input_ready_event);
/* Copy out the main VFO outputs (vfo::decimate[decimateCount], vfo.h:39) of the last
 * process call: cf32 [n_streams][n_blocks*block_out] on the device. */
int sdrb_bank_copy_main(sdrb_bank *bank, int main_idx, int n_blocks, float *d_out_cf32, void *cuda_stream);

/* Spectrum sources of the last process call, as the reference emits them through fftData:
 *   input: the `samples` vector of sdrj::demodData (sdrj.cpp:271-294; shown when "Main" is selected,
 *          sdrj.cpp:296-303): converted and, with correct_dc_bias, DC-corrected input of callback
 *          `cb`, first n samples (n a multiple of 128, <= block): cf32 [n_streams][n]. Bit-identical
 *          to the reference. For the device entry points the d_iq of that call must still be valid.
 *   sub:   vfo::decimate[decimateCount] of sub VFO sub_idx (vfo.cpp:290-293; shown when that VFO is
 *          selected): cf32 [n_streams][n_blocks*block_z], block_z = (in_rate/bufsplit) >> decim. */
int sdrb_bank_copy_input(sdrb_bank *bank, int cb, int n, float *d_out_cf32, void *cuda_stream);
int sdrb_bank_read_input(sdrb_bank *bank, int cb, int n, float *h_out_cf32);
int sdrb_bank_copy_sub(sdrb_bank *bank, int sub_idx, int n_blocks, float *d_out_cf32, void *cuda_stream);
int sdrb_bank_read_sub(sdrb_bank *bank, int sub_idx, int n_blocks, float *h_out_cf32);

/* IQ forwarder output of the last process call (vfo::compress, vfo.cpp:389-424, followed by
 * vfo::transmitData, vfo.cpp:439-451): for main VFO `main_idx` the packed bytes of every stream,
 * uint8 [n_streams][n_blocks*fwd_bytes_per_block]; each fwd_bytes_per_block slice is one ZMQ
 * payload (rate frame = the main VFO's out_rate). Computed on demand from the main VFO output,
 * valid for any main VFO (the reference runs compress() only where there are no sub VFOs). */
int sdrb_bank_copy_forward(sdrb_bank *bank, int main_idx, int n_blocks, uint8_t *d_out, void *cuda_stream);
int sdrb_bank_read_forward(sdrb_bank *bank, int main_idx, int n_blocks, uint8_t *h_out);

/* Inspection: the DC-removal state (sdrj.cpp:280 `avept`) entering every 128th sample of the
 * last process call, float2 (I,Q) [n_streams][n_blocks*block/128] on the device. The kernels
 * reproduce the reference's float recursion bit for bit; tests compare this trace exactly.
 * d_modes (optional, NULL = off): one byte per entry, low nibble I arm, high nibble Q arm:
 * 0/1 = the 128 samples were advanced as one integer translation, 2 = stepped in float. */
int sdrb_bank_copy_dc_trace(sdrb_bank *bank, int n_blocks, float *d_out, uint8_t *d_modes, void *cuda_stream);

/*
 * Host-facing call: same work with HOST buffers (pinned from sdrb_host_alloc for full
 * speed; pageable memory works but is staged by the driver). Copies in, runs, copies out
 * and returns when h_pcm is complete. Streams are split into groups whose H2D copy,
 * kernels and D2H copy overlap on separate CUDA streams.
 */
int sdrb_bank_process_host(sdrb_bank *bank, const uint8_t *h_iq, size_t iq_stride, int n_blocks,
                           int16_t *h_pcm, float *h_tap);
/* The same call without the final wait: returns once everything is enqueued. Several calls may be
 * in flight; the library orders them chunk by chunk, so the copy-in of the next call overlaps the
 * filters and the copy-out of the current one and the PCIe link never idles between calls. Each
 * call in flight needs its own h_iq / h_pcm / h_tap (pinned) until sdrb_bank_host_wait has
 * returned. Every other entry point waits for outstanding asynchronous calls first. */
int sdrb_bank_process_host_async(sdrb_bank *bank, const uint8_t *h_iq, size_t iq_stride, int n_blocks,
                                 int16_t *h_pcm, float *h_tap);
int sdrb_bank_host_wait(sdrb_bank *bank);                               /* all of them */
int sdrb_bank_host_wait_until(sdrb_bank *bank, int max_in_flight);      /* oldest first, until <= max_in_flight remain */
/* vfo::process entry (vfo.cpp:235-296): the caller supplies complex float samples (what
 * sdrj::demodData hands to the main VFOs, i.e. already converted and DC-corrected by the
 * caller); everything from the main-VFO mix on runs on the GPU. h_in: cf32, stream s at
 * h_in + 2*s*stride_samples floats. State is shared with the uint8 entry points, do not mix
 * the two kinds of calls on one bank without a reset. */
int sdrb_bank_process_cf32_host(sdrb_bank *bank, const float *h_in_cf32, size_t stride_samples, int n_blocks,
                                int16_t *h_pcm, float *h_tap);
/* Main VFO outputs of the last call, to host: cf32 [n_streams][n_blocks*block_out]
 * (vfo::decimate[decimateCount], vfo.h:39). */
int sdrb_bank_read_main(sdrb_bank *bank, int main_idx, int n_blocks, float *h_out_cf32);
/* Kernel launches issued by the last process_* call (for bench.py's gpu_launches). */
int sdrb_bank_last_launches(const sdrb_bank *bank);
/* Per-kernel-class device timing (CUDA events on the launching stream), for roofline
 * reporting: classes 0 DC scan, 1 ingest+main VFOs, 2 sub-VFO cascades, 3 /late FIR,
 * 4 USB audio, 5 carry. set_timing(.., 1) starts/clears; kernel_times synchronises the
 * device and returns accumulated milliseconds and number of timed calls per class. */
#define SDRB_N_KERNEL_CLASSES 6
int sdrb_bank_set_timing(sdrb_bank *bank, int on);
int sdrb_bank_kernel_times(sdrb_bank *bank, double *ms, long *calls);

/* FP32 peak of the current device, measured: a register-only loop of independent FMA chains on every
 * SM, timed with CUDA events (best of `reps`). packed = 0: scalar FFMA; 1: FFMA2 (fma.rn.f32x2, the
 * form the half-band and USB kernels use). Result in TFLOP/s (2 flop per FMA lane). This is the FP32
 * denominator of bench.py's roofline (SURVEY 8(d): "measure an FMA-loop peak on the box"). */
int sdrb_probe_fp32_tflops(int packed, int reps, double *tflops);

void *sdrb_host_alloc(size_t bytes);   /* cudaHostAlloc'd (pinned) */
void sdrb_host_free(void *p);

/* ---- per-class primitives backing the C++ facades (device pointers, batch of `n_ch`
 *      independent channels laid out channel-major) ---- */
/* Oscillator (oscillator.cpp:4-50): host-built table, bit-identical to the reference. */
long sdrb_nco_table(double sample_rate, double frequency, float *dst_cf32, long max_entries);
/* vfo::process mix loop (vfo.cpp:237-245): out[i] = table[idx(n0+i)] * in[i]. */
int sdrb_nco_mix(const float *d_table_cf32, int table_len, int64_t n0, const float *d_in_cf32,
                 float *d_out_cf32, int n_ch, int n, void *cuda_stream);
/* HalfBandDecimator::decimate (halfbanddecimator.cpp:43-72), taps = 11: one call = one
 * block of n (even) samples per channel; d_hist holds the 11-sample queue head per channel
 * and is updated with the reference's off-by-one carry (jonti/dsp.cpp:163-173). */
int sdrb_halfband11(const float *d_in_cf32, float *d_out_cf32, float *d_hist_cf32, int n_ch, int n,
                    void *cuda_stream);
/* The same class with its other filter lengths (halfbanddecimator.h:28-63, .cpp:10-34): taps = 11,
 * 23 or 51 use the reference's tables; any other odd length behaves like the reference, whose
 * switch has no case for it (15 and 21 have tables that are never loaded): all outputs are 0.
 * d_hist = `taps` complex samples per channel, zero for a fresh object. Any even n >= 2. */
int sdrb_halfband(int taps, const float *d_in_cf32, float *d_out_cf32, float *d_hist_cf32, int n_ch, int n,
                  void *cuda_stream);
/* FIR::FIRUpdateAndProcess over a block (jonti/dsp.cpp:59-71): newest sample excluded;
 * d_hist = last ntaps inputs per channel (updated); decim >= 1 keeps every decim-th output
 * starting with the first (vfo::usb_decimdemod, vfo.cpp:334-387). Any block length n >= 1. */
int sdrb_fir(const float *d_taps, int ntaps, const float *d_in, float *d_out, float *d_hist, int n_ch,
             int n, int decim, void *cuda_stream);
/* Same with include_newest = 1: the FIRHilbert form y[m] = sum_i taps[i]*x[m - N + 1 + i]
 * (jonti/dsp.cpp:218-231, ring of N with the newest sample included). Any n >= 1. */
int sdrb_fir_ex(const float *d_taps, int ntaps, const float *d_in, float *d_out, float *d_hist, int n_ch,
                int n, int decim, int include_newest, void *cuda_stream);
/* delay(62)(re) - FIRHilbert125(im) (vfo.cpp:316-324; jonti/dsp.cpp:184-231); d_points = the
 * 125 FIRHilbert coefficients on the device (sdrb_hilbert_points), d_hist = last 124 complex
 * inputs per channel (updated). */
int sdrb_usb_demod(const float *d_points, const float *d_in_cf32, float *d_out, float *d_hist_cf32,
                   int n_ch, int n, void *cuda_stream);
/* vfo::compress (vfo.cpp:389-424) on n complex samples per channel. style 1: out[i] =
 * ((signed char)((re/scale)*128) & 0xF0) | (((signed char)((im/scale)*128) & 0xF0) >> 4), n bytes
 * per channel; otherwise out[2i] = (signed char)(re*128), out[2i+1] = (signed char)(im*128), 2n
 * bytes. Conversions truncate toward zero and keep the low 8 bits (what the reference's x86 build
 * does; it is undefined behaviour in C++ outside -128..127). */
int sdrb_compress_iq(const float *d_in_cf32, uint8_t *d_out, int n_ch, int n, int scale, int style, void *cuda_stream);
/* gnuradio firdes low_pass, Hamming (gnuradio/firfilter.cpp:64-108). Returns ntaps or
 * SDRB_E_INVALID where the reference throws std::out_of_range. Host only. */
int sdrb_low_pass(double gain, double fs, double cutoff, double tw, float *taps, int max_taps);
/* FIRHilbert coefficients (jonti/dsp.cpp:198-216). Host only. */
int sdrb_hilbert_points(int len, int fs, float *points);

/* ---- spectrum path: Hann window + 8192-point FFT (mainwindow.cpp:411-455, kiss_fft) ---- */
int sdrb_spectrum_fft(const float *d_in_cf32, float *d_out_cf32, int n_batch, int nfft, int apply_hann,
                      void *cuda_stream);

/* The spectrum display MainWindow keeps (fftHandlerSlot, mainwindow.cpp:411-455; state
 * mainwindow.h:54-72), for n_displays independent displays (e.g. one per receiver of a bank):
 *   inr[a] = data[a]*hann[a] for a < min(nfft, len) -- samples beyond `len` keep their previous
 *            value, as in the reference when a sub VFO's short buffer is shown (cpp:418-425);
 *   X = FFT(inr);  pwr[b] = 0.95*pwr[b] + 0.05*10*log10(max(1e5*|X[i]|/nfft, 1)), b = i + nfft/2 mod nfft;
 *   smooth[i] = mean(pwr[i..i+4]), i < nfft-10;  stats = {maxval, aveval} as used for the y axis.
 * pwr/smooth/stats are double like the reference's QVector<double>. reset = what selecting
 * another VFO in the combo box does (mainwindow.cpp:539-551): pwr and inr to zero. */
typedef struct sdrb_spectrum sdrb_spectrum;
int sdrb_spectrum_create(int device, int n_displays, int nfft, sdrb_spectrum **out);
void sdrb_spectrum_destroy(sdrb_spectrum *sp);
int sdrb_spectrum_reset(sdrb_spectrum *sp, int display /* -1 = all */);
/* One fftHandlerSlot per display. d_in_cf32: display k reads complex samples at
 * d_in + 2*k*in_stride floats; len = data.size() of the reference's signal (any length >= 0).
 * d_fft_out (optional): the complex spectrum X, cf32 [n_displays][nfft]. Only enqueues. */
int sdrb_spectrum_feed_device(sdrb_spectrum *sp, const float *d_in_cf32, size_t in_stride, int len, float *d_fft_out,
                              void *cuda_stream);
int sdrb_spectrum_feed_host(sdrb_spectrum *sp, const float *h_in_cf32, size_t in_stride, int len);
/* The batched form: one fftHandlerSlot per receiver of `bank` (sp must have n_streams displays on
 * the same device) straight from the bank's device buffers, callback `cb` of the last process
 * call. source -1 = "Main": the DC-corrected input samples, emitted by the reference on every
 * 4th callback (sdrj.cpp:296-303); source k >= 0 = sub VFO k's decimate[decimateCount], emitted
 * on every callback while that VFO is selected (vfo.cpp:290-293). Only enqueues. */
int sdrb_bank_spectrum_feed(sdrb_bank *bank, sdrb_spectrum *sp, int source, int cb, float *d_fft_out, void *cuda_stream);
/* Host copies (any pointer may be NULL): smooth double [n][nfft-10], pwr double [n][nfft],
 * stats double [n][2] = {maxval, aveval}. Synchronises the device. */
int sdrb_spectrum_read(sdrb_spectrum *sp, double *h_smooth, double *h_pwr, double *h_stats);

/* ---- ZMQ output (zmqpublisher.cpp:15-96), libzmq loaded at run time ---- */
typedef struct sdrb_publisher sdrb_publisher;
int sdrb_publisher_open(const char *address, int bind, sdrb_publisher **out);
int sdrb_publisher_send(sdrb_publisher *p, const char *topic, uint32_t rate, const void *payload, uint32_t len);
/* One multipart message per sub VFO per callback per stream from a process_host result. */
int sdrb_publisher_send_block(sdrb_publisher *p, const sdrb_plan *plan, const int16_t *h_pcm_record);
/* Closes socket and context. The reference never closes its sockets (they end with the process, queued frames are
 * dropped): close() does the same with ZMQ_LINGER 0. Set SDRB_ZMQ_LINGER_MS (milliseconds, -1 = wait for ever, libzmq's
 * default) before sdrb_publisher_open to let queued frames drain first. */
void sdrb_publisher_close(sdrb_publisher *p);
/* A pool of publishers: n_sockets PUB sockets, one sender thread each. The reference runs one process -- one ZmqPublisher
 * (zmqpublisher.cpp:15-96), one address -- per dongle; a bank holds hundreds of receivers, and a single socket fed by a single
 * thread caps the publish leg far below the rest of the path. Receiver s is sent on socket s % n_sockets, its callbacks in order,
 * every message in the reference's three-frame format. Socket k's address: "%d" in `address` replaced by k; else a tcp port
 * + k; else ".k" appended (n_sockets == 1: `address` as it is). sdrb_publisher_pool_send_call takes the [n_streams][n_blocks]
 * [pcm_per_block] result of one process_host call and returns when every frame has been handed to libzmq; one caller at a time.
 * Socket options are the reference's (zmqpublisher.cpp:24-37) except the send high-water mark: a pool socket queues a whole call's
 * burst before its I/O thread has written any of it, so it is 65536 messages instead of libzmq's 1000 per subscriber
 * (SDRB_ZMQ_SNDHWM overrides it for pool and single publishers alike, 0 = no limit). */
typedef struct sdrb_publisher_pool sdrb_publisher_pool;
int sdrb_publisher_pool_open(const char *address, int bind, int n_sockets, sdrb_publisher_pool **out);
int sdrb_publisher_pool_sockets(const sdrb_publisher_pool *pool);
int sdrb_publisher_pool_address(const sdrb_publisher_pool *pool, int k, char *buf, size_t len);
int sdrb_publisher_pool_send_call(sdrb_publisher_pool *pool, const sdrb_plan *plan, const int16_t *h_pcm, int n_streams, int n_blocks);
void sdrb_publisher_pool_close(sdrb_publisher_pool *pool);

/* ---- ingest front ends, host side (the library opens no socket and no dongle) ---- */
/* rtl_tcp client protocol as spoken by sdrj (sdrj.cpp:31-74, 125-188). Feed whatever the socket
 * delivers: the 12-byte dongle header "RTL0" + tuner type + gain count (big endian, sdrj.cpp:134-149)
 * is recognised at the start of the stream, everything after it is uint8 IQ, cut into callback
 * blocks of block_bytes (0 = the reference's (sample_rate/4)*2, sdrj.cpp:46). A stream that does
 * not start with "RTL0" (a recording) is all samples. */
typedef struct sdrb_rtltcp sdrb_rtltcp;
int sdrb_rtltcp_create(int sample_rate, size_t block_bytes, sdrb_rtltcp **out);
void sdrb_rtltcp_destroy(sdrb_rtltcp *f);
size_t sdrb_rtltcp_block_bytes(const sdrb_rtltcp *f);
int sdrb_rtltcp_feed(sdrb_rtltcp *f, const uint8_t *bytes, size_t n);    /* >= 0: complete blocks waiting */
int sdrb_rtltcp_header(const sdrb_rtltcp *f, uint32_t *tuner_type, uint32_t *gain_count);   /* 1 once seen */
int sdrb_rtltcp_pop(sdrb_rtltcp *f, uint8_t *dst_block);                 /* 1 = one block copied, 0 = none */
/* Commands (sdrj.h:10-16; sdrj::sendCommand, sdrj.cpp:168-188): 1 command byte + value, MSB first. */
#define SDRB_RTLTCP_SET_FREQ 0x01
#define SDRB_RTLTCP_SET_SAMPLE_RATE 0x02
#define SDRB_RTLTCP_SET_TUNER_GAIN_MODE 0x03
#define SDRB_RTLTCP_SET_GAIN 0x04
#define SDRB_RTLTCP_SET_FREQ_COR 0x05
#define SDRB_RTLTCP_SET_AGC_MODE 0x08
#define SDRB_RTLTCP_SET_TUNER_GAIN_INDEX 0x0d
void sdrb_rtltcp_command(uint8_t cmd, uint32_t value, uint8_t out[5]);
/* What sdrj::start_tcp_rtl sends after connecting (sdrj.cpp:56-66): AGC off, manual gain, gain
 * index, sample rate, centre frequency -- 25 bytes. */
int sdrb_rtltcp_start_sequence(int sample_rate, int frequency, int gain_index, uint8_t out[25]);

/* The hand-over ring between the librtlsdr callback thread and the demodulator thread
 * (jonti/sdr.cpp:100-184; N_BUFFERS = 20, jonti/sdr.h:83). push = sdr::rtlsdr_callback: returns 1,
 * or 0 when all buffers are in use and the new one is DROPPED, like the reference. pop =
 * sdr::demod_dispatcher: waits (timeout_ms < 0: for ever) and lends the oldest buffer until
 * sdrb_ring_release. Buffers hold raw bytes and are pinned when `pinned` != 0, so that
 * sdrb_bank_process_host can DMA straight out of them. One producer, one consumer. */
typedef struct sdrb_ring sdrb_ring;
int sdrb_ring_create(size_t block_bytes, int n_buffers /* 0 = 20 */, int pinned, sdrb_ring **out);
void sdrb_ring_destroy(sdrb_ring *r);
int sdrb_ring_push(sdrb_ring *r, const uint8_t *bytes, uint32_t len);
int sdrb_ring_pop(sdrb_ring *r, const uint8_t **bytes, uint32_t *len, int timeout_ms);
int sdrb_ring_release(sdrb_ring *r);
void sdrb_ring_cancel(sdrb_ring *r);
int sdrb_ring_stats(sdrb_ring *r, uint64_t *pushed, uint64_t *dropped, int *used);

const char *sdrb_last_error(void);
const char *sdrb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SDRB200_H */
