"""ctypes binding of libsdrb200.so (include/sdrb200.h).

Thin by design: every call below is one C-ABI entry point. torch is used by callers only
for device memory and streams (tensor.data_ptr(), torch.cuda.current_stream()); nothing
here computes. If the CUDA library is missing this module raises -- there is no fallback.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SDRB_LIB") or os.path.join(_HERE, "libsdrb200.so")   # SDRB_LIB: kernel-variant experiments

SDRB_MAX_MAIN, SDRB_MAX_SUB = 8, 256


class SdrbError(RuntimeError):
    pass


class MainDesc(C.Structure):
    _fields_ = [("mixer_hz", C.c_double), ("decim", C.c_int32), ("topic", C.c_char * 8),
                ("compress_scale", C.c_int32), ("compress_style", C.c_int32)]


class SubDesc(C.Structure):
    _fields_ = [("topic", C.c_char * 8), ("main_idx", C.c_int32), ("mixer_hz", C.c_double),
                ("decim", C.c_int32), ("late", C.c_int32), ("filter_bw", C.c_int32), ("gain", C.c_float)]


class PlanDesc(C.Structure):
    _fields_ = [("sample_rate", C.c_int32), ("block", C.c_int32), ("bufsplit", C.c_int32),
                ("correct_dc", C.c_int32), ("n_main", C.c_int32), ("n_sub", C.c_int32),
                ("mains", MainDesc * SDRB_MAX_MAIN), ("subs", SubDesc * SDRB_MAX_SUB)]


class PlanInfo(C.Structure):
    _fields_ = [("sample_rate", C.c_int32), ("block", C.c_int32), ("bufsplit", C.c_int32),
                ("correct_dc", C.c_int32), ("n_main", C.c_int32), ("n_sub", C.c_int32),
                ("center_frequency", C.c_int32), ("pcm_per_block", C.c_int32),
                ("alg_bytes_per_sample", C.c_double), ("alg_flops_per_sample", C.c_double),
                ("zmq_address", C.c_char * 128)]


class MainInfo(C.Structure):
    _fields_ = [("mixer_hz", C.c_double), ("frequency", C.c_int32), ("decim", C.c_int32),
                ("out_rate", C.c_int32), ("block_out", C.c_int32), ("n_subs", C.c_int32), ("forward", C.c_int32),
                ("compress_scale", C.c_int32), ("compress_style", C.c_int32), ("fwd_bytes_per_block", C.c_int32),
                ("topic", C.c_char * 8), ("zmq_address", C.c_char * 128)]


class SubInfo(C.Structure):
    _fields_ = [("topic", C.c_char * 8), ("frequency", C.c_int32), ("data_rate", C.c_int32),
                ("main_idx", C.c_int32), ("decim", C.c_int32), ("late", C.c_int32), ("filter_bw", C.c_int32),
                ("gain", C.c_float), ("mixer_hz", C.c_double), ("in_rate", C.c_int32), ("out_rate", C.c_int32),
                ("samples_out", C.c_int32), ("pcm_offset", C.c_int32), ("n_dec_taps", C.c_int32),
                ("n_lpf_taps", C.c_int32)]


_lib = None


def lib():
    """Load libsdrb200.so (raises if it has not been built: `python -c 'import __graft_entry__ as g; g.build()'`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SdrbError("%s is missing: build it with __graft_entry__.build(); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i, d, f, l, sz = C.c_void_p, C.c_int, C.c_double, C.c_float, C.c_long, C.c_size_t
    P = C.POINTER
    sig = {
        "sdrb_plan_from_ini": (i, [C.c_char_p, P(vp)]),
        "sdrb_plan_create": (i, [P(PlanDesc), P(vp)]),
        "sdrb_plan_destroy": (None, [vp]),
        "sdrb_plan_get_info": (i, [vp, P(PlanInfo)]),
        "sdrb_plan_get_main": (i, [vp, i, P(MainInfo)]),
        "sdrb_plan_get_sub": (i, [vp, i, P(SubInfo)]),
        "sdrb_plan_copy_table": (l, [vp, i, i, vp, l]),
        "sdrb_plan_get_setting": (i, [vp, C.c_char_p, C.c_char_p, sz]),
        "sdrb_bank_create": (i, [vp, i, i, i, P(vp)]),
        "sdrb_bank_destroy": (None, [vp]),
        "sdrb_bank_reset": (i, [vp, i]),
        "sdrb_bank_blocks_done": (i, [vp, i, P(C.c_int64)]),
        "sdrb_plan_fingerprint": (i, [vp, P(C.c_uint64)]),
        "sdrb_bank_state_bytes": (sz, [vp]),
        "sdrb_bank_save_state": (i, [vp, vp, i, vp, vp]),
        "sdrb_bank_load_state": (i, [vp, vp, i, vp, vp]),
        "sdrb_bank_read_state": (i, [vp, vp, i, vp]),
        "sdrb_bank_write_state": (i, [vp, vp, i, vp]),
        "sdrb_bank_process_device": (i, [vp, vp, sz, i, vp, vp, vp]),
        "sdrb_bank_process_device_ex": (i, [vp, vp, sz, i, vp, vp, vp, vp]),
        "sdrb_bank_process_streams_device": (i, [vp, vp, i, vp, sz, i, vp, vp, vp, vp]),
        "sdrb_bank_process_streams_host": (i, [vp, vp, i, vp, i, vp, vp]),
        "sdrb_bank_copy_main": (i, [vp, i, i, vp, vp]),
        "sdrb_bank_copy_dc_trace": (i, [vp, i, vp, vp, vp]),
        "sdrb_bank_copy_forward": (i, [vp, i, i, vp, vp]),
        "sdrb_bank_read_forward": (i, [vp, i, i, vp]),
        "sdrb_compress_iq": (i, [vp, vp, i, i, i, i, vp]),
        "sdrb_bank_process_host": (i, [vp, vp, sz, i, vp, vp]),
        "sdrb_bank_process_cf32_host": (i, [vp, vp, sz, i, vp, vp]),
        "sdrb_bank_process_host_async": (i, [vp, vp, sz, i, vp, vp]),
        "sdrb_bank_host_wait": (i, [vp]),
        "sdrb_bank_host_wait_until": (i, [vp, i]),
        "sdrb_bank_read_main": (i, [vp, i, i, vp]),
        "sdrb_bank_last_launches": (i, [vp]),
        "sdrb_bank_set_timing": (i, [vp, i]),
        "sdrb_bank_kernel_times": (i, [vp, vp, vp]),
        "sdrb_probe_fp32_tflops": (i, [i, i, P(d)]),
        "sdrb_host_alloc": (vp, [sz]),
        "sdrb_host_free": (None, [vp]),
        "sdrb_nco_table": (l, [d, d, vp, l]),
        "sdrb_nco_mix": (i, [vp, i, C.c_int64, vp, vp, i, i, vp]),
        "sdrb_halfband11": (i, [vp, vp, vp, i, i, vp]),
        "sdrb_halfband": (i, [i, vp, vp, vp, i, i, vp]),
        "sdrb_fir": (i, [vp, i, vp, vp, vp, i, i, i, vp]),
        "sdrb_fir_ex": (i, [vp, i, vp, vp, vp, i, i, i, i, vp]),
        "sdrb_usb_demod": (i, [vp, vp, vp, vp, i, i, vp]),
        "sdrb_low_pass": (i, [d, d, d, d, vp, i]),
        "sdrb_hilbert_points": (i, [i, i, vp]),
        "sdrb_spectrum_fft": (i, [vp, vp, i, i, i, vp]),
        "sdrb_spectrum_create": (i, [i, i, i, P(vp)]),
        "sdrb_spectrum_destroy": (None, [vp]),
        "sdrb_spectrum_reset": (i, [vp, i]),
        "sdrb_spectrum_feed_device": (i, [vp, vp, sz, i, vp, vp]),
        "sdrb_spectrum_feed_host": (i, [vp, vp, sz, i]),
        "sdrb_spectrum_read": (i, [vp, vp, vp, vp]),
        "sdrb_bank_spectrum_feed": (i, [vp, vp, i, i, vp, vp]),
        "sdrb_bank_copy_input": (i, [vp, i, i, vp, vp]),
        "sdrb_bank_read_input": (i, [vp, i, i, vp]),
        "sdrb_bank_copy_sub": (i, [vp, i, i, vp, vp]),
        "sdrb_bank_read_sub": (i, [vp, i, i, vp]),
        "sdrb_rtltcp_create": (i, [i, sz, P(vp)]),
        "sdrb_rtltcp_destroy": (None, [vp]),
        "sdrb_rtltcp_block_bytes": (sz, [vp]),
        "sdrb_rtltcp_feed": (i, [vp, vp, sz]),
        "sdrb_rtltcp_header": (i, [vp, P(C.c_uint32), P(C.c_uint32)]),
        "sdrb_rtltcp_pop": (i, [vp, vp]),
        "sdrb_rtltcp_command": (None, [C.c_uint8, C.c_uint32, vp]),
        "sdrb_rtltcp_start_sequence": (i, [i, i, i, vp]),
        "sdrb_ring_create": (i, [sz, i, i, P(vp)]),
        "sdrb_ring_destroy": (None, [vp]),
        "sdrb_ring_push": (i, [vp, vp, C.c_uint32]),
        "sdrb_ring_pop": (i, [vp, P(vp), P(C.c_uint32), i]),
        "sdrb_ring_release": (i, [vp]),
        "sdrb_ring_cancel": (None, [vp]),
        "sdrb_ring_stats": (i, [vp, P(C.c_uint64), P(C.c_uint64), P(i)]),
        "sdrb_publisher_open": (i, [C.c_char_p, i, P(vp)]),
        "sdrb_publisher_send": (i, [vp, C.c_char_p, C.c_uint32, vp, C.c_uint32]),
        "sdrb_publisher_send_block": (i, [vp, vp, vp]),
        "sdrb_publisher_close": (None, [vp]),
        "sdrb_publisher_pool_open": (i, [C.c_char_p, i, i, P(vp)]),
        "sdrb_publisher_pool_sockets": (i, [vp]),
        "sdrb_publisher_pool_address": (i, [vp, i, C.c_char_p, C.c_size_t]),
        "sdrb_publisher_pool_send_call": (i, [vp, vp, vp, i, i]),
        "sdrb_publisher_pool_send_streams": (i, [vp, vp, vp, vp, i, i]),
        "sdrb_publisher_pool_close": (None, [vp]),
        "sdrb_last_error": (C.c_char_p, []),
        "sdrb_version": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        raise SdrbError("%s failed (%d): %s" % (what, rc, lib().sdrb_last_error().decode("utf-8", "replace")))


class Plan:
    """Immutable VFO plan (ini -> rates, tree, NCO tables, filter taps)."""

    def __init__(self, ini_path=None, desc=None):
        L = lib()
        h = C.c_void_p()
        if ini_path is not None:
            _check(L.sdrb_plan_from_ini(os.fsencode(ini_path), C.byref(h)), "sdrb_plan_from_ini")
        else:
            _check(L.sdrb_plan_create(C.byref(desc), C.byref(h)), "sdrb_plan_create")
        self.h = h
        self.path = None if ini_path is None else os.fspath(ini_path)      # the ini this plan came from (None: built from a descriptor)
        info = PlanInfo()
        _check(L.sdrb_plan_get_info(h, C.byref(info)), "sdrb_plan_get_info")
        self.info = info
        self.fs, self.block, self.bufsplit = info.sample_rate, info.block, info.bufsplit
        self.correct_dc, self.center = bool(info.correct_dc), info.center_frequency
        self.pcm_per_block = info.pcm_per_block
        self.alg_bytes, self.alg_flops = info.alg_bytes_per_sample, info.alg_flops_per_sample
        self.zmq_address = info.zmq_address.decode()
        self.mains, self.subs = [], []
        for k in range(info.n_main):
            m = MainInfo()
            _check(L.sdrb_plan_get_main(h, k, C.byref(m)), "sdrb_plan_get_main")
            self.mains.append({"mixer": m.mixer_hz, "freq": m.frequency, "decim": m.decim,
                               "out_rate": m.out_rate, "block_out": m.block_out, "n_subs": m.n_subs,
                               "forward": bool(m.forward), "scalecomp": m.compress_scale, "cstyle": m.compress_style,
                               "fwd_bytes": m.fwd_bytes_per_block, "topic": m.topic.decode(),
                               "zmq_address": m.zmq_address.decode()})
        for k in range(info.n_sub):
            s = SubInfo()
            _check(L.sdrb_plan_get_sub(h, k, C.byref(s)), "sdrb_plan_get_sub")
            self.subs.append({"topic": s.topic.decode(), "freq": s.frequency, "data_rate": s.data_rate,
                              "main": s.main_idx, "decim": s.decim, "late": s.late, "filterbw": s.filter_bw,
                              "gain": s.gain, "mixer": s.mixer_hz, "Fs": s.in_rate, "out_rate": s.out_rate,
                              "samples_out": s.samples_out, "pcm_offset": s.pcm_offset,
                              "n_dec_taps": s.n_dec_taps, "n_lpf_taps": s.n_lpf_taps})

    @classmethod
    def from_desc(cls, fs, block, bufsplit, correct_dc, mains, subs):
        d = PlanDesc()
        d.sample_rate, d.block, d.bufsplit, d.correct_dc = fs, block, bufsplit, int(correct_dc)
        d.n_main, d.n_sub = len(mains), len(subs)
        for k, m in enumerate(mains):
            d.mains[k].mixer_hz, d.mains[k].decim = m["mixer"], m["decim"]
            d.mains[k].topic = m.get("topic", "").encode()[:7]
            d.mains[k].compress_scale, d.mains[k].compress_style = m.get("scalecomp", 1), m.get("cstyle", 1)
        for k, s in enumerate(subs):
            d.subs[k].topic = s.get("topic", "VFO%02d" % k).encode()[:7]
            d.subs[k].main_idx, d.subs[k].mixer_hz = s["main"], s["mixer"]
            d.subs[k].decim, d.subs[k].late = s["decim"], s.get("late", 0)
            d.subs[k].filter_bw, d.subs[k].gain = s.get("filterbw", 0), s.get("gain", 0.01)
        return cls(desc=d)

    @property
    def fingerprint(self):
        """64-bit hash of everything in the plan that can change an output sample (sdrb_plan_fingerprint)."""
        v = C.c_uint64()
        _check(lib().sdrb_plan_fingerprint(self.h, C.byref(v)), "sdrb_plan_fingerprint")
        return v.value

    def setting(self, key, default=None):
        """Value of an ini key as QSettings names it, or `default`."""
        buf = C.create_string_buffer(512)
        n = lib().sdrb_plan_get_setting(self.h, key.encode(), buf, 512)
        return default if n < 0 else buf.value.decode()

    def table(self, kind, idx):
        L = lib()
        n = L.sdrb_plan_copy_table(self.h, kind, idx, None, 0)
        if n < 0:
            _check(int(n), "sdrb_plan_copy_table")
        width = 2 if kind in (0, 1) else 1
        out = np.zeros(n * width, dtype=np.float32)
        L.sdrb_plan_copy_table(self.h, kind, idx, out.ctypes.data_as(C.c_void_p), n)
        return out.view(np.complex64) if width == 2 else out

    def close(self):
        if getattr(self, "h", None):
            lib().sdrb_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Bank:
    """n_streams receivers of one plan on one GPU (sdrj + vfo tree, batched)."""

    def __init__(self, plan, n_streams, max_blocks, device=0):
        self.plan, self.n_streams, self.max_blocks, self.device = plan, n_streams, max_blocks, device
        h = C.c_void_p()
        _check(lib().sdrb_bank_create(plan.h, device, n_streams, max_blocks, C.byref(h)), "sdrb_bank_create")
        self.h = h

    def reset(self, stream=-1):
        _check(lib().sdrb_bank_reset(self.h, stream), "sdrb_bank_reset")

    def blocks_done(self, stream=0):
        v = C.c_int64()
        _check(lib().sdrb_bank_blocks_done(self.h, stream, C.byref(v)), "sdrb_bank_blocks_done")
        return v.value

    @property
    def state_bytes(self):
        """Size of one receiver state record; the same for every bank of this plan."""
        return lib().sdrb_bank_state_bytes(self.h)

    @staticmethod
    def _streams(streams):
        s = np.ascontiguousarray(streams, dtype=np.int32).reshape(-1)
        return s, s.ctypes.data_as(C.c_void_p)

    def read_state(self, streams):
        """State records of the listed streams: uint8 [len(streams), state_bytes] (sdrb_bank_read_state)."""
        s, sp = self._streams(streams)
        out = np.zeros((s.size, self.state_bytes), dtype=np.uint8)
        _check(lib().sdrb_bank_read_state(self.h, sp, s.size, out.ctypes.data_as(C.c_void_p)), "sdrb_bank_read_state")
        return out

    def write_state(self, streams, records):
        """Load records (uint8 [len(streams), state_bytes]) into the listed streams; all or nothing (sdrb_bank_write_state)."""
        s, sp = self._streams(streams)
        rec = np.ascontiguousarray(records, dtype=np.uint8)
        if rec.size != s.size * self.state_bytes:
            raise SdrbError("write_state: expected %d records of %d bytes" % (s.size, self.state_bytes))
        _check(lib().sdrb_bank_write_state(self.h, sp, s.size, rec.ctypes.data_as(C.c_void_p)), "sdrb_bank_write_state")

    def save_state(self, streams, d_records_ptr, cuda_stream=None):
        """Enqueue the records of the listed streams into device memory (len(streams) * state_bytes bytes)."""
        s, sp = self._streams(streams)
        _check(lib().sdrb_bank_save_state(self.h, sp, s.size, d_records_ptr, cuda_stream), "sdrb_bank_save_state")

    def load_state(self, streams, d_records_ptr, cuda_stream=None):
        """Load device-resident records into the listed streams (synchronises cuda_stream to check the headers)."""
        s, sp = self._streams(streams)
        _check(lib().sdrb_bank_load_state(self.h, sp, s.size, d_records_ptr, cuda_stream), "sdrb_bank_load_state")

    def process_device(self, d_iq_ptr, iq_stride, n_blocks, d_pcm_ptr, d_tap_ptr=None, cuda_stream=None,
                       input_ready_event=None):
        """input_ready_event: raw cudaEvent_t (int) after which d_iq is valid; lets the DC pre-pass of this
        call overlap the previous call (sdrb_bank_process_device_ex)."""
        _check(lib().sdrb_bank_process_device_ex(self.h, d_iq_ptr, iq_stride, n_blocks, d_pcm_ptr, d_tap_ptr,
                                                 cuda_stream, input_ready_event), "sdrb_bank_process_device_ex")

    def process_streams_device(self, streams, d_iq_ptr, iq_stride, n_blocks, d_pcm_ptr, d_tap_ptr=None, cuda_stream=None,
                               input_ready_event=None):
        """n_blocks callbacks for the listed streams only, in the layout of process_device: stream s reads
        d_iq + s*iq_stride and writes PCM row s; every other stream is left as it was (sdrb_bank_process_streams_device)."""
        s, sp = self._streams(streams)
        _check(lib().sdrb_bank_process_streams_device(self.h, sp, s.size, d_iq_ptr, iq_stride, n_blocks, d_pcm_ptr, d_tap_ptr,
                                                      cuda_stream, input_ready_event), "sdrb_bank_process_streams_device")

    def process_streams_host(self, streams, rows, n_blocks, want_tap=False):
        """rows[k]: the uint8 input of stream streams[k] (n_blocks*block*2 bytes: a numpy array, or an int host address) ->
        compact (pcm int16 [len(streams), n_blocks, pcm_per_block], tap) with record k for streams[k]
        (sdrb_bank_process_streams_host)."""
        s, sp = self._streams(streams)
        if len(rows) != s.size:
            raise SdrbError("process_streams_host: %d rows for %d streams" % (len(rows), s.size))
        need = n_blocks * self.plan.block * 2
        keep, ptrs = [], (C.c_void_p * s.size)()
        for k, r in enumerate(rows):
            if isinstance(r, int):
                ptrs[k] = r
                continue
            a = np.ascontiguousarray(r, dtype=np.uint8).reshape(-1)
            if a.size < need:
                raise SdrbError("process_streams_host: row %d has %d bytes, needs %d" % (k, a.size, need))
            keep.append(a)
            ptrs[k] = a.ctypes.data
        pcm = np.zeros((s.size, n_blocks, self.plan.pcm_per_block), dtype=np.int16)
        tap = np.zeros(pcm.shape, dtype=np.float32) if want_tap else None
        _check(lib().sdrb_bank_process_streams_host(self.h, sp, s.size, C.cast(ptrs, C.c_void_p), n_blocks,
                                                    pcm.ctypes.data_as(C.c_void_p),
                                                    tap.ctypes.data_as(C.c_void_p) if want_tap else None),
               "sdrb_bank_process_streams_host")
        return pcm, tap

    def copy_main(self, main_idx, n_blocks, d_out_ptr, cuda_stream=None):
        _check(lib().sdrb_bank_copy_main(self.h, main_idx, n_blocks, d_out_ptr, cuda_stream), "sdrb_bank_copy_main")

    def copy_dc_trace(self, n_blocks, d_out_ptr, d_modes_ptr=None, cuda_stream=None):
        _check(lib().sdrb_bank_copy_dc_trace(self.h, n_blocks, d_out_ptr, d_modes_ptr, cuda_stream),
               "sdrb_bank_copy_dc_trace")

    def read_input(self, cb, n):
        """sdrj::demodData's `samples` of callback cb of the last call: complex64 [n_streams, n]."""
        out = np.zeros((self.n_streams, n), dtype=np.complex64)
        _check(lib().sdrb_bank_read_input(self.h, cb, n, out.ctypes.data_as(C.c_void_p)), "sdrb_bank_read_input")
        return out

    def read_sub(self, sub_idx, n_blocks):
        """vfo::decimate[decimateCount] of a sub VFO for the last call: complex64 [n_streams, n_blocks*block_z]."""
        s = self.plan.subs[sub_idx]
        block_z = s["samples_out"] * (s["late"] or 1)
        out = np.zeros((self.n_streams, n_blocks * block_z), dtype=np.complex64)
        _check(lib().sdrb_bank_read_sub(self.h, sub_idx, n_blocks, out.ctypes.data_as(C.c_void_p)), "sdrb_bank_read_sub")
        return out

    def spectrum_feed(self, spectrum, source, cb, d_fft_out_ptr=None, cuda_stream=None):
        _check(lib().sdrb_bank_spectrum_feed(self.h, spectrum.h, source, cb, d_fft_out_ptr, cuda_stream),
               "sdrb_bank_spectrum_feed")

    def copy_forward(self, main_idx, n_blocks, d_out_ptr, cuda_stream=None):
        _check(lib().sdrb_bank_copy_forward(self.h, main_idx, n_blocks, d_out_ptr, cuda_stream), "sdrb_bank_copy_forward")

    def read_forward(self, main_idx, n_blocks):
        """vfo::compress payloads of the last call: uint8 [n_streams, n_blocks, fwd_bytes]."""
        out = np.zeros((self.n_streams, n_blocks, self.plan.mains[main_idx]["fwd_bytes"]), dtype=np.uint8)
        _check(lib().sdrb_bank_read_forward(self.h, main_idx, n_blocks, out.ctypes.data_as(C.c_void_p)),
               "sdrb_bank_read_forward")
        return out

    def process_host(self, h_iq_ptr, iq_stride, n_blocks, h_pcm_ptr, h_tap_ptr=None):
        _check(lib().sdrb_bank_process_host(self.h, h_iq_ptr, iq_stride, n_blocks, h_pcm_ptr, h_tap_ptr),
               "sdrb_bank_process_host")

    def process_host_async(self, h_iq_ptr, iq_stride, n_blocks, h_pcm_ptr, h_tap_ptr=None):
        _check(lib().sdrb_bank_process_host_async(self.h, h_iq_ptr, iq_stride, n_blocks, h_pcm_ptr, h_tap_ptr),
               "sdrb_bank_process_host_async")

    def host_wait(self, max_in_flight=0):
        _check(lib().sdrb_bank_host_wait_until(self.h, max_in_flight), "sdrb_bank_host_wait_until")

    def process_numpy(self, iq, n_blocks, want_tap=False):
        """iq: uint8 [n_streams, n_blocks*block*2] -> (pcm int16 [n_streams, n_blocks, pcm_per_block], tap)."""
        iq = np.ascontiguousarray(iq, dtype=np.uint8).reshape(self.n_streams, -1)
        row = n_blocks * self.plan.block * 2
        stride = (row + 15) // 16 * 16
        buf = np.zeros((self.n_streams, stride), dtype=np.uint8)
        buf[:, :row] = iq[:, :row]
        pcm = np.zeros((self.n_streams, n_blocks, self.plan.pcm_per_block), dtype=np.int16)
        tap = np.zeros(pcm.shape, dtype=np.float32) if want_tap else None
        self.process_host(buf.ctypes.data_as(C.c_void_p), stride, n_blocks, pcm.ctypes.data_as(C.c_void_p),
                          tap.ctypes.data_as(C.c_void_p) if want_tap else None)
        return pcm, tap

    def set_timing(self, on=True):
        _check(lib().sdrb_bank_set_timing(self.h, int(on)), "sdrb_bank_set_timing")

    def kernel_times(self):
        """{class name: (total ms, timed calls)} since set_timing(True)."""
        ms = (C.c_double * 6)()
        calls = (C.c_long * 6)()
        _check(lib().sdrb_bank_kernel_times(self.h, ms, calls), "sdrb_bank_kernel_times")
        names = ["dc_scan", "ingest_main", "sub_cascade", "late_fir", "usb_audio", "carry"]
        return {n: (ms[k], calls[k]) for k, n in enumerate(names)}

    @property
    def last_launches(self):
        return lib().sdrb_bank_last_launches(self.h)

    def close(self):
        if getattr(self, "h", None):
            lib().sdrb_bank_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Spectrum:
    """MainWindow's spectrum display state for n independent displays (fftHandlerSlot)."""
    NFFT = 8192

    def __init__(self, n_displays, device=0):
        self.n = n_displays
        h = C.c_void_p()
        _check(lib().sdrb_spectrum_create(device, n_displays, self.NFFT, C.byref(h)), "sdrb_spectrum_create")
        self.h = h

    def reset(self, display=-1):
        _check(lib().sdrb_spectrum_reset(self.h, display), "sdrb_spectrum_reset")

    def feed_device(self, d_in_ptr, in_stride, length, d_fft_out_ptr=None, cuda_stream=None):
        _check(lib().sdrb_spectrum_feed_device(self.h, d_in_ptr, in_stride, length, d_fft_out_ptr, cuda_stream),
               "sdrb_spectrum_feed_device")

    def feed_numpy(self, x):
        """x: complex64 [n_displays, len]."""
        x = np.ascontiguousarray(x, dtype=np.complex64).reshape(self.n, -1)
        _check(lib().sdrb_spectrum_feed_host(self.h, x.ctypes.data_as(C.c_void_p), x.shape[1], x.shape[1]),
               "sdrb_spectrum_feed_host")

    def read(self):
        smooth = np.zeros((self.n, self.NFFT - 10)); pwr = np.zeros((self.n, self.NFFT)); stats = np.zeros((self.n, 2))
        _check(lib().sdrb_spectrum_read(self.h, smooth.ctypes.data_as(C.c_void_p), pwr.ctypes.data_as(C.c_void_p),
                                        stats.ctypes.data_as(C.c_void_p)), "sdrb_spectrum_read")
        return smooth, pwr, stats

    def close(self):
        if getattr(self, "h", None):
            lib().sdrb_spectrum_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PinnedBuffer:
    """cudaHostAlloc'd host memory viewed as a numpy array."""

    def __init__(self, nbytes):
        self.ptr = lib().sdrb_host_alloc(nbytes)
        if not self.ptr:
            raise SdrbError("sdrb_host_alloc(%d) failed" % nbytes)
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr))

    def view(self, dtype):
        return self.array.view(dtype)

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            lib().sdrb_host_free(self.ptr)
            self.ptr = None


def probe_fp32_tflops(packed=False, reps=5):
    """Measured FP32 FMA peak of the current device in TFLOP/s (sdrb_probe_fp32_tflops)."""
    v = C.c_double(0.0)
    _check(lib().sdrb_probe_fp32_tflops(1 if packed else 0, reps, C.byref(v)), "sdrb_probe_fp32_tflops")
    return v.value


def split_pcm(plan, pcm):
    """pcm [n_blocks, pcm_per_block] of one stream -> {topic: int16 audio across callbacks}."""
    out = {}
    for s in plan.subs:
        out[s["topic"]] = np.ascontiguousarray(pcm[:, s["pcm_offset"]:s["pcm_offset"] + s["samples_out"]]).reshape(-1)
    return out
