#!/usr/bin/env python
"""bench.py -- aggregate input MS/s of the SDRReceiver channelizer hot path (25E plan).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = `--blocks` callbacks (default 4 = one second of signal) for each of `--streams`
independent 1.536 MS/s uint8-IQ streams per GPU (default 128: the 1024-stream configuration
of BASELINE.json sharded over 8 GPUs; weak scaling, no data-path collective). Rank 0 prints
ONE JSON line:
  value     whole-job input MS/s with the uint8 IQ already resident in HBM (kernels only)
  e2e       same metric through the host-facing C-ABI call sdrb_bank_process_host: pinned
            host uint8 in, H2D, kernels, D2H, pinned int16 out, every step
  roofline  the kernel class with the largest share of the step, algorithmic bytes / its
            CUDA-event time vs the measured HBM copy peak (MEASURED_PEAKS.json)
  cpu_baseline  the unmodified reference (oracle/_ref) on this box's host cores, bounded sample
`--impl reference` times the reference's own CPU code instead (same metric/config).
Every timed loop (kernel leg, end to end, publish leg -- once with n sockets, once with one -- and each of the other
plans, the kernel legs followed by a second pass with per-launch timing) runs `--steps` steps after `--warmup`, so the
wall time of a run grows with --steps in every leg.
`--dump-outputs DIR` writes what the kernel leg's last step computed (rank 0) as DIR/*.npy: the seeded inputs are
identical from run to run, so two builds can be compared output for output. The bank carries state from step to step
and the dumped step is the last of the per-launch timing pass (step warmup + 2*steps), so two dumps are comparable when
--steps, --warmup, --plan, --streams and --blocks agree.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "aggregate input MS/s (uint8 IQ, 25E plan)"
HBM_FALLBACK_GBS = 6650.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--plan", default="25E")
    ap.add_argument("--streams", type=int, default=128, help="streams per GPU")
    ap.add_argument("--blocks", type=int, default=4, help="callbacks per stream per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-zmq", action="store_true", help="skip the publish-inclusive end-to-end leg")
    ap.add_argument("--no-plans", action="store_true", help="skip the short runs of the other BASELINE configurations")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the kernel leg's last-step int16 records as float32 .npy files; two dumps compare only "
                         "at equal --steps/--warmup/--plan/--streams/--blocks (the bank carries state across steps)")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------
# synthetic input: a few fully synthesised base streams, the rest are time-rotated copies
# --------------------------------------------------------------------------------------
def base_streams(plan, n_base, n_samples):
    from sdrreceiver_b200 import synth
    car = synth.carriers_for_plan(plan.center, plan.subs)
    return [synth.make_iq(plan.fs, n_samples, car, stream=s) for s in range(n_base)]


def bind_to_gpu_cpus(index):
    """Pin this process to the CPU cores NVML reports as local to GPU `index`, so that the pinned staging
    buffers of the end-to-end leg live on that GPU's NUMA node (matters from 2 ranks up). Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)),
        }
        getr = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = getr(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)      # NVML queries take driver locks: keep them rare next to ~130 launches per step

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference, one process per host core
# --------------------------------------------------------------------------------------
def run_reference_cpu(plan, plan_path, cores, blocks_timed, skip):
    """Runs `cores` copies of oracle/_ref/sdr_ref_i16 (one stream each) and returns
    (total_samples, seconds = slowest process's time inside demodData)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "sdr_ref_i16")
    if not os.path.exists(exe):
        raise RuntimeError("oracle/_ref/sdr_ref_i16 missing (built from /root/reference by oracle/Makefile)")
    n_blocks = blocks_timed + skip
    base = base_streams(plan, 1, plan.block * n_blocks)[0]
    with tempfile.TemporaryDirectory() as d:
        procs = []
        for c in range(cores):
            fn = os.path.join(d, "s%d.u8" % c)
            np.roll(base, 2 * 977 * c).tofile(fn)
        for c in range(cores):
            procs.append(subprocess.Popen([exe, "--ini", plan_path, "--in", os.path.join(d, "s%d.u8" % c), "--time",
                                           "--skip", str(skip), "--blocks", str(n_blocks)],
                                          stdout=subprocess.PIPE, text=True))
        total, worst = 0, 0.0
        for p in procs:
            out = p.communicate()[0].split()
            if p.returncode != 0 or len(out) != 2:
                raise RuntimeError("reference harness failed")
            total += int(out[0])
            worst = max(worst, float(out[1]))
    return total, worst


class RefPlan:
    """What run_reference_cpu needs of a plan, from oracle/plan.py (reference arm) -- same attribute names as binding.Plan."""

    def __init__(self, op):
        self.fs, self.block, self.center, self.subs = op["Fs"], op["block"], op["center"], op["subs"]


def reference_arm(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    plan_path = os.path.join(ROOT, "plans", args.plan + ".ini")
    # plan arithmetic from the oracle's own ini reader: this arm never loads libsdrb200.so
    from oracle import plan as OP
    plan = RefPlan(OP.build_plan(plan_path))
    op = {"Fs": plan.fs, "block": plan.block}
    cores = os.cpu_count() or 1
    # each step = every core pushes `--blocks` callbacks of its own stream through the reference
    total, secs = run_reference_cpu(plan, plan_path, cores, args.blocks * args.steps, args.blocks * args.warmup)
    value = total / secs / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "realtime_x": value * 1e6 / op["Fs"],
        "config": {"workload": "%s plan, %d host processes x 1 stream, %d callbacks per step" % (args.plan, cores, args.blocks),
                   "plan": args.plan, "streams": cores, "blocks_per_step": args.blocks},
        "cpu_baseline": {"value": value, "unit": "MS/s", "cores": cores, "kind": "reference",
                         "sample": "%d processes x %d timed callbacks (g++ -O2 -ffp-contract=off build of the unmodified reference)" % (cores, args.blocks * args.steps)},
        "e2e": {"value": value, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------
CLASSES = ["dc_scan", "ingest_main", "sub_cascade", "late_fir", "usb_audio", "carry"]


def alg_tables(plan):
    """Algorithmic bytes and flops per input complex sample of every kernel class (DESIGN.md section 4,
    SURVEY.md 8(d)'s counting rule)."""
    fs = plan.fs
    main_out_b = 8.0 * sum(m["out_rate"] for m in plan.mains) / fs
    z_b = 8.0 * sum(s["out_rate"] * (s["late"] or 1) for s in plan.subs) / fs
    d_b = 8.0 * sum(s["out_rate"] for s in plan.subs if s["late"]) / fs
    usb_in_b = 8.0 * sum(s["out_rate"] for s in plan.subs) / fs
    pcm_b = 2.0 * sum(s["out_rate"] for s in plan.subs) / fs
    alg_bytes = {"dc_scan": 2.0, "ingest_main": 2.0 + main_out_b, "sub_cascade": main_out_b + z_b,
                 "late_fir": (z_b + d_b) if d_b else 0.0, "usb_audio": usb_in_b + pcm_b, "carry": 0.0}
    hb = lambda decim: sum(20.0 / 2 ** a for a in range(1, decim + 1))
    alg_flops = {
        "dc_scan": 8.0 if plan.correct_dc else 0.0,
        "ingest_main": 10.0 + sum(6.0 + hb(m["decim"]) for m in plan.mains),     # u8->f32 2 + DC 8 (SURVEY 8(d)) + mains
        "sub_cascade": sum((s["Fs"] / fs) * (6.0 + hb(s["decim"])) for s in plan.subs),
        "late_fir": sum((s["out_rate"] / fs) * 4.0 * s["n_dec_taps"] for s in plan.subs if s["late"]),
        "usb_audio": sum((s["out_rate"] / fs) * (2.0 * 62 + 1 + 2.0 * s["n_lpf_taps"] + 2.0) for s in plan.subs),
        "carry": 0.0,
    }
    return alg_bytes, alg_flops


class Resident:
    """One bank with its input resident in HBM: the kernel-only leg, for the headline plan and the other BASELINE configs."""

    def __init__(self, B, torch, shard, plan, S, NB, dev, local_rank, rank, world, canary):
        self.B, self.torch, self.plan, self.S, self.NB, self.dev = B, torch, plan, S, NB, dev
        Bk = plan.block
        self.row = NB * Bk * 2
        self.samples_per_step = S * NB * Bk
        base = base_streams(plan, 2, NB * Bk)
        self.pin_in = B.PinnedBuffer(S * self.row)
        h_iq = self.pin_in.array.reshape(S, self.row)
        for s, g in enumerate(shard.stream_ids(rank, world, S)):
            # local slot 0 of every rank is the canary: identical bytes everywhere, its digest must agree across ranks
            h_iq[s] = base[0] if (canary and s == 0) else np.roll(base[g % 2], 2 * 977 * g)
        self.d_iq = torch.from_numpy(h_iq).to(dev)
        self.d_pcm = torch.empty((S, NB, plan.pcm_per_block), dtype=torch.int16, device=dev)
        self.bank = B.Bank(plan, S, NB, device=local_rank)
        self.stream = torch.cuda.Stream(device=dev)
        torch.cuda.synchronize()
        self.in_ready = torch.cuda.Event()
        self.in_ready.record(self.stream)
        self.in_ready.synchronize()
        self.after_step = None

    def step(self):
        self.bank.process_device(self.d_iq.data_ptr(), self.row, self.NB, self.d_pcm.data_ptr(), None, self.stream.cuda_stream,
                                 self.in_ready.cuda_event)
        if self.after_step:
            self.after_step()

    def timed(self, steps, warmup, barrier):
        torch = self.torch
        for _ in range(warmup):
            self.step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            self.step()
        e1.record(self.stream)
        barrier()
        launches = self.bank.last_launches * steps
        dev_ms = e0.elapsed_time(e1)
        # second pass over the same steps with a CUDA-event pair around every launch (on the stream it is launched
        # on): per-class durations for the roofline, kept out of the number above
        self.bank.set_timing(True)
        for _ in range(steps):
            self.step()
        torch.cuda.synchronize()
        kt = self.bank.kernel_times()
        self.bank.set_timing(False)
        return dev_ms, launches, {k: v[0] / steps for k, v in kt.items()}, {k: v[1] / steps for k, v in kt.items()}


def class_rooflines(plan, per_step_ms, samples_per_step, hbm_peak_gbs, fp32_peak):
    """Both roofline axes of every kernel class from its CUDA-event time: algorithmic bytes resp. flops / time / peak."""
    alg_bytes, alg_flops = alg_tables(plan)
    out = {}
    for k, ms in per_step_ms.items():
        if ms <= 0:
            continue
        gbs = alg_bytes[k] * samples_per_step / (ms * 1e-3) / 1e9
        tf = alg_flops[k] * samples_per_step / (ms * 1e-3) / 1e12
        out[k] = {"ms_per_step": ms, "hbm_gbs": gbs, "hbm_frac": gbs / hbm_peak_gbs, "fp32_tflops": tf,
                  "fp32_frac": tf / fp32_peak, "alg_bytes_per_sample": alg_bytes[k], "alg_flops_per_sample": alg_flops[k]}
    return out


DUMP_BYTES = 60 << 20        # what --dump-outputs writes at most (float32)


def dump_outputs(out_dir, pcm):
    """pcm [S, NB, pcm_per_block] int16 -- the records a caller of the kernel leg receives for every receiver -- as float32.
    Receivers beyond the DUMP_BYTES budget are left out: a fixed, seeded choice that always keeps receiver 0 (the canary).
    pcm.npy is [k, NB, pcm_per_block], pcm_streams.npy the k receiver indices it holds. When one receiver alone is over the
    budget, k is 1 and pcm.npy is 1-D: the first DUMP_BYTES / 4 samples of receiver 0's records, in memory order."""
    S = pcm.shape[0]
    k = max(1, min(S, DUMP_BYTES // (pcm[0].size * 4)))
    pick = np.sort(np.concatenate([[0], np.random.default_rng(20261020).permutation(np.arange(1, S))[:k - 1]]))
    sel = pcm[pick]
    if sel.size * 4 > DUMP_BYTES:          # one receiver alone is over the budget: its first samples
        sel = sel.reshape(-1)[:DUMP_BYTES // 4]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pcm.npy"), sel.astype(np.float32))
    np.save(os.path.join(out_dir, "pcm_streams.npy"), pick.astype(np.float64))


def canary_check(B, plan, local_rank):
    """Parity verdict of this rank: a fresh one-receiver bank runs the canary's first callback and is compared with
    tests/golden/canary_25E_1block.npz (int16 of the unmodified reference, tools/make_golden.py): +-1 LSB."""
    import hashlib
    from sdrreceiver_b200 import synth
    gold = os.path.join(ROOT, "tests", "golden", "canary_%s_1block.npz" % os.path.basename(plan.path or "").replace(".ini", ""))
    if not os.path.exists(gold):
        return None, "no golden file for this plan"
    g = np.load(gold)
    level = 0.5 if any(s["late"] for s in plan.subs) else 1.0          # as tools/make_golden.py (the /late plans clip at full level)
    iq = synth.make_iq(plan.fs, plan.block, synth.carriers_for_plan(plan.center, plan.subs), level=level, stream=0)
    if not np.array_equal(np.frombuffer(hashlib.sha256(iq.tobytes()).digest(), np.uint8), g["input_sha256"]):
        return None, "synthetic input differs from the golden file's"
    bank = B.Bank(plan, 1, 1, device=local_rank)
    pcm, _ = bank.process_numpy(iq[None, :], 1)
    bank.close()
    got = B.split_pcm(plan, pcm[0])
    worst = 0
    for s in plan.subs:
        worst = max(worst, int(np.abs(got[s["topic"]].astype(np.int32) - g["pcm_" + s["topic"]].astype(np.int32)).max()))
    return worst, "max |int16 difference| over %d sub VFOs x %d samples vs the unmodified reference" % (len(plan.subs), plan.pcm_per_block)


def b200_arm(args):
    import torch
    import torch.distributed as dist
    from sdrreceiver_b200 import binding as B, shard

    rank, local_rank, world = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    numa = bind_to_gpu_cpus(local_rank)          # before the pinned buffers are allocated (first touch)
    plan_path = os.path.join(ROOT, "plans", args.plan + ".ini")
    plan = B.Plan(plan_path)
    S, NB, Bk = args.streams, args.blocks, plan.block

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- input: stream s of rank r is global stream r + world*s (independent units, no exchange)
    R = Resident(B, torch, shard, plan, S, NB, dev, local_rank, rank, world, canary=True)
    row, samples_per_step, bank = R.row, R.samples_per_step, R.bank
    pin_in = R.pin_in
    pin_out = B.PinnedBuffer(S * NB * plan.pcm_per_block * 2)
    # the end-to-end leg keeps two calls in flight: a second pair of pinned host buffers
    pin_in2 = B.PinnedBuffer(S * row)
    pin_in2.array[:] = pin_in.array
    pin_out2 = B.PinnedBuffer(S * NB * plan.pcm_per_block * 2)

    host_bufs = [(pin_in.ptr, pin_out.ptr), (pin_in2.ptr, pin_out2.ptr)]
    host_step = [0]

    def step_host():
        # sdrb_bank_process_host_async: every step copies its own input from pinned host memory and its own result
        # back; at most two steps are in flight, so step i+1's copy-in overlaps step i's filters and copy-out
        i, o = host_bufs[host_step[0] & 1]
        host_step[0] += 1
        bank.process_host_async(i, row, NB, o, None)
        bank.host_wait(1)

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- kernel metric: inputs resident in HBM (393 MB per step > 126 MB L2) ----
    dev_ms, launches, per_step_ms, launches_per_step = R.timed(args.steps, args.warmup, barrier)

    # ---- end to end through the host-facing call ----
    e2e_ms = None
    if not args.no_e2e:
        for _ in range(args.warmup):
            step_host()
        bank.host_wait(0)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host()
        bank.host_wait(0)                                      # the last result is on the host
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- end to end including the ZMQ publish leg (vfo::transmitData, zmqpublisher.cpp:82-96) ----
    zmq_leg = None
    if not args.no_e2e and not args.no_zmq:
        try:
            n_sock = max(1, min(8, (os.cpu_count() or 8) // max(1, 2 * args.gpus)))
            if os.environ.get("SDRB_BENCH_SOCKETS"):
                n_sock = max(1, int(os.environ["SDRB_BENCH_SOCKETS"]))
            zmq_leg = publish_leg(B, plan, bank, host_bufs, row, S, NB, rank, args, n_sock)
            if n_sock > 1:                    # the reference's shape beside it: one socket, one sender thread
                one = publish_leg(B, plan, bank, host_bufs, row, S, NB, rank, args, 1)
                zmq_leg["single_socket"] = {k: one[k] for k in ("value", "ms_per_step", "messages_per_s", "messages_received")}
        except Exception as ex:           # reported, never required for the GPU number
            zmq_leg = {"value": None, "error": str(ex)[:200]}

    # ---- parity verdict: this rank's canary against the reference's golden output, and -- gathered over NCCL with the
    # timings -- the canary digest of every rank, which must agree (identical bytes, identical history on every rank)
    lsb, lsb_what = canary_check(B, plan, local_rank)
    pcm_host = R.d_pcm.cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pcm_host)
    digest = shard.pcm_digest(pcm_host) + shard.pcm_digest(pcm_host[0]) + [-1 if lsb is None else int(lsb)]
    stats_all, digests = shard.gather([dev_ms, e2e_ms if e2e_ms is not None else 0.0, float(samples_per_step)],
                                      digest, device=dev)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    verdict = shard.parity_verdict(digests)

    agg = shard.aggregate(stats_all, args.steps)
    max_dev_ms, max_e2e_ms = agg["dev_ms"], agg["e2e_ms"]
    value = agg["value_msps"]
    e2e_value = agg["e2e_msps"] if e2e_ms is not None else None

    # ---- rooflines (rank 0's events): every class on both axes; the headline object is the class with the largest share
    # of the step ON THE LAUNCHING STREAM; the DC recursion runs beside it on a side stream and is reported with it
    fs = plan.fs
    peak, peak_src = hbm_peak()
    clocks = sampler.summary()
    sm_mhz = clocks["sm_mhz"] or 1965.0
    fp32_nominal = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    # FP32 denominator: an FMA loop measured on this device after the timed region (scalar FFMA and packed
    # FFMA2 chains, the better of the two); the nominal figure is kept beside it
    fp32_probe = {"ffma": B.probe_fp32_tflops(False), "ffma2": B.probe_fp32_tflops(True)}
    fp32_peak = max(fp32_probe.values())
    fp32_src = ("measured FMA loop (sdrb_probe_fp32_tflops): FFMA %.1f, FFMA2 %.1f TFLOP/s; nominal 148 SM x 128 lanes x 2 x "
                "%.0f MHz = %.1f" % (fp32_probe["ffma"], fp32_probe["ffma2"], sm_mhz, fp32_nominal))
    step_ms = max_dev_ms / args.steps
    per_class = class_rooflines(plan, per_step_ms, samples_per_step, peak, fp32_peak)
    longest = max(per_class, key=lambda k: per_class[k]["ms_per_step"])
    dom = max((k for k in per_class if k != "dc_scan"), key=lambda k: per_class[k]["ms_per_step"])
    dc_cls = per_class[dom]
    traffic, traffic_src = None, None
    for fn in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", fn)) as f:
                tj = json.load(f)
            if tj["config"]["plan"] == args.plan and tj["config"]["streams_per_gpu"] == S and dom in tj["per_class_per_callback"]:
                traffic, traffic_src = tj["per_class_per_callback"][dom], "profiles/%s (ncu --set full)" % fn
                break
        except Exception:
            pass
    samples_per_callback = S * Bk
    fp32_bound = dc_cls["fp32_frac"] >= dc_cls["hbm_frac"]
    roofline = {
        "bound": "fp32" if fp32_bound else "hbm", "kernel": dom,
        "achieved": dc_cls["fp32_tflops"] if fp32_bound else dc_cls["hbm_gbs"],
        "peak": fp32_peak if fp32_bound else peak, "unit": "TFLOP/s" if fp32_bound else "GB/s",
        "frac": dc_cls["fp32_frac"] if fp32_bound else dc_cls["hbm_frac"],
        "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": fp32_src if fp32_bound else peak_src,
        "launch": "the %s kernels of one callback (%d streams x %d samples)" % (dom, S, Bk),
        "alg_flops_per_launch": dc_cls["alg_flops_per_sample"] * samples_per_callback,
        "alg_bytes_per_launch": dc_cls["alg_bytes_per_sample"] * samples_per_callback, "launch_ms": dc_cls["ms_per_step"] / NB,
        "kernel_ms_per_step": dc_cls["ms_per_step"], "share_of_step": dc_cls["ms_per_step"] / step_ms if step_ms > 0 else None,
        "hbm": {"achieved": dc_cls["hbm_gbs"], "peak": peak, "unit": "GB/s", "frac": dc_cls["hbm_frac"], "peak_source": peak_src},
        "fp32": {"achieved_tflops": dc_cls["fp32_tflops"], "peak_tflops": fp32_peak, "frac": dc_cls["fp32_frac"],
                 "alg_flops_per_sample": dc_cls["alg_flops_per_sample"], "peak_source": fp32_src},
        "longest_class_any_stream": longest,
        "per_class": per_class,
    }
    line = {
        "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s plan x %d streams per GPU (%d total) x %d callbacks (%.2f s of signal) per step; "
                               "input %.0f MB per GPU per step, larger than L2" % (
                                   args.plan, S, S * world, NB, NB / plan.bufsplit, S * row / 1e6),
                   "plan": args.plan, "streams_per_gpu": S, "blocks_per_step": NB, "sample_rate": fs,
                   "l2_policy": "input larger than L2 (no flush)", "parallelism": "streams sharded, no collective",
                   "cpus_bound_per_rank": numa},
        "realtime_x": value * 1e6 / fs,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "MS/s", "h2d_bytes_per_step": S * row,
                "d2h_bytes_per_step": S * NB * plan.pcm_per_block * 2, "ms_per_step": max_e2e_ms / args.steps,
                "timing": "host wall clock around K sdrb_bank_process_host_async calls, two in flight, last result waited for "
                          "(pinned host buffers in and out every step)",
                "realtime_x": (e2e_value * 1e6 / fs) if e2e_value else None} if e2e_ms is not None else None,
        "e2e_zmq": zmq_leg,
        "gpu_launches": launches,
        "parity_ok": verdict["ok"], "parity": dict(verdict, what=lsb_what),
        "roofline": roofline,
        "roofline_pipeline": {"bound": "fp32", "achieved": plan.alg_flops * samples_per_step / (step_ms * 1e-3) / 1e12,
                              "peak": fp32_peak, "unit": "TFLOP/s",
                              "frac": plan.alg_flops * samples_per_step / (step_ms * 1e-3) / 1e12 / fp32_peak,
                              "alg_flops_per_sample": plan.alg_flops, "peak_source": fp32_src,
                              "hbm": {"achieved": plan.alg_bytes * samples_per_step / (step_ms * 1e-3) / 1e9, "peak": peak,
                                      "unit": "GB/s", "frac": plan.alg_bytes * samples_per_step / (step_ms * 1e-3) / 1e9 / peak,
                                      "alg_bytes_per_sample": plan.alg_bytes}},
        "kernels_ms_per_step": per_step_ms,
        "kernel_launches_per_step": launches_per_step,
        "digests": digests,
    }
    # ---- the other BASELINE.json configurations, --steps steps each: value and per-class times ----
    if world == 1 and not args.no_plans:
        R.bank.close()
        del R
        torch.cuda.empty_cache()
        extra = {}
        for name in EXTRA_PLANS:
            if name == args.plan:
                continue
            try:
                extra[name] = extra_plan(B, torch, shard, name, S, NB, dev, local_rank, peak, fp32_peak, barrier,
                                         args.steps, args.warmup)
            except Exception as ex:
                extra[name] = {"error": str(ex)[:200]}
        line["plans"] = extra
    if world == 1 and not args.no_cpu_baseline:
        try:
            cores = os.cpu_count() or 1
            total, secs = run_reference_cpu(plan, plan_path, cores, 12, 1)
            line["cpu_baseline"] = {"value": total / secs / 1e6, "unit": "MS/s", "cores": cores, "kind": "reference",
                                    "sample": "%d processes x 12 timed callbacks (3 s of signal each), unmodified reference "
                                              "built g++ -O2 -ffp-contract=off" % cores}
        except Exception as ex:   # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "MS/s", "cores": 0, "kind": "reference", "sample": "failed: %s" % ex}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


EXTRA_PLANS = ["54W_288K", "54W_all", "CBAND_143E"]


def extra_plan(B, torch, shard, name, S, NB, dev, local_rank, peak, fp32_peak, barrier, steps, warmup):
    """Kernel-only leg of another BASELINE.json configuration: same bank size, `warmup` + `steps` timed steps. CBAND_143E runs with
    the spectrum path fed as the reference's GUI would (fftHandlerSlot): "Main" on every 4th callback and one selected
    sub VFO on every callback, for every receiver of the bank."""
    plan = B.Plan(os.path.join(ROOT, "plans", name + ".ini"))
    R = Resident(B, torch, shard, plan, S, NB, dev, local_rank, 0, 1, canary=False)
    out = {}
    spec_ms = None
    if name.startswith("CBAND"):
        spec_main, spec_sub = B.Spectrum(S, device=local_rank), B.Spectrum(S, device=local_rank)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        acc = {"ms": 0.0, "n": 0, "count": [0]}

        def feed():
            st = R.stream.cuda_stream
            ev[0].record(R.stream)
            for cb in range(NB):
                acc["count"][0] += 1
                if acc["count"][0] % 4 == 1:                       # sdrj.cpp:296-303: first emit, then every 4th callback
                    R.bank.spectrum_feed(spec_main, -1, cb, None, st)
                R.bank.spectrum_feed(spec_sub, 0, cb, None, st)    # vfo.cpp:290-293: the selected VFO, every callback
            ev[1].record(R.stream)
        R.after_step = feed
    dev_ms, launches, per_step_ms, _ = R.timed(steps, warmup, barrier)
    if name.startswith("CBAND"):
        # the feeds of one step, timed on their own after the run
        torch.cuda.synchronize()
        R.after_step()
        torch.cuda.synchronize()
        spec_ms = ev[0].elapsed_time(ev[1])
        spec_main.close(); spec_sub.close()
    step_ms = dev_ms / steps
    out = {"value": R.samples_per_step / (step_ms * 1e-3) / 1e6, "unit": "MS/s", "ms_per_step": step_ms, "steps": steps, "warmup": warmup,
           "realtime_x": R.samples_per_step / (step_ms * 1e-3) / plan.fs, "kernels_ms_per_step": per_step_ms,
           "per_class": class_rooflines(plan, per_step_ms, R.samples_per_step, peak, fp32_peak), "gpu_launches": launches}
    if spec_ms is not None:
        out["spectrum_feed_ms_per_step"] = spec_ms
        out["spectrum_feeds_per_step"] = "%d displays x (%d sub-VFO feeds + 1 Main feed)" % (S, NB)
    R.bank.close()
    # the same parity check as the headline plan's: one callback of a fresh receiver against the unmodified reference's int16
    lsb, what = canary_check(B, plan, local_rank)
    out["parity_ok"] = lsb is not None and lsb <= 1
    out["canary_max_lsb_vs_reference"] = lsb
    out["parity_what"] = what
    return out


def publish_leg(B, plan, bank, host_bufs, row, S, NB, rank, args, n_sockets=8):
    """The path's last hop: every callback record of every receiver is sent as the reference does (3 frames per sub VFO:
    topic, rate, int16 payload) into SUB sockets of this process over ipc. Timed with the host call that produces the
    records: K steps of process_host_async (two in flight) + sdrb_publisher_pool_send_call for the step that just completed.
    n_sockets PUB sockets with one sender thread each (receiver s on socket s % n_sockets); 1 = the reference's single socket."""
    import ctypes as C
    import threading
    import zmq
    lib = B.lib()
    base = "ipc:///tmp/sdrb_bench_%d_%d_%d" % (os.getpid(), rank, n_sockets)
    pool = C.c_void_p()
    B._check(lib.sdrb_publisher_pool_open(base.encode(), 1, n_sockets, C.byref(pool)), "sdrb_publisher_pool_open")
    addrs = []
    for k in range(n_sockets):
        buf = C.create_string_buffer(256)
        B._check(lib.sdrb_publisher_pool_address(pool, k, buf, 256), "sdrb_publisher_pool_address")
        addrs.append(buf.value.decode())
    # the receiving side: tools/zmq_sink.cpp (built next to the library) in its own process, one thread per address; a python
    # SUB socket per address with a drain thread each if the binary is missing
    sink_bin = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sdrreceiver_b200", "zmq_sink")
    sink = None
    n_rx = [[0, 0] for _ in range(n_sockets)]
    stop = [False]
    subs, threads = [], []
    if os.access(sink_bin, os.X_OK):
        import subprocess
        sink = subprocess.Popen([sink_bin] + addrs, stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
        if sink.stdout.readline().strip() != "ready":
            sink.kill()
            sink = None
    if sink is None:
        ctx = zmq.Context.instance()

        def drain(sub, acc):
            while not stop[0]:
                try:
                    parts = sub.recv_multipart(copy=False)
                    acc[0] += 1
                    acc[1] += len(parts[2].buffer) if len(parts) == 3 else 0
                except zmq.Again:
                    pass

        for k in range(n_sockets):
            sub = ctx.socket(zmq.SUB)
            sub.setsockopt(zmq.RCVHWM, 0)
            sub.setsockopt(zmq.RCVTIMEO, 50)
            sub.setsockopt(zmq.SUBSCRIBE, b"")
            sub.connect(addrs[k])
            subs.append(sub)
            threads.append(threading.Thread(target=drain, args=(sub, n_rx[k]), daemon=True))
        for th in threads:
            th.start()
    time.sleep(0.3)
    steps = args.steps
    sent = 0
    step_no = [0]

    def one():
        i, o = host_bufs[step_no[0] & 1]
        step_no[0] += 1
        bank.process_host_async(i, row, NB, o, None)
        bank.host_wait(1)

    def publish(o):
        B._check(lib.sdrb_publisher_pool_send_call(pool, plan.h, C.c_void_p(o), S, NB), "sdrb_publisher_pool_send_call")
        return S * NB * len(plan.subs)

    one()
    bank.host_wait(0)
    t0 = time.perf_counter()
    for k in range(steps):
        one()                                   # step k+1 is in flight while step k's records are published
        sent += publish(host_bufs[(step_no[0] - 2) & 1][1])
    bank.host_wait(0)
    secs = time.perf_counter() - t0
    time.sleep(0.5)
    if sink is not None:
        out, _ = sink.communicate("", timeout=20)              # EOF on stdin: the sink prints its counts and leaves
        got = json.loads(out.strip().splitlines()[-1])
        received, received_bytes = got["messages"], got["payload_bytes"]
        side = "tools/zmq_sink.cpp in its own process, one SUB socket and thread per address"
    else:
        stop[0] = True
        for th in threads:
            th.join(timeout=2)
        for sub in subs:
            sub.close(0)
        received, received_bytes = sum(a[0] for a in n_rx), sum(a[1] for a in n_rx)
        side = "python SUB sockets in this process, one drain thread per address"
    lib.sdrb_publisher_pool_close(pool)
    samples = S * NB * plan.block * steps
    return {"value": samples / secs / 1e6, "unit": "MS/s", "realtime_x": samples / secs / plan.fs, "steps": steps,
            "messages_sent": sent, "messages_per_s": sent / secs, "messages_received": received,
            "payload_bytes_received": received_bytes, "sockets": n_sockets,
            "transport": "ipc, %d PUB socket(s) with one sender thread each (sdrb_publisher_pool) -> %s" % (n_sockets, side),
            "ms_per_step": 1e3 * secs / steps}


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
