#!/usr/bin/env python
"""bench.py - IQ Msamp/s through xcorr_pss (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the hot path (xcorr_pss: correlate 3 PSS roots x n_f frequency
hypotheses, fold, delay-spread, argmax, signal power) over one batch of synthetic capture
buffers.  Workload = BASELINE.json configs[1]: 153600-sample capture buffers, +-100 ppm grid at
739 MHz (n_f = 31), ds_comb_arm 2, synthetic rtl-sdr-like 8-bit IQ (SURVEY.md 8d).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned, for a fixed sample of its buffers, as DIR/<name>.npy, so
that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.

Launch for N>1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N
Capture buffers shard across ranks with no data-path collective (weak scaling: B buffers per
rank per step); the only collective is the max-over-ranks of the device time.

Prints ONE JSON line (rank 0).  `value` = whole-job Msamp/s with inputs resident in HBM;
`e2e` = same metric through the host-buffer C-ABI call (pinned host cu8 in, results out, copies
inside the timed region); `roofline` = the dominant kernel against the measured peaks;
`cpu_baseline` = the CPU oracle (port of the reference loop nest, OpenMP) on a bounded sample;
`parity_spot` = one buffer of the last timed step against the oracle; `sweep` / `tracker` = BASELINE
configs 4 and 5 (512-channel frequency sweep with an NCCL gather of the cells; 64-channel streaming
searcher) measured in the same run on the same ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "lte-cell-scanner_b200"))

N_CAP = 153600
FC = 739e6
PPM = 100.0
ARM = 2
FS = 1.92e6
SEED0 = 0xC0FFEE
DUMP_SEED = 0xD0
DUMP_BYTES = 32e6                  # room for 8 whole buffers of the n_f = 31 workload, half the 64 MB a dump may take


def synth_cu8(seed, n_cap=N_CAP, sigma=20.0):
    rng = np.random.default_rng(seed)
    v = np.clip(np.round(127.5 + sigma * rng.standard_normal((n_cap, 2))), 0, 255)
    return v.astype(np.uint8)


def f_grid():
    n_extra = int(np.floor((FC * PPM / 1e6 + 2.5e3) / 5e3))       # CellSearch.cpp:463
    return np.arange(-n_extra, n_extra + 1) * 5000.0


def b_alg(n_f, in_bytes_per_sample):
    """Algorithmic bytes per capture buffer (SURVEY.md 8d): input once + production outputs once."""
    return N_CAP * in_bytes_per_sample + 3 * 9600 * n_f * 4 + 3 * 9600 * 8 + 3 * 9600 * 4 + 9600 * 8


def f_alg(n_f, n_comb=15):
    return 8.0 * 137 * 3 * n_f * n_comb * 9600


def ncu_traffic(kernel, capbufs):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full`
    capture (profiles/traffic.json, bytes per capture buffer of the bench workload), scaled to this launch; None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return float(json.load(f)[kernel]["dram_bytes_per_capbuf"]) * capbufs
    except Exception:  # noqa
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  A thread polls NVML every 5 ms
    (pynvml; the GIL is released while the main thread waits on CUDA); if NVML is unavailable one `nvidia-smi -lms 20`
    process runs across the region instead.  Only samples stamped inside the region are kept."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                    0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.t0 = self.t1 = None
        self.nvml_rows = []
        self.thread = None
        self.stop = False

    def _nvml_loop(self, h, nv):
        while not self.stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1e3
                self.nvml_rows.append((time.time(), sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: map through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._nvml_loop, args=(h, nv), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.25)          # let the first samples arrive before the region starts
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def summary(self):
        if self.thread is not None:
            self.stop = True
            self.thread.join(timeout=1)
            inside = [r for r in self.nvml_rows if self.t0 is not None and self.t0 <= r[0] <= self.t1]
            use = inside if inside else self.nvml_rows
            reasons = set()
            for r in use:
                for bit, name in self.NVML_REASONS.items():
                    if r[3] & bit:
                        reasons.add(name)
            return dict(sm_mhz=float(np.median([r[1] for r in use])) if use else None, sm_max_mhz=float(self.sm_max),
                        power_w_max=max([r[2] for r in use]) if use else None, reasons=sorted(reasons), samples=len(inside),
                        samples_total=len(self.nvml_rows), source="nvml, 5 ms period")
        rows = []
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            import datetime
            for line in out.splitlines():
                r = [x.strip() for x in line.split(",")]
                if len(r) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except Exception:
                    ts = None
                rows.append((ts, r))
        inside = [r for ts, r in rows if ts is not None and self.t0 is not None and self.t0 - 0.02 <= ts <= self.t1 + 0.02]
        use = inside if inside else [r for _, r in rows]
        sm = [float(r[1]) for r in use if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in use if r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in use if r[3].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in use:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(pw) if pw else None, reasons=sorted(reasons), samples=len(inside),
                    samples_total=len(rows))


def host_threads():
    """Threads the CPU arm may use: physical cores visible to this process (affinity mask, cgroup quota).
    Hyper-threads only add barrier contention to the 93 OpenMP regions per capture buffer."""
    n = len(os.sched_getaffinity(0))
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    try:
        cores = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
                cores.add((phys, core))
        if cores:
            n = min(n, len(cores))
    except Exception:
        pass
    return max(1, n)


WORKLOAD = "xcorr_pss 153600-sample capbuf, n_f=31 (+-100 ppm @739 MHz), 3 PSS roots, ds_comb_arm=2"


def run_reference(args):
    """--impl reference: the CPU oracle (HEAD-faithful port of searcher.cpp:113-383, OpenMP over
    the lag index like searcher.cpp:153) on this box's host cores.  The reference binary itself
    cannot be built in this image (no IT++/FFTW/Boost - DESIGN.md)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lcs_oracle as O
    f = f_grid()
    cores = host_threads()
    O.set_threads(cores)
    caps = [((synth_cu8(SEED0 + i).astype(np.float64) - 127) / 128).view(np.complex128).reshape(-1) for i in range(2)]
    per_step = 1                                   # bounded sample: one capture buffer per step
    for w in range(args.warmup):
        O.xcorr_pss(caps[w % 2], f, ARM, FC, FC, FS, want_sp=False)
    t0 = time.perf_counter()
    for s in range(args.steps):
        O.xcorr_pss(caps[s % 2], f, ARM, FC, FC, FS, want_sp=False)
    dt = time.perf_counter() - t0
    capbufs_per_s = args.steps * per_step / dt
    val = capbufs_per_s * N_CAP / 1e6
    line = {
        "impl": "reference", "metric": "IQ Msamp/s through xcorr_pss", "value": val, "unit": "Msamp/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "xcorr_pss 153600-sample capbuf, n_f=31 (+-100 ppm @739 MHz), 3 PSS roots, ds_comb_arm=2",
                   "capbufs_per_step": per_step, "capbufs_per_s": capbufs_per_s, "n_f": int(f.size)},
        "cpu_baseline": {"value": val, "unit": "Msamp/s", "cores": cores, "kind": "port",
                         "sample": "%d capture buffers, 1 per step, all %d host threads (OpenMP over lags)" % (args.steps, cores)},
        "e2e": {"value": val, "unit": "Msamp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def cpu_baseline_leg(f, budget_s=12.0):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lcs_oracle as O
    cores = host_threads()
    O.set_threads(cores)
    cap = ((synth_cu8(SEED0).astype(np.float64) - 127) / 128).view(np.complex128).reshape(-1)
    O.xcorr_pss(cap, f, ARM, FC, FC, FS, want_sp=False)           # warm (tables, threads)
    n, t0 = 0, time.perf_counter()
    while True:
        O.xcorr_pss(cap, f, ARM, FC, FC, FS, want_sp=False)
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= 16:
            break
    return {"value": n / dt * N_CAP / 1e6, "unit": "Msamp/s", "cores": cores, "kind": "port",
            "capbufs_per_s": n / dt,
            "sample": "%d capture buffers of the bench workload (n_f=%d), %d host threads, %.1f s" % (n, f.size, cores, dt)}


def load_real_capture():
    """The reference's shipped capture test/capbuf_0000.it in its exact raw 8-bit form (tests/golden, cells 277 and 271)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "capbuf_0000.npz"))
    return g["cu8"].reshape(-1, 2)


def bind_to_gpu_numa(torch, local):
    """Pin this rank to the CPUs of the NUMA node its GPU hangs off, so that the page-locked host buffers of the e2e legs are
    allocated in (and the copy threads run on) memory local to the GPU's PCIe root complex - what `numactl --cpunodebind`
    does for a user.  Returns (original affinity, note); any failure leaves the affinity untouched."""
    orig = os.sched_getaffinity(0)
    try:
        try:
            pr = torch.cuda.get_device_properties(local)
            bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        except AttributeError:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = int(vis.split(",")[local]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else local
            bid = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(idx)).busId
            bid = bid.decode() if isinstance(bid, bytes) else bid
            bus = bid.lower()[-12:]                     # "00000000:9C:00.0" -> "0000:9c:00.0"
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return orig, "gpu %s: no NUMA node reported" % bus
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        use = cpus & orig
        if not use:
            return orig, "gpu %s: NUMA node %d has no CPU in this process' affinity mask" % (bus, node)
        os.sched_setaffinity(0, use)
        return orig, "gpu %s -> NUMA node %d, %d CPUs" % (bus, node, len(use))
    except Exception as e:  # noqa
        return orig, "not bound (%s)" % e


def all_max(torch, dist, world, dev, v):
    t = torch.tensor([v], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def dump_outputs(out_dir, torch, single, pw, frq, spi):
    """Write the outputs lcs_xcorr_pss_device returned for a seeded sample of the batch's buffers, in the layout it writes:
    single [b][3][n_f][9600] float32, pow and frq [b][3][9600] (frq as float32, exact for frequency indices),
    sp_incoherent [b][9600] float64.  Returns the sampled buffer indices."""
    B, _, n_f, _ = single.shape
    per_buf = 9600 * (3 * n_f * 4 + 3 * 8 + 3 * 4 + 8)
    n = max(1, min(B, int(DUMP_BYTES // per_buf)))
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(B, n, replace=False))
    sel = torch.from_numpy(idx).to(single.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t, dt in (("single", single, np.float32), ("pow", pw, np.float64), ("frq", frq, np.float32),
                        ("sp_incoherent", spi, np.float64)):
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, sel).cpu().numpy().astype(dt))
    return idx


def sweep_leg(L, torch, dist, ctx, rank, world, dev, barrier, reps=3):
    """BASELINE config 4: 512-channel frequency sweep (715.0 MHz + k*100 kHz, CellSearch.cpp:465), one capture buffer per
    channel (synthetic 8-bit IQ; channel 240 = 739.0 MHz carries the reference's real capture), channels round-robin over
    the ranks, every rank runs its channels through lcs_sweep_search_cu8 (one plan per centre frequency built on the
    device, one correlator launch per 64 channels, threshold + peak_search on the device, per-peak chain), NCCL all_gather
    of the detected cells, dedup on rank 0.  Timed: host buffers in -> final cell list, max over ranks."""
    import sweep as SW
    n_ch, f_start, ppm = 512, 715e6, 120.0
    f = L.f_search_set(f_start, ppm)                                  # CellSearch.cpp:463-464: one grid, from freq_start
    fcs = f_start + 100e3 * np.arange(n_ch)
    mine = SW.shard(n_ch, rank, world)
    real = load_real_capture()
    base = [synth_cu8(SEED0 + 7000 + i) for i in range(16)]
    iq = torch.empty((len(mine), N_CAP, 2), dtype=torch.uint8).pin_memory()
    iq_np = iq.numpy()
    for k, ch in enumerate(mine):
        iq_np[k] = real if abs(fcs[ch] - 739e6) < 1 else np.roll(base[ch % 16], 31 * ch, axis=0)
    sw = L.Sweep(ctx, N_CAP)
    d = dist if world > 1 else None

    def one():
        return SW.sweep_batched(list(fcs), None, lambda _iq, fc: sw.search_cu8(None, fc, f, FS, host_ptr=iq.data_ptr(), max_cells=4),
                                L.new_cell, L.dedup, dist=d, device=dev)

    res = one()                                                       # warm-up (allocations, module load)
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        res = one()
    torch.cuda.synchronize(dev)
    dt = all_max(torch, dist, world, dev, time.perf_counter() - t0)
    sw.close()
    if rank != 0:
        return None
    ids = sorted(c.n_id_cell() for c in res)
    return {"workload": "512-channel sweep 715.0-766.1 MHz, n_f=%d (ppm=120 at 715 MHz), 1 capbuf per channel, channel 739.0 MHz = "
                        "tests/golden/capbuf_0000" % f.size, "channels": n_ch, "channels_per_s": n_ch * reps / dt,
            "Msamp_per_s": n_ch * reps / dt * N_CAP / 1e6, "s_per_sweep": dt / reps, "reps": reps, "n_gpus": world,
            "cells": ids, "cells_ok": ids == [271, 277], "gather": "torch.distributed all_gather (nccl)" if world > 1 else "none (1 rank)",
            "api": "lcs_sweep_search_cu8 + lcs_dedup", "h2d_bytes_per_sweep": n_ch * N_CAP * 2}


def tracker_leg(L, torch, dist, ctx, rank, world, dev, barrier, cycles=8, reps=3):
    """BASELINE config 5: 64 channels x continuous 1.92 Msps, tracker-mode searcher (searcher_thread.cpp:83-246): every
    80 ms each channel delivers a 153600-sample buffer that is searched at the channel's current frequency-offset
    estimate (n_f = 1).  Channels round-robin over the ranks; a step = `cycles` consecutive searcher cycles of all the
    rank's channels through lcs_sweep_track_cu8 (host buffers in -> new cells + frame timing out).  Channel 0 carries the
    real capture (its two cells are already being tracked: steady state); the others are synthetic."""
    import sweep as SW
    n_ch = 64
    mine = SW.shard(n_ch, rank, world)
    real = load_real_capture()
    rng = np.random.default_rng(99)
    f_off_all = np.round(rng.uniform(-30e3, 30e3, n_ch))
    f_off_all[0] = 35228.0
    fcs_all = 739e6 + 100e3 * np.arange(n_ch)
    base = [synth_cu8(SEED0 + 9000 + i) for i in range(8)]
    iq = torch.empty((len(mine), N_CAP, 2), dtype=torch.uint8).pin_memory()
    for k, ch in enumerate(mine):
        iq.numpy()[k] = real if ch == 0 else np.roll(base[ch % 8], 13 * ch, axis=0)
    tracked = [[277, 271] if ch == 0 else [] for ch in mine]
    sw = L.Sweep(ctx, N_CAP)
    fo, fc = f_off_all[mine], fcs_all[mine]

    def cycle():
        return sw.track_cu8(None, fo, fc, FS, tracked=tracked, host_ptr=iq.data_ptr(), max_cells=4)

    first = sw.track_cu8(None, fo, fc, FS, host_ptr=iq.data_ptr(), max_cells=4)      # untracked: the real channel's cells are NEW
    cycle()
    barrier()
    t0 = time.perf_counter()
    n_new = 0
    for _ in range(reps * cycles):
        n_new += sum(len(c) for c in cycle())
    torch.cuda.synchronize(dev)
    dt = all_max(torch, dist, world, dev, time.perf_counter() - t0)
    sw.close()
    found0 = sorted(c.n_id_cell() for c, _ in first[0]) if (len(mine) and mine[0] == 0) else None
    if rank != 0:
        return None
    rate = n_ch * reps * cycles / dt
    return {"workload": "64 channels x 1.92 Msps streaming, searcher cycle per 153600-sample buffer at the tracked offset (n_f=1)",
            "channels": n_ch, "capbufs_per_s": rate, "Msamp_per_s": rate * N_CAP / 1e6, "realtime_capbufs_per_s": n_ch * 12.5,
            "x_realtime": rate / (n_ch * 12.5), "cycles": reps * cycles, "n_gpus": world, "first_cycle_cells_channel0": found0,
            "new_cells_steady_state": n_new, "api": "lcs_sweep_track_cu8", "h2d_bytes_per_cycle": n_ch * N_CAP * 2}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=384, help="capture buffers per rank per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "fp32", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-legs", action="store_true", help="skip the sweep / tracker / search legs (ncu captures)")
    ap.add_argument("--workload", default="search", choices=["search", "tracker"],
                    help="search: BASELINE configs[1] (n_f=31); tracker: SURVEY 8d config 5 shape (n_f=1 at the tracked offset)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write single / pow / frq / sp_incoherent of the last timed step (rank 0, a seeded sample of its "
                         "buffers) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import lcs_b200 as L

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    orig_affinity, numa_note = bind_to_gpu_numa(torch, local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's log (version banner, communicator lines with rank / nranks) goes to stderr so that stdout stays the one
        # JSON line; a level the environment asked for is kept if it is at least INFO
        if rank == 0:
            print("bench.py: NCCL env before init: %s" % {k: v for k, v in os.environ.items() if k.startswith("NCCL_")}, file=sys.stderr)
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ["NCCL_DEBUG_SUBSYS"] = "INIT"
        os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=dev)

    f = f_grid() if args.workload == "search" else np.array([0.0])      # searcher_thread.cpp:97-98: one offset
    n_f = int(f.size)
    B = args.batch
    wl_name = WORKLOAD if args.workload == "search" else ("tracker shape (SURVEY 8d config 5): xcorr_pss 153600-sample capbuf, n_f=1, "
                                                          "3 PSS roots, ds_comb_arm=2; real time = 12.5 capbufs/s per channel")
    ctx = L.Context(local)
    kern = {"auto": L.KERNEL_AUTO, "fp32": L.KERNEL_FP32, "tc": L.KERNEL_TC}[args.kernel]
    plan = ctx.plan(N_CAP, f, ARM, FC, FC, FS, max_batch=B, kernel=kern)
    kernel_used = {L.KERNEL_FP32: "xcorr_fold_fp32", L.KERNEL_TC: "xcorr_fold_tc"}[plan.kernel_for(L.IQ_CU8)]

    # ---- synthetic inputs: a ring of distinct batches whose inputs+outputs exceed L2 (126 MB) ----
    out_bytes_per_cap = 3 * n_f * 9600 * 4 + 3 * 9600 * 12 + 9600 * 8
    ring = max(2, int(np.ceil(300e6 / (B * (out_bytes_per_cap + N_CAP * 2)))))      # inputs+outputs in flight > L2 (126 MB)
    base = np.stack([synth_cu8(SEED0 + rank * 100003 + i) for i in range(B)])      # [B][n_cap][2] u8
    h_iq = torch.from_numpy(base).pin_memory()
    d_iq, d_single, d_pow, d_frq, d_spi = [], [], [], [], []
    for r in range(ring):
        # distinct contents per ring slot (rolled copies) so nothing is served from a previous slot's lines
        d_iq.append(torch.roll(h_iq.to(dev), shifts=r * 17, dims=1).contiguous())
        d_single.append(torch.empty((B, 3, n_f, 9600), dtype=torch.float32, device=dev))
        d_pow.append(torch.empty((B, 3, 9600), dtype=torch.float64, device=dev))
        d_frq.append(torch.empty((B, 3, 9600), dtype=torch.int32, device=dev))
        d_spi.append(torch.empty((B, 9600), dtype=torch.float64, device=dev))
    stream = torch.cuda.Stream(device=dev)
    sp = stream.cuda_stream

    def step(i):
        r = i % ring
        plan.run_device(d_iq[r].data_ptr(), L.IQ_CU8, B, d_single[r].data_ptr(), d_pow[r].data_ptr(),
                        d_frq[r].data_ptr(), d_spi[r].data_ptr(), None, sp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident timing ----
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    plan.timing_enable(True)
    launches0 = ctx.launches
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for i in range(args.steps):
            step(args.warmup + i)
        e1.record(stream)
    barrier()
    sampler.mark_end()
    ms = e0.elapsed_time(e1)
    kernel_ms, kernel_n = plan.timing_read()
    plan.timing_enable(False)
    launches = ctx.launches - launches0
    clocks = sampler.summary() if rank == 0 else None
    ms_max = all_max(torch, dist, world, dev, ms)
    capbufs_per_s = world * B * args.steps / (ms_max / 1e3)
    value = capbufs_per_s * N_CAP / 1e6
    r_last = (args.warmup + args.steps - 1) % ring      # ring slot the last timed step wrote

    dump = None
    if rank == 0 and args.dump_outputs:
        idx = dump_outputs(args.dump_outputs, torch, d_single[r_last], d_pow[r_last], d_frq[r_last], d_spi[r_last])
        dump = {"dir": os.path.abspath(args.dump_outputs), "ring_slot": r_last, "buffers": idx.tolist()}

    # ---- parity spot check: one buffer of the LAST timed step against the oracle (test infrastructure, after the timing) ----
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import lcs_oracle as O
        os.sched_setaffinity(0, orig_affinity)          # the CPU oracle may use every host core
        O.set_threads(host_threads())
        b_chk = B // 2
        cu8 = d_iq[r_last][b_chk].cpu().numpy()
        ref = O.xcorr_pss(((cu8.astype(np.float64) - 127) / 128).view(np.complex128).reshape(-1), f, ARM, FC, FC, FS, want_sp=False)
        got_s = d_single[r_last][b_chk].cpu().numpy().transpose(0, 2, 1)
        got_p = d_pow[r_last][b_chk].cpu().numpy()
        e_s = float(np.abs(got_s - ref["single"]).max() / np.abs(ref["single"]).max())
        e_p = float(np.abs(got_p - ref["pow"]).max() / ref["pow"].max())
        e_spi = float(np.abs(d_spi[r_last][b_chk].cpu().numpy() / ref["sp_incoherent"] - 1).max())
        frq_bad = int((d_frq[r_last][b_chk].cpu().numpy() != ref["frq"]).sum())
        bind_to_gpu_numa(torch, local)
        parity = {"buffer": "ring slot %d, buffer %d of the last timed step" % (r_last, b_chk), "rel_err_single": e_s, "rel_err_pow": e_p,
                  "rel_err_sp_incoherent": e_spi, "frq_mismatches_of_28800": frq_bad, "tolerance": 1e-6,
                  "ok": bool(e_s < 1e-6 and e_p < 1e-6 and e_spi < 1e-12 and frq_bad < 58)}

    # ---- e2e: host pinned cu8 in -> results to host, through lcs_xcorr_pss_batch_host ----
    h_single = torch.empty((B, 3, n_f, 9600), dtype=torch.float32).pin_memory()
    h_pow = torch.empty((B, 3, 9600), dtype=torch.float64).pin_memory()
    h_frq = torch.empty((B, 3, 9600), dtype=torch.int32).pin_memory()
    h_spi = torch.empty((B, 9600), dtype=torch.float64).pin_memory()
    e2e_steps = max(3, args.steps // 2)

    def timed_host_leg(fn, n_steps):
        for _ in range(min(args.warmup, 3)):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_steps):
            fn()                                   # synchronous: returns after the D2H completed
        torch.cuda.synchronize(dev)
        return all_max(torch, dist, world, dev, time.perf_counter() - t0)

    dt = timed_host_leg(lambda: plan.run_host(h_iq.data_ptr(), L.IQ_CU8, B, h_single.data_ptr(), h_pow.data_ptr(), h_frq.data_ptr(),
                                              h_spi.data_ptr()), e2e_steps)
    e2e_val = world * B * e2e_steps / dt * N_CAP / 1e6
    h2d = B * N_CAP * 2
    d2h = B * out_bytes_per_cap
    # same call without xc_incoherent_single (h_single = NULL): what a caller that only needs pow / frq / sp_incoherent pays
    dt = timed_host_leg(lambda: plan.run_host(h_iq.data_ptr(), L.IQ_CU8, B, None, h_pow.data_ptr(), h_frq.data_ptr(), h_spi.data_ptr()),
                        e2e_steps)
    e2e_ns_val = world * B * e2e_steps / dt * N_CAP / 1e6

    # ---- e2e_search: host buffers through the batched search call (xcorr_pss + threshold + peak_search on the device,
    # per-peak chain for buffers with a PSS; only cells return).  One buffer in 64 is the reference's real capture, so the
    # per-peak stages (sss_detect ... decode_mib) run inside the timed region; cells_found counts them. ----
    search = None
    if not args.no_extra_legs:
        real = load_real_capture()
        h_iq_s = h_iq.clone().pin_memory()
        n_real = 0
        for b in range(0, B, 64):
            h_iq_s.numpy()[b] = real
            n_real += 1
        found = [0]

        def search_step():
            found[0] += sum(len(c) for c in plan.cell_search_batch_cu8(None, max_cells=8, host_ptr=h_iq_s.data_ptr(), batch=B))

        dt_s = timed_host_leg(search_step, e2e_steps)
        n_calls = e2e_steps + min(args.warmup, 3)
        # the same batch without the real capture: the difference is the cost of the per-peak chain
        dt_n = timed_host_leg(lambda: plan.cell_search_batch_cu8(None, max_cells=8, host_ptr=h_iq.data_ptr(), batch=B), e2e_steps)
        search_val = world * B * e2e_steps / dt_s * N_CAP / 1e6
        cells_per_call = found[0] / n_calls
        search = {"value": search_val, "unit": "Msamp/s", "capbufs_per_s": search_val * 1e6 / N_CAP,
                  "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * (4 + 32 * 24), "cells_found": found[0],
                  "buffers_with_cells_per_step": n_real, "cells_per_step": cells_per_call,
                  "noise_only_value": world * B * e2e_steps / dt_n * N_CAP / 1e6,
                  "us_per_detected_cell": max(0.0, (dt_s - dt_n)) / e2e_steps / max(cells_per_call, 1e-9) * 1e6,
                  "api": "lcs_cell_search_batch_cu8 (pinned host cu8 -> cells; xcorr_pss + Z_th1 + peak_search on the "
                         "device, xc_incoherent_single stays in HBM; 1 buffer in 64 = tests/golden/capbuf_0000)"}

    sweep_res = tracker_res = None
    if not args.no_extra_legs and args.workload == "search":
        sweep_res = sweep_leg(L, torch, dist, ctx, rank, world, dev, barrier)
        tracker_res = tracker_leg(L, torch, dist, ctx, rank, world, dev, barrier)

    if rank == 0:
        peaks = load_peaks()
        k_avg_s = (kernel_ms / 1e3) / max(kernel_n, 1)
        in_bps = 2                                   # cu8 staged format
        alg_bytes = B * b_alg(n_f, in_bps)
        alg_flops = B * f_alg(n_f)
        timed_s = ms / 1e3
        if kernel_used == "xcorr_fold_tc":
            # burst cuBLAS figure unless the kernel ran inside a seconds-long power-capped sequence (B200_PROFILING.md)
            long_run = timed_s > 2.0
            pk = peaks["bf16_tflops_sustained"] if long_run else peaks["bf16_tflops"]
            roof = {"bound": "tensor", "achieved": alg_flops / k_avg_s / 1e12, "peak": pk, "unit": "TFLOP/s",
                    "peak_kind": ("sustained bf16 (timed region %.2f s > 2 s)" if long_run else "burst bf16 (timed region %.2f s)") % timed_s,
                    "frac_of_burst": alg_flops / k_avg_s / 1e12 / peaks["bf16_tflops"],
                    "frac_of_sustained": alg_flops / k_avg_s / 1e12 / peaks["bf16_tflops_sustained"],
                    "tensor_mode": "tcgen05 kind::i8 (s8 x s8 -> s32, exact); the driver measures only a bf16 peak, int8 runs at 2x "
                                   "that rate; achieved counts F_alg only - the kernel executes 3 int8 digit planes x 96/93 column padding "
                                   "x 288/274 K padding x 9728/9600 tile rounding = 3.3x more MACs than F_alg"}
        else:
            roof = {"bound": "hbm", "achieved": alg_bytes / k_avg_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
        roof["frac"] = roof["achieved"] / roof["peak"]
        if kernel_used == "xcorr_fold_tc" and args.workload == "search":
            # executed int8 operations: 38 tiles x 15 half frames x 2 sub-tiles x 2 parts x 2 jobs per buffer, 9 UTCIMMA of
            # M=128, N=144, K=32 B per job; against the rate a loop of nothing but these instructions sustains on all SMs
            # (tools/microbench/umma_sustained.cu, profiles/r02_umma_sustained_microbench.txt)
            ops = B * 38 * 15 * 2 * 2 * 2 * 9 * (2.0 * 128 * 144 * 32)
            pops = ops / k_avg_s / 1e15
            ceil_pops = 3.65 if (clocks and clocks.get("sm_mhz") and clocks["sm_mhz"] < 1750) else 4.1
            roof.update({"executed_int8_pops": pops, "pure_mma_ceiling_int8_pops": ceil_pops,
                         "pure_mma_ceiling_note": "4.1 POP/s for a burst at ~1.83 GHz, 3.65 POP/s power-capped at ~1.63 GHz (measured, profiles/r02_umma_sustained_microbench.txt); chosen by the SM clock sampled during this run",
                         "frac_of_pure_mma_ceiling": pops / ceil_pops})
        roof.update({"traffic": ncu_traffic(kernel_used, B), "traffic_source": "profiles/traffic.json (ncu --set full capture of this kernel, scaled to this batch)",
                     "kernel": kernel_used, "kernel_avg_ms": k_avg_s * 1e3, "kernel_launches": kernel_n,
                     "kernel_share_of_step": kernel_ms / ms, "alg_bytes_per_launch": alg_bytes,
                     "alg_flops_per_launch": alg_flops, "alg_tflops": alg_flops / k_avg_s / 1e12,
                     "hbm_frac": alg_bytes / k_avg_s / 1e9 / peaks["hbm_gbs"],
                     "peak_source": peaks["source"],
                     "note": "compute-bound contraction (AI ~3000 FLOP/B, SURVEY 8d): HBM fraction is reported because "
                             "the BASELINE metric asks for it; alg_tflops is the governing figure"})
        line = {
            "metric": "IQ Msamp/s through xcorr_pss", "value": value, "unit": "Msamp/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if kernel_used == "xcorr_fold_fp32" else "s8 (3 exact int8 digits, int32 accumulate)",
            "data": "synthetic",
            "config": {"workload": wl_name,
                       "capbufs_per_step_per_gpu": B, "capbufs_per_s": capbufs_per_s, "n_f": n_f, "iq_format": "cu8",
                       "parallelism": "capbufs sharded across %d rank(s), no data-path collective" % world,
                       "l2": "ring of %d input/output sets (%.0f MB) larger than L2" % (ring, ring * B * (out_bytes_per_cap + N_CAP * 2) / 1e6),
                       "kernel": kernel_used,
                       **({"realtime_channels": capbufs_per_s / 12.5} if args.workload == "tracker" else {})},
            "e2e": {"value": e2e_val, "unit": "Msamp/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "api": "lcs_xcorr_pss_batch_host (pinned host cu8 -> host pow/frq/sp_incoherent/single)"},
            "e2e_nosingle": {"value": e2e_ns_val, "unit": "Msamp/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": B * (3 * 9600 * 12 + 9600 * 8),
                             "steps": e2e_steps, "api": "lcs_xcorr_pss_batch_host with h_single = NULL (pow/frq/sp_incoherent only)"},
            "gpu_launches": int(launches), "roofline": roof, "clocks": clocks,
        }
        if search is not None:
            line["e2e_search"] = search
        if parity is not None:
            line["parity_spot"] = parity
        if dump is not None:
            line["dump_outputs"] = dump
        if sweep_res is not None:
            line["sweep"] = sweep_res
        if tracker_res is not None:
            line["tracker"] = tracker_res
        line["config"]["host_binding"] = numa_note
        if not args.no_cpu_baseline and world == 1:
            os.sched_setaffinity(0, orig_affinity)
            line["cpu_baseline"] = cpu_baseline_leg(f)
        print(json.dumps(line))
    plan.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
