#!/usr/bin/env python
"""Benchmark of the CWT hot path (BASELINE.json metric: CWT scale-points/s and HBM GB/s vs
roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--configs 2,3,4,5] [--kernels-only] [--dump-outputs DIR]

Headline workload (SURVEY 8d config 2): Morlet(6) CWT of a synthetic linear chirp, N = 2^20,
256 scales (s0=2, dj=1/16, J=255), fp64.  One "step" = one full transform of one signal (forward
FFT + every scale).  Under torchrun every rank transforms its own signal on its own GPU (weak
scaling, no data-path collective); `value` = all ranks' scale-points / max time over ranks.

The same JSON line carries, under "configs", one result object per additional BASELINE.json
configuration (3: Paul/DOG fp32, 4: xwt + wct + 200 surrogates, 5: batched channels), each with
its own `e2e`, `roofline` and `cpu_baseline`; under torchrun also the two sharded paths of
SURVEY 8e (config 5 channels over ranks with the NCCL gather of the spectra inside the timed
region; config 2 scales over ranks, strong scaling).  `--configs 2` restricts the run to the
headline.  See DESIGN.md "Measurement" for every field.

`--dump-outputs DIR` writes, after the timed steps, what the headline transform computed in its
last step (see `dump_config2`), so that two builds can be compared output for output: the
inputs depend only on the arguments.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workloads as wl   # noqa: E402

METRIC = "cwt_scale_points_per_sec"
UNIT = "scale-points/s"


# ---------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def source_hash():
    """SHA-256 over the CUDA sources: ties ncu-derived numbers to the build they came from."""
    h = hashlib.sha256()
    for f in ("cplx.cuh", "fft_tile.cuh", "kernels.cuh", "engine.cu"):
        with open(os.path.join(ROOT, "pycwt_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_name` from the committed
    `ncu --set full` captures (profiles/traffic.json, written by profiles/ncu_traffic.py), or None
    when there is no capture of THIS build of the sources (source hash mismatch)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        if t.get("source_hash") != source_hash():
            return None
        k = t["kernels"].get(kernel_name)
        return None if k is None else k
    except Exception:
        return None


class ClockSampler(object):
    """SM clock and throttle reasons of one GPU during the timed region: NVML in a sampling thread
    (one query costs ~0.1 ms, so even a 15 ms region yields samples; `nvidia-smi -lms` needs
    hundreds of ms to start on an 8-GPU box and returned nothing there), nvidia-smi as the
    fallback.  `index` is the CUDA device index of this rank."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index = index
        self.sm, self.bits = [], 0
        self.max_mhz = None
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None
        self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: resolve through the PCI bus id
            bus = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id",
                                           "--format=csv,noheader"], text=True).strip()
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_once(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            self.bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            try:
                self.bits |= int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass

    def _loop(self):
        while not self.stop_flag.is_set():
            try:
                self._sample_once()
            except Exception:
                break
            self.stop_flag.wait(0.002)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if self.nvml is None:
            return self._smi_once()
        self.stop_flag.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        if not self.sm:
            return self._smi_once()
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "samples": len(self.sm),
                "reasons": sorted(nm for nm, bit in self.REASONS if self.bits & bit), "how": "nvml, 2 ms period"}

    def _smi_once(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            f = [x.strip() for x in subprocess.check_output(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                text=True, timeout=20).strip().split(",")]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            return {"sm_mhz": float(f[0]), "sm_max_mhz": float(f[1]), "samples": 1,
                    "reasons": sorted(nm for nm, v in zip(names, f[2:6]) if v.lower().startswith("active")),
                    "how": "one nvidia-smi query right after the timed region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}


class Dist(object):
    """Process-group plumbing: torch.distributed (NCCL) for the barrier / max-over-ranks of the
    bench contract, plus the product's own communicator (NCCL behind the C ABI) for the sharded
    data paths."""

    def __init__(self, n_gpus):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(self.local)
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            import torch
            self.dist.barrier(device_ids=[self.local])
            torch.cuda.synchronize()

    def max(self, value):
        if self.dist is None:
            return value
        import torch
        t = torch.tensor([value], dtype=torch.float64, device="cuda:%d" % self.local)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def broadcast_bytes(self, data):
        """rank 0's bytes object to every rank (the NCCL id of the product communicator)."""
        if self.dist is None:
            return data
        box = [data]
        self.dist.broadcast_object_list(box, src=0)
        return box[0]

    def close(self):
        if self.dist is not None:
            self.dist.barrier(device_ids=[self.local])
            self.dist.destroy_process_group()


def pin_to_gpu_numa_node(local_rank):
    """CPU affinity (and with it first-touch page placement of the pinned result buffers) on the
    NUMA node the GPU hangs off: eight ranks copying 4.3 GB each otherwise contend for one
    socket's memory controllers.  Returns the node or None."""
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id",
                                       "--format=csv,noheader"], text=True).strip().lower()
        bus = bus[-12:] if len(bus) > 12 else bus          # 00000000:1B:00.0 -> 0000:1b:00.0
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def dominant_writer(prof, bytes_per_row):
    """The W-writing kernel type with the largest share of the step and its roofline numbers.
    Writers carry `bytes_per_row` algorithmic bytes per scale row; "fwd:" / "coarse:" launches and
    the first kernels of the two-kernel scales are intermediate work (0 algorithmic bytes)."""
    writers = [k for k in prof if ":" not in k["name"] and k["name"].split("<")[0] in
               ("SingleBody", "DirectBody", "PassBBody", "ExpandBody", "ExpandMmaBody", "PipeAB") and ", -1" not in k["name"]]
    if not writers:
        return None
    kern_ms = sum(k["ms"] for k in prof)
    w = max(writers, key=lambda k: k["ms"])
    nbytes = w["rows"] * bytes_per_row
    t = ncu_traffic(w["name"])
    return {"kernel": w["name"], "launches_per_step": w["launches"], "ms_per_step": w["ms"],
            "share_of_step": w["ms"] / kern_ms, "rows": w["rows"],
            "algorithmic_bytes_per_step": nbytes,
            "algorithmic_bytes_per_launch": nbytes / w["launches"],
            "achieved": nbytes / (w["ms"] * 1e-3) / 1e9,
            "traffic": None if t is None else t["dram_bytes_per_row"] * w["rows"] / w["launches"],
            "largest_kernel_any": max(prof, key=lambda k: k["ms"])["name"]}


def roofline_block(prof, bytes_per_row, step_bytes, step_ms):
    peak, peak_src = measured_peaks()
    dom = dominant_writer(prof, bytes_per_row)
    step_achieved = step_bytes / (step_ms * 1e-3) / 1e9
    out = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src,
           "step": {"achieved": step_achieved, "frac": step_achieved / peak,
                    "algorithmic_bytes": step_bytes},
           "kernels": {k["name"]: {"launches": k["launches"], "ms": round(k["ms"], 4), "rows": k["rows"]}
                       for k in prof},
           "source_hash": source_hash()}
    if dom is not None:
        out.update({"achieved": dom["achieved"], "frac": dom["achieved"] / peak, "traffic": dom["traffic"]})
        out.update({k: dom[k] for k in ("kernel", "launches_per_step", "ms_per_step", "share_of_step", "rows",
                                        "algorithmic_bytes_per_step", "algorithmic_bytes_per_launch",
                                        "largest_kernel_any")})
    return out


# ---------------------------------------------------------------------------------------------
# CPU side: the reference itself (oracle/_ref: unmodified copy of the reference package, built by
# oracle/make_ref.py) or, where that copy is absent, the oracle port
# ---------------------------------------------------------------------------------------------
def reference_module():
    from oracle import make_ref
    if make_ref.available():
        return make_ref.load(), "reference"
    from oracle import cwt_oracle as orc
    return orc, "port"


def subset_freqs(mod, wavelet, sj, count):
    idx = np.linspace(0, len(sj) - 1, count).round().astype(int)
    return 1.0 / (wavelet.flambda() * sj[idx])


def cpu_config2(sample_scales):
    """Stock `pycwt.cwt` (reference wavelet.py:13-124, single-threaded scipy.fftpack) on a bounded
    sample of config 2: `sample_scales` of the 256 scales, evenly spread, full N."""
    mod, kind = reference_module()
    x = wl.config2_signal()
    w = mod.Morlet(wl.C2["f0"])
    fr = subset_freqs(mod, w, wl.config2_scales(), sample_scales)
    t0 = time.perf_counter()
    W = mod.cwt(x, wl.C2["dt"], wavelet=w, freqs=fr)[0]
    dt = time.perf_counter() - t0
    assert W.shape == (sample_scales, wl.C2["n"])
    return sample_scales * wl.C2["n"] / dt, dt, kind


def cpu_port_all_threads(sample_scales):
    """The oracle port with scipy.fft on every host thread (the reference has no threaded path;
    reported beside the stock number for scale)."""
    from oracle import cwt_oracle as orc
    x = wl.config2_signal()
    w = orc.Morlet(wl.C2["f0"])
    fr = subset_freqs(orc, w, wl.config2_scales(), sample_scales)
    t0 = time.perf_counter()
    orc.cwt(x, wl.C2["dt"], wavelet=w, freqs=fr, workers=os.cpu_count() or 1)
    return sample_scales * wl.C2["n"] / (time.perf_counter() - t0)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host
    cores, each step a bounded sample (16 of the 256 scales, full N) of config 2."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = 16
    kind = reference_module()[1]
    for _ in range(min(args.warmup, 1)):
        cpu_config2(4)
    tot_t, tot_pts = 0.0, 0
    for _ in range(args.steps):
        v, dt, kind = cpu_config2(sample)
        tot_t += dt
        tot_pts += sample * wl.C2["n"]
    value = tot_pts / tot_t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config2_description(),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind,
                         "sample": "%d of 256 scales (evenly spread, freqs=...), full N=2^20, per step; "
                                   "stock pycwt.cwt, scipy.fftpack, one thread (the reference has no "
                                   "threaded path)" % sample if kind == "reference" else
                                   "%d of 256 scales, full N=2^20, per step; oracle port (oracle/_ref "
                                   "absent), one thread" % sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def config2_description():
    c = wl.C2
    return {"workload": "config2: Morlet(6) CWT, synthetic chirp N=2^20, 256 scales "
                        "(s0=2, dj=1/16, J=255), fp64, one signal per GPU",
            "n": c["n"], "scales": c["J"] + 1, "wavelet": "morlet(6)",
            "l2": "no explicit flush: each step writes 4.29 GB of coefficients (>> 126 MB L2) "
                  "and re-reads only the 16 MiB spectrum it just produced"}


# ---------------------------------------------------------------------------------------------
# config 2 (headline)
# ---------------------------------------------------------------------------------------------
DUMP_COLUMNS = 8192


def dump_config2(out_dir, eng, n_scales, n):
    """The outputs of the resident transform as a caller fetches them (`Engine.get_w`,
    `Engine.signal_fft`), as float64 .npy files: W at every scale for DUMP_COLUMNS time
    indices drawn once from RandomState(0), sorted (W_real, W_imag: 32 MiB of the 4 GiB), and
    the signal spectrum returned beside it (fft_real, fft_imag)."""
    os.makedirs(out_dir, exist_ok=True)
    cols = np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_COLUMNS), replace=False))
    W = eng.get_w(n_scales, n)
    Ws = W[:, cols]
    del W
    fft = eng.signal_fft()
    for name, a in (("W_real", Ws.real), ("W_imag", Ws.imag), ("fft_real", fft.real), ("fft_imag", fft.imag)):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_config2(args, D, eng, pycwt, _engine):
    c = wl.C2
    sj = wl.config2_scales()
    S = len(sj)
    x = wl.config2_signal(D.rank)
    pts = S * c["n"]

    # ---- value: inputs resident in HBM, kernels only (CUDA events in the engine) ----
    dsig = eng.dev_alloc(x.nbytes)
    eng.h2d(dsig, x)
    eng.cwt_dev(dsig, 0, c["n"], c["dt"], sj, _engine.MORLET, c["f0"], _engine.F64)   # plans + first run
    if args.warmup > 0:
        eng.bench_last(args.warmup)
    launches_per_step = eng.last_launch_count()
    sampler = ClockSampler(D.local)
    D.barrier()
    eng.sync()
    sampler.start()
    ms = eng.bench_last(args.steps)          # mean device ms per step, events on the engine stream
    eng.sync()
    D.barrier()
    clocks = sampler.stop()
    ms_max = D.max(ms)
    if args.dump_outputs and D.rank == 0:
        dump_config2(args.dump_outputs, eng, S, c["n"])
    value = D.world * pts / (ms_max * 1e-3)
    prof = eng.profile_last()    # per-kernel-type event times of one more (untimed, serialised) step
    eng.dev_free(dsig)
    if args.kernels_only:   # for ncu: no e2e leg, no CPU baseline
        return {"kernels_only": True, "ms_per_step": ms_max, "value": value,
                "launches_per_step": launches_per_step,
                "kernels": {k["name"]: [k["launches"], round(k["ms"], 4), k["rows"]] for k in prof}}

    # ---- e2e: public API, host buffers, H2D + D2H inside the timed region ----
    e2e_steps = max(1, min(args.steps, 5))
    mother = pycwt.Morlet(c["f0"])
    for _ in range(2):   # warm-up: default engine, device buffers, the two pinned result buffers
        W, *_ = pycwt.cwt(x, c["dt"], c["dj"], c["s0"], c["J"], mother)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        W, *_ = pycwt.cwt(x, c["dt"], c["dj"], c["s0"], c["J"], mother)
    t_e2e = (time.perf_counter() - t0) / e2e_steps
    assert W.shape == (S, c["n"])
    del W
    t_e2e = D.max(t_e2e)

    # ---- e2e through the device-resident API: only O(S) + O(N) numbers leave the GPU ----
    for _ in range(3):   # warm-up: the pinned O(N) result buffers of the products circulate in pairs
        r = pycwt.cwt_resident(x, c["dt"], c["dj"], c["s0"], c["J"], mother)
        gp, sa, iw = r.global_power(), r.scale_avg_power(2, 8), r.icwt()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r = pycwt.cwt_resident(x, c["dt"], c["dj"], c["s0"], c["J"], mother)
        gp, sa, iw = r.global_power(), r.scale_avg_power(2, 8), r.icwt()
    t_res = D.max((time.perf_counter() - t0) / e2e_steps)
    pycwt.default_engine().trim()

    step_bytes = pts * 16 + c["n"] * 8
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": D.world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config2_description(),
        "e2e": {"value": D.world * pts / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(x.nbytes),
                "d2h_bytes_per_step": int(pts * 16), "ms_per_step": 1e3 * t_e2e, "steps": e2e_steps,
                "resident": {"value": D.world * pts / t_res, "unit": UNIT, "ms_per_step": 1e3 * t_res,
                             "d2h_bytes_per_step": int(S * 8 + 2 * c["n"] * 8),
                             "what": "cwt_resident + global_power + scale_avg_power + icwt: W (4.29 GB) "
                                     "stays in HBM, the products are reduced on the device"}},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roofline_block(prof, c["n"] * 16, step_bytes, ms_max),
        "clocks": clocks,
    }
    line["roofline"]["step"]["nominal_fp64_tflops"] = S * 5.0 * c["n"] * np.log2(c["n"]) / (ms_max * 1e-3) / 1e12
    line["roofline"]["step"]["note"] = "whole step: forward FFT + all per-scale inverse transforms"
    return line


def cpu_baseline_config2(world):
    if world != 1:
        return {"value": None, "unit": UNIT, "cores": 1, "kind": reference_module()[1], "sample": "timed at N=1 only"}
    sample = 8
    v, dt, kind = cpu_config2(sample)
    out = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
           "sample": "%d of 256 scales (evenly spread), full N=2^20, stock pycwt.cwt single-threaded; %.1f s"
                     % (sample, dt)}
    try:
        out["port_all_threads"] = {"value": cpu_port_all_threads(16), "cores": os.cpu_count(),
                                   "what": "oracle port, scipy.fft workers = all host threads, 16 scales"}
    except Exception as exc:   # the port is optional decoration
        out["port_all_threads"] = {"error": str(exc)}
    return out


# ---------------------------------------------------------------------------------------------
# config 3: Paul(4) / DOG(2), N = 2^18, 128 scales, fp32
# ---------------------------------------------------------------------------------------------
def run_config3(args, D, eng, pycwt, _engine):
    c = wl.C3
    x = wl.config3_signal()
    out = {"workload": "config3: Paul(4) and DOG(2) CWT, chirp N=2^18 (float32), 128 scales, fp32 engine",
           "dtype": "f32", "metric": METRIC, "unit": UNIT}
    steps = args.steps
    mod, kind = reference_module()
    os.environ["CWTB_PRECISION"] = "fp32"
    try:
        for fam, code in (("paul", _engine.PAUL), ("dog", _engine.DOG)):
            p = c[fam]
            sj = wl.geometric_scales(p["s0"], p["dj"], p["J"])
            pts = len(sj) * c["n"]
            dsig = eng.dev_alloc(x.nbytes)
            eng.h2d(dsig, x)
            eng.cwt_dev(dsig, 1, c["n"], c["dt"], sj, code, float(p["m"]), _engine.F32)
            eng.bench_last(max(args.warmup, 3))
            ms = eng.bench_last(steps)
            launches = eng.last_launch_count()
            prof = eng.profile_last()
            eng.dev_free(dsig)
            mother = pycwt.Paul(p["m"]) if fam == "paul" else pycwt.DOG(p["m"])
            for _ in range(2):
                W, *_ = pycwt.cwt(x, c["dt"], p["dj"], p["s0"], p["J"], mother)
            t0 = time.perf_counter()
            for _ in range(5):
                W, *_ = pycwt.cwt(x, c["dt"], p["dj"], p["s0"], p["J"], mother)
            t_e2e = (time.perf_counter() - t0) / 5
            assert W.shape == (len(sj), c["n"]) and W.dtype == np.complex128
            del W
            res = {"value": pts / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "gpu_launches": launches * steps,
                   "e2e": {"value": pts / t_e2e, "unit": UNIT, "ms_per_step": 1e3 * t_e2e,
                           "h2d_bytes_per_step": int(x.nbytes), "d2h_bytes_per_step": int(pts * 16),
                           "note": "float32 in, complex128 out like the reference (widened on the device)"},
                   "roofline": roofline_block(prof, c["n"] * 8, pts * 8 + c["n"] * 4, ms)}
            if D.world == 1:
                w = mod.Paul(p["m"]) if fam == "paul" else mod.DOG(p["m"])
                fr = subset_freqs(mod, w, sj, 16)
                t0 = time.perf_counter()
                mod.cwt(x, c["dt"], wavelet=w, freqs=fr)
                dt = time.perf_counter() - t0
                res["cpu_baseline"] = {"value": 16 * c["n"] / dt, "unit": UNIT, "cores": 1, "kind": kind,
                                       "sample": "16 of 128 scales, full N=2^18; %.1f s" % dt}
            out[fam] = res
    finally:
        os.environ.pop("CWTB_PRECISION", None)
    out["value"] = min(out["paul"]["value"], out["dog"]["value"])
    return out


# ---------------------------------------------------------------------------------------------
# config 4: xwt + wct of two N = 2^18 series, Morlet, 200 Monte-Carlo surrogates
# ---------------------------------------------------------------------------------------------
def run_config4(args, D, eng, pycwt, _engine):
    c = wl.C4
    y1, y2 = wl.config4_signals()
    m = pycwt.Morlet(c["f0"])
    S = c["J"] + 1
    pts = S * c["n"]
    peak, _ = measured_peaks()
    deng = pycwt.default_engine()
    out = {"workload": "config4: xwt + wct(sig) of two noisy chirps N=2^18, Morlet(6), s0=2, dj=1/12, J=144 "
                       "(145 scales), 200 Monte-Carlo surrogate pairs of 49152 samples", "dtype": "f64",
           "metric": METRIC, "unit": UNIT}

    def timed(fn, reps=5):
        # three warm-up calls: the second and third bring the two pinned result buffers into the
        # engine's pool that then circulate (the previous result is still referenced while the next
        # call runs); a cold call page-locks 608 MB (~60 ms), which is not the steady state
        for _ in range(3):
            r = fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) / reps, r

    t_x, _ = timed(lambda: pycwt.xwt(y1, y2, c["dt"], c["dj"], c["s0"], c["J"], wavelet=m))
    k_x = deng.last_kernel_ms()
    t_w, _ = timed(lambda: pycwt.wct(y1, y2, c["dt"], c["dj"], c["s0"], c["J"], sig=False, wavelet=m))
    k_w = deng.last_kernel_ms()
    out["xwt"] = {"value": pts / (k_x * 1e-3), "kernels_ms": k_x,
                  "e2e": {"value": pts / t_x, "ms_per_step": 1e3 * t_x, "h2d_bytes_per_step": int(2 * y1.nbytes),
                          "d2h_bytes_per_step": int(pts * 16)},
                  "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak,
                               "algorithmic_bytes": pts * 16 + 2 * y1.nbytes,
                               "achieved": (pts * 16 + 2 * y1.nbytes) / (k_x * 1e-3) / 1e9,
                               "frac": (pts * 16 + 2 * y1.nbytes) / (k_x * 1e-3) / 1e9 / peak,
                               "note": "W12 written once (two transforms, conj-product fused into the second)"}}
    out["wct"] = {"value": pts / (k_w * 1e-3), "kernels_ms": k_w,
                  "e2e": {"value": pts / t_w, "ms_per_step": 1e3 * t_w, "h2d_bytes_per_step": int(2 * y1.nbytes),
                          "d2h_bytes_per_step": int(pts * 16)},
                  "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak,
                               "algorithmic_bytes": pts * 16 + 2 * y1.nbytes,
                               "achieved": (pts * 16 + 2 * y1.nbytes) / (k_w * 1e-3) / 1e9,
                               "frac": (pts * 16 + 2 * y1.nbytes) / (k_w * 1e-3) / 1e9 / peak,
                               "note": "WCT + aWCT (f64) out, two series in (SURVEY 8d); 2 transforms + 4 "
                                       "smoothing transforms + coherence per call"}}
    # Monte-Carlo significance, host RNG in the reference's order (bit-reproducible levels)
    a1, a2 = 0.3, 0.5
    np.random.seed(0)
    pycwt.wct_significance(a1, a2, c["dt"], c["dj"], c["s0"], c["J"], wavelet=m, mc_count=8, progress=False, cache=False)
    np.random.seed(0)
    t0 = time.perf_counter()
    pycwt.wct_significance(a1, a2, c["dt"], c["dj"], c["s0"], c["J"], wavelet=m, mc_count=c["mc_count"],
                           progress=False, cache=False)
    t_mc = time.perf_counter() - t0
    nmc = 49152
    out["mc"] = {"pairs": c["mc_count"], "seconds": t_mc, "pairs_per_s": c["mc_count"] / t_mc,
                 "surrogate_scale_points_per_s": 2 * c["mc_count"] * S * nmc / t_mc,
                 "note": "end to end: host RNG (numpy global stream, reference order) + H2D + 2 transforms, "
                         "3 smoothings, coherence and histogram per pair on the GPU"}
    out["value"] = pts / ((k_x + k_w) * 1e-3)
    if D.world == 1:
        mod, kind = reference_module()
        ns = 2 ** 14
        z1, z2 = wl.config4_signals(ns)
        w = mod.Morlet(c["f0"])
        t0 = time.perf_counter()
        mod.xwt(z1, z2, c["dt"], c["dj"], c["s0"], c["J"], wavelet=w)
        tx = time.perf_counter() - t0
        t0 = time.perf_counter()
        mod.wct(z1, z2, c["dt"], c["dj"], c["s0"], c["J"], sig=False, wavelet=w)
        tw = time.perf_counter() - t0
        out["cpu_baseline"] = {"kind": kind, "cores": 1, "unit": UNIT,
                               "value": S * ns / (tx + tw),
                               "xwt": S * ns / tx, "wct": S * ns / tw,
                               "sample": "stock xwt + wct(sig=False) on N=2^14 slices of the two series, same 145 "
                                         "scales: %.1f s + %.1f s (the full N=2^18 pair takes ~40 s; the "
                                         "reference's Monte-Carlo loop ~23 s per surrogate pair, BASELINE.md)" % (tx, tw)}
    return out


# ---------------------------------------------------------------------------------------------
# config 5: batched channels, N = 2^16, 128 scales, fp32, 1024 channels per GPU
# ---------------------------------------------------------------------------------------------
def run_config5(args, D, eng, pycwt, _engine, comm=None):
    c = wl.C5
    sj = wl.geometric_scales(c["s0"], c["dj"], c["J"])
    S = len(sj)
    nch = c["per_gpu"]
    X = wl.config5_channels(D.rank * nch, nch)
    pts_gpu = nch * S * c["n"]
    out = {"workload": "config5: Morlet(6) CWT of %d channels x N=2^16 (float32), 128 scales, fp32 engine, "
                       "%d channels per GPU; coefficients stay sharded in HBM, [channels, scales] spectra are "
                       "gathered" % (nch * D.world, nch), "dtype": "f32", "metric": METRIC, "unit": UNIT,
           "scaling": "weak"}
    # kernels with the inputs resident: chunks of 256 channels (17 GB of complex64 coefficients each)
    chunk = 256
    dX = eng.dev_alloc(chunk * c["n"] * 4)
    eng.h2d(dX, X[:chunk])
    eng.cwt_batch_dev(dX, chunk, c["n"], c["dt"], sj, _engine.MORLET, c["f0"], _engine.F32)
    eng.bench_last(2)
    D.barrier()
    ms = D.max(eng.bench_last(args.steps))
    launches = eng.last_launch_count()
    prof = eng.profile_last()
    eng.dev_free(dX)
    pts_chunk = chunk * S * c["n"]
    out.update({"value": D.world * pts_chunk / (ms * 1e-3), "ms_per_step": ms, "steps": args.steps,
                "step": "one 256-channel chunk (4 per GPU share)", "gpu_launches": launches * args.steps,
                "roofline": roofline_block(prof, c["n"] * 8, pts_chunk * 8 + chunk * c["n"] * 4, ms)})
    # end to end: host float32 channels in, per-channel spectra out, gathered over the ranks
    from pycwt_b200 import distributed as Dm
    # warm-up: engine buffers and the communicator's first collective (NCCL connects lazily)
    p0, _ = eng.cwt_batch(X[:64], c["dt"], sj, _engine.MORLET, c["f0"], _engine.F32, want_power=True)
    Dm.gather_rows(p0, 64 * D.world, comm)
    Dm.gather_rows(np.zeros((nch, S)), nch * D.world, comm)   # and once at the size of the timed gather
    D.barrier()
    t0 = time.perf_counter()
    power, _ = eng.cwt_batch(X, c["dt"], sj, _engine.MORLET, c["f0"], _engine.F32, want_power=True)
    full = Dm.gather_rows(power, nch * D.world, comm)
    t_e2e = D.max(time.perf_counter() - t0)
    assert full.shape == (nch * D.world, S)
    out["e2e"] = {"value": D.world * pts_gpu / t_e2e, "unit": UNIT, "ms_per_step": 1e3 * t_e2e,
                  "h2d_bytes_per_step": int(X.nbytes), "d2h_bytes_per_step": int(full.nbytes),
                  "collective": "ncclAllGather of the [channels, scales] spectra through the C ABI "
                                "(cwtb_comm_allgather)" if comm is not None and comm.world > 1 else "none (1 GPU)"}
    if D.world == 1:
        mod, kind = reference_module()
        w = mod.Morlet(c["f0"])
        fr = 1.0 / (w.flambda() * sj)
        t0 = time.perf_counter()
        for ch in range(2):
            mod.cwt(X[ch], c["dt"], wavelet=w, freqs=fr)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": 2 * S * c["n"] / dt, "unit": UNIT, "cores": 1, "kind": kind,
                               "sample": "2 of the 8192 channels, all 128 scales; %.1f s" % dt}
    return out


def run_config2_scale_sharded(args, D, eng, pycwt, _engine, comm):
    """SURVEY 8e row 2: ONE config-2 signal, the 256 scales block-partitioned over the ranks
    (strong scaling); the [S] global spectrum is all-gathered through the C ABI."""
    from pycwt_b200 import distributed as Dm
    c = wl.C2
    sj = wl.config2_scales()
    x = wl.config2_signal(0)
    rows = Dm.scale_rows(len(sj), D.rank, D.world)      # cyclic: balances small (costly) and large scales
    dsig = eng.dev_alloc(x.nbytes)
    eng.h2d(dsig, x)
    eng.cwt_dev(dsig, 0, c["n"], c["dt"], sj[rows], _engine.MORLET, c["f0"], _engine.F64)
    eng.bench_last(3)
    D.barrier()
    ms = D.max(eng.bench_last(10))
    eng.dev_free(dsig)
    Dm.cwt_scale_sharded(x, c["dt"], sj, _engine.MORLET, c["f0"], _engine.F64, eng, comm)   # warm-up
    D.barrier()
    t0 = time.perf_counter()
    Dm.cwt_scale_sharded(x, c["dt"], sj, _engine.MORLET, c["f0"], _engine.F64, eng, comm)
    t_e2e = D.max(time.perf_counter() - t0)
    pts = len(sj) * c["n"]
    return {"workload": "config2 scale-sharded: one N=2^20 signal, 256 scales over %d GPUs" % D.world,
            "scaling": "strong", "value": pts / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "e2e": {"value": pts / t_e2e, "ms_per_step": 1e3 * t_e2e,
                    "note": "host signal in, slabs stay resident, [S] spectrum gathered (ncclAllGather)"}}


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    D = Dist(args.gpus)
    numa = pin_to_gpu_numa_node(D.local) if os.environ.get("CWTB_NUMA_PIN", "1") != "0" else None
    import pycwt_b200 as pycwt
    from pycwt_b200 import _engine, distributed as Dm
    eng = _engine.Engine(D.local)
    configs = [int(v) for v in args.configs.split(",") if v]

    line = run_config2(args, D, eng, pycwt, _engine)
    if args.kernels_only:
        if D.rank == 0:
            print(json.dumps(line))
        D.close()
        return
    line["topology"] = {"numa_node_of_gpu": numa, "cpus": len(os.sched_getaffinity(0))}
    line["cpu_baseline"] = cpu_baseline_config2(D.world) if D.rank == 0 else None

    comm = None
    if D.world > 1:
        # the product's communicator: NCCL behind the C ABI; its 128-byte id travels over the
        # bench's own process group
        uid = D.broadcast_bytes(eng.comm_unique_id() if D.rank == 0 else None)
        comm = Dm.NcclComm(eng, D.rank, D.world, exchange=lambda _u: uid)
    extra = {}
    try:
        if 3 in configs and D.world == 1:
            extra["3"] = run_config3(args, D, eng, pycwt, _engine)
        if 4 in configs and D.world == 1:
            extra["4"] = run_config4(args, D, eng, pycwt, _engine)
        if 5 in configs:
            extra["5"] = run_config5(args, D, eng, pycwt, _engine, comm)
        if D.world > 1:
            extra["2_scale_sharded"] = run_config2_scale_sharded(args, D, eng, pycwt, _engine, comm)
    except Exception as exc:       # the headline must survive a failure of an additional config
        extra["error"] = "%s: %s" % (type(exc).__name__, exc)
    if comm is not None:
        comm.close()
    line["configs"] = extra
    D.close()
    if D.rank == 0:
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--configs", default="2,3,4,5",
                    help="BASELINE.json configurations to measure (2 is always the headline)")
    ap.add_argument("--kernels-only", action="store_true",
                    help="profiling aid: time the resident-input kernels of config 2 only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the headline transform's outputs of its last "
                         "timed step to DIR/<name>.npy (float64, 40 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's transform (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
