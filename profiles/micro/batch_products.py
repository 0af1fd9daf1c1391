"""Cost of the per-channel batch products (cwtb_cwt_batch_products) at config 5's geometry:
1024 channels fp32 of 2^16 samples, Morlet(6), s0 = 2, dj = 1/8, J = 127 (S = 128).

Alternates, in one process, after one warm-up call of each:
  (a) spectra only          Engine.cwt_batch (PowerBody per chunk)
  (b) products              COI spectrum, 2 bands, icwt (BatchProductsBody<float, 2> per chunk;
                            2 GiB of column outputs to the host)
  (c) COI spectrum only     BatchProductsBody without column outputs: the kernel's own cost
and reports device time (last_kernel_ms: events around the chunk loop on the engine's stream) and
wall time per call, with their spread; the per-kernel event table of one chunk of (a) and (b);
and the algorithmic read rate of the W chunk for PowerBody and BatchProductsBody.

    python profiles/micro/batch_products.py [--reps 5] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from pycwt_b200 import _engine  # noqa: E402

C, N, S = 1024, 1 << 16, 128


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    say("GPU: %s (name, power limit, max SM clock; read in this run)" % gpu_info())
    e = _engine.Engine(0)
    X = np.random.RandomState(0).randn(C, N).astype(np.float32)
    sj = 2.0 * 2 ** (np.arange(S) / 8)
    lam = 4 * np.pi / (6 + np.sqrt(2 + 36))
    period = lam * sj
    coi_c = lam / np.sqrt(2)
    half = N / 2 - period / coi_c
    mid = (N - 1) / 2
    lo = np.clip(np.ceil(mid - half - 1e-12), 0, N).astype(np.int64)
    hi = np.clip(np.floor(mid + half + 1e-12) + 1, 0, N).astype(np.int64)
    hi[half < 0] = lo[half < 0]
    wt = np.stack([np.where((period >= a) & (period < b), 1 / sj, 0.0) for a, b in [(8, 32), (64, 256)]])
    fac = 0.125 / (0.776 * np.pi ** -0.25) + 0j

    calls = {
        "a spectra only": lambda Xc: e.cwt_batch(Xc, 1.0, sj, _engine.MORLET, 6.0, _engine.F32),
        "b coi+2 bands+icwt": lambda Xc: e.cwt_batch_products(Xc, 1.0, sj, _engine.MORLET, 6.0, _engine.F32,
                                                              coi_ranges=(lo, hi), band_weights=wt,
                                                              icwt_factor=fac),
        "c coi only": lambda Xc: e.cwt_batch_products(Xc, 1.0, sj, _engine.MORLET, 6.0, _engine.F32,
                                                      coi_ranges=(lo, hi)),
    }
    say("config 5 geometry: %d channels x %d samples fp32, S = %d, Morlet(6)" % (C, N, S))
    for f in calls.values():        # warm-up: plans, pinned output pools, module loads
        f(X)
    dev = {k: [] for k in calls}
    wall = {k: [] for k in calls}
    for _ in range(args.reps):       # alternate the three variants
        for k, f in calls.items():
            t0 = time.perf_counter()
            r = f(X)
            wall[k].append((time.perf_counter() - t0) * 1e3)
            dev[k].append(e.last_kernel_ms())
            del r
    say("\n%-22s %28s %28s" % ("call (%d reps)" % args.reps, "device ms: median [min, max]",
                                "wall ms: median [min, max]"))
    for k in calls:
        d, w = np.array(dev[k]), np.array(wall[k])
        say("%-22s %12.1f [%6.1f, %6.1f] %12.1f [%6.1f, %6.1f]" % (k, np.median(d), d.min(), d.max(),
                                                                   np.median(w), w.min(), w.max()))

    # one chunk (64 channels = 4 GiB of fp32 coefficients), every launch bracketed by events
    nb = (4 << 30) // (8 * N * S)
    wbytes = nb * S * N * 8
    say("\nper-kernel event table of one chunk (%d channels, W = %.2f GiB), serialised streams" % (nb, wbytes / 2 ** 30))
    rates = {}
    for k in ("a spectra only", "b coi+2 bands+icwt", "c coi only"):
        calls[k](X[:nb])
        e.profile_begin()
        calls[k](X[:nb])
        prof = e.profile_end()
        say("  %s" % k)
        for p in sorted(prof, key=lambda p: -p["ms"]):
            say("    %-52s %4d launches %9.3f ms" % (p["name"], p["launches"], p["ms"]))
            if p["name"].startswith(("PowerBody", "BatchProductsBody")):
                rates[(k, p["name"])] = wbytes / (p["ms"] * 1e-3) / 1e12
    say("\nalgorithmic read rate of W (chunk bytes / kernel time)")
    for (k, name), r in rates.items():
        say("  %-22s %-32s %6.2f TB/s" % (k, name, r))
    pw = [r for (k, n), r in rates.items() if n.startswith("PowerBody")]
    for (k, name), r in rates.items():
        if name.startswith("BatchProductsBody") and pw:
            say("  %s / PowerBody: %.2f" % (name + " (" + k + ")", r / pw[0]))
    e.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
