"""Helper of tests/test_bench_contract.py: runs bench.py's PRODUCT arm on the host-emulation
build with a small signal, so that the assembly of the JSON line (keys, roofline, e2e, clocks)
is exercised where no GPU is present.  The emulation has no clock, so the device-timing hooks are
given fixed numbers; the printed throughput means nothing.  Extra arguments go to bench.py."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import conftest  # noqa: E402

conftest.use_emulation_library()
from pycwt_b200 import _engine  # noqa: E402

_engine.Engine.bench_last = lambda self, iters: 2.2
_engine.Engine.profile_last = lambda self: [
    {"name": "PassBBody<double, 1, 1024>", "launches": 4, "ms": 0.43, "rows": 72},
    {"name": "SingleBody<double, 1024>", "launches": 1, "ms": 0.08, "rows": 16},
    {"name": "PassABody<double, 1024, 0, 1>", "launches": 1, "ms": 0.25, "rows": 24}]
import bench  # noqa: E402

bench.wl.C2["n"] = 2 ** 12
bench.ClockSampler = type("CS", (), {
    "__init__": lambda s, *a, **k: None, "start": lambda s: None,
    "stop": lambda s: {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "samples": 1, "reasons": []}})
sys.argv = ["bench.py", "--steps", "3", "--warmup", "1", "--configs", "2"] + sys.argv[1:]
bench.main()
