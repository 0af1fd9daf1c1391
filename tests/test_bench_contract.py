"""The bench.py contract the round driver relies on, as far as it can be checked without a GPU:
the reference arm (`--impl reference`) times the CPU oracle and prints ONE JSON line with the
agreed keys; under a multi-rank launch only rank 0 works and prints."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def _run(env_extra, *args):
    env = dict(os.environ)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run({}, "--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "cwt_scale_points_per_sec"
    assert d["unit"] == "scale-points/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    assert d["n_gpus"] == 1 and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("config2") and d["config"]["n"] == 2 ** 20
    e2e = d["e2e"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"]
    cb = d["cpu_baseline"]
    from oracle import make_ref
    # the unmodified reference package where its copy exists (oracle/_ref, built by
    # __graft_entry__.build() from /root/reference), else the oracle port; one thread either way
    assert cb["kind"] == ("reference" if make_ref.available() else "port")
    assert cb["cores"] == 1 and cb["value"] == d["value"] and cb["sample"]


#: SHA-256 of the reference package's files at v0.3.0a22 (commit f88aec2)
REFERENCE_SHA256 = {
    "__init__.py": "568ec8dab26353a2167732d6756fd1efccb3e53e3c625a51de82cd247bb5b30f",
    "wavelet.py": "12aa7178db085ce128b392b0db645d8b4c4093442a431ec2cd3469e69869fcd2",
    "mothers.py": "500111993e025651a935de3dd5f6abd9dd4113b4fea01d981e18c46c7fe39443",
    "helpers.py": "116395fb05b6bf227b6f2463618635c080c090d8851e06b1bf6d7760bb80759f",
}


def test_reference_copy_is_the_unmodified_reference():
    """oracle/_ref/pycwt (the timing arm), where it was built, is byte-identical to the reference."""
    import hashlib
    from oracle import make_ref
    assert sorted(make_ref.FILES) == sorted(REFERENCE_SHA256)
    if not make_ref.available():
        return
    for f in make_ref.FILES:
        b = hashlib.sha256(open(os.path.join(make_ref.DST, "pycwt", f), "rb").read()).hexdigest()
        assert b == REFERENCE_SHA256[f], f
    mod = make_ref.load()
    assert mod.__version__ == "0.3.0a22" and mod.cwt.__module__ == "pycwt.wavelet"


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, "--impl", "reference", "--gpus", "2",
             "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_product_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: without a device the product arm must not print a number."""
    import pycwt_b200._engine as eng
    try:
        have = eng.device_count() > 0
    except Exception:
        have = False
    if have:
        return
    r = _run({}, "--steps", "1", "--warmup", "0")
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_product_arm_json_assembly_on_the_emulation_build():
    """Every key the driver reads is present and well-formed (values are not meaningful here)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_bench_emu_driver.py")], cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline",
              "cpu_baseline", "clocks"):
        assert k in d, k
    assert "impl" not in d and d["scaling"] == "weak" and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["gpu_launches"] > 0 and d["steps"] == 3 and d["warmup"] == 1
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in rf, k
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 1 and cb["value"] > 0 and cb["sample"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["e2e"]["resident"]["value"] > 0 and d["configs"] == {}
    assert rf["kernel"] == "PassBBody<double, 1, 1024>" and rf["source_hash"]


def test_dump_outputs_are_the_headline_transform(tmp_path):
    """--dump-outputs writes the sampled W and the signal spectrum of the timed transform (here
    the emulation build at N = 2^12, where every column is kept) as float64 files."""
    import numpy as np
    import workloads as wl
    from oracle import cwt_oracle as orc
    from conftest import relerr
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_bench_emu_driver.py"),
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert sorted(out) == ["W_imag", "W_real", "fft_imag", "fft_real"]
    assert all(a.dtype == np.float64 for a in out.values())
    c, n = wl.C2, 2 ** 12
    x = wl.chirp(n)
    W, _, _, _, fft, _ = orc.cwt(x, c["dt"], c["dj"], c["s0"], c["J"], orc.Morlet(c["f0"]))
    assert relerr(out["W_real"] + 1j * out["W_imag"], W) < 1e-10
    assert relerr(out["fft_real"] + 1j * out["fft_imag"], fft) < 1e-10
