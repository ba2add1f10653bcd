"""CPU: the parts of bench.py that do not need a GPU -- the algorithmic byte model (SURVEY.md 8d), the peak lookup,
the clock sampler's behaviour without NVML, the workload table -- so that a typo there cannot take the round-end
measurement down."""
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from deblurgs_b200 import synthetic  # noqa: E402


class _Shs:
    shape = (300000, 16, 3)


def test_algorithmic_byte_model_covers_every_hbm_stage():
    w = {"P": 300000, "F": 16, "W": 600, "H": 400, "scene": type("S", (), {"shs": _Shs})}
    st = {"V": 4339284, "D": 19154524, "E": 1777802608, "K": 252057426, "E_b": 1751127673}
    ab = bench.algorithmic_bytes(w, st, 42)
    for k in ["preprocess_fwd", "binning", "bwd_memset", "preprocess_bwd", "render_fwd", "render_bwd", "blur_mean"]:
        assert ab[k] > 0
    G = 44 + 12 * 16
    assert ab["preprocess_fwd"] == 300000 * G + st["V"] * 48
    # binning = scan + duplicate + the reference's single 42-bit sort (6 passes of 12-B pairs) + ranges
    assert ab["binning"] == 8 * 300000 * 16 + (st["V"] * 16 + st["D"] * 12) + st["D"] * 12 * 2 * 6 + st["D"] * 8
    # what this library's binning moves is far less than that, and is reported next to it
    moved = bench.moved_bytes_binning(w, st, 10)
    assert 0 < moved < 0.5 * ab["binning"]
    assert bench.moved_bytes_binning(w, st, 8) < moved < bench.moved_bytes_binning(w, st, 17)


def test_peaks_and_clock_sampler_degrade_gracefully():
    hbm, src = bench.measured_peaks()
    assert hbm > 1000 and isinstance(src, str)
    s = bench.ClockSampler(0)
    s.start()                                             # without NVML run() returns at once; with it, it samples
    time.sleep(0.1)
    s.stop_flag = True
    s.join(timeout=10)
    assert not s.is_alive()
    out = s.summary()
    assert set(out) == {"sm_mhz", "sm_max_mhz", "reasons", "samples"}
    if s.nv is None:
        assert out["reasons"] == [] and out["samples"] == 0
    else:
        assert out["samples"] >= 1 and set(out["reasons"]) <= {"sw_power_cap", "hw_slowdown", "hw_thermal_slowdown",
                                                                "sw_thermal_slowdown", "hw_power_brake"}
    json.dumps(out)


def test_workload_table_matches_baseline_configs():
    assert synthetic.get_config("c2") == (300000, 600, 400, 16, 9)
    assert synthetic.get_config("c1") == (50000, 256, 256, 4, 3)
    assert synthetic.get_config("c3")[:4] == (1000000, 1920, 1080, 16)
    assert synthetic.get_config("c4")[:4] == (3000000, 1280, 720, 32)
    assert synthetic.get_config("P=1000,F=5") == (1000, 600, 400, 5, 9)


def test_bench_cli_declares_the_contract_flags():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0
    for flag in ["--gpus", "--steps", "--warmup", "--impl", "--config", "--loss", "--split", "--no-graph"]:
        assert flag in r.stdout
