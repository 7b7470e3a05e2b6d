"""bench.py's host-side helpers and the committed measurement files they read (no GPU): the line must not fail at the
round-end run because a JSON under profiles/ does not parse or lacks a key."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_probe_ceiling_interpolates_the_committed_measurement():
    pts = json.load(open(os.path.join(ROOT, "profiles", "probe_ceiling.json")))["g_probes_per_s_by_table_mib"]
    assert bench.probe_ceiling(64 << 20) == pts["64"] and bench.probe_ceiling(256 << 20) == pts["256"]
    assert bench.probe_ceiling(1 << 20) == pts["32"] and bench.probe_ceiling(1 << 40) == pts["4096"]   # clamped at both ends
    mid = bench.probe_ceiling(160 << 20)
    assert pts["192"] < mid < pts["128"]                                                              # monotone in between
    last = float("inf")
    for mib in (32, 48, 64, 100, 128, 200, 256, 400, 512, 2048, 4096):
        v = bench.probe_ceiling(mib << 20)
        assert v <= last
        last = v


def test_committed_ncu_counters_have_what_the_line_needs():
    for cfg in (2, 3):
        nc = bench.ncu_counters(cfg)
        assert nc, cfg
        for key in ("warp_instructions_per_read", "dram_bytes_per_read", "l2_bytes_per_read", "issue_active_pct", "step_ms_in_capture", "kernels"):
            assert key in nc, (cfg, key)
        assert any("scan" in k["kernel"] for k in nc["kernels"]) and sum(k["time_ms"] for k in nc["kernels"]) > 0
        assert os.path.exists(os.path.join(ROOT, nc["capture"].split(" ")[0]))           # the capture's summary is committed
    assert bench.ncu_counters(4) is None or isinstance(bench.ncu_counters(4), dict)


def test_algorithmic_bytes_of_a_150_base_read():
    import numpy as np
    assert bench.algorithmic_bytes(np.array([150])) == 3782        # 38 packed + 232 x 16 probe + 32 result (SURVEY 8d)
    assert bench.algorithmic_bytes(np.array([34, 150, 150])) >= 2 * 3782


def test_help_and_argument_defaults():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--gpus" in r.stdout and "--impl" in r.stdout and "--no-config4" in r.stdout
    assert "--dump-outputs" in r.stdout
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
