"""bench.py's DEFAULT flow (`run_b200`: config 3 with the nested config-4 object) end to end on a fake device: the
placements come from the C++ oracle behind a stand-in for ``classeq2_b200.Index``, CUDA events and streams are
host-clock stand-ins, the synthetic models are shrunk.  Nothing here measures anything - it holds that the line the
driver parses at the end of a round is built without a Python error and carries every key of the contract, whatever
was last edited in bench.py.  No GPU."""
import argparse
import contextlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


class _Event:
    def __init__(self, enable_timing=False):
        self.t = 0.0

    def record(self, stream=None):
        self.t = time.perf_counter()

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


class _Stream:
    cuda_stream = 0

    def __init__(self, device=None):
        pass


def _fake_index_class(cq, cpp_oracle):
    class Resident:
        def __init__(self, ix, seqs):
            self.ix, (self.bases, self.offsets) = ix, cq.make_batch(seqs)

        def place(self, params=None, stream=0):
            self.ix.launches = 3

        def fetch(self, stream=0):
            return self.ix.place_batch((self.bases, self.offsets))

        def close(self):
            pass

    class Index:
        def __init__(self, flat, device=0, device_mask=None):
            self.md, self.flat, self.launches, self.nbytes = cpp_oracle.CppModel.from_flat(flat), flat, 0, (0, 0)

        def info(self):
            return {"n_entries": len(self.flat.entry_hash), "table_bytes": 64 << 20, "n_distinct_sets": len(self.flat.set_off) - 1}

        def upload(self, seqs):
            return Resident(self, seqs)

        def place_batch(self, seqs, params=None):
            bases, offsets = cq.make_batch(seqs)
            o = self.md.place_batch(bases, offsets, n_threads=4)
            res = cq.BatchResult(len(offsets) - 1)
            for f, _ in cq.engine.RESULT_DTYPES:
                getattr(res, f)[:] = o[f]
            return res

        def place_batch_into(self, bases, offsets, res, params=None):
            got = self.place_batch((bases, offsets))
            for f, _ in cq.engine.RESULT_DTYPES:
                getattr(res, f)[:] = getattr(got, f)
            self.nbytes = (int(len(bases)), 32 * (len(offsets) - 1))

        def timing(self):
            return {"pack_ms": 1.0, "h2d_ms": 1.0, "kernel_ms": 1.0, "d2h_ms": 1.0, "total_ms": 4.0, "kernel_launches": self.launches,
                    "h2d_bytes": self.nbytes[0], "d2h_bytes": self.nbytes[1], "pack_on_device": 0}

        def close(self):
            self.md.close()

    return Index


def _run_default_flow(monkeypatch, capsys, **overrides):
    """`run_b200` on the fake device with shrunk models; returns the parsed line."""
    import torch

    import classeq2_b200 as cq
    from classeq2_b200 import synth
    from oracle import cpp_oracle

    small = {k: dict(v) for k, v in synth.CONFIGS.items()}
    small[3]["n_tips"], small[4]["n_tips"] = 200, 120
    monkeypatch.setattr(synth, "CONFIGS", small)
    monkeypatch.setattr(cq, "Index", _fake_index_class(cq, cpp_oracle))
    for name, val in (("set_device", lambda d: None), ("Stream", _Stream), ("Event", _Event), ("synchronize", lambda *a: None),
                      ("device_count", lambda: 1), ("stream", lambda s: contextlib.nullcontext())):
        monkeypatch.setattr(torch.cuda, name, val)
    real_empty = torch.empty
    monkeypatch.setattr(torch, "empty", lambda *a, device=None, **k: real_empty(*[min(x, 1 << 16) if isinstance(x, int) else x for x in a], **k)
                        if device is not None else real_empty(*a, **k))
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    args = argparse.Namespace(gpus=1, steps=2, warmup=1, impl="b200", config=3, reads=3000, transport="p2p", cpu_seconds=0.3,
                              no_config4=False, reads4=400, no_config5=False, reads5=1000, no_inprocess=False, device_build=False,
                              dump_outputs=None)
    for k, v in overrides.items():
        setattr(args, k, v)
    bench.run_b200(args, 0, 1, 0)
    lines = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_default_flow_builds_the_whole_line_on_a_fake_device(monkeypatch, capsys):
    d = _run_default_flow(monkeypatch, capsys)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "parity", "config4"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["config"]["reads_total"] == 3000 and d["gpu_launches"] == 6
    assert d["parity"] == {"checked_reads": 3000, "mismatching_fields": 0, "e2e_equals_resident": True}
    r = d["roofline"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic", "peak_nominal", "frac_nominal", "aggregate", "secondary"):
        assert key in r, key
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and abs(r["aggregate"]["frac"] - r["frac"]) < 1e-9 * max(1.0, r["frac"])
    assert r["algorithmic_bytes_per_step"] == 3000 * 3782
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 3000 * 150 and e["d2h_bytes_per_step"] == 3000 * 32 and e["value"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0
    c4 = d["config4"]
    assert "error" not in c4, c4
    assert c4["parity"]["mismatching_fields"] == 0 and c4["config"]["reads"] == 400 and c4["value"] > 0
    assert sum(d["status_histogram"]) == 3000 and np.isfinite(d["value"])


def test_default_flow_times_every_step_and_dumps_the_last_results(monkeypatch, capsys, tmp_path):
    """--steps sets the timed steps of the nested config-4 measurement too; --dump-outputs writes the sampled results of
    the last step, which equal the oracle's placements of the same seeded reads."""
    from classeq2_b200 import engine
    from oracle import cpp_oracle

    assert 9 * 8 * (bench.DUMP_READS + bench.DUMP_READS_CONFIG4) <= 64 << 20
    monkeypatch.setattr(bench, "DUMP_READS", 1000)
    d = _run_default_flow(monkeypatch, capsys, steps=5, dump_outputs=str(tmp_path))
    assert d["steps"] == 5 and len(d["step_ms"]) == 5 and d["gpu_launches"] == 15
    assert d["config4"]["steps"] == 5 and len(d["config4"]["step_ms"]) == 5
    fields = ["read_index"] + [f for f, _ in engine.RESULT_DTYPES]
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(f"{p}{f}.npy" for p in ("", "config4_") for f in fields)
    for prefix, config, n_reads, n_kept in (("", 3, 3000, 1000), ("config4_", 4, 400, 400)):
        got = {f: np.load(tmp_path / f"{prefix}{f}.npy") for f in fields}
        assert all(a.dtype == np.float64 and a.shape == (n_kept,) for a in got.values())
        keep = got["read_index"].astype(np.int64)
        assert (np.diff(keep) > 0).all() and keep[0] >= 0 and keep[-1] < n_reads
        sm, bases, offsets, _, _ = bench.make_workload(config, 0, 1, n_reads)
        md = cpp_oracle.CppModel.from_flat(sm.flat)
        want = md.place_batch(bases, offsets, n_threads=4)
        md.close()
        for f, _ in engine.RESULT_DTYPES:
            assert np.array_equal(got[f], want[f][keep].astype(np.float64)), (prefix, f)


def test_sharded_flow_builds_its_line_on_a_fake_device(monkeypatch, capsys, tmp_path):
    """`run_sharded` (config 5; nested in every multi-GPU run of the default command) with world = 1: a stand-in for
    ``ShardedPlacer`` around the same oracle-backed index; the parity leg runs over every read of every sub-batch."""
    import torch

    import classeq2_b200 as cq
    from classeq2_b200 import parallel, synth
    from oracle import cpp_oracle

    small = {k: dict(v) for k, v in synth.CONFIGS.items()}
    small[5]["n_tips"] = 150
    monkeypatch.setattr(synth, "CONFIGS", small)
    Index = _fake_index_class(cq, cpp_oracle)
    monkeypatch.setattr(cq, "Index", Index)

    class Sharded:
        def __init__(self, flat, device, rank, world, transport="p2p", max_windows=0):
            self.index = Index(flat)
            self.timing = {"route_ms": 1.0, "probe_ms": 1.0, "place_ms": 1.0, "wire_bytes_out": 1000.0}
            up = self.index.upload

            def upload(seqs):
                rb = up(seqs)
                rb.nbytes = lambda: 64 * (len(rb.offsets) - 1)
                return rb
            self.index.upload = upload

        def place_resident(self, rb, params):
            pass

        def place(self, seqs, params):
            return self.index.place_batch(seqs)

        def close(self):
            self.index.close()

    monkeypatch.setattr(parallel, "ShardedPlacer", Sharded)
    for name, val in (("set_device", lambda d: None), ("Event", _Event), ("synchronize", lambda *a: None),
                      ("current_stream", lambda *a: _Stream())):
        monkeypatch.setattr(torch.cuda, name, val)
    real_empty = torch.empty
    monkeypatch.setattr(torch, "empty", lambda *a, device=None, **k: real_empty(*[min(x, 1 << 16) if isinstance(x, int) else x for x in a], **k))
    args = argparse.Namespace(gpus=1, steps=2, warmup=1, impl="b200", config=5, reads=2500, transport="p2p", cpu_seconds=0.3,
                              no_config4=True, reads4=400, no_config5=True, reads5=1000, no_inprocess=True, device_build=False,
                              dump_outputs=str(tmp_path))
    line = bench.run_sharded(args, 0, 1, 0)
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(out) == 1 and json.loads(out[0])["value"] == line["value"]
    assert line["parity"]["checked_reads"] == 2500 and line["parity"]["mismatching_fields"] == 0
    for key in ("metric", "value", "unit", "n_gpus", "ms_per_step", "scaling", "e2e", "gpu_launches", "roofline", "nvlink", "clocks", "config"):
        assert key in line, key
    assert sum(line["status_histogram"]) == 2500
    assert np.array_equal(np.load(tmp_path / "read_index.npy"), np.arange(2500.0))        # every read: fewer than DUMP_READS
    assert np.bincount(np.load(tmp_path / "status.npy").astype(np.int64), minlength=11).tolist() == line["status_histogram"]
    nested = bench.run_sharded(args, 0, 1, 0, embedded=True)        # the nested form: returned, not printed
    assert nested["parity"]["mismatching_fields"] == 0 and not [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
