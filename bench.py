#!/usr/bin/env python
"""Benchmark of the placement hot path (BASELINE.json: "queries placed/s and k-mer lookups/s").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (extract + murmur3 + probe + count + descend) over one batch
of synthetic reads of the named configuration (SURVEY.md section 8d; classeq2_b200/synth.py):

  value   reads placed per second with the packed batch already resident in HBM (kernel-resident),
          CUDA events around every step on the launching stream, L2 flushed between steps,
          max over ranks;
  e2e     the same metric through the reference-facing C-ABI call `cls_place_batch` with HOST
          buffers: 2-bit packing, pinned H2D, kernels and D2H of the result records all inside the
          timed region;
  roofline / cpu_baseline / clocks: see DESIGN.md "Measurement".

The default workload is config 3 - the configuration the north-star target is quoted on (10 M x 150 bp reads,
10k-tip tree): its reads are SHARDED over the ranks ("strong"; it fits one GPU too).  `--config 2|4` run one
batch per GPU ("weak"), `--config 5` the hash-sharded index.
N > 1 (launched by torchrun, one rank per GPU): queries shard across ranks with the index
replicated and NO data-path collective (SURVEY.md 8e).
`--impl reference` times the CPU restatement of the reference (oracle/classeq_oracle.cpp, all host
cores) on a bounded sample of the same workload; the reference itself is Rust and cannot be built
here (DESIGN.md).
Every timed loop runs exactly K steps.

`--dump-outputs DIR` writes, after the timed steps, the result arrays of the last kernel-resident step (the fields of
`cls_result`, one element per read) as DIR/<field>.npy in float64, on a fixed, seeded sample of the reads whose indices
are DIR/read_index.npy; the nested config-4 measurement adds DIR/config4_<field>.npy.  The workload is generated from
fixed seeds, so two builds of the library run with the same arguments can be compared file by file.  Under torchrun
rank 0 writes the results of its own reads.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_SIZE = 35
NOMINAL_HBM_GBS = 8000.0   # B200 HBM3e, nominal (SURVEY.md 8d asks for both denominators; `peak` is the measured one)
NAMES = {2: "config2: synthetic 1,000-tip tree, 1 kb refs, 1M x 150 bp reads, index replicated",
         3: "config3: synthetic 10k-tip tree, ~600 bp refs, 10M x 150 bp reads sharded over the GPUs, index replicated",
         4: "config4: synthetic 5k-tip tree, 1.5 kb refs, 1M reads of skewed length 150-1550 bp",
         5: "config5: synthetic 100k-tip tree, ~600 bp refs, 10M x 150 bp reads sharded over the GPUs, index HASH-SHARDED "
            "(owner = hash >> 61 mod N), query k-mers routed by NCCL all-to-all over NVLink"}


L2_NOTE = "256 MiB memset between steps of the GPU arm (outside the event pairs)"
# --dump-outputs: reads kept of the main batch and of the nested config-4 batch; 9 float64 arrays each, 45 MiB in all
DUMP_READS, DUMP_READS_CONFIG4, DUMP_SEED = 1 << 19, 1 << 17, 0


def dump_outputs(directory: str, fields: dict, n_keep: int, prefix: str = "") -> None:
    """Writes ``fields`` (equal-length per-read arrays) at a fixed, seeded sample of at most ``n_keep`` reads as
    float64 .npy files, with the sampled read indices as ``<prefix>read_index.npy``."""
    n = len(next(iter(fields.values())))
    keep = np.arange(n) if n <= n_keep else np.sort(np.random.default_rng(DUMP_SEED).choice(n, n_keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    for name, a in {"read_index": keep, **{k: v[keep] for k, v in fields.items()}}.items():
        out = a.astype(np.float64)
        if not np.array_equal(out.astype(a.dtype), a):       # node ids are uint64: exact only below 2^53
            raise ValueError(f"--dump-outputs: {name} does not fit float64 exactly")
        np.save(os.path.join(directory, f"{prefix}{name}.npy"), out)


def common_config(config: int, n_total: int, world: int) -> dict:
    """The `config` object both arms print (the driver compares them): the workload and nothing measured."""
    sharded = config in (3, 5)
    return {"workload": NAMES[config], "reads_total": int(n_total * (1 if sharded else world)),
            "reads_per_gpu": int(n_total // world if sharded else n_total), "k": K_SIZE, "m": 4, "l2": L2_NOTE}


def synth_reads(config: int) -> int:
    return int(load_synth_data().CONFIGS[config]["n_reads"])


def load_synth_data():
    """classeq2_b200/synth_data.py by path: the generator is pure numpy, and the reference arm must not map the
    product library (importing the package loads it)."""
    import importlib.util
    name = "classeq_synth_data"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "classeq2_b200", "synth_data.py"))
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


def ncu_counters(config: int):
    """Counters of the committed ncu capture of this config's kernels (profiles/ncu_counters.json), if any."""
    p = os.path.join(ROOT, "profiles", "ncu_counters.json")
    if os.path.exists(p):
        return json.load(open(p)).get(f"config{config}")
    return None


def algorithmic_bytes(lens: np.ndarray) -> int:
    """SURVEY.md 8d: ceil(L/4) packed bases + 16 B per k-mer lookup + 32 B result record."""
    lens = lens[lens >= K_SIZE].astype(np.int64)
    return int(((lens + 3) // 4 + 2 * (lens - K_SIZE + 1) * 16 + 32).sum())


def make_workload(config: int, rank: int, world: int, n_reads_override=None, build_device=None):
    from classeq2_b200 import synth
    c = dict(synth.CONFIGS[config])
    t0 = time.time()
    # build_device: the model's k-mer map is built on that GPU (cls_model_build_device) instead of the host cores;
    # both builders give the same arrays (tests/test_zbuild_device.py), so the workload is the same either way
    sm = synth.make_model(c["n_tips"], c["l_ref"], c["tree_seed"], device=build_device)
    n_total = n_reads_override or c["n_reads"]
    if config in (3, 5):  # the 10M reads of configs 3 and 5 are SHARDED over the ranks (strong)
        n_local = n_total // world + (1 if rank < n_total % world else 0)
        scaling = "strong"
    else:                # configs 2 and 4: every GPU places its own batch of the named size (weak)
        n_local, scaling = n_total, "weak"
    if c["read_len"] == "skewed":
        lens = synth.skewed_lengths(n_local, c["len_seed"] + rank)
    else:
        lens = c["read_len"]
    bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, n_local, lens, c["tree_seed"] + 2 + 1000 * rank)
    return sm, bases, offsets, scaling, time.time() - t0


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, device: int):
        super().__init__(daemon=True)
        self.device, self.samples, self.reasons, self.stop_flag, self.max_mhz = device, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[device]) if vis and vis.split(",")[device].isdigit() else device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def run(self):
        while self.nv is not None and not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                bits = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.02)

    def summary(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def probe_ceiling(table_bytes: int):
    """Measured rate of random 32-byte probes of a table of this size on one B200 (profiles/probe_ceiling.json, from
    tools/micro/probe_bench.cu), interpolated in log(table size).  G probes/s, or None."""
    p = os.path.join(ROOT, "profiles", "probe_ceiling.json")
    try:
        pts = sorted((float(k), float(v)) for k, v in json.load(open(p))["g_probes_per_s_by_table_mib"].items())
    except (OSError, ValueError, KeyError):
        return None
    mib = table_bytes / float(1 << 20)
    if mib <= pts[0][0]:
        return pts[0][1]
    if mib >= pts[-1][0]:
        return pts[-1][1]
    import math
    for (a, va), (b, vb) in zip(pts, pts[1:]):
        if a <= mib <= b:
            t = (math.log(mib) - math.log(a)) / (math.log(b) - math.log(a))
            return va + t * (vb - va)
    return None


def ncu_traffic(config: int):
    """dram bytes per launch of the place kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(f"config{config}")
    return None


def time_cpu_oracle(sm, bases, offsets, seconds: float, threads: int):
    """The C++ restatement on a bounded prefix of the batch sized to take about `seconds`."""
    from oracle import cpp_oracle
    md = cpp_oracle.CppModel.from_flat(sm.flat)
    n_all = len(offsets) - 1

    def run(n):
        off = offsets[: n + 1]
        t0 = time.perf_counter()
        md.place_batch(bases[: int(off[-1])], off, n_threads=threads)
        return time.perf_counter() - t0

    n0 = min(n_all, 2000)
    t = run(n0)
    n = int(min(n_all, max(n0, n0 * seconds / max(t, 1e-6))))
    t = run(n)
    lens = np.diff(offsets[: n + 1].astype(np.int64))
    md.close()
    return n, t, int((2 * (lens[lens >= K_SIZE] - K_SIZE + 1)).sum())


def run_reference(args, rank, world):
    """The reference's CPU path on the host cores: the C++ restatement (oracle/), its model built by the oracle's own
    builder - nothing of the product is imported or mapped here."""
    if rank != 0:
        return
    from oracle import cpp_oracle
    sd = load_synth_data()
    c = dict(sd.CONFIGS[args.config])
    n_total = args.reads or c["n_reads"]
    threads = os.cpu_count() or 1
    tree = sd.make_tree(c["n_tips"], c["tree_seed"])
    codes, rlens = sd.make_refs(tree, c["l_ref"], c["tree_seed"] + 1)
    rb, ro = sd.refs_to_batch(codes, rlens)
    flat = cpp_oracle.build_model(K_SIZE, 4, tree.node_id, tree.node_kind, tree.child_off, tree.child_idx, tree.tip_node, rb, ro,
                                  n_threads=threads)
    md = cpp_oracle.CppModel.from_flat(flat)
    scaling = "strong" if args.config in (3, 5) else "weak"
    # the first chunks of the batch rank 0 of the GPU arm places (whole generator chunks: the same reads)
    n_gen = min(n_total, 400_000)
    if c["read_len"] == "skewed":
        lens_in = sd.skewed_lengths(n_total, c["len_seed"])[:n_gen]
    else:
        lens_in = c["read_len"]
    bases, offsets, _ = sd.make_reads(codes, rlens, n_gen, lens_in, c["tree_seed"] + 2)
    n_all = len(offsets) - 1
    # size the per-step sample so that warmup + steps finish within about two minutes
    n0 = min(n_all, 2000)
    t0 = time.perf_counter()
    md.place_batch(bases[: int(offsets[n0])], offsets[: n0 + 1], n_threads=threads)
    rate = n0 / (time.perf_counter() - t0)
    budget = 120.0 / (args.steps + args.warmup)
    n = int(min(n_all, max(1000, rate * min(budget, 20.0))))
    off = offsets[: n + 1]
    bs = bases[: int(off[-1])]
    for _ in range(args.warmup):
        md.place_batch(bs, off, n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        md.place_batch(bs, off, n_threads=threads)
    dt = (time.perf_counter() - t0) / args.steps
    lens = np.diff(off.astype(np.int64))
    value = n / dt
    sample = (f"first {n} reads of the batch per step, {threads} threads, C++ restatement of the reference "
              "(oracle/classeq_oracle.cpp; the Rust binary cannot be built here), model built by the oracle's own builder")
    line = {"impl": "reference", "metric": "queries placed/s", "value": value, "unit": "reads/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": common_config(args.config, n_total, max(1, args.gpus)),
            "lookups_per_s": float((2 * (lens[lens >= K_SIZE] - K_SIZE + 1)).sum() / dt),
            "cpu_baseline": {"value": value, "unit": "reads/s", "cores": threads, "kind": "port", "sample": sample,
                             "reads_per_step": n},
            "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    md.close()


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import classeq2_b200 as cq

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sm, bases, offsets, scaling, gen_s = make_workload(args.config, rank, world, args.reads,
                                                       local_rank if args.device_build else None)
    n_local = len(offsets) - 1
    lens = np.diff(offsets.astype(np.int64))
    lookups_local = int((2 * (lens[lens >= K_SIZE] - K_SIZE + 1)).sum())
    alg_bytes_local = algorithmic_bytes(lens)

    t0 = time.time()
    index = cq.Index(sm.flat, device=local_rank)
    info = index.info()
    upload_s = time.time() - t0
    params = cq.PlaceParams()
    rb = index.upload((bases, offsets))
    stream = torch.cuda.Stream(device=local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allgather(x: float):
        if world == 1:
            return [x]
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def allsum(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- kernel-resident: `value` ----------------------------------------------------------------------
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            flush.fill_(1)
            rb.place(params, stream.cuda_stream)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    wall0 = time.perf_counter()
    with torch.cuda.stream(stream):
        for a, b in ev:
            flush.fill_(rank + 2)          # L2 flush, outside the event pair
            a.record(stream)
            rb.place(params, stream.cuda_stream)
            b.record(stream)
    barrier()
    wall_resident = time.perf_counter() - wall0
    clocks = sampler.summary()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    ms_local = float(sum(step_ms))
    ms_total = allmax(ms_local)
    launches_per_step = int(index.timing()["kernel_launches"])
    reads_total = allsum(float(n_local))
    lookups_total = allsum(float(lookups_local))
    alg_bytes_total = allsum(float(alg_bytes_local))
    ms_per_step = ms_total / args.steps
    value = reads_total / (ms_per_step / 1e3)

    # parity spot check of what was just timed (bit-exact against the CPU oracle on a sample)
    res = rb.fetch(stream.cuda_stream)
    status_hist = np.bincount(res.status, minlength=11).tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f: getattr(res, f) for f, _ in cq.engine.RESULT_DTYPES}, DUMP_READS)

    # ---- end to end through the C ABI with host buffers: `e2e` ----------------------------------------
    out = cq.BatchResult(n_local)
    # the step's inputs sit in PINNED host memory (what a reader that fills a reusable buffer hands over): with few host
    # cores per GPU the library copies the ASCII bases straight from it and packs on the device (cls_set_pack_mode)
    pinned = torch.empty(len(bases), dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = bases
    bases = pinned.numpy()
    for _ in range(max(1, min(args.warmup, 2))):
        index.place_batch_into(bases, offsets, out, params)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        index.place_batch_into(bases, offsets, out, params)
    torch.cuda.synchronize()
    e2e_local = (time.perf_counter() - t0) / args.steps
    e2e_s = allmax(e2e_local)
    tm = index.timing()
    same = all((getattr(out, f) == getattr(res, f)).all() for f, _ in cq.engine.RESULT_DTYPES)
    e2e = {"value": reads_total / e2e_s, "unit": "reads/s", "h2d_bytes_per_step": int(allsum(float(tm["h2d_bytes"]))),
           "d2h_bytes_per_step": int(allsum(float(tm["d2h_bytes"]))), "ms_per_step": e2e_s * 1e3,
           "breakdown_ms_rank0": {k: round(tm[k], 3) for k in ("pack_ms", "h2d_ms", "kernel_ms", "d2h_ms", "total_ms")},
           "pack": ["host (2-bit words cross PCIe)", "device (ASCII staged through pinned memory)",
                    "device (ASCII copied straight from the caller's pinned memory)",
                    "mixed (the chunks of a call are dealt to the host packer and to the device packer)"][int(tm["pack_on_device"])],
           "ms_per_step_by_rank": [round(x * 1e3, 3) for x in allgather(e2e_local)],
           "host_input": "ASCII bases (pinned host memory) + offsets in caller memory (what the reference's FASTA reader hands over); "
                         "bytes counted by the library from the copies it enqueues, summed over the ranks"}

    # ---- ONE process, ONE handle, every visible GPU (cls_index_create_multi): the reference's callers are single
    #      processes that fan out internally (ports/cli/src/cmds/place_sequences.rs:125-156); N = 1 arm only -----
    e2e_multi = None
    if world == 1 and torch.cuda.device_count() > 1 and not args.no_inprocess:
        try:
            n_dev = torch.cuda.device_count()
            mix = cq.Index(sm.flat, device_mask=0)
            out2 = cq.BatchResult(n_local)
            for _ in range(2):
                mix.place_batch_into(bases, offsets, out2, params)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                mix.place_batch_into(bases, offsets, out2, params)
            dt = (time.perf_counter() - t0) / args.steps
            same2 = all((getattr(out2, f) == getattr(res, f)).all() for f, _ in cq.engine.RESULT_DTYPES)
            e2e_multi = {"value": n_local / dt, "unit": "reads/s", "n_devices": n_dev, "ms_per_step": dt * 1e3,
                         "equals_single_device": bool(same2),
                         "call": "one cls_place_batch on a cls_index_create_multi handle over every visible GPU, host ASCII in / host arrays out"}
            mix.close()
        except Exception as ex:  # noqa: BLE001
            e2e_multi = {"error": repr(ex)[:300]}

    # ---- CPU baseline (rank 0, N = 1 only) + sampled parity ---------------------------------------------
    cpu = None
    parity = None
    if rank == 0:
        from oracle import cpp_oracle
        threads = os.cpu_count() or 1
        if world == 1:
            n_s, t_s, look_s = time_cpu_oracle(sm, bases, offsets, args.cpu_seconds, threads)
            cpu = {"value": n_s / t_s, "unit": "reads/s", "cores": threads, "kind": "port",
                   "lookups_per_s": look_s / t_s,
                   "sample": f"first {n_s} reads of the same batch, {threads} threads, oracle/classeq_oracle.cpp "
                             "(C++ restatement with direct hash lookups - kinder than the Rust reference, which "
                             "clones and scans the whole index per query; the Rust binary cannot be built here)"}
        md = cpp_oracle.CppModel.from_flat(sm.flat)
        n_chk = min(n_local, 20000)
        o = md.place_batch(bases[: int(offsets[n_chk])], offsets[: n_chk + 1], n_threads=threads)
        bad = sum(int((o[f] != getattr(res, f)[:n_chk]).sum()) for f, _ in cq.engine.RESULT_DTYPES)
        parity = {"checked_reads": n_chk, "mismatching_fields": bad, "e2e_equals_resident": bool(same)}
        md.close()

    if rank == 0:
        peak, peak_src = measured_peak()
        step_s = ms_local / args.steps / 1e3
        achieved = alg_bytes_local / step_s / 1e9   # this GPU's kernels, GB/s
        # secondary ceilings (SURVEY.md 8d) from the committed ncu capture of this config's kernels: the path is integer
        # hashing plus random 32-byte probes - instruction issue and (when the table does not fit L2) HBM sectors
        nc = ncu_counters(args.config)
        secondary = None
        traffic = None
        if nc:
            sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
            peak_issue = 148 * 4 * sm_hz
            reads_per_s_gpu = n_local / step_s
            traffic = nc["dram_bytes_per_read"] * n_local
            secondary = {
                "issue": {"warp_instructions_per_read": nc["warp_instructions_per_read"], "peak_warp_instructions_per_s": peak_issue,
                          "frac": nc["warp_instructions_per_read"] * reads_per_s_gpu / peak_issue,
                          "issue_active_pct_in_capture": nc.get("issue_active_pct")},
                "dram_gbs": nc["dram_bytes_per_read"] * reads_per_s_gpu / 1e9,
                "dram_frac_of_peak": nc["dram_bytes_per_read"] * reads_per_s_gpu / 1e9 / peak,
                "l2_gbs": nc["l2_bytes_per_read"] * reads_per_s_gpu / 1e9,
                "limiter": nc.get("limiter"), "capture": nc.get("capture"),
                "note": "per-read counters of the committed capture x this run's reads/s on one GPU"}
        # the ceiling of the table probes themselves: random 32-byte reads of a table of this size (a miss moves a whole
        # 128-byte line from HBM), measured by tools/micro/probe_bench.cu on this GPU model
        pc = probe_ceiling(int(info["table_bytes"]))
        if pc:
            look_gpu = lookups_local / step_s / 1e9
            scan_share = None
            if nc and nc.get("kernels"):
                scan_ms = sum(k["time_ms"] for k in nc["kernels"] if "scan" in k["kernel"])
                scan_share = scan_ms / nc["step_ms_in_capture"] if nc.get("step_ms_in_capture") else None
            probe = {"table_mib": info["table_bytes"] / float(1 << 20), "ceiling_g_probes_per_s": pc,
                     "achieved_g_probes_per_s_whole_step": look_gpu, "frac_whole_step": look_gpu / pc,
                     "source": "profiles/probe_ceiling.json (tools/micro/probe_bench.cu, profiles/r2b/probe_bench.log)"}
            if scan_share:
                probe["achieved_g_probes_per_s_scan_kernel"] = look_gpu / scan_share
                probe["frac_scan_kernel"] = look_gpu / scan_share / pc
                probe["scan_kernel_share_of_step_in_capture"] = scan_share
            secondary = dict(secondary or {}, random_probe=probe)
        cfg = common_config(args.config, args.reads or synth_reads(args.config), world)
        line = {
            "metric": "queries placed/s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": cfg,
            "index": {"index_entries": int(info["n_entries"]), "table_bytes": int(info["table_bytes"]),
                      "distinct_node_sets": int(info["n_distinct_sets"]),
                      "parallelism": f"queries sharded x{world}, index replicated, no collective"},
            "lookups_per_s": lookups_total / (ms_per_step / 1e3),
            "e2e": e2e, "e2e_one_process_all_gpus": e2e_multi, "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         # SURVEY 8d: both denominators (measured copy bandwidth / nominal HBM3e), and the whole job against N GPUs
                         "peak_nominal": NOMINAL_HBM_GBS, "frac_nominal": achieved / NOMINAL_HBM_GBS,
                         "aggregate": {"n_gpus": world, "achieved": alg_bytes_total / (ms_per_step / 1e3) / 1e9, "peak": peak * world,
                                       "frac": alg_bytes_total / (ms_per_step / 1e3) / 1e9 / (peak * world)},
                         "algorithmic_bytes_per_step": alg_bytes_local, "launches_per_step": launches_per_step,
                         "secondary": secondary,
                         "kernel": "cls::scan2_kernel<4> + cls::descend16_kernel (+ cls::descend_kernel<2> for reads with more than 16 node sets, "
                                   "cls::scan_kernel<1> over the overflow list), timed together "
                                   "(config 4: cls::scanfrag_kernel + cls::gather_kernel + cls::descend_kernel<8> / cls::descend_wide_kernel for the kb-scale classes)",
                         "note": "3782 B per 150 bp read = 38 packed + 232 x 16 probe + 32 result; achieved = algorithmic bytes / CUDA-event "
                                 "time of the whole step (all launches of the step); traffic = DRAM bytes per read of the committed ncu "
                                 "capture x reads per step"},
            "cpu_baseline": cpu, "clocks": clocks, "parity": parity,
            "status_histogram": status_hist, "step_ms": [round(x, 4) for x in step_ms],
            "setup_s": {"generate": round(gen_s, 1), "index_upload": round(upload_s, 2)},
            "wall_s_resident_region": round(wall_resident, 4),
        }
    rb.close()
    index.close()
    # ---- N > 1 on the default workload: the hash-sharded index (config 5) rides along, so that the run that measures
    #      the scaling of config 3 also measures the NVLink path (a nested object, not a second line) ------------------
    c5 = None
    if world > 1 and args.config == 3 and not args.no_config5:
        torch.cuda.synchronize()
        dist.barrier()
        try:
            a5 = argparse.Namespace(**vars(args))
            a5.config, a5.reads, a5.warmup, a5.device_build, a5.dump_outputs = 5, args.reads5 * world, 2, True, None
            l5 = run_sharded(a5, rank, world, local_rank, embedded=True)
            if rank == 0 and l5:
                c5 = {k: l5[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "scaling", "lookups_per_s", "e2e", "config", "nvlink",
                                         "stage_ms_per_step_rank0", "parity", "roofline", "status_histogram")}
        except Exception as ex:  # noqa: BLE001
            c5 = {"error": repr(ex)[:300]}
    # ---- N = 1 on the default workload: the kb-scale reads of config 4 ride along (resident value + sampled parity),
    #      so that the driver's one-GPU run also measures the fragment path (scanfrag / gather / wide descent kernels)
    c4 = None
    if world == 1 and args.config == 3 and not args.no_config4:
        try:
            c4 = run_config4_nested(args, local_rank)
        except Exception as ex:  # noqa: BLE001
            c4 = {"error": repr(ex)[:300]}
    if rank == 0:
        line["config5"] = c5
        line["config4"] = c4
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_config4_nested(args, local_rank):
    """Config 4 (5 k tips x 1.5 kb refs, 1 M reads of 150-1 550 bases) kernel-resident on one GPU: value, lookups/s,
    a sampled parity check against the oracle.  A nested object of the default line, not a line of its own."""
    import torch

    import classeq2_b200 as cq
    from oracle import cpp_oracle

    n4 = min(args.reads4, 1_000_000)
    sm, bases, offsets, _, gen_s = make_workload(4, 0, 1, n4, local_rank if args.device_build else None)
    lens = np.diff(offsets.astype(np.int64))
    lookups = int((2 * (lens[lens >= K_SIZE] - K_SIZE + 1)).sum())
    index = cq.Index(sm.flat, device=local_rank)
    info = index.info()
    rb = index.upload((bases, offsets))
    stream = torch.cuda.Stream(device=local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")
    params = cq.PlaceParams()
    with torch.cuda.stream(stream):
        for _ in range(2):
            rb.place(params, stream.cuda_stream)
        ev = []
        for i in range(args.steps):
            flush.fill_(i)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            rb.place(params, stream.cuda_stream)
            b.record(stream)
            ev.append((a, b))
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    ms_per_step = float(np.mean(ms))
    res = rb.fetch(stream.cuda_stream)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f: getattr(res, f) for f, _ in cq.engine.RESULT_DTYPES}, DUMP_READS_CONFIG4, "config4_")
    n_chk = min(len(lens), 2000)
    md = cpp_oracle.CppModel.from_flat(sm.flat)
    o = md.place_batch(bases[: int(offsets[n_chk])], offsets[: n_chk + 1], n_threads=os.cpu_count() or 1)
    md.close()
    bad = sum(int((o[f] != getattr(res, f)[:n_chk]).sum()) for f, _ in cq.engine.RESULT_DTYPES)
    alg = algorithmic_bytes(lens)
    peak, _ = measured_peak()
    pc = probe_ceiling(int(info["table_bytes"]))
    out = {"value": len(lens) / (ms_per_step / 1e3), "unit": "reads/s", "ms_per_step": ms_per_step, "steps": args.steps, "warmup": 2,
           "lookups_per_s": lookups / (ms_per_step / 1e3),
           "config": {"workload": NAMES[4], "reads": int(len(lens)), "mean_read_length": float(lens.mean()),
                      "index_entries": int(info["n_entries"]), "table_bytes": int(info["table_bytes"])},
           "roofline": {"bound": "hbm", "achieved": alg / (ms_per_step / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (ms_per_step / 1e3) / 1e9 / peak,
                        "random_probe_ceiling_g_per_s": pc, "achieved_g_probes_per_s": lookups / (ms_per_step / 1e3) / 1e9,
                        "kernel": "cls::scanfrag_kernel + cls::gather_kernel + cls::descend_kernel<8> + cls::descend_wide_kernel "
                                  "(+ cls::scan2_kernel / descend16_kernel for the classes of up to 290 bases)"},
           "parity": {"checked_reads": n_chk, "mismatching_fields": bad},
           "status_histogram": np.bincount(res.status, minlength=11).tolist(), "step_ms": [round(x, 3) for x in ms],
           "setup_s": round(gen_s, 1)}
    rb.close()
    index.close()
    return out


def run_sharded(args, rank, world, local_rank, embedded=False):
    """Config 5: every rank owns one shard of the k-mer table and is home to its share of the reads.
    embedded=True: called from the default (config 3) run under torchrun, on its process group; returns the line
    (rank 0) instead of printing it."""
    import torch
    import torch.distributed as dist

    import classeq2_b200 as cq
    from classeq2_b200.parallel import ShardedPlacer

    torch.cuda.set_device(local_rank)
    if world > 1 and not embedded:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sm, bases, offsets, scaling, gen_s = make_workload(5, rank, world, args.reads, local_rank if args.device_build else None)
    n_local = len(offsets) - 1
    lens = np.diff(offsets.astype(np.int64))
    lookups_local = int((2 * (lens[lens >= K_SIZE] - K_SIZE + 1)).sum())
    t0 = time.time()
    max_w = int(2 * (lens[lens >= K_SIZE] - K_SIZE + 1)[:1_250_000].sum()) if n_local else 0
    max_w = max(max_w, 2 * 116 * min(n_local, 1_250_000))
    sp = ShardedPlacer(sm.flat, local_rank, rank, world, transport=args.transport, max_windows=max_w)
    info = sp.index.info()
    upload_s = time.time() - t0
    params = cq.PlaceParams()
    dev = f"cuda:{local_rank}"
    # sub-batches bound the exchange buffers (about 20 bytes of wire + 24 bytes of buffers per k-mer)
    sub = 1_250_000
    cuts = list(range(0, n_local, sub)) + [n_local]
    parts = [(bases[int(offsets[a]):int(offsets[b])], (offsets[a:b + 1] - offsets[a]).astype(np.uint64)) for a, b in zip(cuts[:-1], cuts[1:])]
    rbs = [sp.index.upload(p) for p in parts]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allred(x: float, op) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    st = torch.cuda.current_stream()
    stage = {}

    def step():
        for rb in rbs:
            sp.place_resident(rb, params)
            for k, v in sp.timing.items():
                stage[k] = stage.get(k, 0.0) + float(v)

    for _ in range(args.warmup):
        flush.fill_(1)
        step()
    barrier()
    stage.clear()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_local = 0.0
    step_ms = []
    for i in range(args.steps):
        flush.fill_(i + 2)
        if world > 1:
            dist.barrier()       # the all-to-alls couple the ranks: start every step together
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        step()
        b.record(st)
        b.synchronize()
        step_ms.append(a.elapsed_time(b))
        ms_local += step_ms[-1]
    barrier()
    clocks = sampler.summary()
    ms_per_step = allred(ms_local, dist.ReduceOp.MAX) / args.steps
    reads_total = allred(float(n_local), dist.ReduceOp.SUM)
    lookups_total = allred(float(lookups_local), dist.ReduceOp.SUM)
    value = reads_total / (ms_per_step / 1e3)
    res = [rb.fetch(st.cuda_stream) for rb in rbs]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {f: np.concatenate([getattr(r, f) for r in res]) for f, _ in cq.engine.RESULT_DTYPES},
                     DUMP_READS)
    line = None

    # end to end: host ASCII in, host arrays out, every sub-batch uploaded and fetched inside the timed region
    e2e_res = [sp.place(p, params) for p in parts]   # warm-up (first-use registration of the exchange buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_res = [sp.place(p, params) for p in parts]
    torch.cuda.synchronize()
    e2e_s = allred((time.perf_counter() - t0) / args.steps, dist.ReduceOp.MAX)

    # parity: the replicated index on this GPU must give the very same arrays for EVERY read of EVERY sub-batch of this
    # rank (resident and end-to-end results alike); the counts are summed over the ranks
    rep_ix = cq.Index(sm.flat, device=local_rank)
    n_chk = bad = bad_e2e = 0
    for j, p in enumerate(parts):
        want = rep_ix.place_batch(p, params)
        bad += sum(int((getattr(want, f) != getattr(res[j], f)).sum()) for f, _ in cq.engine.RESULT_DTYPES)
        bad_e2e += sum(int((getattr(e2e_res[j], f) != getattr(res[j], f)).sum()) for f, _ in cq.engine.RESULT_DTYPES)
        n_chk += len(p[1]) - 1
    rep_info = rep_ix.info()
    rep_ix.close()
    bad = int(allred(float(bad + bad_e2e), dist.ReduceOp.SUM))
    n_chk = int(allred(float(n_chk), dist.ReduceOp.SUM))

    if rank == 0:
        peak, peak_src = measured_peak()
        per = {k: v / args.steps for k, v in stage.items()}
        n_device = int((lens >= K_SIZE).sum())
        kern_ms = per.get("route_ms", 0) + per.get("probe_ms", 0) + per.get("place_ms", 0)
        alg = algorithmic_bytes(lens)
        wire_ms = (per.get("send_ms", 0) + per.get("reply_ms", 0)) if args.transport == "nccl" else (per.get("route_ms", 0) + per.get("probe_ms", 0))
        line = {
            "metric": "queries placed/s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": NAMES[5], "reads_per_gpu": n_local, "reads_total": int(reads_total), "k": K_SIZE, "m": 4,
                       "index_entries_this_shard": int(info["n_entries"]), "index_entries_total": int(rep_info["n_entries"]),
                       "table_bytes_this_shard": int(info["table_bytes"]), "distinct_node_sets": int(info["n_distinct_sets"]),
                       "parallelism": (f"queries sharded x{world}, k-mer table hash-sharded x{world}, exchange fused into the route / probe "
                                       "kernels over NVLink peer memory (CUDA IPC); NCCL carries 8 counts + 1 barrier per sub-batch")
                       if args.transport == "p2p" else
                       f"queries sharded x{world}, k-mer table hash-sharded x{world}, 2 NCCL all-to-alls per sub-batch",
                       "transport": args.transport,
                       "sub_batch_reads": sub, "l2": "256 MiB memset between steps (outside the event pairs)"},
            "lookups_per_s": lookups_total / (ms_per_step / 1e3),
            "e2e": {"value": reads_total / e2e_s, "unit": "reads/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(sum(rb.nbytes() for rb in rbs) - 32 * n_device), "d2h_bytes_per_step": 32 * n_device,
                    "host_input": "ASCII bases + offsets in caller memory"},
            "gpu_launches": 3 * len(rbs) * args.steps,
            "roofline": {"bound": "hbm", "achieved": alg / (kern_ms / 1e3) / 1e9 if kern_ms else None, "peak": peak, "unit": "GB/s",
                         "frac": alg / (kern_ms / 1e3) / 1e9 / peak if kern_ms else None, "traffic": ncu_traffic(5),
                         "peak_source": peak_src, "algorithmic_bytes_per_step": alg,
                         "kernel": "cls::route_kernel<35> + cls::shard_probe_kernel + cls::place_routed_kernel<1> (rank 0, summed)",
                         "note": "the exchange is NVLink-bound: see `nvlink`"},
            "nvlink": {"wire_ms_per_step_rank0": wire_ms, "bytes_out_per_step_rank0": per.get("wire_bytes_out", 0),
                       "achieved_gbs_out_rank0": per.get("wire_bytes_out", 0) / (wire_ms / 1e3) / 1e9 if wire_ms else None,
                       "peak_gbs_per_direction": 900.0, "bytes_per_routed_kmer": 20,
                       "note": "p2p: the wire time IS the route + probe kernels (stores into peer memory)" if args.transport == "p2p" else "nccl: send + reply all-to-alls"},
            "stage_ms_per_step_rank0": {k: round(v, 3) for k, v in per.items() if k.endswith("_ms")},
            "cpu_baseline": None, "clocks": clocks,
            "parity": {"checked_reads": n_chk, "mismatching_fields": bad,
                       "against": "the replicated index on the same GPU (itself pinned to the CPU oracle by configs 2-4 and the tests)"},
            "status_histogram": np.bincount(np.concatenate([r.status for r in res]), minlength=11).tolist(),
            "step_ms": [round(x, 3) for x in step_ms],
            "setup_s": {"generate": round(gen_s, 1), "index_upload": round(upload_s, 2)},
        }
        if not embedded:
            print(json.dumps(line), flush=True)
    for rb in rbs:
        rb.close()
    if world > 1:
        dist.barrier()
    sp.close()
    if world > 1 and not embedded:
        dist.destroy_process_group()
    return line if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5],
                    help="workload (default 3: the configuration of the north-star target; it fits one GPU)")
    ap.add_argument("--reads", type=int, default=None, help="override the number of reads of the config")
    ap.add_argument("--transport", default="p2p", choices=["p2p", "nccl"], help="config 5: how routed k-mers cross NVLink")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU-baseline sample size in seconds of work")
    ap.add_argument("--no-config4", action="store_true", help="N = 1, default workload: skip the nested config-4 (kb-scale reads) measurement")
    ap.add_argument("--reads4", type=int, default=400_000, help="reads of the nested config-4 measurement")
    ap.add_argument("--no-config5", action="store_true", help="N > 1, default workload: skip the nested config-5 (hash-sharded index) measurement")
    ap.add_argument("--reads5", type=int, default=1_250_000, help="reads per GPU of the nested config-5 measurement")
    ap.add_argument("--no-inprocess", action="store_true", help="N = 1: skip the one-process-all-GPUs end-to-end number")
    ap.add_argument("--device-build", action="store_true",
                    help="set-up only: build the synthetic model's k-mer map on the GPU (cls_model_build_device) instead of the "
                         "host cores - the same arrays, outside every timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (a fixed, seeded sample of the reads) as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm places a timing-sized sample of the batch; dump the b200 arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun (one rank per GPU); running the single-GPU line", file=sys.stderr)
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.config == 5:
        run_sharded(args, rank, world, local_rank)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
