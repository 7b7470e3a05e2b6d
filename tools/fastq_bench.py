#!/usr/bin/env python
"""Times the FASTQ readers on config 3's reads (10 M x 150 bp, 1 % substitutions) written as FASTQ: titles "@r<i>",
random qualities, about 3.3 GB of text.  Reports the host reader (cls_fastq_read), cls_fastq_upload split into the copy
of the text, the kernels and the rest (host bookkeeping: record rules, planning, small copies, allocations), and
place_sequences end to end with host and with device ingest on the first --e2e-reads reads (the writer sets the pace of
that call: every record becomes a JSON line on disk).  The card's name and power limit are printed in the same run.
usage: python tools/fastq_bench.py [--reads N] [--e2e-reads N] [--out result.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import classeq2_b200 as cq  # noqa: E402
from classeq2_b200 import _lib, synth  # noqa: E402
from classeq2_b200.model import Clade, Tree  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        return "unknown"


def tree_of(st) -> Tree:
    """The synthetic topology as the reference's Tree (what the record writer reads)."""
    kinds = {0: "ROOT", 1: "NODE", 2: "LEAF"}
    clades = [None] * len(st.node_id)
    for v in range(len(st.node_id) - 1, -1, -1):      # pre-order: children have larger indices
        kids = [clades[int(c)] for c in st.child_idx[int(st.child_off[v]):int(st.child_off[v + 1])]]
        k = kinds[int(st.node_kind[v])]
        clades[v] = Clade(id=int(st.node_id[v]), parent=None if st.parent[v] < 0 else int(st.node_id[st.parent[v]]), kind=k,
                          name=f"tip_{v}" if k == "LEAF" else None, children=kids if k != "LEAF" else None)
    return Tree(id="synthetic", name="config3", min_branch_support=0.0, root=clades[0])


def fastq_text(bases, n, read_len, seed):
    rng = np.random.default_rng(seed)
    body = bases.reshape(n, read_len)
    out, step = [], 1 << 18
    for a in range(0, n, step):
        b = min(n, a + step)
        qual = rng.integers(33, 75, (b - a, read_len), dtype=np.uint8)
        out.append(b"".join(b"@r%d\n%b\n+\n%b\n" % (a + i, body[a + i].tobytes(), qual[i].tobytes()) for i in range(b - a)))
    return b"".join(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--e2e-reads", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"card": card(), "reads": a.reads, "read_len": 150}
    print("card:", res["card"], flush=True)
    c = synth.CONFIGS[3]
    sm = synth.make_model(c["n_tips"], c["l_ref"], c["tree_seed"], device=0)
    bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, a.reads, 150, c["tree_seed"] + 2)
    t0 = time.time()
    raw = fastq_text(bases, a.reads, 150, 7)
    text = np.frombuffer(raw, dtype=np.uint8)
    res["text_bytes"] = int(text.size)
    print(f"text: {text.size / 1e9:.2f} GB built in {time.time() - t0:.1f} s", flush=True)
    ptr = text.ctypes.data_as(_lib.u8p)

    # ---- host reader ----
    ts = []
    for _ in range(a.reps):
        h, rec = C.c_void_p(), _lib.FastaHostRecords()
        t0 = time.perf_counter()
        _lib.check(_lib.lib.cls_fastq_read(ptr, text.size, C.byref(h), C.byref(rec)))
        ts.append(time.perf_counter() - t0)
        n_host = int(rec.n_records)
        _lib.lib.cls_fasta_text_destroy(h)
    assert n_host == a.reads
    res["host_reader_s"] = ts
    print(f"cls_fastq_read: {min(ts) * 1e3:.0f} ms (runs {[round(t * 1e3) for t in ts]}) = {text.size / min(ts) / 1e9:.2f} GB/s", flush=True)

    # ---- device ingest ----
    ix = cq.Index(sm.flat, device=0)
    ts = []
    for rep in range(a.reps + 1):                        # the first call warms the allocator and loads the module
        h, rec = C.c_void_p(), _lib.FastaRecords()
        t0 = time.perf_counter()
        _lib.check(_lib.lib.cls_fastq_upload(ix._h, ptr, text.size, C.byref(h), C.byref(rec)))
        dt = time.perf_counter() - t0
        rb = cq.ResidentBatch._from_handle(ix, h, int(rec.n_records))
        if rep:
            ts.append(dt)
        if rep == a.reps:
            rb.place()
            got = rb.fetch()
            want = ix.place_batch((bases, offsets))
            res["placements_equal_place_batch"] = bool(all((getattr(got, f) == getattr(want, f)).all() for f, _ in cq.engine.RESULT_DTYPES))
        rb.close()
    res["upload_s"] = ts
    print(f"cls_fastq_upload: {min(ts) * 1e3:.0f} ms (runs {[round(t * 1e3) for t in ts]}) = {a.reads / min(ts) / 1e6:.1f} M reads/s, "
          f"{text.size / min(ts) / 1e9:.2f} GB/s of text; placements equal to cls_place_batch: {res['placements_equal_place_batch']}", flush=True)

    # one more call under the profiler (a run of its own): device time of the copies and of the kernels
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        h, rec = C.c_void_p(), _lib.FastaRecords()
        t0 = time.perf_counter()
        _lib.check(_lib.lib.cls_fastq_upload(ix._h, ptr, text.size, C.byref(h), C.byref(rec)))
        wall = time.perf_counter() - t0
        _lib.lib.cls_resident_destroy(h)
    split = {"h2d_ms": 0.0, "d2h_ms": 0.0, "memset_ms": 0.0, "kernels_ms": {}}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = e.time_range.elapsed_us()
        name = e.name
        if "Memcpy HtoD" in name:
            split["h2d_ms"] += us / 1e3
        elif "Memcpy DtoH" in name:
            split["d2h_ms"] += us / 1e3
        elif "Memset" in name:
            split["memset_ms"] += us / 1e3
        else:
            short = next((k for k in ("fastq_tile_kernel", "fastq_scan_kernel", "fastq_write_kernel", "fastq_record_kernel",
                                      "fasta_pack_kernel") if k in name), name[:60])
            split["kernels_ms"][short] = split["kernels_ms"].get(short, 0.0) + us / 1e3
    k_total = sum(split["kernels_ms"].values())
    split["profiled_wall_ms"] = wall * 1e3
    split["kernels_total_ms"] = k_total
    split["host_bookkeeping_ms"] = wall * 1e3 - split["h2d_ms"] - split["d2h_ms"] - split["memset_ms"] - k_total
    res["upload_split"] = split
    print("cls_fastq_upload under the profiler: " + json.dumps(split), flush=True)

    # ---- place_sequences end to end ----
    ne = min(a.e2e_reads, a.reads)
    tree = tree_of(sm.tree)
    cut = sum(len(str(i)) for i in range(ne)) + 307 * ne          # "@r<i>\n" + 150 + "\n+\n" + 150 + "\n"
    with tempfile.TemporaryDirectory() as d:
        q = os.path.join(d, "q.fastq")
        with open(q, "wb") as f:
            f.write(memoryview(raw)[:cut])
        files = {}
        for ingest in ("host", "device"):
            ts = []
            for rep in range(2):
                out = os.path.join(d, f"{ingest}{rep}", "r")
                t0 = time.perf_counter()
                cq.place_sequences(q, tree, out, output_format="jsonl", index=ix, ingest=ingest, query_format="fastq")
                ts.append(time.perf_counter() - t0)
                files[ingest] = os.path.getsize(out + ".jsonl")
            res[f"place_sequences_{ingest}_s"] = ts
            print(f"place_sequences {ne} reads ({cut / 1e6:.0f} MB of FASTQ), ingest={ingest}: {min(ts) * 1e3:.0f} ms "
                  f"(runs {[round(t * 1e3) for t in ts]}) = {ne / min(ts) / 1e6:.2f} M reads/s", flush=True)
        same = open(os.path.join(d, "host1", "r.jsonl"), "rb").read() == open(os.path.join(d, "device1", "r.jsonl"), "rb").read()
        res["e2e_reads"] = ne
        res["e2e_host_device_files_identical"] = same
        print(f"result files of the two ingests identical: {same} ({files['host'] / 1e6:.0f} MB of JSON lines)", flush=True)
    ix.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
