#!/usr/bin/env python
"""End-to-end timing of cls_place_batch (host ASCII buffers in, host result arrays out) on config 2's workload, under the
host-side knobs CLS_CHUNK_MBASES, CLS_HOST_THREADS and CLS_PACK; CLASSEQ_B200_LIB picks the library.
usage: [ENV=...] python tools/e2e_bench.py [n_reads=1000000]"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import classeq2_b200 as cq  # noqa: E402
from classeq2_b200 import synth  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
cfg = int(sys.argv[2]) if len(sys.argv) > 2 else 2
n_dev = int(sys.argv[3]) if len(sys.argv) > 3 else 0      # > 0: one multi-device handle over that many replicas
c = synth.CONFIGS[cfg]
sm = synth.make_model(c["n_tips"], c["l_ref"], c["tree_seed"])
bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, n, 150, c["tree_seed"] + 2)
import torch  # noqa: E402
ix = cq.Index(sm.flat, device=0) if n_dev == 0 else cq.Index(sm.flat, devices=[d % torch.cuda.device_count() for d in range(n_dev)])
if os.environ.get("PIN"):      # the bases in pinned memory (a device pack then copies straight from them)
    pin = torch.empty(len(bases), dtype=torch.uint8).pin_memory()
    pin.numpy()[:] = bases
    bases = pin.numpy()
out = cq.BatchResult(n)
for _ in range(3):
    ix.place_batch_into(bases, offsets, out)
ts = []
for _ in range(10):
    t0 = time.perf_counter()
    ix.place_batch_into(bases, offsets, out)
    ts.append(time.perf_counter() - t0)
dt = float(np.mean(ts))
knobs = {k: os.environ[k] for k in ("CLS_CHUNK_MBASES", "CLS_HOST_THREADS", "CLASSEQ_B200_LIB", "CLS_PACK", "PIN") if k in os.environ}
print(f"config{cfg} n={n} replicas={n_dev} {knobs} e2e {dt * 1e3:.2f} ms (min {min(ts) * 1e3:.2f})  {n / dt / 1e6:.1f} M reads/s  "
      f"status_hist={np.bincount(out.status, minlength=11).tolist()} sum(node)={int(out.node_id.sum())}",
      {k: round(v, 2) for k, v in ix.timing().items()})
