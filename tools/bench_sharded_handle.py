"""Config 5 (synthetic Tree(100 000, 1005) model, 150 bp reads) through ONE hash-sharded handle in ONE process
(cls_index_create_sharded), next to the replicated handle in the same run.  Prints one JSON line.

    python tools/bench_sharded_handle.py [--reads N] [--steps K] [--warmup W]

Per variant (1 GPU with 1 and with 8 shards, every visible GPU with one shard each, the replicated multi-device handle):
  resident  reads/s of cls_place_resident on a batch uploaded once: CUDA events around every step on the caller's stream
            of the first device, 256 MiB written between steps so that the 126 MB L2 holds nothing of the last step
  e2e       reads/s of cls_place_batch from pinned host memory to host result arrays (host clock; the call ends synchronised)
  check     20 000 reads placed by the variant and by the replicated handle: every result field equal
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FIELDS = ("status", "node_id", "one", "rest", "n_query_kmers", "n_matched", "n_root_matched", "iterations")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "visible_gpus": len(out)}
    except Exception as e:  # noqa: BLE001
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch

    import classeq2_b200 as cq
    from classeq2_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    n_gpu = min(torch.cuda.device_count(), 8)
    c = synth.CONFIGS[5]
    t0 = time.time()
    sm = synth.make_model(c["n_tips"], c["l_ref"], c["tree_seed"], device=0)
    bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, args.reads, c["read_len"], c["tree_seed"] + 2)
    pinned = torch.empty(bases.size, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = bases
    pb = pinned.numpy()
    line = {"workload": "config5: Tree(100000, 1005), 150 bp reads", "reads": args.reads, "steps": args.steps, **card(),
            "model_s": round(time.time() - t0, 1), "l2": "256 MiB memset between resident steps (outside the event pairs)"}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    st = torch.cuda.current_stream(0)
    chk = (pb[: int(offsets[20000])], offsets[:20001])
    ref = cq.Index(sm.flat, device=0)
    want = ref.place_batch(chk)

    def measure(ix, resident=True):
        r = {}
        res = cq.BatchResult(args.reads)
        for i in range(args.warmup):
            ix.place_batch_into(pb, offsets, res)
        t = time.perf_counter()
        for i in range(args.steps):
            ix.place_batch_into(pb, offsets, res)
        r["e2e_reads_per_s"] = args.reads * args.steps / (time.perf_counter() - t)
        r["e2e_ms_per_step"] = (time.perf_counter() - t) * 1e3 / args.steps
        if resident:
            rb = ix.upload((pb, offsets))
            ms = []
            for i in range(args.warmup + args.steps):
                flush.fill_(i & 0xFF)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                rb.place(stream=st.cuda_stream)
                e1.record(st)
                torch.cuda.synchronize(0)
                if i >= args.warmup:
                    ms.append(e0.elapsed_time(e1))
            r["resident_reads_per_s"] = args.reads / (sum(ms) / len(ms) / 1e3)
            r["resident_ms_per_step"] = [round(x, 2) for x in ms]
            rb.close()
        got = ix.place_batch(chk)
        r["check_20k_equal"] = all(bool((getattr(got, f) == getattr(want, f)).all()) for f in FIELDS)
        r["timing"] = {k: v for k, v in ix.timing().items() if k in ("kernel_ms", "total_ms", "kernel_launches")}
        return r

    out = {}
    out["replicated_1gpu"] = measure(ref)
    variants = [("sharded_1gpu_1shard", [0]), ("sharded_1gpu_8shards", [0] * 8)]
    if n_gpu > 1:
        variants.append((f"sharded_{n_gpu}gpu_1shard_each", list(range(n_gpu))))
    for name, devs in variants:
        t = time.time()
        ix = cq.Index(sm.flat, sharded_devices=devs)
        build_s = time.time() - t
        out[name] = dict(measure(ix), create_s=round(build_s, 1))
        ix.close()
    if n_gpu > 1:
        multi = cq.Index(sm.flat, devices=list(range(n_gpu)))
        out[f"replicated_{n_gpu}gpu"] = measure(multi, resident=False)   # (resident batches of that handle use its first device)
        multi.close()
    ref.close()
    line["results"] = out
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
