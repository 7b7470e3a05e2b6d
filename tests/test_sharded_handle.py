"""ONE handle over a HASH-SHARDED index (cls_index_create_sharded): shard s of the k-mer table on devices[s], the
routed stages (route -> probe -> place) chained inside the library by events across devices.  Every result field must
equal that of a replicated index on the same reads.  Shards may share a GPU, so everything here runs on one B200 as
well; the test with one shard per visible GPU skips below two.

Without a GPU the host side runs against the fake CUDA runtime (tests/native/sharded_fake_main.cpp, the peer-access
calls in tests/native/fake_peer_runtime.h, the routed launches restated in tests/native/fake_routed_kernels.cpp) under AddressSanitizer + UBSan and, with every stream a worker thread, under
ThreadSanitizer.  Dropping the owner's wait for a sender's route event (enqueue_routed in capi_sharded.cpp) makes ThreadSanitizer
report races there (checked by mutation)."""
import os
import shutil
import subprocess
import threading

import numpy as np
import pytest

from helpers import CAPI_HOST_SOURCES, CSRC

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FIELDS = ("status", "node_id", "one", "rest", "n_query_kmers", "n_matched", "n_root_matched", "iterations")
SHARDED = os.path.join(CSRC, "capi_sharded.cpp")
SOURCES = [SHARDED] + CAPI_HOST_SOURCES + [os.path.join(HERE, "native", f) for f in ("sharded_fake_main.cpp", "fake_routed_kernels.cpp")]


# ---- host side on the fake runtime ------------------------------------------------------------------------------------------
def _build(tmp, name, san, orc):
    out = tmp / name
    out.mkdir()
    jobs, objs = [], []
    for src in SOURCES:
        obj = str(out / (os.path.basename(src) + ".o"))
        objs.append(obj)
        cmd = ["g++", "-O1", "-g", "-std=c++17", "-pthread", *san, "-I", os.path.join(HERE, "native", "fakecuda")] + \
              (["-include", os.path.join(HERE, "native", "fake_peer_runtime.h")] if src == SHARDED else []) + ["-c", src, "-o", obj]
        jobs.append(subprocess.Popen(cmd, stderr=subprocess.PIPE, text=True))
    for p in jobs:
        _, err = p.communicate()
        assert "error:" not in err, err[-3000:]
        if p.returncode != 0:
            pytest.skip(f"cannot build with {san} here: {err[-300:]}")
    exe = str(out / "sharded_fake")
    r = subprocess.run(["g++", "-pthread", *san, *objs, orc, "-o", exe], capture_output=True, text=True)
    assert "undefined reference" not in r.stderr, r.stderr[-3000:]
    if r.returncode != 0:
        pytest.skip(f"cannot link with {san} here: {r.stderr[-300:]}")
    return exe


@pytest.fixture(scope="module")
def fake_runs(tmp_path_factory):
    """Both builds, then both runs side by side: {name: CompletedProcess}."""
    if shutil.which("g++") is None:
        pytest.skip("needs g++")
    tmp = tmp_path_factory.mktemp("sharded_fake")
    orc = str(tmp / "orc.o")
    subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-c", os.path.join(ROOT, "oracle", "classeq_oracle.cpp"), "-o", orc], check=True)
    exes = {"asan": _build(tmp, "asan", ["-fsanitize=address,undefined", "-fno-sanitize-recover=undefined"], orc),
            "tsan": _build(tmp, "tsan", ["-fsanitize=thread"], orc)}
    procs = {"asan": subprocess.Popen([exes["asan"]], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True),
             "tsan": subprocess.Popen([exes["tsan"], "threads"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                      env=dict(os.environ, FAKE_CUDA_ASYNC="1"))}
    out = {}
    for name, p in procs.items():
        try:
            so, se = p.communicate(timeout=1800)
        except subprocess.TimeoutExpired:
            p.kill()
            so, se = p.communicate()
            se += "\n[timed out]"
        out[name] = subprocess.CompletedProcess(p.args, p.returncode, so, se)
    return out


def test_sharded_host_side_equals_the_oracle_under_asan(fake_runs):
    """1, 3 and 8 shards over one to three fake devices, several sub-batches, host and device packing, an overflowing
    segment, the resident path and the FASTA ingest, refusals, a failing allocation at every position of create and place
    (nothing leaked) and a failing CUDA call at every position of a placement (the handle works afterwards)."""
    r = fake_runs["asan"]
    assert "ERROR: AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[:4000]
    assert r.returncode == 0 and r.stdout.startswith("bad=0 "), (r.returncode, r.stdout, r.stderr[-1500:])


def test_sharded_streams_and_threads_are_race_free_under_tsan(fake_runs):
    """The same with every stream a worker thread (FAKE_CUDA_ASYNC=1): the events between the lanes' streams (route ->
    probe across devices, probe -> place) and the one host wait per sub-batch are what keeps this free of races; four
    concurrent callers on one handle."""
    r = fake_runs["tsan"]
    if "FATAL: ThreadSanitizer" in r.stderr and "unexpected memory mapping" in r.stderr:
        pytest.skip("ThreadSanitizer cannot map its shadow memory in this container")
    assert "WARNING: ThreadSanitizer" not in r.stderr and "[timed out]" not in r.stderr, r.stderr[:4000]
    assert r.returncode == 0 and r.stdout.startswith("bad=0 "), (r.returncode, r.stdout, r.stderr[-1500:])


# ---- on the GPU ---------------------------------------------------------------------------------------------------------------
def _same(a, b):
    for f in FIELDS:
        bad = np.flatnonzero(getattr(a, f) != getattr(b, f))
        assert bad.size == 0, (f, bad[:5], getattr(a, f)[bad[:5]], getattr(b, f)[bad[:5]])


@pytest.fixture(scope="module")
def cq():
    import classeq2_b200
    return classeq2_b200


@pytest.fixture(scope="module")
def synth_case(cq):
    from classeq2_b200 import synth
    sm = synth.make_model(300, 400, 77)
    b, o, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, 3000, np.full(3000, 150), 78)
    return sm, b, o


PARAMS = (dict(), dict(remove_intersection=True), dict(min_match_coverage=0.2, max_iterations=3))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 8])
def test_shards_on_one_gpu_equal_the_replicated_index(cq, synth_case, n):
    sm, b, o = synth_case
    for flat in (sm.flat, sm.flat.with_general_sets()):
        ref = cq.Index(flat, device=0)
        sh = cq.Index(flat, sharded_devices=[0] * n)
        inf = sh.info()
        assert inf["n_devices"] == n and inf["device"] == 0 and inf["n_entries"] == ref.info()["n_entries"]
        assert inf["closed_sets"] == ref.info()["closed_sets"]
        for kn in PARAMS:
            p = cq.PlaceParams(**kn)
            _same(sh.place_batch((b, o), p), ref.place_batch((b, o), p))
        sh.close(), ref.close()


def _col_reads(col_queries):
    """The fixture's queries of up to 160 bases, plus 150-base windows of the longer ones."""
    seqs = []
    for _, s in col_queries:
        if len(s) <= 160:
            seqs.append(s)
        else:
            seqs += [s[i:i + 150] for i in range(0, len(s) - 149, 50)]
    return seqs


@pytest.mark.gpu
def test_colletotrichum_through_four_shards(cq, col_flat, col_queries):
    seqs = _col_reads(col_queries)
    assert len(seqs) > 1000
    ref, sh = cq.Index(col_flat, device=0), cq.Index(col_flat, sharded_devices=[0, 0, 0, 0])
    for kn in PARAMS:
        p = cq.PlaceParams(**kn)
        _same(sh.place_batch(seqs, p), ref.place_batch(seqs, p))
    sh.close(), ref.close()


@pytest.mark.gpu
def test_ragged_lengths_short_reads_and_an_empty_batch(cq, synth_case):
    from classeq2_b200 import synth
    sm, _, _ = synth_case
    lens = np.random.default_rng(5).integers(20, 162, 4000)
    lens[:5] = [0, 1, 34, 35, 161]
    b, o, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, len(lens), lens, 79)
    b = b.copy()
    b[int(o[40]) + 3] = ord("N")
    ref, sh = cq.Index(sm.flat, device=0), cq.Index(sm.flat, sharded_devices=[0, 0, 0])
    _same(sh.place_batch((b, o)), ref.place_batch((b, o)))
    empty = (np.zeros(1, np.uint8), np.zeros(1, np.uint64))
    assert sh.place_batch(empty).status.size == 0
    sh.close(), ref.close()


def _run_child(code, env):
    """A fresh interpreter: the sub-batch bound is read once per process."""
    r = subprocess.run(["python", "-c", code], cwd=ROOT, env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


_CHILD_PRELUDE = """
import numpy as np, classeq2_b200 as cq
from classeq2_b200 import synth
F = ("status", "node_id", "one", "rest", "n_query_kmers", "n_matched", "n_root_matched", "iterations")
def same(a, b):
    for f in F:
        assert (getattr(a, f) == getattr(b, f)).all(), f
sm = synth.make_model(300, 400, 77)
"""


@pytest.mark.gpu
def test_several_sub_batches(cq):
    """CLS_SHARD_SUB_READS (a test knob) lowers the bound on reads per home and sub-batch: 12 000 reads on 3 homes are
    eight sub-batches each, through cls_place_batch and through a resident batch."""
    _run_child(_CHILD_PRELUDE + """
b, o, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, 12000, np.random.default_rng(3).integers(30, 162, 12000), 80)
ref, sh = cq.Index(sm.flat, device=0), cq.Index(sm.flat, sharded_devices=[0, 0, 0])
want = ref.place_batch((b, o))
same(sh.place_batch((b, o)), want)
rb = sh.upload((b, o)); rb.place(); same(rb.fetch(), want)
print("OK")
""", {"CLS_SHARD_SUB_READS": "500"})


def _single_owner_homopolymer(n_max=8):
    """(n_shards, base) such that every window of a 150-base homopolymer of `base` - both strands - has one owner."""
    from oracle import cpp_oracle
    for n in range(2, n_max + 1):
        for c in "ACGT":
            h = np.asarray(cpp_oracle.kmer_hashes((c * 150).encode(), 35), dtype=np.uint64)
            own = (h >> np.uint64(61)) % np.uint64(n)
            if (own == own[0]).all():
                return n, c, h.size
    raise AssertionError("no homopolymer with one owner")


@pytest.mark.gpu
def test_low_complexity_reads_overflow_a_segment(cq, synth_case):
    """Every window of a homopolymer read goes to one owner: 2 000 of them per home exceed the first seg_cap (checked here
    on the host), and the sub-batch runs again with the exact bound."""
    from classeq2_b200 import synth
    sm, _, _ = synth_case
    n, c, w = _single_owner_homopolymer()
    per_home = 2000
    windows = per_home * w
    first_seg_cap = ((int(windows / n * 1.15) + 65536) + 31) & ~31
    assert windows > first_seg_cap
    nb, no, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, 600 * n, np.full(600 * n, 150), 81)
    normal = [nb[int(no[i]):int(no[i + 1])].tobytes().decode() for i in range(600 * n)]
    seqs = []
    for i in range(per_home * n):
        seqs.append(c * 150)
        if i % 10 == 0:
            seqs.append(normal[i // 10])
    ref, sh = cq.Index(sm.flat, device=0), cq.Index(sm.flat, sharded_devices=[0] * n)
    _same(sh.place_batch(seqs), ref.place_batch(seqs))
    sh.close(), ref.close()


@pytest.mark.gpu
def test_resident_fasta_and_place_sequences(cq, col_flat, col_tree, col_queries, tmp_path):
    """Resident path and cls_fasta_upload on the handle; place_sequences with both ingests and place_sequences_native
    write files byte-identical to the replicated handle's."""
    seqs = _col_reads(col_queries)
    ref, sh = cq.Index(col_flat, device=0), cq.Index(col_flat, sharded_devices=[0, 0, 0, 0])
    rb = sh.upload(seqs)
    rb.place()
    _same(rb.fetch(), ref.place_batch(seqs))
    rb.close()
    text = "".join(f">q{i} window\n{s}\n" for i, s in enumerate(seqs)) + ">empty\n\n>short\nACGT\n>tail\nACGTACGTAC\n"
    fa = tmp_path / "q.fasta"
    fa.write_text(text)
    frb, headers, lens = sh.upload_fasta(text.encode())
    frb.place()
    rrb, _, _ = ref.upload_fasta(text.encode())
    rrb.place()
    _same(frb.fetch(), rrb.fetch())
    frb.close(), rrb.close()
    tree = cq.Tree.from_obj(col_tree.to_obj())
    for kw in (dict(), dict(ingest="device")):
        a, b = tmp_path / f"ref{len(kw)}" / "r.yaml", tmp_path / f"sh{len(kw)}" / "r.yaml"
        cq.place_sequences(str(fa), tree, a, index=ref, **kw)
        cq.place_sequences(str(fa), tree, b, index=sh, **kw)
        assert a.read_bytes() == b.read_bytes() and len(a.read_bytes()) > 10000
        assert a.with_suffix(".error").read_bytes() == b.with_suffix(".error").read_bytes()
    a, b = tmp_path / "nref" / "r.yaml", tmp_path / "nsh" / "r.yaml"
    cq.place_sequences_native(str(fa), tree, a, index=ref)
    cq.place_sequences_native(str(fa), tree, b, index=sh)
    assert a.read_bytes() == b.read_bytes() and len(a.read_bytes()) > 10000
    sh.close(), ref.close()


@pytest.mark.gpu
def test_four_concurrent_callers(cq, synth_case):
    from classeq2_b200 import synth
    sm, _, _ = synth_case
    ref, sh = cq.Index(sm.flat, device=0), cq.Index(sm.flat, sharded_devices=[0, 0, 0])
    batches = [synth.make_reads(sm.ref_codes, sm.ref_lens, 2000, np.full(2000, 140 + t), 90 + t)[:2] for t in range(4)]
    want = [ref.place_batch(bo) for bo in batches]
    errors = []

    def run(t):
        try:
            for _ in range(3):
                _same(sh.place_batch(batches[t]), want[t])
        except Exception as e:   # noqa: BLE001 - reported below
            errors.append(e)
    th = [threading.Thread(target=run, args=(t,)) for t in range(4)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors[0]
    sh.close(), ref.close()


@pytest.mark.gpu
def test_refusals(cq, synth_case):
    from classeq2_b200 import _lib
    sm, b, o = synth_case
    sh = cq.Index(sm.flat, sharded_devices=[0, 0])
    ref = cq.Index(sm.flat, device=0)
    with pytest.raises(_lib.ClsError) as e:
        sh.place_batch(["A" * 162, "ACGT" * 40])
    assert e.value.code == _lib.CLS_ERR_UNSUPPORTED and "161" in e.value.message
    _same(sh.place_batch((b, o)), ref.place_batch((b, o)))   # the handle still works
    for n in (0, 9):
        with pytest.raises(_lib.ClsError) as e:
            cq.Index(sm.flat, sharded_devices=[0] * n)
        assert e.value.code == _lib.CLS_ERR_INVALID_ARGUMENT
    rb = sh.upload((b, o))
    with pytest.raises(_lib.ClsError) as e:
        rb.routed_windows()
    assert e.value.code == _lib.CLS_ERR_INVALID_ARGUMENT
    buf = np.zeros(1 << 16, np.uint64)
    p = buf.ctypes.data
    for call in (lambda: rb.route_hashes(2, 1024, p, p), lambda: rb.route_hashes_p2p(2, 1024, [p, p], p),
                 lambda: rb.place_routed(p, p, 2, 1024), lambda: sh.shard_probe(p, 1, p), lambda: sh.debug_node_counts("ACGT" * 40)):
        with pytest.raises(_lib.ClsError) as e:
            call()
        assert e.value.code == _lib.CLS_ERR_INVALID_ARGUMENT
    rb.close(), sh.close(), ref.close()


@pytest.mark.gpu
def test_one_shard_per_visible_gpu(cq, synth_case):
    import torch
    n_gpu = min(torch.cuda.device_count(), 8)
    if n_gpu < 2:
        pytest.skip("needs two GPUs")
    sm, b, o = synth_case
    ref, sh = cq.Index(sm.flat, device=0), cq.Index(sm.flat, sharded_devices=list(range(n_gpu)))
    assert sh.info()["n_devices"] == n_gpu
    for kn in PARAMS:
        p = cq.PlaceParams(**kn)
        _same(sh.place_batch((b, o), p), ref.place_batch((b, o), p))
    rb = sh.upload((b, o))
    rb.place()
    _same(rb.fetch(), ref.place_batch((b, o)))
    rb.close(), sh.close(), ref.close()
