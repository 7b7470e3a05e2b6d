"""The HOST side of the hot path's public call - ``cls_place_batch`` and its neighbours (classeq2_b200/csrc/capi.cpp,
place_batch.cpp, resident.cpp, routed.cpp):
planning (general and just in time, with its fallback), host / device / mixed packing from pageable and pinned memory,
the chunked pipeline, scatter into the caller's arrays, resident batches, one handle over several devices, concurrent
callers, a failing launch - end to end WITHOUT a GPU.  They are compiled with g++ against a fake CUDA runtime
(tests/native/fakecuda/cuda_runtime.h: device memory is host memory, every call completes before it returns); the
placement launch unpacks the reads it is handed and gives them to the C++ oracle (tests/native/fake_kernels.cpp); the
results must equal the oracle's on the caller's ASCII batch (tests/native/capi_fake_main.cpp).  Run under
AddressSanitizer + UBSan (a copy past a "device" buffer is a report) and, with every stream of the fake runtime a
worker thread, under ThreadSanitizer (a missing stream dependency is a data race).  The kernels themselves are what the ``-m gpu`` tests are for."""
import os
import shutil
import subprocess

import pytest

from helpers import CAPI_HOST_SOURCES

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FAKE = os.path.join(HERE, "native", "fakecuda")
SOURCES = CAPI_HOST_SOURCES + [os.path.join(HERE, "native", f) for f in ("capi_fake_main.cpp", "fake_kernels.cpp")]


def _compile(tmp_path, name, san):
    """Starts the compilers: one object per source, side by side.  The oracle is compiled once, without a sanitizer (it is
    the checker, and its allocations dominate the run time under one)."""
    out = tmp_path / name
    out.mkdir()
    jobs, objs = [], []
    orc = tmp_path / "orc.o"
    if not getattr(_compile, "orc_started", False):
        _compile.orc_started = True
        jobs.append(subprocess.Popen(["g++", "-O2", "-std=c++17", "-pthread", "-c", os.path.join(ROOT, "oracle", "classeq_oracle.cpp"), "-o", str(orc)],
                                     stderr=subprocess.PIPE, text=True))
    for src in SOURCES:
        obj = str(out / (os.path.basename(src) + ".o"))
        objs.append(obj)
        cmd = ["g++", "-O1", "-g", "-std=c++17", "-pthread", *san, "-I", FAKE, "-c", src, "-o", obj]
        jobs.append(subprocess.Popen(cmd, stderr=subprocess.PIPE, text=True))
    return jobs, objs, str(orc), str(out / "capi_fake"), san


def _link(jobs, objs, orc, exe, san):
    for p in jobs:
        _, err = p.communicate()
        assert "error:" not in err, err[-3000:]                      # a real build error is a failure
        if p.returncode != 0:
            pytest.skip(f"cannot build with {san} here: {err[-300:]}")
    r = subprocess.run(["g++", "-pthread", *san, *objs, orc, "-o", exe], capture_output=True, text=True)
    assert "undefined reference" not in r.stderr, r.stderr[-3000:]
    if r.returncode != 0:
        pytest.skip(f"cannot link with {san} here: {r.stderr[-300:]}")
    return exe


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """Both builds side by side, then both runs side by side (the oracle dominates either): {name: CompletedProcess}."""
    if shutil.which("g++") is None:
        pytest.skip("needs g++")
    tmp = tmp_path_factory.mktemp("capi_fake")
    _compile.orc_started = False
    started = [_compile(tmp, "asan", ["-fsanitize=address,undefined", "-fno-sanitize-recover=undefined"]), _compile(tmp, "tsan", ["-fsanitize=thread"])]
    exes = {"asan": _link(*started[0]), "tsan": _link(*started[1])}
    # asan: the synchronous runtime (host logic, buffer sizes); tsan: every stream a worker thread (FAKE_CUDA_ASYNC=1) - a
    # missing dependency between streams, or between a stream and the host, is a data race there
    procs = {"asan": subprocess.Popen([exes["asan"]], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True),
             "tsan": subprocess.Popen([exes["tsan"]], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                      env=dict(os.environ, FAKE_CUDA_ASYNC="1"))}
    out = {}
    for name, p in procs.items():
        try:
            so, se = p.communicate(timeout=1200)
        except subprocess.TimeoutExpired:
            p.kill()
            so, se = p.communicate()
            se += "\n[timed out]"
        out[name] = subprocess.CompletedProcess(p.args, p.returncode, so, se)
    return out


def test_place_batch_host_side_equals_the_oracle_under_asan(runs):
    r = runs["asan"]
    assert "ERROR: AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[:4000]
    assert r.returncode == 0 and r.stdout.startswith("bad=0 "), (r.returncode, r.stdout, r.stderr[-1500:])


def test_place_batch_streams_and_threads_are_race_free_under_tsan(runs):
    """Every scenario again with the streams of the fake runtime as worker threads: copies, fake kernels and event waits run
    in stream order next to the host thread, so the dependencies of the three-stream pipeline (copies in -> kernels ->
    copies out, the staging ring, the scratch buffer, the scatter of finished chunks) are what keeps this free of races.
    Dropping the kernel stream's wait for the copy-in of the later chunks is reported here (checked by mutation)."""
    r = runs["tsan"]
    if "FATAL: ThreadSanitizer" in r.stderr and "unexpected memory mapping" in r.stderr:
        pytest.skip("ThreadSanitizer cannot map its shadow memory in this container")
    assert "WARNING: ThreadSanitizer" not in r.stderr and "[timed out]" not in r.stderr, r.stderr[:4000]
    assert r.returncode == 0 and r.stdout.startswith("bad=0 "), (r.returncode, r.stdout, r.stderr[-1500:])
