"""The host-side planner of ``cls_place_batch`` / ``cls_batch_upload`` (place_batch.cpp: plan_batch) through
``cls_debug_plan_batch``: host-decided statuses, length classes, device order and packed layout.  No GPU."""
import ctypes as C

import numpy as np
import pytest

from classeq2_b200 import _lib

TOO_SHORT = _lib.STATUS_ERR_TOO_SHORT


def plan(lens, k):
    lens = np.asarray(lens, np.uint64)
    n = len(lens)
    offsets = np.zeros(n + 1, np.uint64)
    offsets[1:] = np.cumsum(lens)
    bases = np.zeros(1, np.uint8)            # the planner never reads the bases
    b = _lib.Batch(n, bases.ctypes.data_as(_lib.u8p), offsets.ctypes.data_as(_lib.u64p))
    pre = np.zeros(max(n, 1), np.uint8)
    perm = np.zeros(max(n, 1), np.uint32)
    woff = np.zeros(n + 1, np.uint32)
    classes = (_lib.PlanClass * 64)()
    nc, nd, nw = C.c_uint32(), C.c_uint32(), C.c_uint64()
    rc = _lib.lib.cls_debug_plan_batch(k, C.byref(b), pre.ctypes.data_as(_lib.u8p), perm.ctypes.data_as(_lib.u32p),
                                       woff.ctypes.data_as(_lib.u32p), classes, 64, C.byref(nc), C.byref(nd), C.byref(nw))
    _lib.check(rc)
    return dict(pre=pre[:n], perm=perm[:nd.value], woff=woff[:nd.value + 1], n_words=nw.value,
                classes=[(classes[c].first, classes[c].count, classes[c].max_len) for c in range(nc.value)])


def class_of(length, k):
    """Table geometry shared by a class: log2 of the de-duplication table size for that length (place_batch.cpp)."""
    h2, c = 4 * (length - k + 1), 6
    while (1 << c) < h2:
        c += 1
    return c


def check(lens, k):
    lens = np.asarray(lens, np.int64)
    p = plan(lens, k)
    on_dev = np.flatnonzero(lens >= k)
    assert (p["pre"] == np.where(lens >= k, 0xFF, TOO_SHORT)).all()
    assert sorted(p["perm"].tolist()) == on_dev.tolist()                         # every long-enough read, once
    first = 0
    prev_class = None
    for f, cnt, mx in p["classes"]:
        assert f == first and cnt > 0
        members = p["perm"][f:f + cnt]
        assert (np.diff(members.astype(np.int64)) > 0).all()                      # input order inside a class
        cl = {class_of(int(lens[i]), k) for i in members}
        assert len(cl) == 1                                                       # one table geometry per class
        assert mx == lens[members].max()
        if prev_class is not None:
            assert cl.pop() < prev_class                                          # longest class first
            prev_class = class_of(int(lens[members[0]]), k)
        else:
            prev_class = cl.pop()
        first += cnt
    assert first == len(on_dev)
    words = (lens[p["perm"]] + 15) // 16
    assert (p["woff"] == np.concatenate([[0], np.cumsum(words)])).all() and p["n_words"] == int(words.sum())
    return p


def test_plan_uniform_short_reads():
    p = check(np.full(100_000, 150), 35)
    assert len(p["classes"]) == 1 and (p["perm"] == np.arange(100_000)).all()     # one class, caller order


def test_plan_mixed_lengths_and_short_queries():
    rng = np.random.default_rng(3)
    for k in (35, 12, 5):
        lens = np.concatenate([rng.integers(0, 60, 3000), rng.integers(100, 400, 3000), rng.integers(1000, 3000, 500),
                               [k - 1, k, k + 1, 0, 150, 151, 161, 162]])
        rng.shuffle(lens)
        p = check(lens, k)
        assert len(p["classes"]) >= 4


def test_plan_many_blocks():
    """More reads than one planner block (2^15): the per-block histograms and the scan over (class, block)."""
    rng = np.random.default_rng(4)
    lens = rng.choice([20, 150, 150, 150, 300, 1500], size=200_001)
    check(lens, 35)


def test_plan_degenerate_batches():
    assert plan([], 35)["classes"] == [] and plan([], 35)["n_words"] == 0
    p = plan([3, 0, 34], 35)
    assert p["classes"] == [] and (p["pre"] == TOO_SHORT).all()
    offsets = np.array([0, 10, 5], np.uint64)                                      # decreasing offsets are refused
    bases = np.zeros(16, np.uint8)
    b = _lib.Batch(2, bases.ctypes.data_as(_lib.u8p), offsets.ctypes.data_as(_lib.u64p))
    nc, nd, nw = C.c_uint32(), C.c_uint32(), C.c_uint64()
    rc = _lib.lib.cls_debug_plan_batch(35, C.byref(b), None, None, None, None, 0, C.byref(nc), C.byref(nd), C.byref(nw))
    assert rc == _lib.CLS_ERR_INVALID_ARGUMENT


# ---- the just-in-time plan of short-read batches (place_batch.cpp: plan_reads_fast) ---------------------------------
def plan_fast(lens, k, chunk, first_offset=0):
    lens = np.asarray(lens, np.uint64)
    n = len(lens)
    offsets = np.full(n + 1, first_offset, np.uint64)
    offsets[1:] += np.cumsum(lens)
    bases = np.zeros(1, np.uint8)
    b = _lib.Batch(n, bases.ctypes.data_as(_lib.u8p), offsets.ctypes.data_as(_lib.u64p))
    woff, ln, src = np.zeros(n + 1, np.uint32), np.zeros(max(n, 1), np.uint32), np.zeros(max(n, 1), np.uint64)
    mx, npl = C.c_uint32(), C.c_uint64()
    _lib.check(_lib.lib.cls_debug_plan_fast(k, C.byref(b), chunk, woff.ctypes.data_as(_lib.u32p), ln.ctypes.data_as(_lib.u32p),
                                            src.ctypes.data_as(_lib.u64p), C.byref(mx), C.byref(npl)))
    p = npl.value
    return dict(n_planned=p, woff=woff[:p + 1], lens=ln[:p], src=src[:p], max_len=mx.value)


@pytest.mark.parametrize("chunk", [1, 7, 8192, 10_000, 1 << 20])
def test_fast_plan_equals_the_general_plan_on_short_reads(chunk):
    """Every read within 35 .. 162 bases: the device order is the input order, the word offsets are those of the
    general plan laid out in input order, whatever the chunking."""
    rng = np.random.default_rng(chunk)
    for lens in (np.full(30_000, 150), rng.integers(35, 163, 30_000), np.array([35]), np.array([162, 35, 162])):
        f = plan_fast(lens, 35, chunk, first_offset=12345)
        assert f["n_planned"] == len(lens) and f["max_len"] == lens.max()
        assert (f["lens"] == lens).all()
        words = (np.asarray(lens) + 15) // 16
        assert (f["woff"] == np.concatenate([[0], np.cumsum(words)])).all()
        assert (f["src"] == np.concatenate([[0], np.cumsum(lens)[:-1]])).all()
        g = plan(lens, 35)                         # the general plan: the same reads, grouped by length class
        assert sorted(g["perm"].tolist()) == list(range(len(lens))) and g["n_words"] == int(words.sum())


def test_fast_plan_stops_at_the_first_chunk_with_a_read_out_of_range():
    lens = np.full(1000, 150)
    for bad_at, bad_len in ((0, 34), (499, 163), (999, 0), (500, 5000)):
        l2 = lens.copy()
        l2[bad_at] = bad_len
        for chunk in (1, 64, 1000):
            f = plan_fast(l2, 35, chunk)
            assert f["n_planned"] == (bad_at // chunk) * chunk, (bad_at, bad_len, chunk)
    # decreasing offsets are refused like any read out of range (the general plan then reports them)
    offsets = np.array([0, 150, 100, 250], np.uint64)
    b = _lib.Batch(3, np.zeros(1, np.uint8).ctypes.data_as(_lib.u8p), offsets.ctypes.data_as(_lib.u64p))
    npl = C.c_uint64(99)
    _lib.check(_lib.lib.cls_debug_plan_fast(35, C.byref(b), 8, None, None, None, None, C.byref(npl)))
    assert npl.value == 0
    # and the empty batch
    assert plan_fast([], 35, 8)["n_planned"] == 0


def test_fast_plan_survives_arbitrary_offsets():
    """Offsets that decrease, jump by 2^40 or wrap: never a crash, never more reads planned than there are, and what is
    planned obeys the 35 .. 162 rule."""
    rng = np.random.default_rng(99)
    for it in range(300):
        n = int(rng.integers(1, 400))
        lens = rng.integers(35, 163, n).astype(np.int64)
        offsets = np.zeros(n + 1, np.int64)
        offsets[1:] = np.cumsum(lens)
        for _ in range(int(rng.integers(0, 4))):          # damage a few entries
            j = int(rng.integers(0, n + 1))
            offsets[j] = int(rng.choice([0, offsets[j] - 1000, offsets[j] + (1 << 40), -1, offsets[j] + 500]))
        off_u = offsets.astype(np.uint64)
        b = _lib.Batch(n, np.zeros(1, np.uint8).ctypes.data_as(_lib.u8p), off_u.ctypes.data_as(_lib.u64p))
        woff, ln = np.zeros(n + 1, np.uint32), np.zeros(n, np.uint32)
        npl = C.c_uint64()
        chunk = int(rng.choice([1, 3, 64, 1000]))
        _lib.check(_lib.lib.cls_debug_plan_fast(35, C.byref(b), chunk, woff.ctypes.data_as(_lib.u32p), ln.ctypes.data_as(_lib.u32p),
                                                None, None, C.byref(npl)))
        p = npl.value
        assert p <= n and p % chunk == 0 or p == n
        true_len = np.diff(off_u[: p + 1].astype(np.int64)) if p else np.zeros(0, np.int64)
        assert ((true_len >= 35) & (true_len <= 162)).all() and (ln[:p] == true_len).all()
