"""Every device walk of the k-mer table against the C++ oracle, on tables planted with long chains, wrap-around, filter
false positives and shared homes, and on tables larger than L2.

Six kernels probe the table with one of two walks (DESIGN.md section 3): walk B (scan2_kernel, scanfrag_kernel) chases
the overflow chain only if the home bucket's filter has the hash's bit (bits 40..42); walk A (place_kernel,
scan_kernel, giant_scan_kernel, shard_probe_kernel) chases while the overflow bit is set.  Models built from real
k-mers leave long chains, wrap-around and filter false positives to chance, so the models here start from a closed
synthetic model and its reads and add DECOYS: entries whose hash no query window produces, with chosen hash bits
(random elsewhere), a valid bucket key, an existing root-containing node set and the target's top three bits (so a
decoy lands in its target's shard for any shard count).  The builder inserts entries in array order, so the decoys go
first and the model's entries end up down the chains:
  (a) long chains to a hit: D in {2, 3, 8, 31, 64, 200} decoys with the low 30 bits of a hit window;
  (b) wrap-around: a run of decoys whose low 30 bits are all ones (home: the last bucket), and chains that push the
      hits with the largest homes past the end of the table;
  (c) filter false positives: decoys with the low 30 bits and bits 40..42 of a window that is not in the model (walk B
      chases to a miss), and the same with bits 40..42 different (walk B stops after one probe, walk A chases);
  (d) two distinct hits of one read behind one home bucket, both down the chain (de-duplication keys on the slot at the
      end of the chase), and tandem repeats of a chained k-mer (the repeats of one chained slot count once).
The cases are defined by hash bits, not by slot positions, so they stay adversarial under another table layout.  What
does depend on today's layout - that each case really happens - is checked first on the host by
tests/native/table_layout.cpp (build_host_index and the two walks restated, under ASan + UBSan), before any GPU runs."""
import functools
import os
import shutil
import subprocess

import numpy as np
import pytest

gpu = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "classeq2_b200", "csrc")
FIELDS = ("status", "node_id", "one", "rest", "n_query_kmers", "n_matched", "n_root_matched")
KNOBS = (dict(), dict(remove_intersection=True), dict(min_match_coverage=0.3, max_iterations=4))
LOW30 = np.uint64((1 << 30) - 1)
TOP3 = np.uint64(7 << 61)
BITS40 = np.uint64(7 << 40)
CHAIN_D = (2, 3, 8, 31, 64, 200)
N_CASE = 8          # the least number of planted instances of every case the host preconditions accept
_COMP = bytes.maketrans(b"ACGT", b"TGCA")


@pytest.fixture(scope="module")
def cq():
    import classeq2_b200
    return classeq2_b200


def _rc(s):
    return s.translate(_COMP)[::-1]


def _next_pow2(n):
    nb = 4
    while nb < n:
        nb <<= 1
    return nb


# ---- the host driver --------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _driver(out_dir):
    exe = os.path.join(out_dir, "table_layout")
    r = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-pthread",
                        os.path.join(HERE, "native", "table_layout.cpp"), os.path.join(CSRC, "index_build.cpp"),
                        os.path.join(CSRC, "host_api.cpp"), os.path.join(CSRC, "host_pool.cpp"), "-o", exe], capture_output=True, text=True)
    assert "undefined reference" not in r.stderr and "error:" not in r.stderr, r.stderr[-2000:]   # a real build error is a failure
    if r.returncode != 0:
        pytest.skip(f"cannot build with the sanitizers here: {r.stderr[-300:]}")
    return exe


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("needs g++")
    return _driver(str(tmp_path_factory.mktemp("table_layout")))


def layout(exe, flat, probes, shard=0, n_shards=1):
    """(n_buckets, kept, rows): rows[i] = (hit, bucket, wrapped, probes of walk A, probes of walk B) of probes[i]."""
    import tempfile
    probes = np.ascontiguousarray(probes, np.uint64)
    n = len(flat.node_id)
    head = np.array([flat.k_size, flat.m_size, n, len(flat.entry_hash), len(flat.set_off) - 1, len(probes), shard, n_shards], np.uint64)
    parts = [head, flat.node_id, flat.node_kind.astype(np.uint64), flat.child_off, flat.child_idx, flat.entry_bucket, flat.entry_hash,
             flat.entry_set, flat.set_off, flat.set_node_ids, probes]
    with tempfile.NamedTemporaryFile(suffix=".bin") as f:
        f.write(b"".join(np.ascontiguousarray(p, np.uint64).tobytes() for p in parts))
        f.flush()
        r = subprocess.run([exe, f.name], capture_output=True, text=True, timeout=1200)
    assert "ERROR: AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[:3000]
    assert r.returncode == 0, (r.returncode, r.stdout[:500], r.stderr[-500:])   # 2: a walk that does not end
    lines = r.stdout.split("\n", 1)
    _, nb, _, kept = lines[0].split()
    rows = np.array(lines[1].split(), np.int64).reshape(-1, 5) if len(probes) else np.zeros((0, 5), np.int64)
    return int(nb), int(kept), rows


# ---- planted models ---------------------------------------------------------------------------------------------------
class Planted:
    """A synthetic model with decoys in front of its entries, its reads and what was planted where."""

    def __init__(self, sm, reads, seed, n_random=0, wrap_run=64, foreign=False):
        from classeq2_b200.model import FlatModel
        from oracle import cpp_oracle
        f0 = sm.flat
        rng = np.random.default_rng(seed)
        k = f0.k_size
        self.k, self.reads = k, list(reads)
        self.read_hashes = [cpp_oracle.kmer_hashes(s.encode(), k) for s in self.reads]
        qh = np.unique(np.concatenate(self.read_hashes))
        model_h = np.unique(f0.entry_hash)
        hit = qh[np.isin(qh, model_h)]
        miss = qh[~np.isin(qh, model_h)]
        used = set()

        def pick(pool, n):
            pool = np.array([h for h in rng.permutation(pool).tolist() if h not in used][:n], np.uint64)
            used.update(pool.tolist())
            assert len(pool) == n, "too few windows to plant on"
            return pool

        hashes, self.plan = [], {}

        def decoys(like, n, mask, flip40=0):
            like = np.uint64(int(like) ^ (flip40 << 40))
            r = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
            hashes.append((r & ~(mask | TOP3)) | (like & (mask | TOP3)))

        # (a) long chains to a hit
        for D in CHAIN_D:
            for t in pick(hit, 4):
                decoys(t, D, LOW30)
                self.plan.setdefault("chain", []).append((int(t), D))
        # (c) filter false positives: the window's bits 40..42, then other ones
        for t in pick(miss, 3 * N_CASE):
            decoys(t, 20, LOW30 | BITS40)
        for t in pick(miss, 3 * N_CASE):
            decoys(t, 12, LOW30 | BITS40, flip40=int(rng.integers(1, 8)))
        # (b) the run whose home is the last bucket
        decoys(np.uint64(LOW30) | (rng.integers(0, 8, dtype=np.uint64) << np.uint64(61)), wrap_run, LOW30)
        n_planned = len(f0.entry_hash) + sum(len(h) for h in hashes) + n_random
        # room for the decoys of (d) and (b), which depend on the table size: checked once they are all there
        nb = self.nb = _next_pow2(n_planned + 256 + 16 * N_CASE)
        mask = np.uint64(nb - 1)
        # (d) two distinct hits of one read with one home: both go down the chain behind 4 decoys of the first one's bits
        pairs = []
        for rh in self.read_hashes:
            h = np.unique(rh[np.isin(rh, hit)])
            h = h[[x not in used for x in h.tolist()]]
            home = h & mask
            order = np.argsort(home, kind="stable")
            same = np.flatnonzero(home[order][1:] == home[order][:-1])
            if len(same):
                a, b = int(h[order][same[0]]), int(h[order][same[0] + 1])
                used.update((a, b))
                pairs.append((a, b))
                decoys(a, 4, LOW30)
            if len(pairs) == 6 * N_CASE:
                break
        self.plan["pairs"] = pairs
        # (b) the hits with the largest homes, each pushed past the last bucket by its own chain
        free = np.array([x for x in hit.tolist() if x not in used], np.uint64)
        last = free[np.argsort(free & mask)[::-1][:2 * N_CASE]]
        used.update(last.tolist())
        for t in last:
            decoys(t, 2 * (nb - 1 - int(t & mask)) + 2, LOW30)
        self.plan["wrap"] = last.tolist()
        if n_random:
            r = rng.integers(0, 1 << 63, n_random, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n_random, dtype=np.uint64)
            hashes.append(r)
        dh = np.concatenate(hashes)
        assert len(np.unique(dh)) == len(dh) and not np.isin(dh, qh).any() and not np.isin(dh, model_h).any()
        self.n_decoys = len(dh)
        keys = np.unique(f0.entry_bucket)
        eb = np.concatenate([keys[rng.integers(0, len(keys), len(dh))], f0.entry_bucket])
        if foreign:   # keys of other entries for 1/40 of the model's own entries: all of them keys of real ACGT prefixes
            idx = len(dh) + rng.choice(len(f0.entry_bucket), len(f0.entry_bucket) // 40, replace=False)
            eb[idx] = eb[rng.permutation(idx)]
        es = np.concatenate([f0.entry_set[rng.integers(0, len(f0.entry_set), len(dh))], f0.entry_set])
        self.flat = FlatModel(k, f0.m_size, f0.node_id, f0.node_kind, f0.child_off, f0.child_idx, eb,
                              np.concatenate([dh, f0.entry_hash]), es, f0.set_off, f0.set_node_ids)
        assert _next_pow2(len(self.flat.entry_hash)) == nb, (len(self.flat.entry_hash), nb)

def _reads(sm, lens, seed):
    from classeq2_b200 import synth
    bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, len(lens), np.asarray(lens), seed)
    return [bases[int(offsets[i]):int(offsets[i + 1])].tobytes().decode() for i in range(len(lens))]


def _tandem(rng, sm_reads, read_hashes, targets, k):
    """Reads of four tandem copies of a chained k-mer between random flanks (at most 162 bases)."""
    out = []
    for t, _ in targets:
        for s, rh in zip(sm_reads, read_hashes):
            w = np.flatnonzero(rh == np.uint64(t))
            if len(w):
                W = len(s) - k + 1
                i = int(w[0])
                kmer = s[i:i + k] if i < W else _rc(s)[i - W:i - W + k]
                fl = "".join("ACGT"[x] for x in rng.integers(0, 4, 162 - 4 * k))
                cut = int(rng.integers(0, len(fl) + 1))
                out.append(fl[:cut] + kmer * 4 + fl[cut:])
                break
    return out


@functools.lru_cache(maxsize=None)
def short_model(n_random=0, foreign=False):
    """16 tips with 1.5 kb references: 1 600 reads of 35-162 bases, 600 of 163-290, tandem repeats of chained k-mers;
    kb-scale reads are drawn separately (kb_reads).  `foreign` moves bucket keys only; `n_random` keeps
    the decoys of (a) and (c), and plants (b) and (d) for its larger table."""
    from classeq2_b200 import synth
    from oracle import cpp_oracle
    sm = synth.make_model(16, 1500, 4101)
    rng = np.random.default_rng(4102)
    reads = _reads(sm, rng.integers(35, 163, 1600), 4103) + _reads(sm, rng.integers(163, 291, 600), 4104)
    p = Planted(sm, reads, 4105, n_random=n_random, foreign=foreign)
    p.tandem = _tandem(rng, reads, p.read_hashes, [c for c in p.plan["chain"] if c[1] >= 31], 35)
    p.reads += p.tandem
    p.read_hashes += [cpp_oracle.kmer_hashes(s.encode(), 35) for s in p.tandem]
    p.sm = sm
    return p


@functools.lru_cache(maxsize=None)
def giant_model():
    """4 tips with 12 kb references, 24 reads of 5-9 kb."""
    from classeq2_b200 import synth
    sm = synth.make_model(4, 12000, 4201)
    rng = np.random.default_rng(4202)
    p = Planted(sm, _reads(sm, rng.integers(5000, 9001, 24), 4203), 4204)
    p.sm = sm
    return p


@functools.lru_cache(maxsize=None)
def k21_model():
    """k = 21, m = 3: 600 reads of 35-290 bases and 60 kb-scale ones."""
    from classeq2_b200 import synth
    sm = synth.make_model(16, 1500, 4301, k_size=21, m_size=3)
    rng = np.random.default_rng(4302)
    lens = np.concatenate([rng.integers(35, 291, 600), rng.integers(291, 1500, 60)])
    p = Planted(sm, _reads(sm, lens, 4303), 4304)
    p.sm = sm
    return p


def kb_reads(p, seed):
    """Skewed kb-scale lengths (config 4's mix above 290 bases) and a few long ones past the references' end."""
    from classeq2_b200 import synth
    lens = synth.skewed_lengths(400, seed)
    lens = np.concatenate([lens[lens >= 291][:150], np.array([291, 1500, 2600, 4100])])
    return _reads(p.sm, lens, seed + 1)


# ---- host preconditions -----------------------------------------------------------------------------------------------
def walk_stats(exe, p, shard=0, n_shards=1):
    """What the planted cases amount to in today's table (the probes: every window of every read that the shard owns)."""
    qh = np.unique(np.concatenate(p.read_hashes))
    if n_shards > 1:
        qh = qh[(qh >> np.uint64(61)) % np.uint64(n_shards) == shard]
    nb, kept, rows = layout(exe, p.flat, qh, shard, n_shards)
    hit = rows[:, 0] == 1
    home = (qh & np.uint64(nb - 1)).astype(np.int64)
    dist = np.where(hit, (rows[:, 1] - home) % nb, -1)
    pa, pb = rows[:, 3], rows[:, 4]
    where = dict(zip(qh.tolist(), range(len(qh))))
    pairs = 0
    for a, b in p.plan["pairs"]:
        ia, ib = where.get(a), where.get(b)
        if ia is not None and ib is not None and home[ia] == home[ib] and dist[ia] > 0 and dist[ib] > 0:
            pairs += 1
    return dict(nb=nb, kept=kept, far=int((dist >= 16).sum()), longest=int(dist.max()), wrapped=int((hit & (rows[:, 2] == 1)).sum()),
                b_long_miss=int((~hit & (pb >= 8)).sum()), b_short_miss=int((~hit & (pb == 1) & (pa >= 4)).sum()), pairs=pairs)


def _assert_cases(st, nb, pairs=True):
    assert st["nb"] == nb, st
    assert st["far"] >= N_CASE and st["longest"] >= 64, st
    assert st["wrapped"] >= N_CASE, st
    assert st["b_long_miss"] >= N_CASE and st["b_short_miss"] >= N_CASE, st
    if pairs:
        assert st["pairs"] >= N_CASE, st


@pytest.mark.parametrize("which", ["short", "giant", "k21"])
def test_planted_cases_happen(driver, which):
    """Host only: n_buckets is the designed one, every walk ends, and every planted case is there - hits at distance
    >= 16 (the longest >= 64), wrapped hits, misses that walk B chases for >= 8 probes, misses where walk B stops after
    one probe while walk A chases >= 4, pairs of distinct hits of one read behind one home, both chained."""
    p = {"short": short_model, "giant": giant_model, "k21": k21_model}[which]()
    _assert_cases(walk_stats(driver, p), p.nb)
    if which == "short":
        assert len(p.tandem) >= N_CASE


@pytest.mark.parametrize("n_shards", [2, 3])
def test_planted_cases_happen_per_shard(driver, n_shards):
    """Host only: the same on every shard of a hash-sharded index (a decoy carries its target's top three bits)."""
    p = short_model()
    tot = dict.fromkeys(("far", "wrapped", "b_long_miss", "b_short_miss", "pairs"), 0)
    for s in range(n_shards):
        st = walk_stats(driver, p, s, n_shards)
        assert st["far"] >= 1 and st["b_long_miss"] >= 1 and st["b_short_miss"] >= 1, (s, st)
        for key in tot:
            tot[key] += st[key]
    assert min(tot.values()) >= N_CASE, tot


def test_planted_cases_happen_beyond_l2(driver):
    """Host only: with 2.2 M random decoys the table has 2^22 buckets (128 MiB), and the planted cases are still there."""
    p = short_model(2_200_000)
    assert p.nb == 1 << 22
    _assert_cases(walk_stats(driver, p), 1 << 22, pairs=False)


# ---- GPU legs ---------------------------------------------------------------------------------------------------------
def _compare(got, want, kn, tag):
    for f in FIELDS:
        bad = np.flatnonzero(getattr(got, f) != want[f])
        assert bad.size == 0, (tag, f, kn, bad[:5], getattr(got, f)[bad[:5]], want[f][bad[:5]])
    assert ((got.iterations == want["iterations"]) | (want["status"] == 8)).all(), (tag, kn)


def _check(cq, flat, reads, nb=None, closed=1, resident=True, index=None, knobs=KNOBS):
    """Index.place_batch (and a resident batch) against the C++ oracle, every field, under every knob set."""
    from oracle import cpp_oracle
    md = cpp_oracle.CppModel.from_flat(flat)
    b, o = cq.make_batch(reads)
    ix = index or cq.Index(flat, device=0)
    info = ix.info()
    assert info["closed_sets"] == closed
    if nb is not None:
        assert info["n_buckets"] == nb
    wants = []
    for kn in knobs:
        want = md.place_batch(b, o, kn.get("max_iterations"), kn.get("min_match_coverage"), kn.get("remove_intersection"))
        _compare(ix.place_batch((b, o), cq.PlaceParams(**kn)), want, kn, "place_batch")
        if resident:
            rb = ix.upload((b, o))
            rb.place(cq.PlaceParams(**kn))
            _compare(rb.fetch(), want, kn, "resident")
            rb.close()
        wants.append(want)
    md.close()
    if index is None:
        ix.close()
    return wants


def _short(p):
    return [s for s in p.reads if len(s) <= 162]


def _medium(p):
    return [s for s in p.reads if len(s) > 162]


@gpu
@pytest.mark.parametrize("band", ["35-162", "163-290"])
def test_short_reads(cq, band):
    """scan2_kernel<4, 4> + descend16 (35-162 bases) and scan2_kernel<8, 4> (163-290), each in its own batch."""
    p = short_model()
    reads = _short(p) if band == "35-162" else _medium(p)
    wants = _check(cq, p.flat, reads, p.nb)
    assert (wants[0]["n_matched"] > 0).mean() > 0.8


@gpu
def test_general_sets(cq):
    """The same model on the general node-set records: scan_kernel<false>."""
    p = short_model()
    flat = p.flat.with_general_sets()
    _check(cq, flat, _short(p), p.nb, closed=0, resident=False)
    _check(cq, flat, _medium(p), p.nb, closed=0, resident=False)


@gpu
@pytest.mark.parametrize("foreign", [False, True])
def test_kb_reads(cq, foreign):
    """scanfrag_kernel (walk B) on 291-4 100 base reads; `foreign`: 1/40 of the model's entries under the bucket key of
    another prefix, so that reads go back to place_kernel<35, *, true> (walk A)."""
    from oracle import cpp_oracle
    p = short_model(foreign=foreign)
    reads = kb_reads(p, 4106)
    if foreign:
        b, o = cq.make_batch(reads)
        moved = cpp_oracle.CppModel.from_flat(p.flat).place_batch(b, o)["n_matched"]
        assert (moved != cpp_oracle.CppModel.from_flat(short_model().flat).place_batch(b, o)["n_matched"]).any()   # the moved keys count
    _check(cq, p.flat, reads, p.nb)


@gpu
def test_giant_reads(cq):
    """giant_scan_kernel (walk A) on 5-9 kb reads of a planted model with 12 kb references."""
    p = giant_model()
    _check(cq, p.flat, p.reads, p.nb)


@gpu
def test_other_k(cq):
    """k = 21, m = 3: place_kernel<0> in warp mode (short reads) and CTA mode (kb-scale reads)."""
    p = k21_model()
    _check(cq, p.flat, [s for s in p.reads if len(s) <= 290], p.nb)
    _check(cq, p.flat, [s for s in p.reads if len(s) > 290], p.nb, resident=False)


@gpu
@pytest.mark.parametrize("n_shards", [2, 3])
def test_sharded_handle(cq, n_shards):
    """shard_probe_kernel (walk A) on every shard of a hash-sharded handle, reads of at most 161 bases."""
    p = short_model()
    reads = [s for s in p.reads if len(s) <= 161]
    ix = cq.Index(p.flat, sharded_devices=[0] * n_shards)
    _check(cq, p.flat, reads, index=ix)
    ix.close()


@gpu
def test_node_counts_on_chained_reads(cq, oracle):
    """cls_debug_node_counts against the Python oracle's trace on reads whose hits sit at the end of long chains."""
    from test_gpu_parity import oracle_tree_from_flat
    p = short_model()
    tree = oracle_tree_from_flat(oracle, p.flat)
    far = {t for t, D in p.plan["chain"] if D >= 31} | set(p.plan["wrap"])
    picked = [s for s, rh in zip(p.reads, p.read_hashes) if len(s) <= 162 and far & set(rh.tolist())][:8] + p.tandem[:4]
    assert len(picked) >= 8
    ix = cq.Index(p.flat, device=0)
    for s in picked:
        trace = []
        try:
            oracle.place_sequence("q", s, tree, trace=trace)
        except oracle.PlacementError:
            pass
        trace.sort(key=lambda r: (r["level"], r["child_id"]))
        rows, _ = ix.debug_node_counts(s)
        assert rows == trace, (s, rows[:3], trace[:3])
    ix.close()


@gpu
def test_table_beyond_l2(cq):
    """The short-read leg on the planted model plus 2.2 M random decoys: 2^22 buckets, a 128 MiB table, more than the
    96 MiB up to which the launcher takes scan2_kernel<4, 4>: scan2_kernel<4, 5> runs."""
    p = short_model(2_200_000)
    ix = cq.Index(p.flat, device=0)
    assert ix.info()["table_bytes"] > 96 << 20
    _check(cq, p.flat, _short(p), 1 << 22, index=ix)
    ix.close()


@gpu
def test_scale_device_built_model(cq):
    """An unplanted model built on the device, past both size limits of the other tests: 65 600 tips (65 599 non-leaf
    nodes, more than 65 536) with references of 45-90 bases give 2.63 M entries, 2^22 buckets and a 128 MiB table
    (scan2_kernel<4, 5>).  200 000 reads of 150 bases and 2 000 of config 4's skewed kb-scale lengths, every read against
    the C++ oracle.  The sizes were measured with the host builder; the model is built in seconds on the device, and
    the oracle takes most of the test's time."""
    from classeq2_b200 import synth
    from oracle import cpp_oracle
    sm = synth.make_model(65_600, (45, 90), 4401, device=0)
    ix = cq.Index(sm.flat, device=0)
    info = ix.info()
    assert info["n_nonleaf_nodes"] > 65_536 and info["table_bytes"] > 96 << 20, info
    md = cpp_oracle.CppModel.from_flat(sm.flat)
    for lens, seed in ((np.full(200_000, 150), 4402), (synth.skewed_lengths(2_000, 4403), 4404)):
        bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, len(lens), lens, seed)
        want = md.place_batch(bases, offsets)
        got = ix.place_batch((bases, offsets))
        _compare(got, want, {}, f"max length {lens.max()}")
        assert (want["n_matched"] > 0).mean() > 0.5
    md.close(), ix.close()
