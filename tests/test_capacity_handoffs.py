"""Every capacity hand-off of the kb-scale and giant read paths, against the C++ oracle.

Most branches of these paths are taken only when a read outgrows a fixed table:
  * gather_kernel (frag_kernels.cuh): up to kPairCapWide = 256 distinct node-set records go to descend_kernel<8>, up to
    kGListCap = 1024 to descend_wide_kernel, more (or D + 1 > 2(L - 34), or more than kGSetSlots = 1024 distinct table
    slots behind collided filter bits) back to place_kernel<35, true, true>;
  * the short-read path: the four- and two-per-warp groups of descend16_kernel, its one-read-per-warp walk, and the
    kPairCap = 64 overflow into scan_kernel;
  * launch_place_t / launch_giant (kernels.cu): second and later scratch waves.
Real models make reads that reach them rare, so the models here are built to a given number of records per read:
a tree with multifurcations, a pool of upward-closed node sets per template read, and hit i of template t filed under
pool_t[i mod D_t].  Every test first checks on the host that its reads reach the branch it is named for."""
import numpy as np
import pytest

gpu = pytest.mark.gpu

FIELDS = ("status", "node_id", "one", "rest", "n_query_kmers", "n_matched", "n_root_matched")
KNOBS = (dict(), dict(remove_intersection=True), dict(min_match_coverage=0.3, max_iterations=4))
KIND_ROOT, KIND_NODE, KIND_LEAF = 0, 1, 2
PAIR_CAP, PAIR_CAP_WIDE, LIST_CAP = 64, 256, 1024      # kPairCap, kPairCapWide (kernels.cu), kGListCap (frag_kernels.cuh)
_COMP = bytes.maketrans(b"ACGT", b"TGCA")


@pytest.fixture(scope="module")
def cq():
    import classeq2_b200
    return classeq2_b200


def _rand_seq(rng, n):
    return bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)]).decode()


def _rc(s):
    return s.encode().translate(_COMP)[::-1].decode()


def _mutate(rng, s, n_sub):
    b = bytearray(s.encode())
    for i in rng.choice(len(b), n_sub, replace=False):
        b[int(i)] = b"ACGT"[("ACGT".index(chr(b[int(i)])) + int(rng.integers(1, 4))) % 4]
    return b.decode()


# ---- 1. a model builder with an exact number of node-set records per template read ----------------------------------
class _Tree:
    """A random tree whose internal nodes have 2 to 6 children (pre-order, node id == index, root 0)."""

    def __init__(self, rng, n_tips):
        kind, parent, kids = [], [], []
        stack = [(n_tips, -1)]
        while stack:
            n, p = stack.pop()
            v = len(kind)
            kind.append(KIND_LEAF if n == 1 else KIND_NODE)
            parent.append(p)
            kids.append([])
            if p >= 0:
                kids[p].append(v)
            if n > 1:
                f = min(n, 2 if rng.random() < 0.55 else int(rng.integers(3, 7)))
                cuts = np.sort(rng.choice(np.arange(1, n), f - 1, replace=False))
                parts = np.diff(np.concatenate([[0], cuts, [n]]))
                stack.extend((int(x), v) for x in parts[::-1])   # the first part is visited first
        kind[0] = KIND_ROOT
        self.node_kind = np.array(kind, np.uint8)
        self.parent = np.array(parent, np.int64)
        self.kids = kids
        self.child_off = np.zeros(len(kind) + 1, np.uint64)
        self.child_off[1:] = np.cumsum([len(c) for c in kids])
        self.child_idx = np.array([c for cs in kids for c in cs], np.uint64)
        self.internal = np.flatnonzero(self.node_kind != KIND_LEAF)
        self.fanout = np.array([len(c) for c in kids])

    def path(self, v):
        out = []
        while v >= 0:
            out.append(int(v))
            v = int(self.parent[v])
        return out

    def subtree_internal(self, v):
        out, stack = [], [int(v)]
        while stack:
            u = stack.pop()
            if self.node_kind[u] != KIND_LEAF:
                out.append(u)
                stack.extend(self.kids[u])
        return out


def _template_pool(rng, tree, D, rootless_frac, n_hits):
    """D node sets with D distinct records (contents restricted to non-leaf nodes): closures to the root of one to three
    internal nodes, drawn mostly inside one subtree; some carry a leaf child of a member (dropped by the upload).  With
    `rootless_frac`, one record is the record of every rootless set, and about that fraction of the hits lands on it (less
    where the read has too few windows: every set of the pool must keep a hit)."""
    sizes = np.array([len(tree.subtree_internal(v)) for v in tree.internal])
    cands = tree.internal[(sizes >= 30) & (sizes <= 150)]
    inside = tree.subtree_internal(int(rng.choice(cands if len(cands) else tree.internal)))
    n_rooted = D - 1 if rootless_frac else D
    seen, pool = set(), []
    while len(pool) < n_rooted:
        picks = [int(rng.choice(inside)) if rng.random() < 0.85 else int(rng.choice(tree.internal))
                 for _ in range(int(rng.integers(1, 4)))]
        members = sorted({u for v in picks for u in tree.path(v)})
        key = tuple(members)
        if key in seen:
            continue
        seen.add(key)
        if rng.random() < 0.2:
            leaves = [c for m in members for c in tree.kids[m] if tree.node_kind[c] == KIND_LEAF]
            if leaves:
                members.append(int(rng.choice(leaves)))
        pool.append(members)
    if rootless_frac:
        n_rl = max(1, min(n_hits - n_rooted, int(round(rootless_frac * n_rooted / (1 - rootless_frac)))))
        rootless = [tree.path(int(rng.choice(inside)))[:-1] or [int(rng.choice(inside))] for _ in range(n_rl)]
        pool += rootless
        order = rng.permutation(len(pool))
        pool = [pool[i] for i in order]
    return pool


_KEYS = {}


def _bucket_keys(seq, k, m=4):
    """Bucket key of every window (forward strand, then reverse complement): h1 of its m-base prefix."""
    from oracle import cpp_oracle
    out = []
    for s in (seq, _rc(seq)):
        for i in range(len(s) - k + 1):
            p = s[i:i + m]
            if p not in _KEYS:
                _KEYS[p] = cpp_oracle.murmur3_x64_128(p.encode())[0]
            out.append(_KEYS[p])
    return np.array(out, np.uint64)


def build_model(tree, templates, pools, k=35, m=4):
    """FlatModel whose entries are the window hashes of both strands of every template, hit i of template t filed under
    pools[t][i mod len(pools[t])] (a hash already filed by an earlier template keeps its set)."""
    from classeq2_b200.model import FlatModel
    from oracle import cpp_oracle
    sets, eb, eh, es, seen = [], [], [], [], set()
    for seq, pool in zip(templates, pools):
        base = len(sets)
        sets += pool
        hs = cpp_oracle.kmer_hashes(seq.encode(), k)
        keys = _bucket_keys(seq, k, m)
        for i, (h, key) in enumerate(zip(hs.tolist(), keys.tolist())):
            if h in seen:
                continue
            seen.add(h)
            eb.append(key), eh.append(h), es.append(base + i % len(pool))
    set_off = np.zeros(len(sets) + 1, np.uint64)
    set_off[1:] = np.cumsum([len(x) for x in sets])
    n = len(tree.node_kind)
    return FlatModel(k, m, np.arange(n, dtype=np.uint64), tree.node_kind, tree.child_off, tree.child_idx,
                     np.array(eb, np.uint64), np.array(eh, np.uint64), np.array(es, np.uint64), set_off,
                     np.array([v for x in sets for v in x], np.uint64))


_REC = {}


def _records(flat):
    """(entry order by hash, sorted hashes, record id of every set, number of distinct records): a set's record is its
    content restricted to non-leaf nodes, and one shared record for every set without the root (index_build.cpp)."""
    key = id(flat)
    if key not in _REC:
        nonleaf = flat.node_kind != KIND_LEAF
        ids, rec = {}, np.zeros(len(flat.set_off) - 1, np.int64)
        for s in range(len(rec)):
            mem = flat.set_node_ids[int(flat.set_off[s]):int(flat.set_off[s + 1])]
            r = tuple(sorted(int(v) for v in mem if nonleaf[int(v)])) if 0 in mem else ()
            rec[s] = ids.setdefault(r, len(ids))
        order = np.argsort(flat.entry_hash, kind="stable")
        _REC[key] = (flat, order, flat.entry_hash[order], rec, len(ids))
    return _REC[key][1:]


def records_per_read(flat, seq):
    """D of a read as the kernels count it: distinct records among the distinct entries its windows hit, an entry
    counting when its bucket key is the key of any window of the read (kmers_map.rs:55-70)."""
    from oracle import cpp_oracle
    order, sh, rec, _ = _records(flat)
    h = np.unique(cpp_oracle.kmer_hashes(seq.encode(), flat.k_size))
    pos = np.minimum(np.searchsorted(sh, h), len(sh) - 1)
    e = order[pos[sh[pos] == h]]
    e = e[np.isin(flat.entry_bucket[e], _bucket_keys(seq, flat.k_size, flat.m_size))]
    return int(np.unique(rec[flat.entry_set[e].astype(np.int64)]).size)


def _make(seed, spec, k=35, n_tips=500):
    """spec: [(L, D, rootless fraction)] -> (tree, templates, flat).  The same seed gives the same tree, templates and
    pools at every k."""
    rng = np.random.default_rng(seed)
    tree = _Tree(rng, n_tips)
    templates = [_rand_seq(rng, L) for L, _, _ in spec]
    pools = [_template_pool(rng, tree, D, frac, 2 * (L - 34)) for L, D, frac in spec]
    return tree, templates, build_model(tree, templates, pools, k=k)


def _kb_spec(rng):
    """Record counts at and around every threshold of the kb-scale path, three templates each.  Reads up to 2.5 kb for
    D <= 1024 keep the filter collisions of gather_kernel well under kGSetSlots (the `bad` branch has its own test);
    and D = 2(L - 34) - 1, D = 2(L - 34) at L = 291-300, where D + 1 > n_ent decides the hand-back."""
    spec = []
    for D in (1, 32, 33, 255, 256, 257, 600, 1023, 1024, 1025, 2049):
        for j in range(3):
            lo, hi = (max(300, D // 2 + 36), 2500) if D <= LIST_CAP else (max(1100, D // 2 + 36), 4000)
            spec.append((int(rng.integers(lo, hi + 1)), D, (0.0, 0.3, 0.7)[j] if D >= 32 else 0.0))
    for _ in range(11):
        L = int(rng.integers(291, 301))
        spec += [(L, 2 * (L - 34) - 1, 0.0), (L, 2 * (L - 34), 0.0)]
    return spec


def _kb_queries(rng, templates):
    """The templates on both strands, copies with three substitutions, chimeras of two templates; shuffled."""
    qs = []
    for s in templates:
        qs += [s, _rc(s), _mutate(rng, s, 3), _rc(_mutate(rng, s, 3))]
    perm = rng.permutation(len(templates))
    for i, j in enumerate(perm):
        a, b = templates[i], templates[int(j)]
        qs.append(a[:len(a) // 2] + b[len(b) // 2:])
    return [qs[i] for i in rng.permutation(len(qs))]


def test_builder_gives_exact_record_counts():
    """Host only: every template of the builder has exactly the D it was built for, at k = 35 and k = 21; the tree
    multifurcates within the split path's fan-out limit; the node sets are upward closed; some are rootless."""
    rng = np.random.default_rng(1)
    spec = _kb_spec(rng)
    for k in (35, 21):
        tree, templates, flat = _make(11, spec, k=k)
        assert 3 <= tree.fanout[tree.internal].max() <= 768 and len(tree.internal) >= 200
        for (L, D, _), s in zip(spec, templates):
            assert len(s) == L and records_per_read(flat, s) == D, (k, L, D)
        for s in range(len(flat.set_off) - 1):
            mem = set(flat.set_node_ids[int(flat.set_off[s]):int(flat.set_off[s + 1])].tolist())
            if 0 in mem:
                assert all(tree.parent[v] in mem for v in mem if v != 0)
        rootless = np.array([0 not in flat.set_node_ids[int(flat.set_off[s]):int(flat.set_off[s + 1])]
                             for s in range(len(flat.set_off) - 1)])
        assert 0.05 < rootless[flat.entry_set.astype(np.int64)].mean() < 0.5
    # the short-read and single-template builders too
    tree, templates, flat = _make(12, [(150, D, 0.0) for D in (1, 8, 9, 16, 17, 32, 33, 64, 65)])
    assert [records_per_read(flat, s) for s in templates] == [1, 8, 9, 16, 17, 32, 33, 64, 65]


# ---- comparison with the oracle ---------------------------------------------------------------------------------------
def _compare(got, want, kn, lens, tag):
    for f in FIELDS:
        bad = np.flatnonzero(getattr(got, f) != want[f])
        assert bad.size == 0, (tag, f, kn, bad[:5], lens[bad[:5]], getattr(got, f)[bad[:5]], want[f][bad[:5]])
    assert ((got.iterations == want["iterations"]) | (want["status"] == 8)).all(), (tag, kn)


def _check(cq, flat, qs, closed=1, sharded=False, knobs=KNOBS):
    """Index.place_batch, a resident batch (and the routed pipeline on three shards) against the oracle, every field."""
    from oracle import cpp_oracle
    md = cpp_oracle.CppModel.from_flat(flat)
    b, o = cq.make_batch(qs)
    lens = np.diff(o.astype(np.int64))
    ix = cq.Index(flat, device=0)
    info = ix.info()
    assert info["closed_sets"] == closed
    if closed:
        assert info["n_distinct_sets"] == _records(flat)[3]
    sh = None
    if sharded:
        from classeq2_b200.parallel import LocalShardedPlacer
        sh = LocalShardedPlacer(flat, 0, 3)
    out = []
    for kn in knobs:
        want = md.place_batch(b, o, kn.get("max_iterations"), kn.get("min_match_coverage"), kn.get("remove_intersection"))
        rb = ix.upload((b, o))
        rb.place(cq.PlaceParams(**kn))
        _compare(rb.fetch(), want, kn, lens, "resident")
        rb.close()
        _compare(ix.place_batch((b, o), cq.PlaceParams(**kn)), want, kn, lens, "place_batch")
        if sh is not None:
            _compare(sh.place((b, o), cq.PlaceParams(**kn)), want, kn, lens, "sharded")
        out.append(want)
    md.close(), ix.close()
    return out


# ---- 2. record-count boundaries of the kb-scale path -------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("variant", ["closed", "general", "k21"])
def test_kb_record_count_boundaries(cq, variant):
    """One shuffled batch of kb-scale reads at every record-count threshold of gather_kernel: descend_kernel<8>
    (D <= 256), descend_wide_kernel (257-1024; one warp walks many wide reads in turn, so its counters must return to
    zero between reads), the hand-back to place_kernel (D > 1024, or D + 1 > n_ent).  `general`: the same reads in the
    one-CTA place_kernel<35, false, true>; `k21`: place_kernel<0, true, true>, which hands up to 256 records over and
    finishes larger reads itself."""
    rng = np.random.default_rng(2)
    spec = _kb_spec(rng)
    tree, templates, flat = _make(11, spec, k=21 if variant == "k21" else 35)
    qs = _kb_queries(rng, templates)
    assert min(len(q) for q in qs) >= 291 and max(len(q) for q in qs) <= 4000   # one CTA per read, below the giant path
    if variant != "k21":   # the thresholds count k = 35 windows
        D = np.array([records_per_read(flat, q) for q in qs])
        n_ent = 2 * (np.array([len(q) for q in qs]) - 34)
        hand_back_n_ent = (D <= LIST_CAP) & (D + 1 > n_ent)
        regular = ~hand_back_n_ent
        bands = [regular & (D <= PAIR_CAP_WIDE), regular & (D > PAIR_CAP_WIDE) & (D <= LIST_CAP), D > LIST_CAP, hand_back_n_ent]
        assert min(int(x.sum()) for x in bands) >= 20, [int(x.sum()) for x in bands]
    if variant == "general":
        flat = flat.with_general_sets()
    wants = _check(cq, flat, qs, closed=0 if variant == "general" else 1)
    assert (wants[0]["n_root_matched"] < wants[0]["n_matched"]).sum() >= 20   # rootless records take part
    assert min((w["status"] == 3).sum() for w in wants) >= 3                   # the coverage gate decides some reads


# ---- 3. the exact-set overflow of gather_kernel -----------------------------------------------------------------------
@gpu
def test_gather_exact_set_overflow(cq):
    """A model of the windows of ONE 3-4 kb read has under 32 768 entries, so its table has at most 65 536 buckets: the
    filter bit of a hit is its bucket, every slot holds one of this read's hashes, and a bucket that two of them call
    home has both slots hit.  More than 1024 such slots overflow gather_kernel's exact set (`bad`) and the read goes
    back to place_kernel.  In the same batch: shorter and mutated copies and random kb reads (the ordinary paths)."""
    rng = np.random.default_rng(3)
    for t, (L, D) in enumerate([(3000, 40), (3500, 200), (4000, 600)]):
        tree, (tmpl,), flat = _make(30 + t, [(L, D, 0.3)])
        n = len(flat.entry_hash)
        nb = 4
        while nb < n:
            nb <<= 1
        assert n < 32768 and nb <= 65536
        home = np.bincount((flat.entry_hash & np.uint64(nb - 1)).astype(np.int64), minlength=nb)
        assert 2 * int((home >= 2).sum()) > 1024, (L, int((home >= 2).sum()))
        assert records_per_read(flat, tmpl) == D <= LIST_CAP
        qs = [tmpl, _rc(tmpl), _mutate(rng, tmpl, 4), _rc(_mutate(rng, tmpl, 2))]
        for _ in range(8):
            a = int(rng.integers(0, L - 1200))
            c = tmpl[a:a + int(rng.integers(291, 1200))]
            qs += [c, _rc(_mutate(rng, c, 2))]
        qs += [_rand_seq(rng, int(rng.integers(300, 4000))) for _ in range(6)]
        qs = [qs[i] for i in rng.permutation(len(qs))]
        ix = cq.Index(flat, device=0)
        assert ix.info()["n_buckets"] == nb
        ix.close()
        _check(cq, flat, qs)


# ---- 4. short-read hand-off boundaries ----------------------------------------------------------------------------------
@gpu
def test_short_read_record_count_boundaries(cq):
    """150-base reads with D around the groups of descend16_kernel (8, 16), its one-read-per-warp walk (32 records per
    register slot) and the kPairCap = 64 overflow into scan_kernel, interleaved so that groups mix record counts; also through the routed pipeline."""
    rng = np.random.default_rng(4)
    Ds = (1, 8, 9, 16, 17, 32, 33, 64, 65)
    spec = [(150, D, 0.3 if D >= 32 and j == 1 else 0.0) for D in Ds for j in range(4)]
    tree, templates, flat = _make(40, spec)
    qs = []
    for s in templates:
        qs += [s, _rc(s), _mutate(rng, s, 2)]
    perm = rng.permutation(len(templates))
    qs += [templates[i][:75] + templates[int(j)][75:] for i, j in enumerate(perm)]
    qs = [qs[i] for i in rng.permutation(len(qs))]
    D = np.array([records_per_read(flat, q) for q in qs])
    edges = [0, 8, 16, 32, PAIR_CAP, 1 << 30]
    counts = [int(((D > a) & (D <= b)).sum()) for a, b in zip(edges, edges[1:])]
    assert min(counts) >= 12, counts
    _check(cq, flat, qs, sharded=True)


# ---- 5. second and later scratch waves --------------------------------------------------------------------------------
def _wave_batch(rng, flat, templates, n_reads):
    """n_reads reads cycled from a small pool (the templates, their reverse complements, mutated copies), so that the
    oracle places each distinct read once; neighbours come from different templates."""
    pool = []
    for s in templates:
        pool += [s, _rc(s), _mutate(rng, s, 3), _rc(_mutate(rng, s, 5))]
    order = np.concatenate([rng.permutation(len(pool)) for _ in range(n_reads // len(pool) + 1)])[:n_reads]
    arrs = [np.frombuffer(p.encode(), np.uint8) for p in pool]
    bases = np.concatenate([arrs[i] for i in order])
    offsets = np.zeros(n_reads + 1, np.uint64)
    offsets[1:] = np.cumsum([len(pool[i]) for i in order])
    D = np.array([records_per_read(flat, p) for p in pool])
    return pool, order, bases, offsets, D


def _check_waves(cq, flat, pool, order, bases, offsets, launches):
    from oracle import cpp_oracle
    md = cpp_oracle.CppModel.from_flat(flat)
    pb, po = cq.make_batch(pool)
    lens = np.diff(offsets.astype(np.int64))
    ix = cq.Index(flat, device=0)
    rb = ix.upload((bases, offsets))
    for kn in KNOBS:
        want = md.place_batch(pb, po, kn.get("max_iterations"), kn.get("min_match_coverage"), kn.get("remove_intersection"))
        rb.place(cq.PlaceParams(**kn))
        assert ix.timing()["kernel_launches"] == launches, (ix.timing()["kernel_launches"], launches)
        _compare(rb.fetch(), {f: v[order] for f, v in want.items()}, kn, lens, "resident")
    rb.close(), ix.close(), md.close()


@gpu
def test_fragment_path_second_wave(cq):
    """One length class of L = 4000 reads, a few hundred more than one 1 GiB wave of fragment hits holds
    (launch_place_t: 2^30 // (2(L - 34) * 8 + 1) reads): scanfrag, gather, descend_wide and place_kernel run once per
    wave, then descend_kernel<8> once over the class; the wide and handed-back reads sit on both sides of the cut."""
    rng = np.random.default_rng(5)
    L = 4000
    spec = [(L, D, 0.3 if j % 2 else 0.0) for j, D in enumerate([1, 100, 256, 257, 700, 1024, 1025, 1600, 3000] * 3)]
    tree, templates, flat = _make(50, spec)
    wave = (1 << 30) // (2 * (L - 34) * 8 + 1)
    n = wave + 300
    pool, order, bases, offsets, D = _wave_batch(rng, flat, templates, n)
    d = D[order]
    for part in (d[wave - 64:wave], d[wave:wave + 64]):
        assert ((part > PAIR_CAP_WIDE) & (part <= LIST_CAP)).any() and (part > LIST_CAP).any() and (part <= PAIR_CAP_WIDE).any()
    _check_waves(cq, flat, pool, order, bases, offsets, launches=4 * 2 + 1)


def _giant_words(L, fanout, k=35):
    """PlaceGeom::words_per_warp of make_place_geom (kernels.cu)."""
    H = 2 * (L - k + 1)
    t1 = 1 << max(6, int(np.ceil(np.log2(2 * H))))
    t2 = 1 << max(5, int(np.ceil(np.log2(H + 1))))
    str_words = ((L + 15) // 16) * 4 + 4
    pk_words = (((L + 15) // 16) + 4 + 3) & ~3
    w = t1 + 3 * t2 + 2 * str_words + 2 * pk_words + 2 * max(1, fanout) + 2
    return (w + 3) & ~3


@gpu
def test_giant_path_second_wave(cq):
    """L = 5000 reads (tables in global memory), half again as many as one 1 GiB wave of arenas holds: the prepare,
    scan and finish kernels run once per wave.  launch_giant cuts waves by the scratch it is given, and the device
    buffers round every request up by an eighth, so a batch of wave + a few hundred reads would still be ONE wave;
    1.5 waves of 2^30 bytes fall on two waves either way."""
    rng = np.random.default_rng(6)
    L = 5000
    spec = [(L, D, 0.3 if j % 2 else 0.0) for j, D in enumerate([1, 100, 256, 257, 700, 1024, 1025, 1600, 3000] * 3)]
    tree, templates, flat = _make(60, spec)
    ix = cq.Index(flat, device=0)
    fan = ix.info()["max_nonleaf_fanout"]
    ix.close()
    per = 4 * _giant_words(L, fan)
    assert per + 4 * 64 * 4 * 8 > 226 * 1024            # needs_giant
    wave = (1 << 30) // per
    n = wave * 3 // 2
    pool, order, bases, offsets, D = _wave_batch(rng, flat, templates, n)
    _check_waves(cq, flat, pool, order, bases, offsets, launches=3 * 2)
