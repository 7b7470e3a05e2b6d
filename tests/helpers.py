"""Comparison helpers shared by the parity tests, and the host sources the fake-runtime drivers compile."""
import os

from classeq2_b200 import _lib

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "classeq2_b200", "csrc")
# The C ABI's host side without the sharded handle (capi_sharded.cpp) and the FASTQ ingest (fastq_ingest.cpp), which the
# drivers that need them add: compiled with g++ against the fake CUDA runtime of tests/native/fakecuda.
CAPI_HOST_SOURCES = [os.path.join(CSRC, f) for f in ("capi.cpp", "place_batch.cpp", "resident.cpp", "routed.cpp", "index_build.cpp",
                                                     "host_api.cpp", "host_pack.cpp", "host_pool.cpp", "record_writer.cpp")]

UNCL_BY_MESSAGE_PREFIX = {
    "Query sequence SequenceHeader(": _lib.STATUS_UNCL_NO_MATCH,
    "Query sequence has no overlapping kmers": _lib.STATUS_UNCL_NO_ROOT,
    "Insufficient kmers coverage": _lib.STATUS_UNCL_COVERAGE,
    "Tree introspection not possible": _lib.STATUS_UNCL_NO_INTROSPECTION,
}
ERR_BY_MESSAGE = {
    "The sequence does not contain enough kmers.": _lib.STATUS_ERR_TOO_SHORT,
    "The maximum number of iterations has been reached.": _lib.STATUS_ERR_MAX_ITERATIONS,
    "The root node does not have children. This is unexpected.": _lib.STATUS_ERR_ROOT_NO_CHILDREN,
}


def expected_row(e: dict) -> dict:
    """Oracle outcome (dict as stored in colletotrichum_expected.json / made by outcome_of) ->
    the exact values every cls_result array must hold for that query."""
    if "error" in e:
        st = ERR_BY_MESSAGE[e["error"]]
        row = {"status": st, "node_id": 0, "one": 0, "rest": 0}
        if st == _lib.STATUS_ERR_TOO_SHORT:
            row.update(n_query_kmers=0, n_matched=0, n_root_matched=0, iterations=0)
        return row
    row = {"n_query_kmers": e["n_query_kmers"], "n_matched": e["n_matched"],
           "n_root_matched": e["n_root_matched"], "iterations": e["iterations"], "node_id": 0, "one": 0, "rest": 0}
    if e["status"] == "Unclassifiable":
        for prefix, st in UNCL_BY_MESSAGE_PREFIX.items():
            if e["message"].startswith(prefix):
                row["status"] = st
        if row.get("status") == _lib.STATUS_UNCL_COVERAGE:
            assert e["message"] == f"Insufficient kmers coverage: {e['n_root_matched']}"
    elif e["status"] == "IdentityFound":
        row.update(status=_lib.STATUS_IDENTITY_FOUND, node_id=e["clade"], one=e["one"], rest=e["rest"])
    elif e["status"] == "MaxResolutionReached":
        row.update(status=_lib.STATUS_MAX_RESOLUTION, node_id=e["clade"])
    elif e["status"] == "Inconclusive":
        row.update(status=_lib.STATUS_INCONCLUSIVE)
        row.pop("node_id")
    return row


def outcome_of(oracle, header, seq, tree, max_iterations=None, min_match_coverage=None, remove_intersection=None):
    try:
        p = oracle.place_sequence(header, seq, tree, max_iterations, min_match_coverage, remove_intersection)
    except oracle.PlacementError as err:
        return {"error": str(err)}
    return {"status": p.status, "message": p.message, "clade": p.clade, "one": p.one, "rest": p.rest,
            "n_query_kmers": p.n_query_kmers, "n_matched": p.n_matched, "n_root_matched": p.n_root_matched,
            "iterations": p.iterations}


def assert_rows_equal(res, expected_outcomes, headers=None):
    bad = []
    for i, e in enumerate(expected_outcomes):
        want, got = expected_row(e), res.row(i)
        diff = {k: (got[k], v) for k, v in want.items() if got[k] != v}
        if diff:
            bad.append((i, headers[i] if headers else None, diff))
    assert not bad, f"{len(bad)} of {len(expected_outcomes)} queries differ (got, want): {bad[:5]}"


# ---- model-builder cases (host builder vs. device builder vs. the CPU walk through the device steps) ----
def random_build_case(rng, n_internal, k, m, max_len=300, shuffle_nodes=True, letters=b"ACGT", dup_tips=0,
                      internal_tips=0):
    """A random tree (multifurcating, node indices in random order when ``shuffle_nodes``) and one sequence per
    tip: related sequences (so that tips share k-mers), some shorter than k, ``dup_tips`` extra sequences mapped to
    tips that already have one, ``internal_tips`` sequences mapped to internal nodes.  Returns
    ``(FlatModel tree_only, tip_node, bases, offsets)``."""
    import numpy as np
    from classeq2_b200 import _lib
    from classeq2_b200.model import FlatModel
    children = {0: []}
    n = 1
    internal = [0]
    for _ in range(n_internal):
        p = internal[int(rng.integers(len(internal)))]
        children[p].append(n)
        children[n] = []
        internal.append(n)
        n += 1
    for p in list(internal):                      # every internal node gets 1-3 leaves
        for _ in range(int(rng.integers(1, 4))):
            children[p].append(n)
            children[n] = None
            n += 1
    perm = rng.permutation(n) if shuffle_nodes else np.arange(n)
    perm = np.concatenate([[0], perm[perm != 0]])      # node 0 stays the root
    new_of = np.empty(n, np.int64)
    new_of[perm] = np.arange(n)
    node_id = np.zeros(n, np.uint64)
    kind = np.zeros(n, np.uint8)
    lists = [[] for _ in range(n)]
    for old in range(n):
        i = int(new_of[old])
        node_id[i] = 1000 + 7 * old                    # sparse ids
        ch = children[old]
        kind[i] = _lib.KIND_ROOT if old == 0 else (_lib.KIND_LEAF if ch is None else _lib.KIND_NODE)
        lists[i] = [int(new_of[c]) for c in (ch or [])]
    child_off = np.zeros(n + 1, np.uint64)
    child_off[1:] = np.cumsum([len(c) for c in lists])
    child_idx = np.array([c for cl in lists for c in cl], np.uint64)
    tflat = FlatModel(k, m, node_id, kind, child_off, child_idx)
    leaves = [int(new_of[o]) for o in range(n) if children[o] is None]
    inner = [int(new_of[o]) for o in range(n) if children[o] is not None]
    tip_nodes = list(leaves)
    tip_nodes += [leaves[int(rng.integers(len(leaves)))] for _ in range(dup_tips)]
    tip_nodes += [inner[int(rng.integers(len(inner)))] for _ in range(internal_tips)]
    order = rng.permutation(len(tip_nodes))
    tip_nodes = [tip_nodes[int(i)] for i in order]
    lut = np.frombuffer(letters, np.uint8)
    base = lut[rng.integers(0, len(lut), max_len)]
    seqs = []
    for _ in tip_nodes:
        s = base.copy()
        mut = rng.random(max_len) < 0.03
        s[mut] = lut[rng.integers(0, len(lut), int(mut.sum()))]
        ln = int(rng.integers(0, max_len + 1)) if rng.random() < 0.3 else max_len
        start = int(rng.integers(0, max_len - ln + 1))
        seqs.append(s[start:start + ln])
    offsets = np.zeros(len(seqs) + 1, np.uint64)
    offsets[1:] = np.cumsum([len(s) for s in seqs])
    bases = np.concatenate(seqs) if seqs else np.zeros(0, np.uint8)
    if len(bases) == 0:
        bases = np.zeros(1, np.uint8)
    return tflat, np.array(tip_nodes, np.uint64), bases, offsets


def assert_built_equal(a: dict, b: dict):
    """Two ``BuiltModel.arrays()`` results describe the same map: same entries in the same order, same set
    numbering, same ids in every set (the order inside a set is free)."""
    import numpy as np
    for key in ("entry_hash", "entry_bucket", "entry_set"):
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(a["set_off"], b["set_off"])
    so = a["set_off"].astype(np.int64)
    if len(so) > 1 and so[-1] > 0:
        seg = np.repeat(np.arange(len(so) - 1), np.diff(so))
        ka = np.lexsort((a["set_node_ids"], seg))
        kb = np.lexsort((b["set_node_ids"], seg))
        assert np.array_equal(a["set_node_ids"][ka], b["set_node_ids"][kb])


# ---- the reference's own build output (tests/golden/reference_built_model_k12.json.gz) ----
def load_reference_built_model():
    import gzip
    import json
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    return json.loads(gzip.decompress(open(os.path.join(here, "golden", "reference_built_model_k12.json.gz"), "rb").read()))


def reference_built_case(tips):
    """The reference-written k = 12 model as a builder case: (pin, FlatModel tree_only (uncollapsed tree, m = 0),
    tip_node, bases, offsets) with the REFERENCE's pairing (sequence i-1 under header i, last sequence dropped,
    build_database/mod.rs:93-116), and ``want`` = {k-mer hash: node-id set} a BOTH-strand builder must produce:
    the reference wrote the model before it indexed reverse complements (v0.2.3), so the set of k-mer s is
    golden[s] | golden[revcomp(s)]."""
    import os
    import numpy as np
    from classeq2_b200 import build, host_murmur3_h1
    from classeq2_b200.model import FlatModel
    pin = load_reference_built_model()
    here = os.path.dirname(os.path.abspath(__file__))
    nwk = open(os.path.join(here, "golden", pin["name"])).read()
    tree = build.tree_from_newick(nwk, pin["name"], -1e9)           # nothing is collapsed, as in the golden
    clades, node_id, node_kind, child_off, child_idx = FlatModel.tree_arrays(tree.root)
    tflat = FlatModel(pin["k_size"], 0, node_id, node_kind, child_off, child_idx)
    idx = {c.name: i for i, c in enumerate(clades) if c.is_leaf()}
    pairs = [(tips[i][0], tips[i - 1][1]) for i in range(1, len(tips))]   # header 0 gets the empty string: no k-mers
    tip_node = np.array([idx[h] for h, _ in pairs], np.uint64)
    bases = np.frombuffer("".join(s for _, s in pairs).encode(), np.uint8).copy()
    offsets = np.zeros(len(pairs) + 1, np.uint64)
    offsets[1:] = np.cumsum([len(s) for _, s in pairs])
    comp = str.maketrans("ACGT", "TGCA")
    want = {}
    for s, ids in pin["kmers"].items():
        rc = s[::-1].translate(comp)
        both = set(ids) | set(pin["kmers"].get(rc, []))
        want[host_murmur3_h1(s.encode(), 0)] = both
        want[host_murmur3_h1(rc.encode(), 0)] = both
    return pin, tflat, tip_node, bases, offsets, want


def built_as_map(a: dict) -> dict:
    """``BuiltModel.arrays()`` -> {hash: set of node ids} (m = 0: a single bucket)."""
    so, sn = a["set_off"], a["set_node_ids"]
    return {int(h): set(sn[int(so[s]):int(so[s + 1])].tolist()) for h, s in zip(a["entry_hash"].tolist(), a["entry_set"].tolist())}
