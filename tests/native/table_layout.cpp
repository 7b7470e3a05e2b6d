// TEST INFRASTRUCTURE.  Where the entries of a given model land in the k-mer table that cls_index_create uploads
// (classeq2_b200/csrc/index_build.cpp: build_host_index), and what the kernels' two probe walks make of a list of
// hashes over it - the host preconditions of tests/test_table_walks.py, which plants long chains, wrap-around and
// filter false positives by hash bits and must know, before any GPU runs, that each planted case really happens.
//
// The walks are those of tests/native/table_probe.cpp:
//   walk A (place_kernel / scan_kernel / giant_scan_kernel / shard_probe_kernel): home bucket; on no match follow the
//          chain while the bucket just looked at carries the overflow bit;
//   walk B (scan2_kernel / scanfrag_kernel): home bucket; on no match follow the chain only if the home bucket's filter
//          has the hash's bit (bits 40..42), then while the overflow bit says so.
// Either walk going round the whole table is an error (exit 2): a GPU walk on such a table would not end.
//
// Input (argv[1]): little-endian uint64 words
//   k, m, n_nodes, n_entries, n_sets, n_probes, shard, n_shards,
//   node_id[n_nodes], node_kind[n_nodes], child_off[n_nodes + 1], child_idx[child_off[n_nodes]],
//   entry_bucket[n_entries], entry_hash[n_entries], entry_set[n_entries], set_off[n_sets + 1],
//   set_node_ids[set_off[n_sets]], probe_hash[n_probes].
// Output (stdout): "n_buckets <nb> kept <n>", then one line per probe hash
//   "<hit> <bucket> <wrapped> <probes of walk A> <probes of walk B>"
// where bucket is the bucket that holds the hash (-1 on a miss) and wrapped says that walk A went past the last bucket
// into bucket 0 before it ended.  Both walks must agree on hit and slot (exit 3 otherwise).
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/classeq_b200.h"
#include "../../classeq2_b200/csrc/index_build.hpp"
#include "../../classeq2_b200/csrc/murmur3_host.hpp"

namespace cls {
int set_last_error(int code, const std::string &) { return code; }   // capi.cu's, stubbed
}
extern "C" uint64_t cls_debug_host_murmur3_x64_128_h1(const uint8_t *d, uint64_t n, uint64_t s) { return cls::murmur3_x64_128_h1(d, n, s); }
extern "C" const char *cls_last_error(void) { return ""; }

using cls::Slot;

struct Found { bool hit; uint64_t slot; uint64_t probes; bool wrapped; };

static Found walk_a(const cls::HostIndex &h, uint64_t hash) {
    const uint64_t mask = h.n_buckets - 1;
    uint64_t b = hash & mask;
    bool wrapped = false;
    for (uint64_t probes = 1;; ++probes) {
        const Slot *s = &h.table[2 * b];
        if (s[0].hash == hash) return {true, 2 * b, probes, wrapped};
        if (s[1].hash == hash) return {true, 2 * b + 1, probes, wrapped};
        if (!(s[0].code & cls::kOverflowBit)) return {false, 0, probes, wrapped};
        if (probes > h.n_buckets) { printf("walk A does not end\n"); exit(2); }
        b = (b + 1) & mask;
        wrapped |= b == 0;
    }
}

static Found walk_b(const cls::HostIndex &h, uint64_t hash) {
    const uint64_t mask = h.n_buckets - 1;
    uint64_t b = hash & mask;
    const Slot *s = &h.table[2 * b];
    if (s[0].hash == hash) return {true, 2 * b, 1, false};
    if (s[1].hash == hash) return {true, 2 * b + 1, 1, false};
    bool chase = (s[1].code >> (cls::kBloomShift + (uint32_t)((hash >> 40) & 7u))) & 1u;
    uint64_t probes = 1;
    while (chase) {
        b = (b + 1) & mask;
        s = &h.table[2 * b];
        ++probes;
        if (s[0].hash == hash) return {true, 2 * b, probes, false};
        if (s[1].hash == hash) return {true, 2 * b + 1, probes, false};
        chase = s[0].code & cls::kOverflowBit;
        if (probes > h.n_buckets) { printf("walk B does not end\n"); exit(2); }
    }
    return {false, 0, probes, false};
}

int main(int argc, char **argv) {
    if (argc != 2) { fprintf(stderr, "usage: table_layout <model file>\n"); return 1; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", argv[1]); return 1; }
    std::vector<uint64_t> w;
    uint64_t buf[4096];
    for (size_t n; (n = fread(buf, 8, 4096, f)) > 0;) w.insert(w.end(), buf, buf + n);
    fclose(f);
    size_t at = 0;
    auto take = [&](uint64_t n) -> const uint64_t * {
        if (at + n > w.size()) { fprintf(stderr, "model file is short\n"); exit(1); }
        const uint64_t *p = w.data() + at;
        at += n;
        return p;
    };
    const uint64_t *hdr = take(8);
    const uint64_t n_nodes = hdr[2], n_entries = hdr[3], n_sets = hdr[4], n_probes = hdr[5];
    const uint64_t *node_id = take(n_nodes), *kind64 = take(n_nodes), *child_off = take(n_nodes + 1);
    const uint64_t *child_idx = take(child_off[n_nodes]);
    const uint64_t *eb = take(n_entries), *eh = take(n_entries), *es = take(n_entries);
    const uint64_t *set_off = take(n_sets + 1);
    const uint64_t *set_ids = take(set_off[n_sets]);
    const uint64_t *probe = take(n_probes);
    if (at != w.size()) { fprintf(stderr, "model file is long\n"); return 1; }
    std::vector<uint8_t> kind(kind64, kind64 + n_nodes);

    cls_model_view mv{};
    mv.k_size = (uint32_t)hdr[0]; mv.m_size = (uint32_t)hdr[1];
    mv.n_nodes = n_nodes; mv.node_id = node_id; mv.node_kind = kind.data(); mv.child_off = child_off; mv.child_idx = child_idx;
    mv.n_entries = n_entries; mv.entry_bucket = eb; mv.entry_hash = eh; mv.entry_set = es;
    mv.n_sets = n_sets; mv.set_off = set_off; mv.set_node_ids = set_ids;
    cls::HostIndex h;
    std::string err;
    if (cls::build_host_index(&mv, h, err, (uint32_t)hdr[6], (uint32_t)hdr[7]) != CLS_OK) { printf("refused: %s\n", err.c_str()); return 1; }
    printf("n_buckets %llu kept %llu\n", (unsigned long long)h.n_buckets, (unsigned long long)h.n_entries_kept);
    std::string out;
    char line[96];
    for (uint64_t i = 0; i < n_probes; ++i) {
        const Found a = walk_a(h, probe[i]), b = walk_b(h, probe[i]);
        if (a.hit != b.hit || (a.hit && a.slot != b.slot)) { printf("the walks disagree on hash %llu\n", (unsigned long long)probe[i]); return 3; }
        snprintf(line, sizeof line, "%d %lld %d %llu %llu\n", a.hit ? 1 : 0, a.hit ? (long long)(a.slot / 2) : -1LL, a.wrapped ? 1 : 0,
                 (unsigned long long)a.probes, (unsigned long long)b.probes);
        out += line;
    }
    fwrite(out.data(), 1, out.size(), stdout);
    return 0;
}
