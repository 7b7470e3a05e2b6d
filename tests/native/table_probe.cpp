// TEST INFRASTRUCTURE.  The k-mer table that cls_index_create uploads (classeq2_b200/csrc/index_build.cpp:
// build_host_index) against the two probe walks the kernels make over it, restated here on the host:
//   walk A (place_kernel / scan_kernel / giant_scan_kernel / shard_probe_kernel): home bucket; on no match follow the
//          chain while the bucket just looked at carries the overflow bit (slot 0, bit 31);
//   walk B (scan2_kernel / scanfrag_kernel): home bucket; on no match follow the chain only if the home bucket's filter
//          (slot 1, bits 24..31; bit (hash >> 40) & 7) has the hash's bit, then while the overflow bit says so.
// Held for random, clustered (long chains) and tiny-valued hashes (equal to the fillers of free slots), one shard or
// three: every kept entry is found by both walks with its own prefix code and its set's record; an entry under a
// bucket key no A/C/G/T prefix produces, an entry of another shard and a hash that is not in the model are missed by
// both; every free slot carries the filler of its bucket; overflow bits sit on full buckets only; a miss whose filter
// bit is clear costs walk B exactly one probe.  Built and run by tests/test_text_fuzz.py (ASan + UBSan).
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "../../include/classeq_b200.h"
#include "../../classeq2_b200/csrc/index_build.hpp"
#include "../../classeq2_b200/csrc/murmur3_host.hpp"

namespace cls {
int set_last_error(int code, const std::string &) { return code; }   // capi.cpp's, stubbed
}
extern "C" uint64_t cls_debug_host_murmur3_x64_128_h1(const uint8_t *d, uint64_t n, uint64_t s) { return cls::murmur3_x64_128_h1(d, n, s); }
extern "C" const char *cls_last_error(void) { return ""; }

using cls::Slot;

static uint64_t rng_state = 0x2545F4914F6CDD1Dull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

struct Found { bool hit; uint64_t slot; uint32_t probes; };

static Found walk_a(const cls::HostIndex &h, uint64_t hash) {
    const uint64_t mask = h.n_buckets - 1;
    uint64_t b = hash & mask;
    for (uint32_t probes = 1;; ++probes) {
        const Slot *s = &h.table[2 * b];
        if (s[0].hash == hash) return {true, 2 * b, probes};
        if (s[1].hash == hash) return {true, 2 * b + 1, probes};
        if (!(s[0].code & cls::kOverflowBit)) return {false, 0, probes};
        if (probes > h.n_buckets) { printf("walk A does not end\n"); exit(1); }
        b = (b + 1) & mask;
    }
}

static Found walk_b(const cls::HostIndex &h, uint64_t hash) {
    const uint64_t mask = h.n_buckets - 1;
    uint64_t b = hash & mask;
    const Slot *s = &h.table[2 * b];
    if (s[0].hash == hash) return {true, 2 * b, 1};
    if (s[1].hash == hash) return {true, 2 * b + 1, 1};
    bool chase = (s[1].code >> (cls::kBloomShift + (uint32_t)((hash >> 40) & 7u))) & 1u;
    uint32_t probes = 1;
    while (chase) {
        b = (b + 1) & mask;
        s = &h.table[2 * b];
        ++probes;
        if (s[0].hash == hash) return {true, 2 * b, probes};
        if (s[1].hash == hash) return {true, 2 * b + 1, probes};
        chase = s[0].code & cls::kOverflowBit;
        if (probes > h.n_buckets) { printf("walk B does not end\n"); exit(1); }
    }
    return {false, 0, probes};
}

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 60;
    long bad = 0, checked = 0, misses = 0, one_probe_misses = 0, chained = 0;
    // a small valid tree: root with two inner nodes, leaves below; sets are root-to-leaf paths or pieces of them
    const uint64_t n_nodes = 7;
    const uint64_t node_id[n_nodes] = {0, 1, 2, 3, 4, 5, 6};
    const uint8_t kind[n_nodes] = {CLS_KIND_ROOT, CLS_KIND_NODE, CLS_KIND_LEAF, CLS_KIND_LEAF, CLS_KIND_NODE, CLS_KIND_LEAF, CLS_KIND_LEAF};
    const uint64_t child_off[n_nodes + 1] = {0, 2, 4, 4, 4, 6, 6, 6};
    const uint64_t child_idx[6] = {1, 4, 2, 3, 5, 6};
    const std::vector<std::vector<uint64_t>> sets = {{0, 1, 2}, {0, 1, 3}, {0, 4, 5}, {0, 4, 6}, {0, 1, 2, 3}, {0, 1, 4, 2, 5}, {1, 2}};
    std::vector<uint64_t> set_off{0}, set_ids;
    for (const auto &s : sets) { set_ids.insert(set_ids.end(), s.begin(), s.end()); set_off.push_back(set_ids.size()); }
    const uint64_t sizes[] = {0, 1, 2, 3, 5, 17, 100, 1000, 3000, 20000};
    for (int r = 0; r < rounds; ++r) {
        const int mode = r % 4;                         // 0 random, 1 clustered low bits, 2 tiny values, 3 one filter bit / one chain
        uint64_t n = sizes[rnd() % 10];
        if (mode == 1 || mode == 3) n = std::min<uint64_t>(n, 1500);   // the builder walks the chains entry by entry
        const uint32_t m_size = (uint32_t)(rnd() % 5), k = 35;
        std::set<uint64_t> used;
        std::vector<uint64_t> eb, eh, es;
        std::vector<uint32_t> want_code;             // expected prefix code, or ~0u for an entry no probe may find
        for (uint64_t e = 0; e < n; ++e) {
            uint64_t hash;
            do {
                switch (mode) {
                    case 0: hash = rnd(); break;
                    case 1: hash = (rnd() << 12) | (rnd() % 3); break;
                    case 2: hash = rnd() % (4 * n + 8); break;
                    default: hash = (rnd() & ~(7ull << 40) & ~0xFFFull) | 5; break;
                }
            } while (!used.insert(hash).second);
            uint8_t pre[4];
            uint32_t code = 0;
            for (uint32_t j = 0; j < m_size; ++j) { pre[j] = (uint8_t)"ACGT"[rnd() & 3]; code |= ((uint32_t)(pre[j] >> 1) & 3u) << (2 * j); }
            uint64_t key = m_size == 0 ? 0 : cls::murmur3_x64_128_h1(pre, m_size, 0);
            if (m_size && rnd() % 13 == 0) { key = rnd() | 1; code = ~0u; }        // a bucket key no prefix produces
            eb.push_back(key); eh.push_back(hash); es.push_back(rnd() % sets.size()); want_code.push_back(code);
        }
        if (eb.empty()) { eb.push_back(0); eh.push_back(0); es.push_back(0); }
        cls_model_view mv{};
        mv.k_size = k; mv.m_size = m_size;
        mv.n_nodes = n_nodes; mv.node_id = node_id; mv.node_kind = kind; mv.child_off = child_off; mv.child_idx = child_idx;
        mv.n_entries = n; mv.entry_bucket = eb.data(); mv.entry_hash = eh.data(); mv.entry_set = es.data();
        mv.n_sets = sets.size(); mv.set_off = set_off.data(); mv.set_node_ids = set_ids.data();
        for (uint32_t shards : {1u, 3u}) {
            const uint32_t shard = (uint32_t)(rnd() % shards);
            cls::HostIndex h;
            std::string err;
            if (cls::build_host_index(&mv, h, err, shard, shards) != CLS_OK) { printf("refused: %s\n", err.c_str()); ++bad; continue; }
            const uint64_t nb = h.n_buckets, mask = nb - 1;
            if (nb < 4 || (nb & mask) || h.table.size() != 2 * nb) { ++bad; continue; }
            // structure: fillers, overflow bits, occupancy
            uint64_t occupied = 0;
            for (uint64_t j = 0; j < nb; ++j) {
                const Slot *s = &h.table[2 * j];
                const bool full = s[0].set_off != cls::kEmpty && s[1].set_off != cls::kEmpty;
                for (int q = 0; q < 2; ++q) {
                    if (s[q].set_off == cls::kEmpty) { if (s[q].hash != ((j + 1) & mask)) ++bad; }
                    else ++occupied;
                }
                if (s[0].set_off == cls::kEmpty && s[1].set_off != cls::kEmpty) ++bad;          // slot 0 fills first
                if ((s[0].code & cls::kOverflowBit) && !full) ++bad;
                if ((s[1].code >> cls::kBloomShift) && !(s[0].code & cls::kOverflowBit)) ++bad;   // a filter bit means an entry moved on
            }
            uint64_t kept = 0;
            std::map<uint64_t, uint32_t> off_of_set;
            for (uint64_t e = 0; e < n; ++e) {
                const bool mine = shards == 1 || (uint32_t)(eh[e] >> 61) % shards == shard;
                const bool reachable = want_code[e] != ~0u;
                const Found a = walk_a(h, eh[e]), b = walk_b(h, eh[e]);
                ++checked;
                if (!(mine && reachable)) { if (a.hit || b.hit) ++bad; continue; }
                ++kept;
                if (!a.hit || !b.hit || a.slot != b.slot) { ++bad; continue; }
                const Slot &s = h.table[a.slot];
                if ((s.code & cls::kCodeMask) != want_code[e] || s.set_off == cls::kEmpty) ++bad;
                auto it = off_of_set.emplace(es[e], s.set_off).first;
                if (it->second != s.set_off) ++bad;                                               // one record per set
                if (a.probes > 1) ++chained;
                if (a.probes != b.probes) ++bad;                                                  // a hit: the same buckets
            }
            if (kept != h.n_entries_kept || occupied != kept) ++bad;
            for (int t = 0; t < 2000; ++t) {                                                       // hashes that are not there
                uint64_t hash;
                switch (t % 4) {
                    case 0: hash = rnd(); break;
                    case 1: hash = rnd() % (4 * n + 8); break;                                     // fillers and their neighbours
                    case 2: hash = n ? eh[rnd() % n] ^ (1ull << (12 + rnd() % 50)) : rnd(); break;  // the home of an entry, another hash
                    default: hash = (rnd() << 12) | (rnd() % 3); break;
                }
                if (used.count(hash)) continue;
                const Found a = walk_a(h, hash), b = walk_b(h, hash);
                ++misses;
                if (a.hit || b.hit || b.probes > a.probes) ++bad;
                const Slot *home = &h.table[2 * (hash & mask)];
                const bool bit = (home[1].code >> (cls::kBloomShift + (uint32_t)((hash >> 40) & 7u))) & 1u;
                if (!bit && b.probes != 1) ++bad;
                if (b.probes == 1) ++one_probe_misses;
            }
        }
    }
    printf("bad=%ld checked=%ld chained_hits=%ld misses=%ld one_probe_misses=%ld\n", bad, checked, chained, misses, one_probe_misses);
    return bad == 0 && checked > 1000 && chained > 0 && misses > 1000 ? 0 : 1;
}
