// TEST INFRASTRUCTURE.  What build_host_index (classeq2_b200/csrc/index_build.cpp) hands the descent kernels for a
// "closed" model - non-leaf nodes renumbered in DFS pre-order (q), subtree intervals, depths, the Euler tour + sparse
// table behind lca_depth_node (kernels.cu), and one TERMINAL LIST per distinct node set - against the tree and the sets
// themselves, on random trees (dense and sparse Clade ids, inner nodes without children, leaves among the members):
//   * the non-leaf children of q tile [q + 1, q_end[q]) in order; depth and child_count agree with the tree;
//   * lca_depth_node(u, v), restated here with the kernel's index arithmetic, is the lowest common ancestor (and its
//     depth) of every pair tried;
//   * a set that holds the root: terminals ascending, the copy of the last one in word 1, and "some terminal lies in
//     [x, q_end[x])" is exactly "x is a member" for EVERY non-leaf node x (device_types.hpp); a set without the root
//     carries an empty list;
//   * the same tree with arbitrary (not upward closed) sets: the mini-tree records, decoded back, hold exactly the sets.
// Built and run by tests/test_text_fuzz.py (ASan + UBSan).
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

static uint64_t rng_state = 0xD1B54A32D192ED03ull;
static uint64_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return rng_state; }

// kernels.cu: lca_depth_node
static uint64_t lca_depth_node(const cls::HostIndex &h, uint32_t u, uint32_t v) {
    const uint32_t fu = h.qinfo[u].euler_first, fv = h.qinfo[v].euler_first;
    const uint32_t j = 31u - (uint32_t)__builtin_clz(fv - fu + 1u);
    const uint64_t row = (uint64_t)j * h.euler_len;
    const uint64_t a = h.lca_table[row + fu], b = h.lca_table[row + fv + 1u - (1u << j)];
    return a < b ? a : b;
}

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 60;
    long bad = 0, sets_checked = 0, pairs = 0, rooted = 0, general = 0;
    for (int r = 0; r < rounds; ++r) {
        const uint64_t n = 1 + rnd() % (r % 5 == 0 ? 600 : 60);
        const bool sparse_ids = r % 3 == 1;
        std::vector<uint64_t> node_id(n), parent(n, 0), child_off(n + 1, 0), child_idx;
        std::vector<uint8_t> kind(n);
        std::vector<std::vector<uint64_t>> kids(n);
        for (uint64_t i = 1; i < n; ++i) {
            parent[i] = r % 4 == 2 ? i - 1 - (rnd() % 2 && i > 1 ? 1 : 0) : rnd() % i;     // r % 4 == 2: deep, narrow trees
            kids[parent[i]].push_back(i);
        }
        for (uint64_t i = 0; i < n; ++i) {
            node_id[i] = sparse_ids ? (i * 0x9E3779B97ull + 12345) | (1ull << 40) : i * 3 + 1;
            kind[i] = i == 0 ? CLS_KIND_ROOT : (!kids[i].empty() || rnd() % 5 == 0) ? CLS_KIND_NODE : CLS_KIND_LEAF;
            for (uint64_t c : kids[i]) child_idx.push_back(c);
            child_off[i + 1] = child_idx.size();
        }
        if (child_idx.empty()) child_idx.push_back(0);
        auto nonleaf = [&](uint64_t i) { return kind[i] != CLS_KIND_LEAF; };
        // sets: unions of root -> node paths (upward closed), some with leaves among the members, some without the root
        const uint64_t n_sets = 1 + rnd() % 40;
        std::vector<std::set<uint64_t>> members(n_sets);
        std::vector<uint64_t> set_off{0}, set_ids;
        for (uint64_t s = 0; s < n_sets; ++s) {
            const bool no_root = rnd() % 6 == 0;
            const uint64_t picks = 1 + rnd() % 5;
            for (uint64_t p = 0; p < picks; ++p) {
                uint64_t i = rnd() % n;
                for (;;) { members[s].insert(i); if (i == 0) break; i = parent[i]; }
            }
            if (no_root) members[s].erase(0);
            std::vector<uint64_t> order(members[s].begin(), members[s].end());
            for (size_t j = order.size(); j > 1; --j) std::swap(order[j - 1], order[rnd() % j]);   // any order, with a repeat
            if (!order.empty() && rnd() % 3 == 0) order.push_back(order[0]);
            for (uint64_t i : order) set_ids.push_back(node_id[i]);
            set_off.push_back(set_ids.size());
        }
        if (set_ids.empty()) set_ids.push_back(0);
        std::vector<uint64_t> eb(n_sets, 0), eh(n_sets), es(n_sets);
        for (uint64_t s = 0; s < n_sets; ++s) { eh[s] = (s + 1) * 0x9E3779B97F4A7C15ull; es[s] = s; }
        cls_model_view mv{};
        mv.k_size = 35; mv.m_size = 0;
        mv.n_nodes = n; mv.node_id = node_id.data(); mv.node_kind = kind.data(); mv.child_off = child_off.data(); mv.child_idx = child_idx.data();
        mv.n_entries = n_sets; mv.entry_bucket = eb.data(); mv.entry_hash = eh.data(); mv.entry_set = es.data();
        mv.n_sets = n_sets; mv.set_off = set_off.data(); mv.set_node_ids = set_ids.data();
        cls::HostIndex h;
        std::string err;
        if (cls::build_host_index(&mv, h, err) != CLS_OK) { printf("refused: %s\n", err.c_str()); ++bad; continue; }
        // sets without the root are never consulted, so they do not decide the mode: every rooted set here is upward closed
        if (!h.closed) { printf("not closed\n"); ++bad; continue; }
        // ---- the q numbering
        const uint32_t nq = (uint32_t)h.qnodes.size();
        std::map<uint64_t, uint32_t> q_of_id;
        for (uint32_t q = 0; q < nq; ++q) q_of_id[h.q_node_id[q]] = q;
        std::vector<uint32_t> q_of(n, ~0u);
        std::vector<uint64_t> node_of_q(nq, 0);
        uint64_t n_nonleaf_reachable = 0;
        for (uint64_t i = 0; i < n; ++i) {
            bool reach = nonleaf(i);                        // a non-leaf node below a LEAF is not part of the non-leaf tree
            for (uint64_t a = i; reach && a != 0; a = parent[a]) reach = nonleaf(parent[a]);
            if (!reach) continue;
            ++n_nonleaf_reachable;
            auto it = q_of_id.find(node_id[i]);
            if (it == q_of_id.end()) { ++bad; continue; }
            q_of[i] = it->second; node_of_q[it->second] = i;
        }
        if (n_nonleaf_reachable != nq || h.qinfo.size() != nq || q_of[0] != 0) { ++bad; continue; }
        for (uint32_t q = 0; q < nq; ++q) {
            const uint64_t i = node_of_q[q];
            std::vector<uint32_t> want;                                       // non-leaf children, in child order
            for (uint64_t c : kids[i]) if (nonleaf(c)) want.push_back(q_of[c]);
            const cls::QInfo &qi = h.qinfo[q];
            if (qi.child_count != want.size() || h.qnodes[q].child_count != want.size()) { ++bad; continue; }
            uint32_t at = q + 1;
            for (uint32_t c : want) { if (c != at) ++bad; at = h.qinfo[c].q_end; }   // they tile [q + 1, q_end)
            if (at != qi.q_end) ++bad;
            uint32_t depth = 0;
            for (uint64_t a = i; a != 0; a = parent[a]) ++depth;
            if (qi.depth != depth || qi.euler_first >= h.euler_len) ++bad;
            if ((uint32_t)h.lca_table[qi.euler_first] != q) ++bad;               // level 0 of the table is the tour itself
        }
        // ---- lowest common ancestors
        for (int t = 0; t < 400 && nq; ++t) {
            uint32_t u = (uint32_t)(rnd() % nq), v = (uint32_t)(rnd() % nq);
            if (u > v) std::swap(u, v);
            uint64_t a = node_of_q[u], b = node_of_q[v];
            auto depth_of = [&](uint64_t x) { return h.qinfo[q_of[x]].depth; };
            while (a != b) { if (depth_of(a) >= depth_of(b)) a = parent[a]; else b = parent[b]; }
            const uint64_t dn = lca_depth_node(h, u, v);
            if ((uint32_t)dn != q_of[a] || (uint32_t)(dn >> 32) != depth_of(a)) ++bad;
            ++pairs;
        }
        // ---- terminal lists
        const uint64_t mask = h.n_buckets - 1;
        for (uint64_t s = 0; s < n_sets; ++s) {
            uint64_t b = eh[s] & mask;
            const cls::Slot *slot = nullptr;
            for (uint64_t step = 0; step < h.n_buckets && !slot; ++step, b = (b + 1) & mask)
                for (int q = 0; q < 2; ++q)
                    if (h.table[2 * b + q].hash == eh[s] && h.table[2 * b + q].set_off != cls::kEmpty) slot = &h.table[2 * b + q];
            if (!slot || slot->set_off + 2 > h.terms.size()) { ++bad; continue; }
            const uint32_t *rec = &h.terms[slot->set_off];
            const uint32_t nt = rec[0] & ~cls::kTermHasRoot;
            ++sets_checked;
            if (!members[s].count(0)) { if (rec[0] != 0) ++bad; continue; }
            ++rooted;
            if (!(rec[0] & cls::kTermHasRoot) || nt == 0 || slot->set_off + 2 + nt > h.terms.size() || rec[1] != rec[1 + nt]) { ++bad; continue; }
            for (uint32_t j = 1; j < nt; ++j) if (rec[2 + j - 1] >= rec[2 + j]) ++bad;
            for (uint32_t x = 0; x < nq; ++x) {
                const uint32_t *lo = std::lower_bound(rec + 2, rec + 2 + nt, x);
                const bool in_list = lo != rec + 2 + nt && *lo < h.qinfo[x].q_end;
                if (in_list != (members[s].count(node_of_q[x]) != 0)) ++bad;
            }
        }
        // ---- the same tree with ARBITRARY node sets (not upward closed): mini-tree records.  Decoded back - entry 0 is the
        //      root, the children of entry e are e + 1, e + 1 + size(e + 1), ... below e + size(e), an entry names its node
        //      by its ordinal among the parent's non-leaf children - the PRESENT entries are exactly the set's non-leaf members
        {
            std::vector<std::set<uint64_t>> mem2(n_sets);
            std::vector<uint64_t> off2{0}, ids2;
            for (uint64_t s2 = 0; s2 < n_sets; ++s2) {
                const uint64_t picks = rnd() % 7;
                for (uint64_t p2 = 0; p2 < picks; ++p2) mem2[s2].insert(rnd() % n);
                if (s2 % 4 == 0) mem2[s2] = members[s2];                     // some closed ones among them
                for (uint64_t i : mem2[s2]) ids2.push_back(node_id[i]);
                if (rnd() % 4 == 0) ids2.push_back(0xFFFFFFFFFFull + rnd() % 9);   // an id that is not in the tree: ignored
                off2.push_back(ids2.size());
            }
            if (ids2.empty()) ids2.push_back(0);
            cls_model_view mv2 = mv;
            mv2.set_off = off2.data(); mv2.set_node_ids = ids2.data();
            mv2.flags = r % 2 ? CLS_MODEL_FORCE_GENERAL_SETS : 0;
            cls::HostIndex g;
            if (cls::build_host_index(&mv2, g, err) != CLS_OK) { printf("refused: %s\n", err.c_str()); ++bad; continue; }
            if (mv2.flags && g.closed) ++bad;
            if (g.closed) continue;                                            // by chance every rooted set was closed
            const uint64_t gmask = g.n_buckets - 1;
            for (uint64_t s2 = 0; s2 < n_sets; ++s2) {
                uint64_t b = eh[s2] & gmask;
                const cls::Slot *slot = nullptr;
                for (uint64_t step = 0; step < g.n_buckets && !slot; ++step, b = (b + 1) & gmask)
                    for (int q = 0; q < 2; ++q)
                        if (g.table[2 * b + q].hash == eh[s2] && g.table[2 * b + q].set_off != cls::kEmpty) slot = &g.table[2 * b + q];
                if (!slot || slot->set_off >= g.arena.size()) { ++bad; continue; }
                const cls::SetWord *rec = &g.arena[slot->set_off];
                const uint32_t ne = rec[0].y;
                if (ne == 0 || slot->set_off + 1 + ne > g.arena.size()) { ++bad; continue; }
                if (((rec[0].x & cls::kSetHasRoot) != 0) != (mem2[s2].count(0) != 0)) ++bad;
                std::set<uint32_t> present;
                std::vector<std::pair<uint32_t, uint32_t>> stack{{0u, 0u}};  // (entry, q)
                uint32_t visited = 0;
                while (!stack.empty()) {
                    const auto [e, q] = stack.back();
                    stack.pop_back();
                    ++visited;
                    if (rec[1 + e].x & cls::kPresentBit) present.insert(q);
                    const uint32_t size = rec[1 + e].y;
                    if (size == 0 || e + size > ne) { ++bad; break; }
                    uint32_t last_ord = 0;
                    bool first = true;
                    for (uint32_t c = e + 1; c < e + size; c += rec[1 + c].y) {
                        const uint32_t ord = rec[1 + c].x & ~cls::kPresentBit;
                        if (rec[1 + c].y == 0 || ord >= g.qnodes[q].child_count || (!first && ord <= last_ord)) { ++bad; break; }
                        first = false; last_ord = ord;
                        stack.push_back({c, g.q_child_list[g.qnodes[q].child_first + ord]});
                    }
                }
                if (visited != ne) ++bad;
                std::set<uint32_t> want;
                for (uint64_t i : mem2[s2]) if (nonleaf(i)) want.insert(q_of[i]);   // same tree, same q numbering as above
                if (present != want) ++bad;
                ++general;
            }
        }
    }
    printf("bad=%ld sets=%ld rooted=%ld lca_pairs=%ld general_sets=%ld\n", bad, sets_checked, rooted, pairs, general);
    return bad == 0 && rooted > 100 && pairs > 1000 && general > 100 ? 0 : 1;
}
