// TEST INFRASTRUCTURE.  The launch functions of tests/native/fake_kernels.cpp with its routed stubs replaced by host
// restatements of the routed kernels (routed_kernels.cuh), for the sharded handle (classeq2_b200/csrc/capi_sharded.cu)
// without a GPU:
//   launch_route                hashes every window with the oracle's hash and appends it to its owner's segment (one run
//                               per read and owner, the window behind every slot, the cursors, the overflow flag) as
//                               route_kernel does;
//   launch_shard_probe_counted  reads the sender's cursor, clamps it to the segment and walks the shard's uploaded table
//                               (host memory here) as table_probe.cpp restates the kernels' walk;
//   launch_place_routed         checks every reply of every read against a direct probe of the hash's owner shard and that
//                               the read's runs cover each of its windows once, then hands the read to the oracle (a read
//                               whose runs are incomplete - a run that did not fit - gets a status no placement has, 0xEE).
// Linked instead of fake_kernels.cpp by tests/test_sharded_handle.py.
#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../classeq2_b200/csrc/kernels.hpp"   // (first: its declarations keep their names below)

extern "C" uint64_t orc_kmer_hashes(const uint8_t *bases, uint64_t len, uint32_t k, uint64_t *out, uint64_t cap);

// fake_kernels.cpp's stubs of the two routed launches are renamed out of the way
#define launch_route fake_stub_launch_route
#define launch_place_routed fake_stub_launch_place_routed
#include "fake_kernels.cpp"
#undef launch_route
#undef launch_place_routed

namespace cls {

// ---- the routed path ------------------------------------------------------------------------------------------------------
namespace {
struct Reply { uint32_t set_off, slot, code; };   // ProbeReply of routed_kernels.cuh
inline bool operator!=(const Reply &a, const Reply &b) { return a.set_off != b.set_off || a.slot != b.slot || a.code != b.code; }
uint32_t owner_of(uint64_t h, uint32_t n_shards) { return (uint32_t)(h >> 61) % n_shards; }
std::string unpack(const uint32_t *packed, const ReadDesc &d) {
    std::string s(d.len, 'A');
    for (uint32_t i = 0; i < d.len; ++i) s[i] = "ACTG"[(packed[d.word_off + i / 16] >> (2 * (i % 16))) & 3u];
    return s;
}
std::vector<uint64_t> window_hashes(const std::string &s, uint32_t k) {
    std::vector<uint64_t> h(s.size() >= k ? 2 * (s.size() - k + 1) : 0);
    if (!h.empty()) orc_kmer_hashes(reinterpret_cast<const uint8_t *>(s.data()), s.size(), k, h.data(), h.size());
    return h;
}
// walk A over one shard's table (home bucket, then along the chain while the bucket's overflow bit is set)
Reply probe(const DeviceIndex &ix, uint32_t shard, uint64_t h) {
    const uint32_t mask = (uint32_t)ix.bucket_mask;
    for (uint32_t b = (uint32_t)h & mask;; b = (b + 1) & mask) {
        const Slot *s = ix.table + 2 * (uint64_t)b;
        if (s[0].hash == h && s[0].set_off != kEmpty) return Reply{s[0].set_off, ((2u * b) << 3) | shard, s[0].code & kCodeMask};
        if (s[1].hash == h && s[1].set_off != kEmpty) return Reply{s[1].set_off, ((2u * b + 1u) << 3) | shard, s[1].code & kCodeMask};
        if (!(s[0].code & kOverflowBit)) return Reply{kEmpty, 0u, 0u};
    }
}
// the table of every shard a probe was launched on (shard number -> its index), for the direct probes of place_routed
std::mutex g_shards_mu;
std::map<uint32_t, DeviceIndex> g_shards;
}  // namespace

cudaError_t launch_route(uint32_t k, const uint32_t *packed, const ReadDesc *reads, uint32_t first_read, uint32_t n_reads, const PlaceGeom &g,
                         uint32_t n_shards, uint64_t seg_cap, uint64_t *const *seg_ptrs, uint16_t *slot_win, uint2 *runs,
                         unsigned long long *cursor, uint32_t *overflow, int, cudaStream_t stream) {
    if (n_reads == 0) return cudaSuccess;
    if (n_shards == 0 || n_shards > kMaxShards) return cudaErrorInvalidConfiguration;
    std::vector<uint64_t *> seg(seg_ptrs, seg_ptrs + n_shards);
    const uint32_t max_len = g.max_len;
    fakecuda::enqueue(stream, [=] {
        for (uint32_t r = first_read; r < first_read + n_reads; ++r) {
            if (reads[r].len > max_len) { ++fakek::async_errors; return; }
            const std::vector<uint64_t> h = window_hashes(unpack(packed, reads[r]), k);
            for (uint32_t o = 0; o < n_shards; ++o) {
                uint32_t cnt = 0;
                for (uint64_t x : h) cnt += owner_of(x, n_shards) == o;
                const uint64_t base = cnt ? cursor[o] : 0;
                cursor[o] += cnt;
                const bool fits = base + cnt <= seg_cap;
                if (!fits) *overflow = 1;
                runs[(size_t)r * 8 + o] = uint2{(unsigned)base, fits ? cnt : 0u};
                if (!fits) continue;
                uint64_t at = base;
                for (uint32_t w = 0; w < h.size(); ++w)
                    if (owner_of(h[w], n_shards) == o) { seg[o][at] = h[w]; slot_win[o * seg_cap + at] = (uint16_t)w; ++at; }
            }
        }
    });
    return cudaSuccess;
}

cudaError_t launch_shard_probe_counted(const DeviceIndex &ix, uint32_t shard, const uint64_t *hashes, uint64_t n,
                                       const unsigned long long *d_count, void *replies, int, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    { std::lock_guard<std::mutex> lk(g_shards_mu); g_shards[shard] = ix; }
    fakecuda::enqueue(stream, [=] {
        const uint64_t cnt = std::min<uint64_t>(*d_count, n);
        Reply *out = static_cast<Reply *>(replies);
        for (uint64_t i = 0; i < cnt; ++i) out[i] = probe(ix, shard, hashes[i]);
    });
    return cudaSuccess;
}

cudaError_t launch_place_routed(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads, uint32_t first_read,
                                uint32_t n_reads, ResultRec *results, const PlaceGeom &g, uint32_t n_shards, uint64_t seg_cap, const uint2 *runs,
                                const uint16_t *slot_win, const void *replies, int, cudaStream_t stream, void *scratch, size_t scratch_bytes) {
    if (n_reads == 0) return cudaSuccess;
    const void *model = fakek::oracle_model;
    if (!model) return cudaErrorUnknown;
    const size_t want = place_scratch_bytes(n_reads, g.max_len, 0, 0);
    if (!scratch || scratch_bytes < want) return cudaErrorInvalidValue;
    std::vector<DeviceIndex> owners(n_shards);
    {
        std::lock_guard<std::mutex> lk(g_shards_mu);
        for (uint32_t o = 0; o < n_shards; ++o) {
            if (!g_shards.count(o)) return cudaErrorUnknown;   // every owner is probed before any home places
            owners[o] = g_shards[o];
        }
    }
    const uint32_t k = ix.k_size, max_len = g.max_len;
    fakecuda::enqueue(stream, [=] {
        static_cast<volatile char *>(scratch)[want - 1] = 1;
        const Reply *rep = static_cast<const Reply *>(replies);
        std::string bases;
        std::vector<uint64_t> offsets{0};
        std::vector<uint32_t> which;   // reads whose replies are complete
        for (uint32_t r = first_read; r < first_read + n_reads; ++r) {
            if (reads[r].len > max_len) { ++fakek::async_errors; return; }
            const std::string s = unpack(packed, reads[r]);
            const std::vector<uint64_t> h = window_hashes(s, k);
            std::vector<uint8_t> seen(h.size(), 0);
            bool complete = true;
            for (uint32_t o = 0; o < n_shards; ++o) {
                const uint2 run = runs[(size_t)r * 8 + o];
                for (uint32_t i = 0; i < run.y; ++i) {
                    const uint64_t idx = o * seg_cap + run.x + i;
                    const uint32_t w = slot_win[idx];
                    if (w >= h.size() || seen[w]) { ++fakek::async_errors; complete = false; continue; }
                    seen[w] = 1;
                    if (owner_of(h[w], n_shards) != o || rep[idx] != probe(owners[o], o, h[w])) ++fakek::async_errors;
                }
            }
            for (uint8_t x : seen) complete &= x != 0;
            if (!complete) { results[r] = ResultRec{0, 0, 0, 0, 0, 0, 0xEE}; continue; }
            bases += s;
            offsets.push_back(bases.size());
            which.push_back(r);
        }
        const uint64_t m = which.size();
        if (!m) return;
        std::vector<uint8_t> status(m);
        std::vector<uint64_t> node(m);
        std::vector<int32_t> one(m), rest(m);
        std::vector<uint32_t> nq(m), nm(m), nr(m), it(m);
        orc_place_batch(model, reinterpret_cast<const uint8_t *>(bases.data()), offsets.data(), m, pp.max_iterations, pp.min_match_coverage,
                        pp.remove_intersection, m >= 256 ? 4 : 1, status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(),
                        nr.data(), it.data());
        for (uint64_t j = 0; j < m; ++j) results[which[j]] = ResultRec{node[j], one[j], rest[j], nm[j], nr[j], it[j], status[j]};
        fakek::reads_placed += m;
    });
    ++fakek::place_launches;
    return cudaSuccess;
}

}  // namespace cls
