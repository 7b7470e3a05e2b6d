// TEST INFRASTRUCTURE.  The launch functions of kernels.hpp / fasta_kernels.hpp for the fake CUDA runtime
// (tests/native/fakecuda/cuda_runtime.h), so that the C ABI's host side runs without a GPU:
//   launch_place        unpacks every read of the launch from the 2-bit words at its descriptor and hands it to the C++
//                       oracle (oracle/classeq_oracle.cpp, linked into the test) - what the placement kernels compute,
//                       by other means; the result records land where the kernels would write them;
//   launch_ascii_pack   pack_kernels.cu's job on the host (ASCII -> 2-bit words at the descriptors' offsets, bad flags);
//   launch_fasta_*      fasta_kernels.cu's passes as serial walks (the host side of cls_fasta_upload is what is tested);
//   the routed / trace launches are not part of these tests and report an error.
// Everything the HOST side hands over - word offsets, descriptors, source offsets, chunk ranges, scratch sizes - has to
// be right for the results to equal the oracle's on the caller's ASCII batch.
#include <atomic>
#include <cstdint>
#include <string>
#include <vector>

#include "../../classeq2_b200/csrc/fasta_kernels.hpp"
#include "../../classeq2_b200/csrc/kernels.hpp"

extern "C" void orc_place_batch(const void *model, const uint8_t *bases, const uint64_t *offsets, uint64_t n, int32_t max_iterations,
                                double min_match_coverage, uint32_t remove_intersection, int n_threads, uint8_t *status, uint64_t *node_id,
                                int32_t *one, int32_t *rest, uint32_t *n_query_kmers, uint32_t *n_matched, uint32_t *n_root_matched,
                                uint32_t *iterations);

namespace fakek {
const void *oracle_model = nullptr;          // set by the test before the first placement
std::atomic<uint64_t> place_launches{0}, pack_launches{0}, reads_placed{0};
std::atomic<uint32_t> fail_above_len{0};     // launch_place reports cudaErrorInvalidConfiguration for longer reads (0: never)
std::atomic<uint64_t> async_errors{0};        // a launch body met a descriptor its launch does not cover
std::atomic<bool> null_placement{false};     // host-overhead timing: the launch writes "no match" records and returns
}  // namespace fakek

namespace cls {

PlaceGeom make_place_geom(uint32_t max_len, uint32_t, uint32_t max_fanout) {
    PlaceGeom g{};
    g.max_len = max_len;
    g.fan_cap = max_fanout;
    return g;
}

size_t place_scratch_bytes(uint32_t n_reads, uint32_t max_len, uint32_t, uint32_t) { return 64 + (size_t)n_reads * 8 + max_len; }

// A launch is checked here and runs IN STREAM ORDER (fakecuda::enqueue: on the stream's worker thread in the
// asynchronous mode of the fake runtime), like a kernel.
cudaError_t launch_place(const DeviceIndex &, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads, uint32_t first_read,
                         uint32_t n_reads, ResultRec *results, const PlaceGeom &g, int, cudaStream_t stream, void *scratch, size_t scratch_bytes,
                         uint32_t *n_launches) {
    if (fakek::fail_above_len && g.max_len > fakek::fail_above_len) return cudaErrorInvalidConfiguration;
    if (fakek::null_placement) {
        fakecuda::enqueue(stream, [=] { for (uint32_t j = first_read; j < first_read + n_reads; ++j) results[j] = ResultRec{0, 0, 0, 0, 0, 0, CLS_DEV_UNCL_NO_MATCH}; });
        if (n_launches) *n_launches += 2;
        return cudaSuccess;
    }
    const void *model = fakek::oracle_model;
    if (!model) return cudaErrorUnknown;
    const size_t want = place_scratch_bytes(n_reads, g.max_len, 0, 0);
    if (!scratch || scratch_bytes < want) return cudaErrorInvalidValue;       // the host must have reserved what it was told to
    const uint32_t max_len = g.max_len;
    fakecuda::enqueue(stream, [=] {
        static_cast<volatile char *>(scratch)[want - 1] = 1;                    // the scratch is really there (ASan), and nobody else uses it now (TSan)
        std::vector<uint8_t> bases;
        std::vector<uint64_t> offsets{0};
        for (uint32_t j = first_read; j < first_read + n_reads; ++j) {
            const ReadDesc d = reads[j];
            if (d.len > max_len) { ++fakek::async_errors; return; }             // the geometry of a launch covers its longest read
            for (uint32_t i = 0; i < d.len; ++i) bases.push_back((uint8_t)"ACTG"[(packed[d.word_off + i / 16] >> (2 * (i % 16))) & 3u]);
            offsets.push_back(bases.size());
        }
        if (bases.empty()) bases.push_back('A');
        std::vector<uint8_t> status(n_reads);
        std::vector<uint64_t> node(n_reads);
        std::vector<int32_t> one(n_reads), rest(n_reads);
        std::vector<uint32_t> nq(n_reads), nm(n_reads), nr(n_reads), it(n_reads);
        orc_place_batch(model, bases.data(), offsets.data(), n_reads, pp.max_iterations, pp.min_match_coverage, pp.remove_intersection,
                        n_reads >= 256 ? 4 : 1, status.data(), node.data(), one.data(), rest.data(), nq.data(), nm.data(), nr.data(), it.data());
        for (uint32_t j = 0; j < n_reads; ++j)
            results[first_read + j] = ResultRec{node[j], one[j], rest[j], nm[j], nr[j], it[j], status[j]};
        fakek::reads_placed += n_reads;
    });
    if (n_launches) *n_launches += 2;
    ++fakek::place_launches;
    return cudaSuccess;
}

cudaError_t launch_ascii_pack(const uint8_t *ascii, const uint64_t *src_off, const ReadDesc *descs, uint32_t first, uint32_t count,
                              uint32_t max_len, uint32_t *words, uint8_t *bad, cudaStream_t stream) {
    if (fakecuda::skip_copies()) return cudaSuccess;      // host-overhead timing
    fakecuda::enqueue(stream, [=] {
        for (uint32_t j = first; j < first + count; ++j) {
            const ReadDesc d = descs[j];
            if (d.len > max_len) { ++fakek::async_errors; return; }
            const uint8_t *s = ascii + src_off[j];
            uint8_t any_bad = 0;
            for (uint32_t w = 0; w < (d.len + 15) / 16; ++w) {
                uint32_t v = 0;
                for (uint32_t i = 16 * w; i < d.len && i < 16 * w + 16; ++i) {
                    const uint8_t c = s[i] & 0xDF;
                    if (c != 'A' && c != 'C' && c != 'G' && c != 'T') any_bad = 1;
                    v |= ((uint32_t)(s[i] >> 1) & 3u) << (2 * (i % 16));
                }
                words[d.word_off + w] = v;
            }
            if (any_bad) bad[j] = 1;
        }
    });
    ++fakek::pack_launches;
    return cudaSuccess;
}

cudaError_t launch_trace(const DeviceIndex &, const PlaceParams &, const uint32_t *, const ReadDesc *, ResultRec *, const PlaceGeom &, int,
                         cudaStream_t, TraceBuf) { return cudaErrorUnknown; }
cudaError_t launch_route(uint32_t, const uint32_t *, const ReadDesc *, uint32_t, uint32_t, const PlaceGeom &, uint32_t, uint64_t,
                         uint64_t *const *, uint16_t *, uint2 *, unsigned long long *, uint32_t *, int, cudaStream_t) { return cudaErrorUnknown; }
cudaError_t launch_shard_probe(const DeviceIndex &, uint32_t, const uint64_t *, uint64_t, void *, cudaStream_t) { return cudaErrorUnknown; }
cudaError_t launch_place_routed(const DeviceIndex &, const PlaceParams &, const uint32_t *, const ReadDesc *, uint32_t, uint32_t, ResultRec *,
                                const PlaceGeom &, uint32_t, uint64_t, const uint2 *, const uint16_t *, const void *, int, cudaStream_t, void *,
                                size_t) { return cudaErrorUnknown; }
cudaError_t launch_hash_only(const uint32_t *, uint32_t, uint32_t, uint64_t *, cudaStream_t) { return cudaErrorUnknown; }

// fasta_kernels.cu's three passes as one serial walk each: what cls_fasta_upload's host side consumes is the totals,
// the per-header-line facts and the compacted 2-bit codes - the tile summaries in between stay unused here.
size_t fasta_tile_bytes() { return 64; }
uint32_t fasta_n_tiles(uint64_t n) { return (uint32_t)((n + 4095) / 4096); }
namespace {
bool fasta_is_base(uint8_t c) { const uint8_t u = c & 0xDFu; return c < 0x80 && (u == 'A' || u == 'C' || u == 'G' || u == 'T'); }
template <class H, class B>
void fasta_walk(const uint8_t *text, uint64_t n, H on_header_byte, B on_base) {
    bool at_start = true, in_hdr = false;
    for (uint64_t i = 0; i < n; ++i) {
        const uint8_t c = text[i];
        const bool line_start = at_start;
        if (at_start) in_hdr = c == '>';
        if (in_hdr) on_header_byte(i, c, line_start);
        else if (fasta_is_base(c)) on_base(c);
        at_start = c == '\n';
    }
}
}  // namespace
cudaError_t launch_fasta_scan(const uint8_t *text, uint64_t n, void *, TileBase *, TileBase *totals, uint32_t *non_ascii, cudaStream_t) {
    uint64_t kept = 0, hdrs = 0;
    for (uint64_t i = 0; i < n; ++i) if (text[i] & 0x80u) *non_ascii = 1;
    fasta_walk(text, n, [&](uint64_t, uint8_t, bool line_start) { hdrs += line_start; }, [&](uint8_t) { ++kept; });
    *totals = TileBase{kept, hdrs, 0u, 0u};
    return cudaSuccess;
}
cudaError_t launch_fasta_write(const uint8_t *text, uint64_t n, const TileBase *, uint8_t *codes, uint64_t *hdr_pos, uint64_t *hdr_kept,
                               uint32_t *hdr_flag, cudaStream_t) {
    uint64_t kept = 0, hdrs = 0;
    fasta_walk(text, n,
               [&](uint64_t i, uint8_t c, bool line_start) {
                   if (line_start) { hdr_pos[hdrs] = i; hdr_kept[hdrs] = kept; ++hdrs; }
                   const bool terminator = c == '\n' || (c == '\r' && i + 1 < n && text[i + 1] == '\n');
                   if (c != '>' && !terminator) hdr_flag[hdrs - 1] |= 1u;
               },
               [&](uint8_t c) { codes[kept++] = (uint8_t)((c >> 1) & 3u); });
    return cudaSuccess;
}
cudaError_t launch_fasta_pack(const uint8_t *codes, const uint64_t *src, const uint32_t *word_off, const uint32_t *len, uint32_t n_records,
                              uint32_t *words, int, cudaStream_t) {
    for (uint32_t r = 0; r < n_records; ++r)
        for (uint32_t w = 0; w < (len[r] + 15) / 16; ++w) {
            uint32_t v = 0;
            for (uint32_t j = 16 * w; j < len[r] && j < 16 * w + 16; ++j) v |= (uint32_t)codes[src[r] + j] << (2 * (j % 16));
            words[word_off[r] + w] = v;
        }
    return cudaSuccess;
}

}  // namespace cls
