// TEST INFRASTRUCTURE.  fastq_kernels.cu's launches for the fake CUDA runtime (tests/native/fakecuda/cuda_runtime.h) as
// serial walks over the text: what cls_fastq_upload's host side consumes is the totals, the line starts, the compacted
// 2-bit codes and the per-record facts - the tile summaries in between stay unused here.
#include <cstdint>

#include "../../classeq2_b200/csrc/fastq_kernels.hpp"
#include "../../classeq2_b200/csrc/fastq_rules.hpp"

namespace cls {
namespace {
bool fq_is_base(uint8_t c) { const uint8_t u = c & 0xDFu; return c < 0x80 && (u == 'A' || u == 'C' || u == 'G' || u == 'T'); }
}  // namespace

size_t fastq_tile_bytes() { return 64; }
uint32_t fastq_n_tiles(uint64_t n) { return (uint32_t)((n + 4095) / 4096); }

cudaError_t launch_fastq_scan(const uint8_t *text, uint64_t n, void *, FastqTileBase *, FastqTileBase *totals, cudaStream_t) {
    uint64_t kept = 0, line = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if ((line & 3) == 1 && fq_is_base(text[i])) ++kept;
        if (text[i] == '\n') ++line;
    }
    *totals = FastqTileBase{kept, line};
    return cudaSuccess;
}

cudaError_t launch_fastq_write(const uint8_t *text, uint64_t n, const FastqTileBase *, uint8_t *codes, uint64_t *line_start, uint64_t *seq_kept,
                               cudaStream_t) {
    uint64_t kept = 0, line = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (i == 0 || text[i - 1] == '\n') {
            line_start[line] = i;
            if ((line & 3) == 1) seq_kept[line >> 2] = kept;
        }
        if ((line & 3) == 1 && fq_is_base(text[i])) codes[kept++] = (uint8_t)((text[i] >> 1) & 3u);
        if (text[i] == '\n') ++line;
    }
    return cudaSuccess;
}

cudaError_t launch_fastq_records(const uint8_t *text, const uint64_t *line_start, uint64_t n_lines, uint64_t n_newlines, uint64_t n_records,
                                 const uint64_t *seq_kept, uint64_t *hb, uint64_t *he, uint64_t *src, unsigned long long *first_bad, int,
                                 cudaStream_t) {
    auto end = [&](uint64_t i) {
        uint64_t e = line_start[i + 1] - 1;
        if (i < n_newlines && e > line_start[i] && text[e - 1] == '\r') --e;
        return e;
    };
    for (uint64_t r = 0; r < n_records; ++r) {
        const uint64_t L = 4 * r;
        int code = 0;
        if (end(L) == line_start[L]) code = kFastqBlankLine;
        else if (text[line_start[L]] != '@') code = kFastqNoAt;
        else if (L + 3 >= n_lines) code = kFastqTruncated;
        else if (end(L + 2) == line_start[L + 2] || text[line_start[L + 2]] != '+') code = kFastqNoPlus;
        else if (end(L + 3) - line_start[L + 3] != end(L + 1) - line_start[L + 1]) code = kFastqQualityLength;
        if (code) {
            const unsigned long long key = (unsigned long long)(r << 3 | (uint64_t)code);
            if (key < *first_bad) *first_bad = key;
            continue;
        }
        hb[r] = line_start[L] + 1;
        he[r] = end(L);
        src[r] = seq_kept[r];
    }
    return cudaSuccess;
}

}  // namespace cls
