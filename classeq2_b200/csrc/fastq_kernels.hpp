// Launch interface of the FASTQ ingest kernels (fastq_kernels.cu), used by cls_fastq_upload (capi.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace cls {

// Reader state at the start of a 4 KiB tile of the text.
struct FastqTileBase {
    uint64_t kept;    // A/C/G/T bytes of sequence lines before the tile
    uint64_t lines;   // newlines before the tile (the number of the line open at its first byte)
};

size_t fastq_tile_bytes();             // size of one per-tile summary (device scratch of launch_fastq_scan)
uint32_t fastq_n_tiles(uint64_t n);

// Pass 1 + 2: per-tile summaries and their exclusive scan.  totals->kept / totals->lines receive the kept bases and the
// newlines of the whole text.  n < 2^32.
cudaError_t launch_fastq_scan(const uint8_t *text, uint64_t n, void *tiles, FastqTileBase *bases, FastqTileBase *totals, cudaStream_t stream);
// Pass 3: codes[i] = 2-bit code of the i-th kept base; line_start[l] = first byte of line l; seq_kept[j] = kept bases
// before sequence line 4j + 1.
cudaError_t launch_fastq_write(const uint8_t *text, uint64_t n, const FastqTileBase *bases, uint8_t *codes, uint64_t *line_start,
                               uint64_t *seq_kept, cudaStream_t stream);
// One thread per record r < n_records: *first_bad = min over malformed records of (r << 3 | FastqReason) (set it to ~0 first);
// for a well-formed record hb[r] / he[r] = its title after the '@', src[r] = seq_kept[r].  line_start has n_lines + 1
// entries, the last one n + 1 when the text does not end with a newline, else n.
cudaError_t launch_fastq_records(const uint8_t *text, const uint64_t *line_start, uint64_t n_lines, uint64_t n_newlines, uint64_t n_records,
                                 const uint64_t *seq_kept, uint64_t *hb, uint64_t *he, uint64_t *src, unsigned long long *first_bad,
                                 int sm_count, cudaStream_t stream);

}  // namespace cls
