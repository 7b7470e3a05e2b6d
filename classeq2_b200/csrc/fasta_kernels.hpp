// Launch interface of the FASTA ingest kernels (fasta_kernels.cu), used by cls_fasta_upload (resident.cpp).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace cls {

// Reader state at the start of a 4 KiB tile of the text.
struct TileBase {
    uint64_t kept;    // A/C/G/T bytes of sequence lines before the tile
    uint64_t hdrs;    // header lines started before the tile
    uint32_t state;   // 1: the line open at the start of the tile is a header line
    uint32_t pad;
};

size_t fasta_tile_bytes();             // size of one per-tile summary (device scratch of launch_fasta_scan)
uint32_t fasta_n_tiles(uint64_t n);

// Pass 1 + 2: per-tile summaries and their exclusive scan.  `totals->kept` / `totals->hdrs` receive the number
// of kept bases and of header lines of the whole text; *non_ascii is set if a byte >= 0x80 was seen.
cudaError_t launch_fasta_scan(const uint8_t *text, uint64_t n, void *tiles, TileBase *bases, TileBase *totals, uint32_t *non_ascii,
                              cudaStream_t stream);
// Pass 3: codes[i] = 2-bit code of the i-th kept base; for header line j: hdr_pos[j] = byte offset of its '>',
// hdr_kept[j] = kept bases before it, hdr_flag[j] != 0 iff its header text is not empty.
cudaError_t launch_fasta_write(const uint8_t *text, uint64_t n, const TileBase *bases, uint8_t *codes, uint64_t *hdr_pos,
                               uint64_t *hdr_kept, uint32_t *hdr_flag, cudaStream_t stream);
// Packs record r = codes[src[r] .. src[r] + len[r]) into words[word_off[r] ..], 16 bases per word.
cudaError_t launch_fasta_pack(const uint8_t *codes, const uint64_t *src, const uint32_t *word_off, const uint32_t *len,
                              uint32_t n_records, uint32_t *words, int sm_count, cudaStream_t stream);

}  // namespace cls
