// FASTA ingest on the device (SURVEY.md section 8f, row 3): raw file bytes -> filtered, upper-cased,
// 2-bit packed reads, with the exact record rules of the reference's reader
// (core/src/domain/dtos/file_or_stdin.rs:76-116, sequence.rs:47-56):
//   * lines end at '\n'; a '\r' right before the '\n' belongs to the terminator;
//   * a line whose first byte is '>' is a header line (its text, minus every '>', is the header);
//   * every other line contributes its A/C/G/T bytes (either case) to the current record;
//     everything else - N, IUPAC codes, gaps, blanks - is DELETED and the flanks are joined.
// The device does the per-byte work (classification, filtering, compaction, packing) with two
// reduce-then-scan passes over 4 KiB tiles; the record-level rules (empty headers, the trailing
// record, "sequence without header") are a few comparisons per record on the host (resident.cpp).
// Non-ASCII bytes are reported, not interpreted: Rust's to_uppercase() maps a handful of non-ASCII
// scalars to strings containing A/C/G/T, and the caller then uses the host reader.
#include <cuda_runtime.h>

#include <cstdint>

#include "fasta_kernels.hpp"

namespace cls {
namespace {

constexpr uint32_t kChunk = 16;                      // bytes per thread
constexpr uint32_t kThreads = 256;
constexpr uint32_t kTile = kChunk * kThreads;        // 4 KiB per CTA

// What a stretch of bytes does to the reader's state, for either state it may start in.
struct Piece {
    uint32_t kept_nh;   // kept bases if the line open at the start of the piece is NOT a header line
    uint32_t kept_h;    // ... if it IS a header line
    uint32_t n_hdr;     // header lines that start inside the piece
    uint32_t det;       // 1: a line starts inside the piece, so the state after it is known locally
    uint32_t hdr_out;   // (det) the line open at the end of the piece is a header line
};

__device__ __forceinline__ Piece combine(const Piece &a, const Piece &b) {   // a then b
    Piece c;
    // b starts in state: a.det ? a.hdr_out : (incoming state of a)
    const uint32_t b_if_nh = a.det ? (a.hdr_out ? b.kept_h : b.kept_nh) : b.kept_nh;
    const uint32_t b_if_h = a.det ? (a.hdr_out ? b.kept_h : b.kept_nh) : b.kept_h;
    c.kept_nh = a.kept_nh + b_if_nh;
    c.kept_h = a.kept_h + b_if_h;
    c.n_hdr = a.n_hdr + b.n_hdr;
    c.det = a.det | b.det;
    c.hdr_out = b.det ? b.hdr_out : a.hdr_out;
    return c;
}

__device__ __forceinline__ bool is_base(uint8_t c) {
    const uint8_t u = c & 0xDFu;   // ASCII upper-casing of letters; other bytes map to values that are not A/C/G/T
    return (c >= 'A') && (u == 'A' || u == 'C' || u == 'G' || u == 'T') && ((c & 0x80u) == 0);
}

// Walks bytes [a, b) of the text.  `hdr` is the state of the line open at `a` (ignored when `a` is a
// line start).  emit(i, byte, in_header_line, is_line_start) is called for every byte.
template <class F>
__device__ __forceinline__ Piece walk(const uint8_t *__restrict__ text, uint64_t a, uint64_t b, bool hdr, F emit) {
    Piece p{0, 0, 0, 0, 0};
    bool at_start = a == 0 || text[a - 1] == '\n';
    uint32_t kept_carried = 0;   // bases of the line open at `a`, before any line start in the piece
    bool cur = hdr;
    for (uint64_t i = a; i < b; ++i) {
        const uint8_t c = text[i];
        if (at_start) {
            cur = c == '>';
            p.det = 1;
            p.n_hdr += cur ? 1u : 0u;
        }
        emit(i, c, cur, at_start);
        if (!cur && is_base(c)) {
            if (p.det) ++p.kept_nh; else ++kept_carried;
        }
        at_start = c == '\n';
    }
    p.kept_h = p.kept_nh;            // bases after the first line start do not depend on the incoming state
    p.kept_nh += kept_carried;
    p.hdr_out = cur ? 1u : 0u;
    return p;
}

// Exclusive scan of Pieces over the threads of a CTA (ordered by thread id); returns the piece made of all
// threads before this one and, in `total`, the whole tile.
__device__ __forceinline__ Piece block_exclusive(const Piece &mine, Piece *smem, Piece &total) {
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    // inclusive scan inside the warp
    Piece inc = mine;
    for (int d = 1; d < 32; d <<= 1) {
        Piece o;
        o.kept_nh = __shfl_up_sync(0xFFFFFFFFu, inc.kept_nh, d);
        o.kept_h = __shfl_up_sync(0xFFFFFFFFu, inc.kept_h, d);
        o.n_hdr = __shfl_up_sync(0xFFFFFFFFu, inc.n_hdr, d);
        o.det = __shfl_up_sync(0xFFFFFFFFu, inc.det, d);
        o.hdr_out = __shfl_up_sync(0xFFFFFFFFu, inc.hdr_out, d);
        if ((int)lane >= d) inc = combine(o, inc);
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    Piece before_warp{0, 0, 0, 0, 0};
    Piece all{0, 0, 0, 0, 0};
    for (uint32_t w = 0; w < kThreads / 32; ++w) {
        if (w == warp) before_warp = all;
        all = w == 0 ? smem[0] : combine(all, smem[w]);
    }
    total = all;
    __syncthreads();
    // exclusive within the warp = inclusive of the previous lane
    Piece prev;
    prev.kept_nh = __shfl_up_sync(0xFFFFFFFFu, inc.kept_nh, 1);
    prev.kept_h = __shfl_up_sync(0xFFFFFFFFu, inc.kept_h, 1);
    prev.n_hdr = __shfl_up_sync(0xFFFFFFFFu, inc.n_hdr, 1);
    prev.det = __shfl_up_sync(0xFFFFFFFFu, inc.det, 1);
    prev.hdr_out = __shfl_up_sync(0xFFFFFFFFu, inc.hdr_out, 1);
    if (lane == 0) return before_warp;
    return warp == 0 ? prev : combine(before_warp, prev);
}

// ---- pass 1: one Piece per tile ------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) fasta_tile_kernel(const uint8_t *__restrict__ text, uint64_t n, Piece *__restrict__ tiles,
                                                              uint32_t *__restrict__ non_ascii) {
    __shared__ Piece smem[kThreads / 32];
    const uint64_t a = (uint64_t)blockIdx.x * kTile + (uint64_t)threadIdx.x * kChunk;
    const uint64_t b = a + kChunk < n ? a + kChunk : n;
    bool bad = false;
    Piece mine{0, 0, 0, 0, 0};
    if (a < n) mine = walk(text, a, b, false, [&](uint64_t, uint8_t c, bool, bool) { bad |= (c & 0x80u) != 0; });
    if (bad) atomicOr(non_ascii, 1u);
    // the walk assumed "not a header line" for the carried part; kept_h already excludes it
    Piece total;
    block_exclusive(mine, smem, total);
    if (threadIdx.x == 0) tiles[blockIdx.x] = total;
}

// ---- pass 2: exclusive scan of the tile pieces (one CTA; each thread owns a run of consecutive tiles) ---
__global__ void __launch_bounds__(kThreads) fasta_scan_kernel(const Piece *__restrict__ tiles, uint32_t n_tiles, TileBase *__restrict__ bases,
                                                              TileBase *__restrict__ totals) {
    __shared__ Piece smem[kThreads / 32];
    const uint32_t per = (n_tiles + kThreads - 1) / kThreads;
    const uint32_t t0 = threadIdx.x * per, t1 = t0 + per < n_tiles ? t0 + per : n_tiles;
    Piece mine{0, 0, 0, 0, 0};
    for (uint32_t t = t0; t < t1; ++t) mine = t == t0 ? tiles[t] : combine(mine, tiles[t]);
    Piece total;
    Piece before = block_exclusive(mine, smem, total);
    // the file starts outside any header line with nothing kept: state "nh"
    uint64_t kept = before.kept_nh, hdrs = before.n_hdr;
    bool state = before.det ? before.hdr_out != 0 : false;
    for (uint32_t t = t0; t < t1; ++t) {
        const Piece p = tiles[t];
        bases[t] = TileBase{kept, hdrs, state ? 1u : 0u, 0u};
        kept += state ? p.kept_h : p.kept_nh;
        hdrs += p.n_hdr;
        if (p.det) state = p.hdr_out != 0;
    }
    if (threadIdx.x == 0) *totals = TileBase{total.kept_nh, total.n_hdr, 0u, 0u};
}

// ---- pass 3: write the compacted 2-bit codes, the header-line starts and the header flags ------------------
__global__ void __launch_bounds__(kThreads) fasta_write_kernel(const uint8_t *__restrict__ text, uint64_t n, const TileBase *__restrict__ bases,
                                                               uint8_t *__restrict__ codes, uint64_t *__restrict__ hdr_pos,
                                                               uint64_t *__restrict__ hdr_kept, uint32_t *__restrict__ hdr_flag) {
    __shared__ Piece smem[kThreads / 32];
    const TileBase tb = bases[blockIdx.x];
    const uint64_t a = (uint64_t)blockIdx.x * kTile + (uint64_t)threadIdx.x * kChunk;
    const uint64_t b = a + kChunk < n ? a + kChunk : n;
    Piece mine{0, 0, 0, 0, 0};
    if (a < n) mine = walk(text, a, b, false, [](uint64_t, uint8_t, bool, bool) {});
    Piece total;
    const Piece before = block_exclusive(mine, smem, total);
    if (a >= n) return;
    const bool tile_state = tb.state != 0;
    const bool state = before.det ? before.hdr_out != 0 : tile_state;
    uint64_t kept = tb.kept + (tile_state ? before.kept_h : before.kept_nh);
    uint64_t hdrs = tb.hdrs + before.n_hdr;
    walk(text, a, b, state, [&](uint64_t i, uint8_t c, bool in_hdr, bool line_start) {
        if (in_hdr) {
            if (line_start) { hdr_pos[hdrs] = i; hdr_kept[hdrs] = kept; ++hdrs; }
            // a header is empty when its line holds nothing but '>' (the terminator is "\n" or "\r\n")
            const bool terminator = c == '\n' || (c == '\r' && i + 1 < n && text[i + 1] == '\n');
            if (c != '>' && !terminator) atomicOr(&hdr_flag[hdrs - 1], 1u);
        } else if (is_base(c)) {
            codes[kept++] = (uint8_t)((c >> 1) & 3u);   // A=0 C=1 T=2 G=3, either case
        }
    });
}

// ---- pack the records the reader sends: 16 bases per word, every record at a word boundary --------------
__global__ void __launch_bounds__(256) fasta_pack_kernel(const uint8_t *__restrict__ codes, const uint64_t *__restrict__ src,
                                                         const uint32_t *__restrict__ word_off, const uint32_t *__restrict__ len,
                                                         uint32_t n_records, uint32_t *__restrict__ words) {
    // one warp per record: lanes stride over its words
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = gw; r < n_records; r += nw) {
        const uint8_t *c = codes + src[r];
        const uint32_t L = len[r], n_words = (L + 15u) >> 4;
        uint32_t *out = words + word_off[r];
        for (uint32_t w = lane; w < n_words; w += 32) {
            uint32_t v = 0;
            const uint32_t base = 16u * w, m = L - base < 16u ? L - base : 16u;
            for (uint32_t j = 0; j < m; ++j) v |= (uint32_t)c[base + j] << (2u * j);
            out[w] = v;
        }
    }
}

}  // namespace

size_t fasta_tile_bytes() { return sizeof(Piece); }
uint32_t fasta_n_tiles(uint64_t n) { return (uint32_t)((n + kTile - 1) / kTile); }

cudaError_t launch_fasta_scan(const uint8_t *text, uint64_t n, void *tiles, TileBase *bases, TileBase *totals, uint32_t *non_ascii,
                              cudaStream_t stream) {
    const uint32_t nt = fasta_n_tiles(n);
    if (nt == 0) return cudaSuccess;
    fasta_tile_kernel<<<nt, kThreads, 0, stream>>>(text, n, reinterpret_cast<Piece *>(tiles), non_ascii);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    fasta_scan_kernel<<<1, kThreads, 0, stream>>>(reinterpret_cast<const Piece *>(tiles), nt, bases, totals);
    return cudaGetLastError();
}

cudaError_t launch_fasta_write(const uint8_t *text, uint64_t n, const TileBase *bases, uint8_t *codes, uint64_t *hdr_pos,
                               uint64_t *hdr_kept, uint32_t *hdr_flag, cudaStream_t stream) {
    const uint32_t nt = fasta_n_tiles(n);
    if (nt == 0) return cudaSuccess;
    fasta_write_kernel<<<nt, kThreads, 0, stream>>>(text, n, bases, codes, hdr_pos, hdr_kept, hdr_flag);
    return cudaGetLastError();
}

cudaError_t launch_fasta_pack(const uint8_t *codes, const uint64_t *src, const uint32_t *word_off, const uint32_t *len,
                              uint32_t n_records, uint32_t *words, int sm_count, cudaStream_t stream) {
    if (n_records == 0) return cudaSuccess;
    uint32_t grid = (uint32_t)sm_count * 8;
    const uint32_t need = (n_records + 7) / 8;
    if (grid > need) grid = need;
    fasta_pack_kernel<<<grid, 256, 0, stream>>>(codes, src, word_off, len, n_records, words);
    return cudaGetLastError();
}

}  // namespace cls
