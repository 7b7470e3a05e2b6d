// FASTQ ingest on the device: raw file bytes -> line starts, compacted 2-bit codes of the sequence lines, and per record
// its title slice, its first kept base and the first malformed record (rules: include/classeq_b200.h, cls_fastq_upload).
// In FASTQ the role of a line is its line number mod 4 (0 title, 1 sequence, 2 separator, 3 quality); its first byte
// cannot tell, because a quality line may start with '@' or '+'.  So the state of the reader at a byte is the number of
// lines before it mod 4, and a stretch of bytes is summarised by its newlines and by its kept bases for each of the four
// phases it may start in - two reduce-then-scan passes over 4 KiB tiles, as fasta_kernels.cu does for FASTA.  Then one
// thread per record checks the record's four lines and reduces the first bad one with atomicMin.  Packing reuses
// launch_fasta_pack.
#include <cuda_runtime.h>

#include <cstdint>

#include "fastq_kernels.hpp"
#include "fastq_rules.hpp"

namespace cls {
namespace {

constexpr uint32_t kChunk = 16;                      // bytes per thread
constexpr uint32_t kThreads = 256;
constexpr uint32_t kTile = kChunk * kThreads;        // 4 KiB per CTA

// What a stretch of bytes does: its newlines, and the sequence bases it keeps if it starts in phase p (the line open at
// its first byte has a line number = p mod 4).
struct Piece {
    uint32_t nl;
    uint32_t kept[4];
};

__device__ __forceinline__ Piece combine(const Piece &a, const Piece &b) {   // a then b
    Piece c;
    c.nl = a.nl + b.nl;
#pragma unroll
    for (uint32_t p = 0; p < 4; ++p) c.kept[p] = a.kept[p] + b.kept[(p + a.nl) & 3u];
    return c;
}

__device__ __forceinline__ bool is_base(uint8_t c) {
    const uint8_t u = c & 0xDFu;
    return (c >= 'A') && (u == 'A' || u == 'C' || u == 'G' || u == 'T') && ((c & 0x80u) == 0);
}

// Bytes [a, b): bases counted by the line they sit in relative to the line open at `a` (mod 4), then turned into the
// per-starting-phase form: the piece keeps the bases of its lines whose (start phase + relative line) mod 4 is 1.
__device__ __forceinline__ Piece summarise(const uint8_t *__restrict__ text, uint64_t a, uint64_t b) {
    uint32_t by_rel[4] = {0, 0, 0, 0};
    uint32_t rel = 0;
    for (uint64_t i = a; i < b; ++i) {
        const uint8_t c = text[i];
        const uint32_t base = is_base(c) ? 1u : 0u;
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j) by_rel[j] += (rel & 3u) == j ? base : 0u;
        rel += c == '\n' ? 1u : 0u;
    }
    Piece p;
    p.nl = rel;
#pragma unroll
    for (uint32_t s = 0; s < 4; ++s) p.kept[s] = by_rel[(1u - s) & 3u];
    return p;
}

__device__ __forceinline__ Piece shfl_up(const Piece &v, int d) {
    Piece o;
    o.nl = __shfl_up_sync(0xFFFFFFFFu, v.nl, d);
#pragma unroll
    for (uint32_t p = 0; p < 4; ++p) o.kept[p] = __shfl_up_sync(0xFFFFFFFFu, v.kept[p], d);
    return o;
}

// Exclusive scan of Pieces over the threads of a CTA; returns the piece of all threads before this one and, in `total`,
// the whole CTA.
__device__ __forceinline__ Piece block_exclusive(const Piece &mine, Piece *smem, Piece &total) {
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    Piece inc = mine;
    for (int d = 1; d < 32; d <<= 1) {
        const Piece o = shfl_up(inc, d);
        if ((int)lane >= d) inc = combine(o, inc);
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    Piece before_warp{0, {0, 0, 0, 0}};
    Piece all{0, {0, 0, 0, 0}};
    for (uint32_t w = 0; w < kThreads / 32; ++w) {
        if (w == warp) before_warp = all;
        all = combine(all, smem[w]);
    }
    total = all;
    __syncthreads();
    const Piece prev = shfl_up(inc, 1);
    if (lane == 0) return before_warp;
    return combine(before_warp, prev);
}

// ---- pass 1: one Piece per tile ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) fastq_tile_kernel(const uint8_t *__restrict__ text, uint64_t n, Piece *__restrict__ tiles) {
    __shared__ Piece smem[kThreads / 32];
    const uint64_t a = (uint64_t)blockIdx.x * kTile + (uint64_t)threadIdx.x * kChunk;
    const uint64_t b = a + kChunk < n ? a + kChunk : n;
    Piece mine{0, {0, 0, 0, 0}};
    if (a < n) mine = summarise(text, a, b);
    Piece total;
    block_exclusive(mine, smem, total);
    if (threadIdx.x == 0) tiles[blockIdx.x] = total;
}

// ---- pass 2: exclusive scan of the tile pieces (one CTA; each thread owns a run of consecutive tiles) ---------------
__global__ void __launch_bounds__(kThreads) fastq_scan_kernel(const Piece *__restrict__ tiles, uint32_t n_tiles, FastqTileBase *__restrict__ bases,
                                                              FastqTileBase *__restrict__ totals) {
    __shared__ Piece smem[kThreads / 32];
    const uint32_t per = (n_tiles + kThreads - 1) / kThreads;
    const uint32_t t0 = threadIdx.x * per, t1 = t0 + per < n_tiles ? t0 + per : n_tiles;
    Piece mine{0, {0, 0, 0, 0}};
    for (uint32_t t = t0; t < t1; ++t) mine = combine(mine, tiles[t]);
    Piece total;
    const Piece before = block_exclusive(mine, smem, total);
    uint64_t kept = before.kept[0], lines = before.nl;   // the text starts in phase 0 (a title line)
    for (uint32_t t = t0; t < t1; ++t) {
        const Piece p = tiles[t];
        bases[t] = FastqTileBase{kept, lines};
        kept += p.kept[lines & 3u];
        lines += p.nl;
    }
    if (threadIdx.x == 0) *totals = FastqTileBase{total.kept[0], total.nl};
}

// ---- pass 3: the compacted 2-bit codes, the start of every line, the first kept base of every sequence line ---------
__global__ void __launch_bounds__(kThreads) fastq_write_kernel(const uint8_t *__restrict__ text, uint64_t n, const FastqTileBase *__restrict__ bases,
                                                               uint8_t *__restrict__ codes, uint64_t *__restrict__ line_start,
                                                               uint64_t *__restrict__ seq_kept) {
    __shared__ Piece smem[kThreads / 32];
    const FastqTileBase tb = bases[blockIdx.x];
    const uint64_t a = (uint64_t)blockIdx.x * kTile + (uint64_t)threadIdx.x * kChunk;
    const uint64_t b = a + kChunk < n ? a + kChunk : n;
    Piece mine{0, {0, 0, 0, 0}};
    if (a < n) mine = summarise(text, a, b);
    Piece total;
    const Piece before = block_exclusive(mine, smem, total);
    if (a >= n) return;
    uint64_t line = tb.lines + before.nl;                  // number of the line open at `a`
    uint64_t kept = tb.kept + before.kept[tb.lines & 3u];
    bool at_start = a == 0 || text[a - 1] == '\n';
    for (uint64_t i = a; i < b; ++i) {
        const uint8_t c = text[i];
        if (at_start) {
            line_start[line] = i;
            if ((line & 3u) == 1u) seq_kept[line >> 2] = kept;
        }
        if ((line & 3u) == 1u && is_base(c)) codes[kept++] = (uint8_t)((c >> 1) & 3u);   // A=0 C=1 T=2 G=3, either case
        at_start = c == '\n';
        line += at_start ? 1u : 0u;
    }
}

// ---- one thread per record: its four lines against the rules; titles and first kept bases for the host --------------
// line_start[0 .. n_lines] with line_start[n_lines] = n + 1 if the last line has no terminator, else n: the content of
// line i ends at line_start[i + 1] - 1, less a '\r' before a terminating '\n'.
__device__ __forceinline__ uint64_t content_end(const uint8_t *__restrict__ text, const uint64_t *__restrict__ line_start, uint64_t i,
                                                uint64_t n_newlines) {
    uint64_t e = line_start[i + 1] - 1;
    if (i < n_newlines && e > line_start[i] && text[e - 1] == '\r') --e;
    return e;
}

__global__ void __launch_bounds__(256) fastq_record_kernel(const uint8_t *__restrict__ text, const uint64_t *__restrict__ line_start,
                                                           uint64_t n_lines, uint64_t n_newlines, uint64_t n_records,
                                                           const uint64_t *__restrict__ seq_kept, uint64_t *__restrict__ hb,
                                                           uint64_t *__restrict__ he, uint64_t *__restrict__ src,
                                                           unsigned long long *__restrict__ first_bad) {
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_records; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t L = 4 * r;
        const uint64_t t0 = line_start[L], t1 = content_end(text, line_start, L, n_newlines);
        int code = 0;
        if (t1 == t0) code = kFastqBlankLine;
        else if (text[t0] != '@') code = kFastqNoAt;
        else if (L + 3 >= n_lines) code = kFastqTruncated;
        else {
            const uint64_t s0 = line_start[L + 1], s1 = content_end(text, line_start, L + 1, n_newlines);
            const uint64_t p0 = line_start[L + 2], p1 = content_end(text, line_start, L + 2, n_newlines);
            const uint64_t q0 = line_start[L + 3], q1 = content_end(text, line_start, L + 3, n_newlines);
            if (p1 == p0 || text[p0] != '+') code = kFastqNoPlus;
            else if (q1 - q0 != s1 - s0) code = kFastqQualityLength;
        }
        if (code) {
            atomicMin(first_bad, (unsigned long long)(r << 3 | (uint64_t)code));
            continue;
        }
        hb[r] = t0 + 1;
        he[r] = t1;
        src[r] = seq_kept[r];
    }
}

}  // namespace

size_t fastq_tile_bytes() { return sizeof(Piece); }
uint32_t fastq_n_tiles(uint64_t n) { return (uint32_t)((n + kTile - 1) / kTile); }

cudaError_t launch_fastq_scan(const uint8_t *text, uint64_t n, void *tiles, FastqTileBase *bases, FastqTileBase *totals, cudaStream_t stream) {
    const uint32_t nt = fastq_n_tiles(n);
    if (nt == 0) return cudaSuccess;
    fastq_tile_kernel<<<nt, kThreads, 0, stream>>>(text, n, reinterpret_cast<Piece *>(tiles));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    fastq_scan_kernel<<<1, kThreads, 0, stream>>>(reinterpret_cast<const Piece *>(tiles), nt, bases, totals);
    return cudaGetLastError();
}

cudaError_t launch_fastq_write(const uint8_t *text, uint64_t n, const FastqTileBase *bases, uint8_t *codes, uint64_t *line_start,
                               uint64_t *seq_kept, cudaStream_t stream) {
    const uint32_t nt = fastq_n_tiles(n);
    if (nt == 0) return cudaSuccess;
    fastq_write_kernel<<<nt, kThreads, 0, stream>>>(text, n, bases, codes, line_start, seq_kept);
    return cudaGetLastError();
}

cudaError_t launch_fastq_records(const uint8_t *text, const uint64_t *line_start, uint64_t n_lines, uint64_t n_newlines, uint64_t n_records,
                                 const uint64_t *seq_kept, uint64_t *hb, uint64_t *he, uint64_t *src, unsigned long long *first_bad,
                                 int sm_count, cudaStream_t stream) {
    if (n_records == 0) return cudaSuccess;
    uint64_t grid = (n_records + 255) / 256;
    if (grid > (uint64_t)sm_count * 16) grid = (uint64_t)sm_count * 16;
    fastq_record_kernel<<<(uint32_t)grid, 256, 0, stream>>>(text, line_start, n_lines, n_newlines, n_records, seq_kept, hb, he, src, first_bad);
    return cudaGetLastError();
}

}  // namespace cls
