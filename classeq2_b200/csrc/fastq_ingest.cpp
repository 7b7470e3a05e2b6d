// cls_fastq_upload: FASTQ ingest on the device (rules: include/classeq_b200.h; the host reader cls_fastq_read in
// record_writer.cpp is the reference).  The text goes to the GPU once; fastq_kernels.cu finds its lines, compacts the bases
// of its sequence lines and checks every record; the host turns the per-record facts into lengths, checks the titles as
// UTF-8 up to the first structurally bad record, and hands the records to the packer cls_fasta_upload uses (resident.cpp).
#include "capi_internal.hpp"
#include "fastq_kernels.hpp"
#include "fastq_rules.hpp"

namespace {

int fastq_upload(cls_index *ix, const uint8_t *text, uint64_t n_bytes, cls_resident_batch **out, cls_fasta_records *records) {
    using namespace cls;
    cls_index *home = resident_home(ix);
    const int device = home->device, sm_count = home->sm_count;
    CU_TRY(cudaSetDevice(device));
    cudaStream_t st = nullptr;
    // (allocated at their exact sizes with cudaMalloc, not grown with reserve)
    DevBuf d_text, d_tiles, d_bases, d_misc, d_codes, d_lines, d_seqk, d_hb, d_he, d_src;
    const uint32_t nt = fastq_n_tiles(n_bytes);
    FastqTileBase totals{0, 0};
    if (n_bytes) {
        CU_TRY(cudaMalloc(&d_text.p, n_bytes + 16));
        CU_TRY(cudaMalloc(&d_tiles.p, (size_t)nt * fastq_tile_bytes()));
        CU_TRY(cudaMalloc(&d_bases.p, (size_t)nt * sizeof(FastqTileBase)));
        CU_TRY(cudaMalloc(&d_misc.p, 256));
        CU_TRY(cudaMemcpyAsync(d_text.p, text, n_bytes, cudaMemcpyHostToDevice, st));
        CU_TRY(launch_fastq_scan(d_text.as<const uint8_t>(), n_bytes, d_tiles.p, d_bases.as<FastqTileBase>(), d_misc.as<FastqTileBase>(), st));
        CU_TRY(cudaMemcpyAsync(&totals, d_misc.p, sizeof totals, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
    }
    const uint64_t n_newlines = totals.lines, n_kept = totals.kept;
    const bool unterminated = n_bytes && text[n_bytes - 1] != '\n';
    const uint64_t n_lines = n_newlines + (unterminated ? 1 : 0);
    const uint64_t n_rec = fastq_n_records(text, n_bytes, n_newlines);
    if (n_rec >= 0xFFFFFFFFull) return set_last_error(CLS_ERR_UNSUPPORTED, "more than 2^32-1 records");
    std::vector<uint64_t> hb(n_rec), he(n_rec), src(n_rec);
    std::vector<uint32_t> ln(n_rec);
    unsigned long long first_bad = ~0ull;
    if (n_rec) {
        const uint64_t sentinel = n_bytes + (unterminated ? 1 : 0);   // line_start[n_lines]: one past the last line's terminator
        CU_TRY(cudaMalloc(&d_codes.p, n_kept + 16));
        CU_TRY(cudaMalloc(&d_lines.p, (n_lines + 1) * 8));
        CU_TRY(cudaMalloc(&d_seqk.p, (n_lines / 4 + 1) * 8));
        CU_TRY(cudaMalloc(&d_hb.p, n_rec * 8));
        CU_TRY(cudaMalloc(&d_he.p, n_rec * 8));
        CU_TRY(cudaMalloc(&d_src.p, n_rec * 8));
        unsigned long long *d_first_bad = reinterpret_cast<unsigned long long *>(d_misc.as<char>() + 128);
        CU_TRY(cudaMemcpyAsync(d_lines.as<uint64_t>() + n_lines, &sentinel, 8, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_first_bad, &first_bad, 8, cudaMemcpyHostToDevice, st));
        CU_TRY(launch_fastq_write(d_text.as<const uint8_t>(), n_bytes, d_bases.as<const FastqTileBase>(), d_codes.as<uint8_t>(), d_lines.as<uint64_t>(),
                                  d_seqk.as<uint64_t>(), st));
        CU_TRY(launch_fastq_records(d_text.as<const uint8_t>(), d_lines.as<const uint64_t>(), n_lines, n_newlines, n_rec, d_seqk.as<const uint64_t>(),
                                    d_hb.as<uint64_t>(), d_he.as<uint64_t>(), d_src.as<uint64_t>(), d_first_bad, sm_count, st));
        CU_TRY(cudaMemcpyAsync(&first_bad, d_first_bad, 8, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(hb.data(), d_hb.p, n_rec * 8, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(he.data(), d_he.p, n_rec * 8, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(src.data(), d_src.p, n_rec * 8, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
    }
    // the first bad record: the device's checks of the lines, then the titles before it as UTF-8 (on the host pool)
    const uint64_t bad = first_bad == ~0ull ? n_rec : (uint64_t)(first_bad >> 3);
    const uint64_t bad_title = fastq_first_bad_title(text, hb.data(), he.data(), bad);
    if (bad_title < bad) return fastq_fail(bad_title, kFastqTitleUtf8);
    if (bad < n_rec) return fastq_fail(bad, (int)(first_bad & 7u));
    for (uint64_t r = 0; r < n_rec; ++r) {
        const uint64_t kept = (r + 1 < n_rec ? src[r + 1] : n_kept) - src[r];
        if (kept >= (1ull << 31)) return set_last_error(CLS_ERR_INVALID_ARGUMENT, "query longer than 2^31 bases");
        ln[r] = (uint32_t)kept;
    }
    return ingest_finish(home, d_codes.as<const uint8_t>(), hb, he, ln, src, st, out, records);
}

}  // namespace

extern "C" int cls_fastq_upload(cls_index *ix, const uint8_t *text, uint64_t n_bytes, cls_resident_batch **out, cls_fasta_records *records) {
    if (!ix || !out || !records || (n_bytes && !text)) return cls::set_last_error(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    std::memset(records, 0, sizeof *records);
    if (n_bytes >= (1ull << 32)) return cls::set_last_error(CLS_ERR_UNSUPPORTED, "FASTQ text of 4 GiB or more: split it (the tile summaries count in 32 bits)");
    try {
        return fastq_upload(ix, text, n_bytes, out, records);
    } catch (const std::bad_alloc &) {
        return cls::set_last_error(CLS_ERR_OUT_OF_MEMORY, "host allocation failed");
    }
}
