// Resident batches (cls_batch_upload, cls_place_resident, cls_resident_fetch) and the device ingest of FASTA text; the
// FASTQ ingest (fastq_ingest.cpp) ends in ingest_finish as well.
#include "capi_internal.hpp"
#include "fasta_kernels.hpp"

using namespace cls;

namespace cls {

cls_index *resident_home(cls_index *ix) {
    if (!ix->shards.empty()) ix = ix->shards[0].get();       // a sharded handle: resident batches live on its first shard's device
    if (!ix->replicas.empty()) ix = ix->replicas[0].get();   // a multi-device handle: resident batches live on its first device
    return ix;
}

// The tail of both text ingests: the records become a resident batch, planned with the planner of cls_batch_upload and
// packed from the compacted codes on the device (`src`: every record's first kept base in them).
int ingest_finish(cls_index *home, const uint8_t *d_codes, std::vector<uint64_t> &hb, std::vector<uint64_t> &he, std::vector<uint32_t> &ln,
                  const std::vector<uint64_t> &src, cudaStream_t st, cls_resident_batch **out, cls_fasta_records *records) try {
    auto rb = std::make_unique<cls_resident_batch>();
    rb->device = home->device;
    rb->fa_header_begin.swap(hb);
    rb->fa_header_end.swap(he);
    rb->fa_length.swap(ln);
    const auto &lens = rb->fa_length;
    const uint64_t n = lens.size();
    std::vector<uint64_t> offsets(n + 1, 0);
    for (uint64_t i = 0; i < n; ++i) offsets[i + 1] = offsets[i] + lens[i];
    cls_batch fake{n, reinterpret_cast<const uint8_t *>(offsets.data()), offsets.data()};   // plan_batch never reads the bases
    std::vector<uint32_t> word_off;
    int rc = plan_batch(&fake, home->dix.k_size, home->dix.max_fanout, rb->lay, word_off);
    if (rc != CLS_OK) return rc;
    const PackedLayout &lay = rb->lay;
    const size_t words_b = (size_t)lay.n_words * 4, descs_b = (size_t)lay.n_device * sizeof(ReadDesc), res_b = (size_t)lay.n_device * sizeof(ResultRec);
    CU_TRY(rb->d_words.reserve(words_b + 16)); CU_TRY(rb->d_descs.reserve(descs_b + 16)); CU_TRY(rb->d_results.reserve(res_b + 32));
    if (lay.n_device) {   // the pinned result buffer is allocated by the first cls_resident_fetch
        DevBuf d_src, d_woff, d_len;
        std::vector<ReadDesc> descs(lay.n_device);
        std::vector<uint64_t> src_dev(lay.n_device);
        std::vector<uint32_t> len_dev(lay.n_device);
        parallel_for(lay.n_device, 1 << 15, [&](uint64_t j0, uint64_t j1) {
            for (uint64_t j = j0; j < j1; ++j) {
                const uint32_t i = lay.perm[j];
                descs[j] = ReadDesc{word_off[j], lens[i]};
                src_dev[j] = src[i];
                len_dev[j] = lens[i];
            }
        });
        CU_TRY(d_src.reserve(src_dev.size() * 8)); CU_TRY(d_woff.reserve(word_off.size() * 4)); CU_TRY(d_len.reserve(len_dev.size() * 4));
        CU_TRY(cudaMemcpyAsync(d_src.p, src_dev.data(), src_dev.size() * 8, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_woff.p, word_off.data(), (size_t)lay.n_device * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_len.p, len_dev.data(), len_dev.size() * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(rb->d_descs.p, descs.data(), descs_b, cudaMemcpyHostToDevice, st));
        CU_TRY(launch_fasta_pack(d_codes, (const uint64_t *)d_src.p, (const uint32_t *)d_woff.p, (const uint32_t *)d_len.p,
                                 lay.n_device, (uint32_t *)rb->d_words.p, home->sm_count, st));
        CU_TRY(cudaMemsetAsync(rb->d_results.p, 0xFF, res_b, st));
        CU_TRY(cudaStreamSynchronize(st));
    }
    records->n_records = rb->fa_length.size();
    records->header_begin = rb->fa_header_begin.data();
    records->header_end = rb->fa_header_end.data();
    records->length = rb->fa_length.data();
    *out = rb.release();
    return CLS_OK;
} CLS_ABI_CATCH

}  // namespace cls

extern "C" {

int cls_batch_upload(cls_index *ix, const cls_batch *batch, cls_resident_batch **out) try {
    if (!ix || !batch || !out) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    ix = resident_home(ix);
    *out = nullptr;
    CU_TRY(cudaSetDevice(ix->device));
    auto rb = std::make_unique<cls_resident_batch>();
    rb->device = ix->device;
    std::vector<uint32_t> word_off;
    int rc = plan_batch(batch, ix->dix.k_size, ix->dix.max_fanout, rb->lay, word_off);
    if (rc != CLS_OK) return rc;
    const PackedLayout &lay = rb->lay;
    const size_t words_b = (size_t)lay.n_words * 4, descs_b = (size_t)lay.n_device * sizeof(ReadDesc),
                 res_b = (size_t)lay.n_device * sizeof(ResultRec);
    std::vector<uint32_t> words(lay.n_words + 4);
    std::vector<ReadDesc> descs(lay.n_device);
    pack_batch(batch, rb->lay, word_off, words.data(), descs.data());
    CU_TRY(rb->d_words.reserve(words_b + 16)); CU_TRY(rb->d_descs.reserve(descs_b + 16)); CU_TRY(rb->d_results.reserve(res_b + 32));
    CU_TRY(rb->h_results.reserve(res_b + 32));
    CU_TRY(cudaMemcpy(rb->d_words.p, words.data(), words_b, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(rb->d_descs.p, descs.data(), descs_b, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(rb->d_results.p, 0xFF, res_b));
    *out = rb.release();
    return CLS_OK;
} CLS_ABI_CATCH

// ---- FASTA ingest on the device (SURVEY.md section 8f row 3; file_or_stdin.rs:76-116, sequence.rs:47-56) -----------
int cls_fasta_upload(cls_index *ix, const uint8_t *text, uint64_t n_bytes, cls_resident_batch **out, cls_fasta_records *records) try {
    if (!ix || !out || !records || (n_bytes && !text)) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    ix = resident_home(ix);
    *out = nullptr;
    std::memset(records, 0, sizeof *records);
    if (n_bytes >= (1ull << 32)) return fail(CLS_ERR_UNSUPPORTED, "FASTA text of 4 GiB or more: split it (the tile summaries count in 32 bits)");
    CU_TRY(cudaSetDevice(ix->device));
    static const bool dbg = getenv("CLS_DEBUG_TIMING") != nullptr;
    double tlast = now_ms();
    auto lap = [&](const char *what) { if (dbg) { const double t = now_ms(); fprintf(stderr, "[fasta] %-22s %8.2f ms\n", what, t - tlast); tlast = t; } };
    cudaStream_t st = nullptr;
    DevBuf d_text, d_tiles, d_bases, d_misc, d_codes, d_hpos, d_hkept, d_hflag;
    const uint32_t nt = fasta_n_tiles(n_bytes);
    TileBase totals{0, 0, 0, 0};
    uint32_t non_ascii = 0;
    if (n_bytes) {
        CU_TRY(d_text.reserve(n_bytes + 16)); CU_TRY(d_tiles.reserve((size_t)nt * fasta_tile_bytes())); CU_TRY(d_bases.reserve((size_t)nt * sizeof(TileBase)));
        CU_TRY(d_misc.reserve(256));
        lap("alloc");
        CU_TRY(cudaMemcpyAsync(d_text.p, text, n_bytes, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemsetAsync(d_misc.p, 0, 256, st));
        TileBase *d_totals = (TileBase *)d_misc.p;
        uint32_t *d_non_ascii = (uint32_t *)((char *)d_misc.p + 128);
        CU_TRY(launch_fasta_scan((const uint8_t *)d_text.p, n_bytes, d_tiles.p, (TileBase *)d_bases.p, d_totals, d_non_ascii, st));
        CU_TRY(cudaMemcpyAsync(&totals, d_totals, sizeof totals, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(&non_ascii, d_non_ascii, 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        lap("h2d + scan");
    }
    if (non_ascii)
        return fail(CLS_ERR_UNSUPPORTED, "non-ASCII byte in the FASTA text: Rust's to_uppercase() is Unicode-aware - use the host reader for this file");
    const uint64_t n_hdr = totals.hdrs, n_kept = totals.kept;
    if (n_hdr >= 0xFFFFFFFFull) return fail(CLS_ERR_UNSUPPORTED, "more than 2^32-1 header lines");
    std::vector<uint64_t> hpos(n_hdr), hkept(n_hdr);
    std::vector<uint32_t> hflag(n_hdr);
    if (n_hdr || n_kept) {
        CU_TRY(d_codes.reserve(n_kept + 16)); CU_TRY(d_hpos.reserve(n_hdr * 8 + 8)); CU_TRY(d_hkept.reserve(n_hdr * 8 + 8)); CU_TRY(d_hflag.reserve(n_hdr * 4 + 4));
        CU_TRY(cudaMemsetAsync(d_hflag.p, 0, n_hdr * 4 + 4, st));
        CU_TRY(launch_fasta_write((const uint8_t *)d_text.p, n_bytes, (const TileBase *)d_bases.p, (uint8_t *)d_codes.p, (uint64_t *)d_hpos.p,
                                  (uint64_t *)d_hkept.p, (uint32_t *)d_hflag.p, st));
        if (n_hdr) {
            CU_TRY(cudaMemcpyAsync(hpos.data(), d_hpos.p, n_hdr * 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaMemcpyAsync(hkept.data(), d_hkept.p, n_hdr * 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaMemcpyAsync(hflag.data(), d_hflag.p, n_hdr * 4, cudaMemcpyDeviceToHost, st));
        }
        CU_TRY(cudaStreamSynchronize(st));
        lap("write + d2h");
    }
    // ---- the record rules of the reader (file_or_stdin.rs:91-113) on the per-header-line facts -----------------
    std::vector<uint64_t> src, hb, he;   // first kept base, header line of every record that is sent
    std::vector<uint32_t> ln;
    hb.reserve(n_hdr); src.reserve(n_hdr); ln.reserve(n_hdr);
    const bool orphan_sequence = n_hdr && hkept[0] > 0;   // bases before the first header: the reader errors out at that header (:96-100)
    if (n_hdr && !orphan_sequence) {
        for (uint64_t j = 0; j < n_hdr; ++j) {
            const bool last = j + 1 == n_hdr;
            const uint64_t kept = (last ? n_kept : hkept[j + 1]) - hkept[j];
            if (kept >= (1ull << 31)) return fail(CLS_ERR_INVALID_ARGUMENT, "query longer than 2^31 bases");
            if (!hflag[j]) {                    // header text empty after removing '>': the reader holds no header
                if (kept && !last) break;       // ... and errors out at the next header line (:96-100)
                continue;
            }
            if (last && kept == 0) continue;    // trailing record without sequence is dropped (:111-113)
            hb.push_back(hpos[j]);
            src.push_back(hkept[j]);
            ln.push_back((uint32_t)kept);
        }
    }
    lap("record rules");
    const uint64_t n = hb.size();
    he.resize(n);
    parallel_for(n, 4096, [&](uint64_t a, uint64_t b) {   // end of the header line's content: "\n" or "\r\n" excluded
        for (uint64_t i = a; i < b; ++i) {
            const uint8_t *s = text + hb[i];
            const void *nl = std::memchr(s, '\n', n_bytes - hb[i]);
            uint64_t e = nl ? (uint64_t)((const uint8_t *)nl - text) : n_bytes;
            if (nl && e > hb[i] && text[e - 1] == '\r') --e;
            he[i] = e;
        }
    });
    lap("header ends");
    const int rc = ingest_finish(ix, (const uint8_t *)d_codes.p, hb, he, ln, src, st, out, records);
    if (rc != CLS_OK) return rc;
    lap("pack");
    return CLS_OK;
} CLS_ABI_CATCH

int cls_place_resident(cls_index *ix, cls_resident_batch *rb, const cls_params *params, void *stream) try {
    if (!ix || !rb || !params) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    if (ix->sharded) return ix->sharded->place_resident(ix, rb, params, (cudaStream_t)stream);
    ix = resident_home(ix);
    if (rb->device != ix->device) return fail(CLS_ERR_INVALID_ARGUMENT, "resident batch lives on another device");
    if (ix->n_shards > 1) return fail(CLS_ERR_INVALID_ARGUMENT, "this handle holds one shard of the index: use the routed calls");
    CU_TRY(cudaSetDevice(ix->device));
    uint64_t launches = 0;
    int rc = launch_classes(ix, rb->lay, params, (const uint32_t *)rb->d_words.p, (const ReadDesc *)rb->d_descs.p,
                            (ResultRec *)rb->d_results.p, (cudaStream_t)stream, rb->d_scratch, &launches);
    if (rc == CLS_OK) { std::lock_guard<std::mutex> lk(ix->mu); ix->timing.kernel_launches = launches; }
    return rc;
} CLS_ABI_CATCH

int cls_resident_fetch(cls_index *ix, cls_resident_batch *rb, void *stream, cls_result *result) try {
    if (!ix || !rb || !result) return fail(CLS_ERR_INVALID_ARGUMENT, "NULL argument");
    ix = resident_home(ix);
    CU_TRY(cudaSetDevice(ix->device));
    const size_t res_b = (size_t)rb->lay.n_device * sizeof(ResultRec);
    if (res_b) {
        CU_TRY(rb->h_results.reserve(res_b + 32));
        CU_TRY(cudaMemcpyAsync(rb->h_results.p, rb->d_results.p, res_b, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    }
    CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    scatter_host_decided(rb->lay, ix->dix.k_size, result);
    scatter_device_range(rb->lay, (const ResultRec *)rb->h_results.p, result, 0, rb->lay.n_device);
    return CLS_OK;
} CLS_ABI_CATCH

void cls_resident_destroy(cls_resident_batch *rb) { delete rb; }

uint64_t cls_resident_bytes(const cls_resident_batch *rb) {
    if (!rb) return 0;
    return (uint64_t)rb->lay.n_words * 4 + (uint64_t)rb->lay.n_device * (sizeof(ReadDesc) + sizeof(ResultRec));
}

}  // extern "C"
