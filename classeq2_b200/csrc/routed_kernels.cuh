// Kernels of the HASH-SHARDED index (config 5 of BASELINE.json, SURVEY.md section 8e): the k-mer table is
// split over the GPUs of a box by `owner = (hash >> 61) % n_shards`; node-set records and the
// tree stay replicated (they are small).  A batch goes through three kernels with an all-to-all
// (NCCL over NVLink, done by the caller on the device buffers) between them:
//
//   route_kernel         home GPU, one warp per read: decode + hash every window (the same code as the
//                        placement kernel), group the hashes by owner and append each group to that
//                        owner's segment of the send buffer; the read's run in every segment and the window
//                        of every slot are kept at home
//   shard_probe_kernel   owner GPU, one thread per received hash: probe the local table shard, answer
//                        {node-set record offset | kEmpty, globally unique slot id, bucket prefix code}
//   place_routed_kernel  home GPU, one warp per read: the placement kernel with the table probe replaced
//                        by coalesced reads of the read's runs of replies; gating, de-duplication, histogram
//                        and descent are the shared code (insert_hits, finish_read_reg, finish_read)
//
// Included at the end of kernels.cu (inside namespace cls): it shares that file's device helpers.
#pragma once

struct ProbeReply {      // 12 bytes per routed k-mer on the way back
    uint32_t set_off;    // kEmpty: the hash is not in the index
    uint32_t slot;       // (slot in the owner's table << 3) | owner: equal hashes <=> equal slot ids
    uint32_t code;       // 2-bit prefix code of the entry's bucket key (bucket gating happens at home)
};
static_assert(sizeof(ProbeReply) == 12, "reply must be 12 bytes");

__device__ __forceinline__ uint32_t owner_of(uint64_t h, uint32_t n_shards) { return (uint32_t)(h >> 61) % n_shards; }

// Shared-memory carve-up of one warp (same geometry as the placement kernels).
struct WarpLayout {
    WarpMem wm;
    uint32_t *t1, *t2k, *t2c, *lst, *cnt, *excl, *n_sets;
};
__device__ __forceinline__ WarpLayout carve_warp(uint32_t *smem, const PlaceGeom &g, uint32_t warp, uint32_t warps_per_cta) {
    WarpLayout w;
    uint32_t *gbase = smem + 4 * kRing * warps_per_cta + (size_t)warp * g.words_per_warp;
    w.wm.ring_a = reinterpret_cast<uint64_t *>(smem + 4 * kRing * warp);
    w.wm.ring_b = w.wm.ring_a + kRing;
    w.t1 = gbase;
    w.t2k = w.t1 + g.t1_size;
    w.t2c = w.t2k + g.t2_size;
    w.lst = w.t2c + g.t2_size;
    w.wm.str_f = w.lst + g.t2_size;
    w.wm.str_r = w.wm.str_f + g.str_words;
    w.wm.pk_f = w.wm.str_r + g.str_words;
    w.wm.pk_r = w.wm.pk_f + g.pk_words;
    w.cnt = w.wm.pk_r + g.pk_words;
    w.excl = w.cnt + g.fan_cap;
    w.n_sets = w.excl + g.fan_cap;
    return w;
}

// ---- stage 1 + 2: hash and route ---------------------------------------------------------------
// seg.p[o][i], i < cursor[o]: the hashes owned by shard o, in no particular order.  seg.p[o] is either
// this GPU's send buffer + o * seg_cap (the exchange is then an NCCL all-to-all) or a PEER pointer into
// owner o's inbox (CUDA IPC over NVLink): the stores of this kernel then ARE the exchange, overlapped with
// the hashing of the next reads, and no collective moves the payload.
// The hashes of one read occupy one contiguous RUN per owner: runs[r * 8 + o] = {first slot, count}, and
// slot_win[o * seg_cap + i] = strand * W + pos of the window behind slot i (the reply comes back at the same index).
// *overflow is set when a segment would exceed seg_cap (the caller retries with a larger one).
struct SegPtrs {
    uint64_t *p[8];
};
template <int K>
__global__ void __launch_bounds__(256, 4) route_kernel(uint32_t k, const uint32_t *__restrict__ packed,
                                                       const ReadDesc *__restrict__ reads, uint32_t first_read,
                                                       uint32_t n_reads, PlaceGeom g,
                                                       uint32_t n_shards, uint64_t seg_cap, SegPtrs seg,
                                                       uint16_t *__restrict__ slot_win, uint2 *__restrict__ runs,
                                                       unsigned long long *__restrict__ cursor, uint32_t *__restrict__ overflow) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint64_t tail_lut[64];
    init_tail_lut(tail_lut);
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5, warps_per_cta = blockDim.x >> 5;
    WarpLayout wl = carve_warp(smem, g, warp, warps_per_cta);
    uint64_t *hs = reinterpret_cast<uint64_t *>(wl.t1);  // 2W hashes: t1 holds 2H 32-bit words
    uint64_t *sorted_h = reinterpret_cast<uint64_t *>(wl.t2k);  // the same hashes grouped by owner (t2k + t2c: 2 x t2_size words)
    uint16_t *sorted_w = reinterpret_cast<uint16_t *>(wl.lst);   // the window of every sorted hash
    uint32_t *own_cnt = wl.lst + (g.t2_size >> 1);               // per-owner counts, then running positions
    __syncthreads();
    const uint32_t gwarp = blockIdx.x * warps_per_cta + warp, gstride = gridDim.x * warps_per_cta;
#pragma unroll 1
    for (uint32_t r = gwarp; r < n_reads; r += gstride) {
        const ReadDesc rd = reads[first_read + r];
        const uint32_t L = rd.len, W = L - k + 1;
        if (lane < 16) own_cnt[lane] = 0;
        decode_read(packed + rd.word_off, L, wl.wm, g.pk_words);
        __syncwarp();
        WindowHasher<K> wh(wl.wm, tail_lut, L, k);
        for (uint32_t strand = 0; strand < 2; ++strand) {
            wh.begin_strand(strand);
            for (uint32_t c = 0; c < wh.n_chunks(); ++c) {
                uint32_t pos;
                uint64_t h = 0;
                const bool valid = wh.pass(c, pos, h);
                if (valid) hs[strand * W + pos] = h;
                const uint32_t o = valid ? owner_of(h, n_shards) : 0xFFu;
                const uint32_t peers = __match_any_sync(kFull, o);
                if (valid && (uint32_t)(__ffs(peers) - 1) == lane) atomicAdd(&own_cnt[o], (uint32_t)__popc(peers));
            }
        }
        __syncwarp();
        // reserve this read's share of every owner's segment; own_loc = start of the owner's run in the sorted copy
        uint32_t my_cnt = 0, my_loc = 0;
        uint64_t my_base = 0;
        if (lane < n_shards) my_cnt = own_cnt[lane];
        {
            uint32_t inc = my_cnt;
            for (int d = 1; d < 8; d <<= 1) {
                const uint32_t t = __shfl_up_sync(kFull, inc, d);
                if ((int)lane >= d) inc += t;
            }
            my_loc = inc - my_cnt;
        }
        if (lane < n_shards) {
            my_base = my_cnt ? atomicAdd(&cursor[lane], (unsigned long long)my_cnt) : 0ull;
            const bool fits = my_base + my_cnt <= seg_cap;
            if (!fits) *overflow = 1u;
            runs[(size_t)(first_read + r) * 8 + lane] = make_uint2((uint32_t)my_base, fits ? my_cnt : 0u);
            if (!fits) my_cnt = 0;
            own_cnt[lane] = my_loc;   // running position of the owner inside the sorted copy
        }
        __syncwarp();
        // counting sort by owner into shared memory (window order is kept inside an owner)
        for (uint32_t w0 = 0; w0 < 2 * W; w0 += 32) {
            const uint32_t w = w0 + lane;
            const bool valid = w < 2 * W;
            const uint64_t h = valid ? hs[w] : 0;
            const uint32_t o = valid ? owner_of(h, n_shards) : 0xFFu;
            const uint32_t peers = __match_any_sync(kFull, o);
            const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
            uint32_t cur = 0;
            if (valid) cur = own_cnt[o];
            __syncwarp();
            if (valid) {
                sorted_h[cur + rank] = h;
                sorted_w[cur + rank] = (uint16_t)w;
                if ((uint32_t)(__ffs(peers) - 1) == lane) own_cnt[o] = cur + __popc(peers);
            }
            __syncwarp();
        }
        // one contiguous run per owner: coalesced stores, local or over NVLink
        for (uint32_t o = 0; o < n_shards; ++o) {
            const uint32_t c = __shfl_sync(kFull, my_cnt, o), loc = __shfl_sync(kFull, my_loc, o);
            const uint64_t base = __shfl_sync(kFull, my_base, o);
            uint64_t *dst = seg.p[o] + base;
            uint16_t *dw = slot_win + (uint64_t)o * seg_cap + base;
            for (uint32_t i = lane; i < c; i += 32) {
                dst[i] = sorted_h[loc + i];
                dw[i] = sorted_w[loc + i];
            }
        }
        __syncwarp();
    }
}

// ---- stage 4: the owner answers ---------------------------------------------------------------
// Hashes [blk, blk + blockDim.x) of a segment of `n`: one thread per hash probes the local table shard.
__device__ __forceinline__ void probe_block(const DeviceIndex &ix, uint32_t shard, const uint64_t *__restrict__ hashes, uint64_t n,
                                            ProbeReply *__restrict__ replies, uint64_t blk, uint32_t (*stage)[96]) {
    const uint64_t i = blk + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    ProbeReply rep{kEmpty, 0u, 0u};
    if (i < n) {
        const uint64_t h = hashes[i];
        const uint32_t bmask = (uint32_t)ix.bucket_mask;
        uint32_t b = (uint32_t)h & bmask;
        for (;;) {
            uint64_t h0, m0, h1, m1;
            ld_bucket(ix.table, b, h0, m0, h1, m1);
            if (h0 == h && (uint32_t)m0 != kEmpty) { rep = ProbeReply{(uint32_t)m0, ((2u * b) << 3) | shard, (uint32_t)(m0 >> 32) & kCodeMask}; break; }
            if (h1 == h && (uint32_t)m1 != kEmpty) { rep = ProbeReply{(uint32_t)m1, ((2u * b + 1u) << 3) | shard, (uint32_t)(m1 >> 32) & kCodeMask}; break; }
            if (!((uint32_t)(m0 >> 32) & kOverflowBit)) break;
            b = (b + 1) & bmask;
        }
    }
    // the 32 replies of a warp are 384 contiguous bytes: store them as 24 aligned 16-byte vectors (whole
    // sectors - the destination may be a peer's memory across NVLink, where partial-sector stores cost a packet each)
    const uint64_t i0 = i - lane;
    const bool vector_ok = i0 + 32 <= n && ((reinterpret_cast<uintptr_t>(replies + i0) & 15u) == 0);
    if (vector_ok) {   // (i0 is the same for the whole warp: a full warp of replies takes this path, or none of it)
        stage[warp][3 * lane] = rep.set_off; stage[warp][3 * lane + 1] = rep.slot; stage[warp][3 * lane + 2] = rep.code;
        __syncwarp();
        if (lane < 24) reinterpret_cast<uint4 *>(replies + i0)[lane] = reinterpret_cast<const uint4 *>(stage[warp])[lane];
        __syncwarp();  // a later stride writes the stage again
    } else if (i < n) {
        replies[i] = rep;
    }
}

// DEVICE_COUNT = false: `n` hashes, counted on the host; one thread per hash.  DEVICE_COUNT = true: the count is the sender's
// cursor for this owner, read from device memory (a peer pointer into the sender's route state) and clamped to `n` =
// seg_cap - a cursor that overflowed runs past the segment, and the clamp keeps the probe inside the inbox; the grid is
// sized before the count is known and strides over the segment.
template <bool DEVICE_COUNT>
__global__ void __launch_bounds__(256) shard_probe_kernel(DeviceIndex ix, uint32_t shard, const uint64_t *__restrict__ hashes,
                                                          uint64_t n, const unsigned long long *__restrict__ d_count,
                                                          ProbeReply *__restrict__ replies) {
    __shared__ __align__(16) uint32_t stage[8][96];
    if constexpr (DEVICE_COUNT) {
        __shared__ unsigned long long s_count;
        if (threadIdx.x == 0) s_count = *d_count;   // one load per block (it may cross NVLink)
        __syncthreads();
        if (s_count < n) n = s_count;
#pragma unroll 1
        for (uint64_t blk = (uint64_t)blockIdx.x * blockDim.x; blk < n; blk += (uint64_t)gridDim.x * blockDim.x)
            probe_block(ix, shard, hashes, n, replies, blk, stage);
    } else {
        probe_block(ix, shard, hashes, n, replies, (uint64_t)blockIdx.x * blockDim.x, stage);
    }
}

// ---- stage 6: count and descend at home -------------------------------------------------------
template <bool CLOSED, bool SPLIT>
__global__ void __launch_bounds__(256, 4) place_routed_kernel(DeviceIndex ix, PlaceParams pp, const uint32_t *__restrict__ packed,
                                                              const ReadDesc *__restrict__ reads, uint32_t first_read,
                                                              uint32_t n_reads, ResultRec *__restrict__ results, PlaceGeom g,
                                                              uint32_t n_shards, uint64_t seg_cap, const uint2 *__restrict__ runs,
                                                              const uint16_t *__restrict__ slot_win,
                                                              const ProbeReply *__restrict__ replies, ScanOut so) {
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5, warps_per_cta = blockDim.x >> 5;
    WarpLayout wl = carve_warp(smem, g, warp, warps_per_cta);
    const ReadTables tb{wl.t1, wl.t2k, wl.t2c, wl.lst, wl.cnt, wl.excl, wl.n_sets, g.t1_size - 1u, g.t2_size - 1u, 32u - g.t2_log2};
    const uint32_t k = ix.k_size;
    const uint32_t code_mask = ix.m_eff >= 16 ? 0xFFFFFFFFu : ((1u << (2 * ix.m_eff)) - 1u);
    for (uint32_t o = lane; o < g.fan_cap; o += 32) { wl.cnt[o] = 0; wl.excl[o] = 0; }
    __syncthreads();
    const uint32_t gwarp = blockIdx.x * warps_per_cta + warp, gstride = gridDim.x * warps_per_cta;
#pragma unroll 1
    for (uint32_t r = gwarp; r < n_reads; r += gstride) {
        const ReadDesc rd = reads[first_read + r];
        const uint32_t L = rd.len, W = L - k + 1;
        {
            uint4 *z = reinterpret_cast<uint4 *>(wl.t1);
            const uint32_t n4 = (g.t1_size + g.t2_size) >> 2;
            for (uint32_t i = lane; i < n4; i += 32) z[i] = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
            if (lane == 0) *wl.n_sets = 0;
        }
        decode_read(packed + rd.word_off, L, wl.wm, g.pk_words);  // the packed strands gate the hits
        const uint2 my_run = lane < n_shards ? runs[(size_t)(first_read + r) * 8 + lane] : make_uint2(0u, 0u);
        __syncwarp();
        uint32_t n_matched = 0;
        // the replies of this read come back as one contiguous run per owner: coalesced loads
        for (uint32_t o = 0; o < n_shards; ++o) {
            const uint32_t base = __shfl_sync(kFull, my_run.x, o), cnt = __shfl_sync(kFull, my_run.y, o);
            for (uint32_t i0 = 0; i0 < cnt; i0 += 32) {
                const uint32_t i = i0 + lane;
                const bool valid = i < cnt;
                ProbeReply rep{kEmpty, 0u, 0u};
                uint32_t w = 0;
                if (valid) {
                    const uint64_t idx = (uint64_t)o * seg_cap + base + i;
                    rep = replies[idx];
                    w = slot_win[idx];
                }
                bool hit = valid && rep.set_off != kEmpty;
                if (hit) {
                    // bucket gating: the entry's bucket key must be among the query's prefix keys
                    const bool rc = w >= W;
                    const uint32_t pos = rc ? w - W : w;
                    hit = packed_bits(rc ? wl.wm.pk_r : wl.wm.pk_f, pos, code_mask) == rep.code;
                    if (!hit) {
                        for (uint32_t q = 0; q < W && !hit; ++q)
                            hit = packed_bits(wl.wm.pk_f, q, code_mask) == rep.code || packed_bits(wl.wm.pk_r, q, code_mask) == rep.code;
                    }
                }
                n_matched += insert_hits<false>(tb, hit, rep.slot, rep.set_off);
            }
        }
        __syncwarp();
        const uint32_t D = *wl.n_sets;
        if constexpr (SPLIT) {  // hand the read over to descend_kernel, like scan_kernel does
            if (D <= so.cap) {
                for (uint32_t j = lane; j < D; j += 32) {
                    const uint32_t p2 = wl.lst[j];
                    so.pairs[(size_t)r * so.cap + j] = make_uint2(wl.t2k[p2], wl.t2c[p2]);
                }
                if (lane == 0) so.meta[r] = make_uint2(n_matched, D);
            } else {
                finish_read<CLOSED>(ix, pp, tb, D, n_matched, results + first_read + r);
                if (lane == 0) so.meta[r] = make_uint2(n_matched, kDone);
            }
        } else {
            if (CLOSED && D <= 32) finish_read_reg<1>(ix, pp, tb, D, n_matched, results + first_read + r);
            else if (CLOSED && D <= 64) finish_read_reg<2>(ix, pp, tb, D, n_matched, results + first_read + r);
            else finish_read<CLOSED>(ix, pp, tb, D, n_matched, results + first_read + r);
        }
        __syncwarp();
    }
}

// ---- host launchers -----------------------------------------------------------------------------
static inline cudaError_t routed_smem(const PlaceGeom &g, int &warps, size_t &smem) {
    const size_t ring = (size_t)4 * kRing * 4, group = (size_t)g.words_per_warp * 4;
    warps = 8;
    while (warps > 1 && (group + ring) * warps > 200 * 1024) warps >>= 1;
    smem = (group + ring) * warps;
    return smem > 226 * 1024 ? cudaErrorInvalidConfiguration : cudaSuccess;
}

cudaError_t launch_route(uint32_t k, const uint32_t *packed, const ReadDesc *reads, uint32_t first_read, uint32_t n_reads,
                         const PlaceGeom &g, uint32_t n_shards, uint64_t seg_cap, uint64_t *const *seg_ptrs,
                         uint16_t *slot_win, uint2 *runs, unsigned long long *cursor, uint32_t *overflow, int sm_count, cudaStream_t stream) {
    SegPtrs seg{};
    for (uint32_t o = 0; o < n_shards && o < 8; ++o) seg.p[o] = seg_ptrs[o];
    if (n_reads == 0) return cudaSuccess;
    if (g.cta_per_read || n_shards == 0 || n_shards > 8) return cudaErrorInvalidConfiguration;
    int warps;
    size_t smem;
    cudaError_t e = routed_smem(g, warps, smem);
    if (e != cudaSuccess) return e;
    uint32_t grid = (uint32_t)(sm_count * 4);
    const uint32_t need = (n_reads + warps - 1) / warps;
    if (grid > need) grid = need;
    if (k == 35) {
        if ((e = cudaFuncSetAttribute(route_kernel<35>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024)) != cudaSuccess) return e;
        route_kernel<35><<<grid, warps * 32, smem, stream>>>(k, packed, reads, first_read, n_reads, g, n_shards, seg_cap, seg,
                                                             slot_win, runs, cursor, overflow);
    } else {
        if ((e = cudaFuncSetAttribute(route_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024)) != cudaSuccess) return e;
        route_kernel<0><<<grid, warps * 32, smem, stream>>>(k, packed, reads, first_read, n_reads, g, n_shards, seg_cap, seg,
                                                            slot_win, runs, cursor, overflow);
    }
    return cudaGetLastError();
}

cudaError_t launch_shard_probe(const DeviceIndex &ix, uint32_t shard, const uint64_t *hashes, uint64_t n, void *replies,
                               cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const uint64_t blocks = (n + 255) / 256;
    if (blocks > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
    shard_probe_kernel<false><<<(uint32_t)blocks, 256, 0, stream>>>(ix, shard, hashes, n, nullptr, reinterpret_cast<ProbeReply *>(replies));
    return cudaGetLastError();
}

cudaError_t launch_shard_probe_counted(const DeviceIndex &ix, uint32_t shard, const uint64_t *hashes, uint64_t seg_cap,
                                       const unsigned long long *d_count, void *replies, int sm_count, cudaStream_t stream) {
    if (seg_cap == 0) return cudaSuccess;
    const uint64_t blocks = std::min<uint64_t>((seg_cap + 255) / 256, (uint64_t)sm_count * 8);   // a full SM of 256-thread blocks, grid-stride
    shard_probe_kernel<true><<<(uint32_t)blocks, 256, 0, stream>>>(ix, shard, hashes, seg_cap, d_count, reinterpret_cast<ProbeReply *>(replies));
    return cudaGetLastError();
}

cudaError_t launch_place_routed(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads,
                                uint32_t first_read, uint32_t n_reads, ResultRec *results, const PlaceGeom &g,
                                uint32_t n_shards, uint64_t seg_cap, const uint2 *runs, const uint16_t *slot_win, const void *replies,
                                int sm_count, cudaStream_t stream, void *scratch, size_t scratch_bytes) {
    if (n_reads == 0) return cudaSuccess;
    if (g.cta_per_read) return cudaErrorInvalidConfiguration;
    int warps;
    size_t smem;
    cudaError_t e = routed_smem(g, warps, smem);
    if (e != cudaSuccess) return e;
    uint32_t grid = (uint32_t)(sm_count * 4);
    const uint32_t need = (n_reads + warps - 1) / warps;
    if (grid > need) grid = need;
    const ProbeReply *rp = reinterpret_cast<const ProbeReply *>(replies);
    const bool split = ix.closed && scratch && scratch_bytes >= scratch_bytes_for(n_reads, kPairCap) &&
                       (size_t)2 * g.fan_cap * 4 * 8 <= 48 * 1024;
    ScanOut so = no_scan_out();
    if (split) {
        so = carve_scratch(scratch, n_reads, kPairCap);
        if ((e = cudaMemsetAsync(so.counters, 0, 64, stream)) != cudaSuccess) return e;
    }
    auto kern = split ? place_routed_kernel<true, true> : (ix.closed ? place_routed_kernel<true, false> : place_routed_kernel<false, false>);
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024)) != cudaSuccess) return e;
    kern<<<grid, warps * 32, smem, stream>>>(ix, pp, packed, reads, first_read, n_reads, results, g, n_shards, seg_cap, runs, slot_win, rp, so);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (split) e = launch_descend16(ix, pp, so, first_read, n_reads, results, g.fan_cap, sm_count, stream);
    return e;
}
