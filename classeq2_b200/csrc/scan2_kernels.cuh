// scan2_kernel: the scan kernel of the short-read path (k = 35, closed models, reads of up to 290 bases),
// second generation.  One warp per read; per read it leaves the distinct {node-set record, number of distinct
// hits} pairs for descend_kernel, as scan_kernel<true, true> did, but the per-hit work is cut to a few
// instructions that every lane executes together:
//
//   hash      one pass (32 windows) per loop iteration, the pass's bucket load stays IN FLIGHT while the next pass
//             is hashed; the pre-mix ring halves alternate by an XOR on the shared-memory addresses
//   dedup     (distinct-hash semantics of the reference's HashSets, kmers_map.rs:273-311) a per-warp 8 192-bit
//             test-and-set filter indexed by hash bits: one ATOMS.OR per lane and pass.  A set bit only means
//             "maybe seen": those lanes (about 1.4 % of the hits) compare their table slot against the slots of
//             all earlier hits of the read, which are kept in a list - exact.
//   histogram one match.any per pass elects a leader per node-set record of the pass; the leaders APPEND
//             {record, count} to a list (ballot + popc, no atomics, no probing).  At the end of the read the list
//             (about 30 entries for a 150-base read) is merged by node-set record in a 128-slot table, 32 entries
//             per round with every lane active, and written out compacted.
//   overflow  reads with more than kListCap list entries or more than so.cap distinct node sets go to a list; the
//             first-generation kernel (scan_kernel<true, false>) finishes them after the descent kernel.
//
// Reads are handed out in blocks of kReadBlock from a global counter: a static stride left the SMs that drew
// cheap (unrelated) reads idle at the end of the launch (12 % of the step, measured).
//
// Included by kernels.cu inside namespace cls { namespace { ... } }.
#pragma once

// ---- explicit shared-state-space accesses: 32-bit addresses, register + immediate operands --------------
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t lds_u64(uint32_t a) {
    uint64_t v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds_v2(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u64(uint32_t a, uint64_t v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void sts_v2(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void sts_v4(uint32_t a, uint32_t v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atoms_or(uint32_t a, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.or.b32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ uint32_t atoms_cas(uint32_t a, uint32_t cmp, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "r"(a), "r"(cmp), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ void reds_add(uint32_t a, uint32_t v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// the bucket load of the lanes that have a window in the pass (the others keep their registers)
__device__ __forceinline__ void ld_bucket_if(bool p, uint64_t table, uint32_t bucket, uint64_t &h0, uint64_t &m0, uint64_t &h1,
                                             uint64_t &m1);
constexpr uint32_t kListCap = 128;     // list area in entries
constexpr uint32_t kListUse = 128;     // {node-set record, count} entries a read may append before the merge
constexpr uint32_t kMergeSlots = 128;  // slots of the merge table (> kListUse: probing always terminates)
// reads a warp takes from the global counter at a time: small, so that the last block of a launch is a small share of
// a warp's work even in the chunked launches of cls_place_batch (about 30 reads per warp)
constexpr uint32_t kScanBlock = 2;

// Per-warp shared memory, byte offsets from the warp's base (a multiple of 512: the ring halves alternate by
// an XOR with 256 on the address).  PPS = passes per strand the geometry allows: 4 (reads of up to 162 bases)
// or 8 (up to 290).
template <int PPS>
struct Scan2Layout {
    static constexpr uint32_t kStrWords = PPS == 4 ? 48 : 80;   // ASCII strand: 16-base groups + over-read pad
    static constexpr uint32_t kPkWords = PPS == 4 ? 16 : 24;    // 2-bit packed strand, padded
    static constexpr uint32_t oRingA = 0;                        // 64 x u64: k1 pre-mixes by byte offset mod 64
    static constexpr uint32_t oRingB = 512;                      // 64 x u64: k2 pre-mixes
    static constexpr uint32_t oLut = 1024;                       // 64 x u64: pre-mix of the 3-byte tail by 2-bit codes
    static constexpr uint32_t oFilter = 1536;                    // 256 words: the test-and-set filter; after the last pass
    static constexpr uint32_t oMergeKey = oFilter;               //   the merge table: 128 keys ...
    static constexpr uint32_t oMergeCnt = oFilter + 512;         //   ... and 128 counts
    static constexpr uint32_t oKeys = 2560;                      // 64 * PPS words: table slot of the hit of (pass, lane)
    static constexpr uint32_t oList = oKeys + 256 * PPS;         // kListCap x {record, count}
    static constexpr uint32_t oStrF = oList + 8 * kListCap;
    static constexpr uint32_t oStrR = oStrF + 4 * kStrWords;
    static constexpr uint32_t oPkF = oStrR + 4 * kStrWords;
    static constexpr uint32_t oPkR = oPkF + 4 * kPkWords;
    static constexpr uint32_t kBytes = (oPkR + 4 * kPkWords + 511u) & ~511u;

    static constexpr uint32_t kMaxLen = 32 * PPS + 34;
};

// pre-mixes of the 8-byte word at this lane's byte offset of a strand (three aligned words at `src`), both
// murmur lanes, into the ring entry at `dst`
__device__ __forceinline__ void premix_ring(uint32_t src, uint32_t sh8, uint32_t dst) {
    const uint32_t r0 = lds_u32(src), r1 = lds_u32(src + 4), r2 = lds_u32(src + 8);
    const uint64_t x = pack64(__funnelshift_r(r0, r1, sh8), __funnelshift_r(r1, r2, sh8));
    sts_u64(dst, premix_k1(x));
    sts_u64(dst + 512, premix_k2(x));
}

__device__ __forceinline__ void ld_bucket_if(bool p, uint64_t table, uint32_t bucket, uint64_t &h0, uint64_t &m0, uint64_t &h1,
                                             uint64_t &m1) {
    asm volatile("{\n\t"
                 ".reg .pred p;\n\t"
                 ".reg .u64 a;\n\t"
                 "setp.ne.u32 p, %6, 0;\n\t"
                 "mad.wide.u32 a, %5, 32, %4;\n\t"
                 "@p ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [a];\n\t"
                 "}"
                 : "+l"(h0), "+l"(m0), "+l"(h1), "+l"(m1)
                 : "l"(table), "r"(bucket), "r"((uint32_t)p));
}

// 16 two-bit codes -> 16 ASCII letters (four words), by spreading the codes into nibbles for PRMT on "ACTG"
__device__ __forceinline__ void decode16(uint32_t v, uint32_t (&out)[4]) {
#pragma unroll
    for (int hlf = 0; hlf < 2; ++hlf) {
        uint32_t x = hlf ? v >> 16 : v & 0xFFFFu;
        x = (x | (x << 8)) & 0x00FF00FFu;
        x = (x | (x << 4)) & 0x0F0F0F0Fu;
        x = (x | (x << 2)) & 0x33333333u;
        out[2 * hlf] = __byte_perm(kAsciiLut, 0u, x & 0xFFFFu);
        out[2 * hlf + 1] = __byte_perm(kAsciiLut, 0u, x >> 16);
    }
}

// decode_read for reads of at most 16 packed words (PPS = 4 geometry): lanes 0-15 own the forward words, lanes
// 16-31 the reverse-complement words (built from the forward ones by shuffles); one 16-byte store per lane.
template <int PPS>
__device__ __forceinline__ void decode_read16(const uint32_t *__restrict__ packed, uint32_t len, uint32_t wb) {
    using Ly = Scan2Layout<PPS>;
    const uint32_t lane = threadIdx.x & 31u, t = lane & 15u;
    const uint32_t nw = (len + 15u) >> 4;
    const uint32_t pad2 = 2u * (nw * 16u - len);  // unused bits at the top of the last word
    uint32_t w = 0;
    if (lane < nw) w = __ldg(packed + lane);
    const uint32_t r = revcomp16(w);
    // reverse-complement word t = bases [16t, 16t + 16) of the reversed string
    const uint32_t a = __shfl_sync(kFull, r, (nw - 1u - t) & 31u), b = __shfl_sync(kFull, r, (nw - 2u - t) & 31u);
    uint32_t v = w;
    if (lane >= 16) v = t < nw ? __funnelshift_r(a, t + 1u < nw ? b : 0u, pad2) : 0u;
    uint32_t q[4];
    decode16(v, q);
    const uint32_t sbase = wb + (lane >= 16 ? Ly::oStrR : Ly::oStrF) + 16u * t;
    if (t < Ly::kStrWords / 4)
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(sbase), "r"(q[0]), "r"(q[1]), "r"(q[2]), "r"(q[3]) : "memory");
    sts_u32(wb + (lane >= 16 ? Ly::oPkR : Ly::oPkF) + 4u * t, v);
}

// One pass (32 windows) whose bucket load is in flight.
struct Flight {
    uint64_t h, q0, qm0, q1, qm1;   // window hash of this lane; the two slots {hash, set_off | code << 32} of its bucket
    uint32_t gate;                  // the window's bucket-key prefix code
    int32_t lim;                    // windows left in the strand when the pass began (warp-uniform): lane < lim has a window
};

// Per-lane constants and per-read state of the scan loop.
struct Scan2Ctx {
    uint32_t wb;                    // shared-memory address of the warp's area
    uint32_t A0, O1, O2, O3;        // ring entries: A0 + immediates when a pass's chunk sits in half 0; the three wrapped ones for half 1
    uint32_t sh8, sh2, lt, str_lane, pk_lane;
    uint32_t code_mask, bmask;
    uint32_t W, n_chunks, n_total;
    uint32_t n_list, gate_next;
    uint32_t sb, pb;                // running shared-memory addresses: the next 32 offsets of the strand, the next tail words
    int32_t lim;                    // windows of the strand not hashed yet
    uint64_t table;                 // global address of the k-mer table
};

// Hash part of pass `it` (HALF = it & 1 = the ring half that holds the pass's own 32 offsets).
template <int PPS, int HALF>
__device__ __forceinline__ void scan2_hash(Scan2Ctx &cx, uint32_t it, Flight &f) {
    using Ly = Scan2Layout<PPS>;
    if (it == 0 || it == cx.n_chunks) {  // a strand begins: its first 32 offsets go to the half this pass reads first
        const bool rc = it != 0;
        const uint32_t s0 = cx.wb + (rc ? Ly::oStrR : Ly::oStrF) + cx.str_lane, p0 = cx.wb + (rc ? Ly::oPkR : Ly::oPkF) + cx.pk_lane;
        premix_ring(s0, cx.sh8, cx.A0 + 256u * HALF);
        cx.gate_next = __funnelshift_r(lds_u32(p0), lds_u32(p0 + 4), cx.sh2);
        cx.sb = s0 + 32u; cx.pb = p0 + 8u; cx.lim = (int32_t)cx.W;
    }
    premix_ring(cx.sb, cx.sh8, cx.A0 + 256u * (1 - HALF));  // the next 32 offsets -> the other half
    __syncwarp();
    uint64_t a0, b1, a2, b3;
    if (HALF == 0) {
        a0 = lds_u64(cx.A0); b1 = lds_u64(cx.A0 + 512u + 64u); a2 = lds_u64(cx.A0 + 128u); b3 = lds_u64(cx.A0 + 512u + 192u);
    } else {
        a0 = lds_u64(cx.A0 + 256u); b1 = lds_u64(cx.O1); a2 = lds_u64(cx.O2); b3 = lds_u64(cx.O3);
    }
    // bases pos + 32 ...: the 3-base tail of this pass's windows, and the bucket-key prefix of the next pass's
    const uint32_t tv = __funnelshift_r(lds_u32(cx.pb), lds_u32(cx.pb + 4u), cx.sh2);
    __syncwarp();
    f.h = window_hash35(a0, b1, a2, b3, lds_u64(cx.wb + Ly::oLut + ((tv << 3) & 0x1F8u)));
    f.gate = cx.gate_next & cx.code_mask;
    f.lim = cx.lim;
    cx.gate_next = tv;
    cx.sb += 32u; cx.pb += 8u; cx.lim -= 32;
}

// Consume the bucket of pass `pi`: match, gate by bucket key, de-duplicate, append to the read's list.
template <int PPS>
__device__ __forceinline__ void scan2_consume(Scan2Ctx &cx, const DeviceIndex &ix, const WarpMem &wm, uint32_t pi, Flight &f) {
    using Ly = Scan2Layout<PPS>;
    const uint32_t lane = threadIdx.x & 31u;
    // lanes past the last window of the strand hashed whatever the strings hold there: ignored
    const bool valid = (int32_t)lane < f.lim;
    uint32_t b = (uint32_t)f.h & cx.bmask;
    // free slots carry a hash that no probe of their bucket can ask for (index_build.cpp), so equality is a hit
    bool e0 = f.q0 == f.h, e1 = f.q1 == f.h;
    // rare: the bucket overflowed at build time and the hash is not in it - follow the chain (all lanes stay together)
    // ... and the home bucket's filter (index_build.cpp: one of eight bits per entry that went elsewhere) has its bit
    bool chase = valid && !(e0 || e1) && (((uint32_t)(f.qm1 >> 32) >> (kBloomShift + (((uint32_t)(f.h >> 32) >> 8) & 7u))) & 1u);
    while (__any_sync(kFull, chase)) {
        if (chase) {
            b = (b + 1) & cx.bmask;
            ld_bucket_if(true, cx.table, b, f.q0, f.qm0, f.q1, f.qm1);
            e0 = f.q0 == f.h; e1 = f.q1 == f.h;
            chase = !(e0 || e1) && ((uint32_t)(f.qm0 >> 32) & kOverflowBit);
        }
    }
    bool hit = valid && (e0 || e1);
    const uint64_t mm = e0 ? f.qm0 : f.qm1;
    const uint32_t want = (uint32_t)(mm >> 32) & kCodeMask;
    // rarer still: the entry's bucket key is not the one of this window's own prefix (models whose bucket keys disagree
    // with their k-mers; kmers_map.rs:55-70 accepts the key of ANY window of the query)
    if (__any_sync(kFull, hit && f.gate != want)) {
        if (hit && f.gate != want) {
            hit = false;
            for (uint32_t q = 0; q < cx.W && !hit; ++q)
                hit = packed_bits(wm.pk_f, q, cx.code_mask) == want || packed_bits(wm.pk_r, q, cx.code_mask) == want;
        }
        __syncwarp();
    }
    const uint32_t set_off = (uint32_t)mm;
    const uint32_t slot_key = 2u * b + (e0 ? 0u : 1u);
    // test-and-set filter on 13 hash bits the bucket index does not use first; a miss ORs nothing in
    const uint32_t hh = (uint32_t)(f.h >> 32);
    const uint32_t fbit = hit ? 1u << ((hh >> 8) & 31u) : 0u;
    const uint32_t old = atoms_or(cx.wb + Ly::oFilter + ((hh >> 11) & 0x3FCu), fbit);
    const uint32_t key_row = cx.wb + Ly::oKeys + 128u * pi + 4u * lane;
    sts_u32(key_row, hit ? slot_key : kEmpty);
    const uint32_t cm = __ballot_sync(kFull, (old & fbit) != 0);
    bool fresh = hit;
    if (cm) {  // warp-uniform, rare: the exact answer for the lanes whose filter bit was already set
        __syncwarp();
        uint32_t todo = cm;
        while (todo) {
            const uint32_t src = (uint32_t)__ffs(todo) - 1u;
            todo &= todo - 1u;
            const uint32_t key = __shfl_sync(kFull, slot_key, src);
            bool found = false;
            for (uint32_t a = cx.wb + Ly::oKeys + 4u * lane; a < key_row; a += 128u) found |= lds_u32(a) == key;
            const uint32_t earlier = __ballot_sync(kFull, found);
            const uint32_t same = __ballot_sync(kFull, hit && slot_key == key) & ~(1u << src);
            // a duplicate if the slot was hit in an earlier pass, or in this pass by a lane that found the bit clear
            // (there is at most one), or - all of them candidates - by a lower lane
            const bool dup = earlier != 0 || (same & ~cm) != 0 || (same & ((1u << src) - 1u)) != 0;
            if (lane == src && dup) fresh = false;
        }
    }
    // one leader per node-set record of the pass appends {record, distinct hits}; lanes without a fresh hit hold unique keys
    const uint32_t peers = __match_any_sync(kFull, fresh ? set_off : (0x80000000u | lane));
    const bool lead = fresh && (peers & cx.lt) == 0;
    const uint32_t lm = __ballot_sync(kFull, lead);
    const uint32_t at = cx.n_list + (uint32_t)__popc(lm & cx.lt);
    if (lead && at < kListUse) sts_v2(cx.wb + Ly::oList + 8u * at, set_off, (uint32_t)__popc(peers));
    cx.n_list += (uint32_t)__popc(lm);
}

template <int PPS, int HALF>
__device__ __forceinline__ void scan2_step(Scan2Ctx &cx, const DeviceIndex &ix, const WarpMem &wm, uint32_t it, Flight &cur, Flight &prev) {
    const bool more = it < cx.n_total;   // warp-uniform
    if (more) scan2_hash<PPS, HALF>(cx, it, cur);
    if (it > 0 && it <= cx.n_total) scan2_consume<PPS>(cx, ix, wm, it - 1u, prev);
    if (more) {
        const bool valid = (int32_t)(threadIdx.x & 31u) < cur.lim;
        ld_bucket_if(valid, cx.table, (uint32_t)cur.h & cx.bmask, cur.q0, cur.qm0, cur.q1, cur.qm1);
    }
}

// MINB = resident CTAs per SM ptxas is asked for: 5 (48 registers, 40 warps per SM) hides the HBM latency of a table that
// does not fit L2 (config 3: 5.14 against 5.36 ms per 1 M reads); 4 (64 registers, no re-materialised constants) is the
// faster one when the table is L2-resident (config 2: 4.14 against 4.24 ms).  The launcher picks by table size.
template <int PPS, int MINB>
__global__ void __launch_bounds__(256, MINB)
    scan2_kernel(DeviceIndex ix, const uint32_t *__restrict__ packed, const ReadDesc *__restrict__ reads, uint32_t first_read,
                 uint32_t n_reads, ScanOut so) {
    using Ly = Scan2Layout<PPS>;
    extern __shared__ __align__(1024) uint32_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    uint32_t *wbase = smem + (size_t)warp * (Ly::kBytes / 4);
    Scan2Ctx cx;
    cx.wb = smem_addr(wbase);
    for (uint32_t i = lane; i < 64; i += 32) {
        const uint64_t t = (uint64_t)((kAsciiLut >> (8 * (i & 3))) & 0xFF) | ((uint64_t)((kAsciiLut >> (8 * ((i >> 2) & 3))) & 0xFF) << 8) |
                           ((uint64_t)((kAsciiLut >> (8 * ((i >> 4) & 3))) & 0xFF) << 16);
        sts_u64(cx.wb + Ly::oLut + 8 * i, premix_k1(t));
    }
    WarpMem wm;
    wm.ring_a = nullptr; wm.ring_b = nullptr;
    wm.str_f = wbase + Ly::oStrF / 4; wm.str_r = wbase + Ly::oStrR / 4;
    wm.pk_f = wbase + Ly::oPkF / 4; wm.pk_r = wbase + Ly::oPkR / 4;
    cx.code_mask = ix.m_eff >= 16 ? 0xFFFFFFFFu : ((1u << (2 * ix.m_eff)) - 1u);
    cx.bmask = (uint32_t)ix.bucket_mask;  // at most 2^30 buckets (cls_index_create)
    cx.table = reinterpret_cast<uint64_t>(ix.table);
    cx.sh8 = (lane & 3u) * 8u; cx.sh2 = (lane & 15u) * 2u;
    cx.lt = (1u << lane) - 1u;
    cx.A0 = cx.wb + Ly::oRingA + 8u * lane;
    cx.O1 = cx.wb + Ly::oRingB + 8u * ((lane + 40u) & 63u);
    cx.O2 = cx.wb + Ly::oRingA + 8u * ((lane + 48u) & 63u);
    cx.O3 = cx.wb + Ly::oRingB + 8u * ((lane + 56u) & 63u);
    cx.str_lane = 4u * (lane >> 2); cx.pk_lane = 4u * (lane >> 4);
    __syncwarp();

    uint32_t blk_base = 0, blk_used = kScanBlock;
#pragma unroll 1
    for (;;) {
        if (blk_used == kScanBlock) {
            // a new block of reads: their descriptors (64 bytes) are requested now, in one go
            uint32_t b0 = 0;
            if (lane == 0) b0 = atomicAdd(so.counters, kScanBlock);
            blk_base = __shfl_sync(kFull, b0, 0);
            blk_used = 0;
            if (blk_base >= n_reads) break;
            if (lane < (kScanBlock * 8u + 31u) / 32u) asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char *>(reads + first_read + blk_base) + 32u * lane));
        }
        const uint32_t r = blk_base + blk_used;
        if (r >= n_reads) break;
        ++blk_used;
        // warp-uniform loads: the loop bounds derived from the descriptor live in uniform registers
        const ReadDesc rd = reads[first_read + r];
        const uint32_t L = rd.len;
        if (blk_used < kScanBlock && r + 1u < n_reads) {   // the next read's packed bases, while this one is placed
            const uint32_t nxt = reads[first_read + r + 1u].word_off;
            if (lane < 3) asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char *>(packed + nxt) + 32u * lane));
        }
        cx.W = L - 34u;  // host guarantees 35 <= L <= Ly::kMaxLen
        sts_v4(cx.wb + Ly::oFilter + 16u * lane, 0u);
        sts_v4(cx.wb + Ly::oFilter + 512u + 16u * lane, 0u);
        if constexpr (PPS == 4) decode_read16<PPS>(packed + rd.word_off, L, cx.wb);
        else decode_read(packed + rd.word_off, L, wm, Ly::kPkWords);
        cx.n_chunks = (cx.W + 31u) >> 5; cx.n_total = 2u * cx.n_chunks;
        cx.n_list = 0; cx.gate_next = 0;
        Flight fa, fb;
        fa.h = fa.q0 = fa.qm0 = fa.q1 = fa.qm1 = 0; fa.gate = 0; fa.lim = 0;
        cx.sb = cx.pb = 0; cx.lim = 0;
        fb = fa;
        __syncwarp();
        // two passes per iteration: the ring halves and the two register sets alternate; pass `it` is hashed, the
        // bucket of pass it - 1 (in flight meanwhile) is consumed, then the bucket of pass `it` is requested
#pragma unroll 1
        for (uint32_t it = 0; it <= cx.n_total; it += 2) {   // n_total is even: the last iteration only consumes
            scan2_step<PPS, 0>(cx, ix, wm, it, fa, fb);
            scan2_step<PPS, 1>(cx, ix, wm, it + 1u, fb, fa);
        }
        // ---- hand the read over: the list itself, or merged by node-set record when it is long --------------------
        __syncwarp();
        bool overflow = cx.n_list > kListUse;
        uint32_t D = 0, n_matched = 0;
        uint2 *row = so.pairs + (size_t)r * so.cap;
        if (cx.n_list <= 32) {
            // one entry per lane: entries of the same node-set record are summed into the lowest lane that holds it (the
            // descent kernel runs several reads side by side when they have few node sets, so fewer pairs pay)
            const bool valid = lane < cx.n_list;
            uint2 e = make_uint2(0u, 0u);
            if (valid) e = lds_v2(cx.wb + Ly::oList + 8u * lane);
            const uint32_t peers = __match_any_sync(kFull, valid ? e.x : (0x80000000u | lane));
            const uint32_t leader = (uint32_t)__ffs(peers) - 1u;
            const bool is_lead = valid && leader == lane;
            if (valid && !is_lead) reds_add(cx.wb + Ly::oList + 8u * leader + 4u, e.y);
            __syncwarp();
            uint32_t wsum = 0;
            if (is_lead) wsum = lds_u32(cx.wb + Ly::oList + 8u * lane + 4u);
            const uint32_t lm = __ballot_sync(kFull, is_lead);
            if (is_lead) row[__popc(lm & cx.lt)] = make_uint2(e.x, wsum);
            n_matched = __reduce_add_sync(kFull, wsum);   // every distinct hit is in exactly one count
            D = (uint32_t)__popc(lm);
        } else if (!overflow) {
            sts_v4(cx.wb + Ly::oMergeKey + 16u * lane, kEmpty);
            sts_v4(cx.wb + Ly::oMergeCnt + 16u * lane, 0u);
            __syncwarp();
            for (uint32_t base = 0; base < cx.n_list; base += 32) {
                const uint32_t j = base + lane;
                bool pending = j < cx.n_list;
                uint2 e = make_uint2(0u, 0u);
                if (pending) e = lds_v2(cx.wb + Ly::oList + 8u * j);
                uint32_t p = (e.x * 0x9E3779B1u) >> 25;
                while (__any_sync(kFull, pending)) {
                    if (pending) {
                        const uint32_t was = atoms_cas(cx.wb + Ly::oMergeKey + 4u * p, kEmpty, e.x);
                        if (was == kEmpty || was == e.x) { reds_add(cx.wb + Ly::oMergeCnt + 4u * p, e.y); pending = false; }
                        else p = (p + 1u) & (kMergeSlots - 1u);
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (uint32_t q = 0; q < kMergeSlots / 32; ++q) {
                const uint32_t sl = 32u * q + lane;
                const uint32_t key = lds_u32(cx.wb + Ly::oMergeKey + 4u * sl), cnt = lds_u32(cx.wb + Ly::oMergeCnt + 4u * sl);
                const bool has = key != kEmpty;
                const uint32_t bm = __ballot_sync(kFull, has);
                const uint32_t at = D + (uint32_t)__popc(bm & cx.lt);
                if (has && at < so.cap) row[at] = make_uint2(key, cnt);
                D += (uint32_t)__popc(bm);
                n_matched += cnt;
            }
            n_matched = __reduce_add_sync(kFull, n_matched);
            overflow = D > so.cap;
        }
        if (lane == 0) {
            so.meta[r] = make_uint2(n_matched, overflow ? kDone : D);
            if (overflow) so.ov_list[atomicAdd(so.counters + 2, 1u)] = r;
        }
        __syncwarp();  // the merge table is the next read's filter
    }
}
