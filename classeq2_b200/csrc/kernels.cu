// sm_100a kernels of the placement path.  The stages of one query (one warp per query for short reads -
// scan_kernel then descend_kernel - or one CTA per query for kb-scale reads - place_kernel):
//
//   decode   2-bit packed bases -> forward + reverse-complement ASCII strings (and the packed
//            reverse complement) in shared memory
//            (reference: kmers_map.rs:375-398 build_kmer_from_string, :431-443 reverse_complement)
//   hash     murmur3_x64_128(window).0 for every window of both strands, one window per lane
//            (kmers_map.rs:405-424, :157-159).  k = 35: the two per-word pre-mixes of every
//            8-byte word are computed ONCE per byte offset and shared between the four windows
//            that use them through a shared-memory ring; the 3-byte tail mix is a 64-entry table.
//   probe    one 32-byte bucket (a single DRAM sector, one 256-bit load) of the open-addressed
//            table per window; bucket-key gating by 2-bit prefix code (kmers_map.rs:273-311, :55-70)
//   dedup    distinct-hash semantics of the reference's HashSets: hits de-duplicated by table
//            slot in a per-warp shared-memory set, then histogrammed by node-set record
//   descend  one-vs-rest walk from the root (place_sequence.rs:279-601,
//            update_introspection_node.rs:13-91):
//            cnt(c)  = #hits whose node set contains child c
//            excl(c) = #hits whose node set contains c and no other non-leaf sibling
//            U       = #hits whose node set contains any non-leaf child of the current node
//            default mode: one = cnt(c), rest = U - excl(c); remove_intersection: one = excl(c),
//            rest = U - cnt(c); a single candidate -> (cnt(c), 0)   (place_sequence.rs:353-418)
//            CLOSED models (every set upward closed - the builder's invariant): sets are sorted
//            terminal lists over pre-order ids; all levels between the current node and the LCA of
//            the live terminals are unanimous (one candidate, rest = 0) and are skipped in one jump.
//            GENERAL models: sets are mini-trees walked level by level with shared-memory counters.
//
// Integer/byte work bound by instruction issue (murmur3) and the HBM/L2 sector rate - no tensor cores.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstdint>

#include "device_types.hpp"
#include "kernels.hpp"
#include "murmur3_device.cuh"

namespace cls {

namespace {

constexpr uint32_t kFull = 0xFFFFFFFFu;
constexpr uint32_t kUndecided = 0xFFFFFFFFu;
constexpr uint32_t kRing = 64;  // pre-mix ring entries per warp (two 32-offset chunks)

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// 4 two-bit codes (one byte) -> 4 ASCII letters via a byte permute on the "ACTG" LUT.
__device__ __forceinline__ uint32_t decode4(uint32_t b) {
    uint32_t sel = (b & 0x03u) | ((b & 0x0Cu) << 2) | ((b & 0x30u) << 4) | ((b & 0xC0u) << 6);
    return __byte_perm(kAsciiLut, 0u, sel);
}

// Reverse the order of the sixteen 2-bit bases of a word and complement them (code ^ 2).
__device__ __forceinline__ uint32_t revcomp16(uint32_t w) {
    uint32_t r = __brev(w);
    r = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);
    return r ^ 0xAAAAAAAAu;
}

// Per-warp shared-memory view.
struct WarpMem {
    uint32_t *str_f, *str_r;  // ASCII strands, 4-byte aligned, zero padded
    uint32_t *pk_f, *pk_r;    // 2-bit packed strands (16 bases / word), zero padded
    uint64_t *ring_a, *ring_b;  // pre-mix ring (k = 35 path)
};

// Decode one read into the two ASCII strands and the two packed strands.  One (word, strand) item per
// thread: a 150-base read is 10 words per strand, i.e. 20 items - all of a warp's lanes get work.
__device__ __forceinline__ void decode_read(const uint32_t *__restrict__ packed, uint32_t len, const WarpMem &m,
                                            uint32_t pk_words, uint32_t tid = threadIdx.x & 31u, uint32_t nthreads = 32u) {
    const uint32_t nw = (len + 15u) >> 4;
    const uint32_t pad = nw * 16u - len;  // unused base slots at the top of the last word
    for (uint32_t it = tid; it < 2 * pk_words; it += nthreads) {
        const bool rc = it >= pk_words;
        const uint32_t t = rc ? it - pk_words : it;
        uint32_t v = 0;
        if (t < nw) {
            if (!rc) {
                v = __ldg(packed + t);
            } else {
                // reverse-complement word t = bases [16t, 16t+16) of the reversed string
                const uint32_t a = revcomp16(__ldg(packed + (nw - 1 - t)));
                const uint32_t b = (t + 1 < nw) ? revcomp16(__ldg(packed + (nw - 2 - t))) : 0u;
                v = __funnelshift_r(a, b, 2u * pad);
            }
        }
        uint32_t *str = rc ? m.str_r : m.str_f;
        if (t <= nw) {  // word nw is the over-read pad of the strings
#pragma unroll
            for (int q = 0; q < 4; ++q) str[4 * t + q] = t < nw ? decode4((v >> (8 * q)) & 0xFFu) : 0u;
        }
        (rc ? m.pk_r : m.pk_f)[t] = v;
    }
}

__device__ __forceinline__ void ld_bucket(const Slot *table, uint64_t bucket, uint64_t &h0, uint64_t &m0,
                                          uint64_t &h1, uint64_t &m1) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(h0), "=l"(m0), "=l"(h1), "=l"(m1)
                 : "l"(table + 2 * bucket));
}

// `mask`-selected low bits (<= 24 of them) of a packed strand starting at base `pos`.
__device__ __forceinline__ uint32_t packed_bits(const uint32_t *pk, uint32_t pos, uint32_t mask) {
    const uint32_t j = pos >> 4;
    return __funnelshift_r(pk[j], pk[j + 1], (2u * pos) & 31u) & mask;
}

// Pre-mixes of the 8-byte little-endian word at byte offset q of an ASCII strand, into the ring.
__device__ __forceinline__ void premix_to_ring(const WarpMem &m, const uint32_t *s32, uint32_t q) {
    const uint32_t *w = s32 + (q >> 2);
    const uint32_t sh = (q & 3u) * 8u;
    const uint32_t r0 = w[0], r1 = w[1], r2 = w[2];
    const uint64_t x = pack64(__funnelshift_r(r0, r1, sh), __funnelshift_r(r1, r2, sh));
    m.ring_a[q & (kRing - 1)] = premix_k1(x);
    m.ring_b[q & (kRing - 1)] = premix_k2(x);
}

// Window hashing, one window per lane and pass.  Usage, by all 32 lanes:
//     for strand in {0, 1}: begin_strand(strand); for c in [0, n_chunks): valid = pass(c, pos, h)
//   K == 35: every 8-byte word of the strand is pre-mixed once (both murmur lanes) into a 64-entry
//            shared-memory ring and reused by the four windows that contain it at block offsets
//            0 / 8 / 16 / 24; block 0 starts from h1 = h2 = 0; the 3-byte tail mix is a table.
//   K == 0 : generic byte-wise hash for any runtime k.
template <int K>
struct WindowHasher {
    const WarpMem &m;
    const uint64_t *tail_lut;
    uint32_t W, k, lane;
    const uint32_t *s32, *pk;

    __device__ __forceinline__ WindowHasher(const WarpMem &m_, const uint64_t *lut, uint32_t len, uint32_t k_)
        : m(m_), tail_lut(lut), W(len - k_ + 1), k(k_), lane(threadIdx.x & 31u), s32(nullptr), pk(nullptr) {}

    __device__ __forceinline__ uint32_t n_chunks() const { return (W + 31u) >> 5; }

    // start hashing a strand at chunk `first_chunk` (chunks are then taken consecutively)
    __device__ __forceinline__ void begin_strand(uint32_t strand, uint32_t first_chunk = 0) {
        s32 = strand ? m.str_r : m.str_f;
        pk = strand ? m.pk_r : m.pk_f;
        if constexpr (K == 35) {
            __syncwarp();
            const uint32_t q = 32u * first_chunk + lane;
            if (q < W + 24u) premix_to_ring(m, s32, q);  // offsets 0 .. W+23 carry a needed pre-mix
        }
    }

    __device__ __forceinline__ bool pass(uint32_t c, uint32_t &pos, uint64_t &h) {
        pos = 32u * c + lane;
        const bool valid = pos < W;
        if constexpr (K == 35) {
            const uint32_t q = pos + 32u;
            if (q < W + 24u) premix_to_ring(m, s32, q);
            __syncwarp();
            if (valid) {
                const uint64_t a0 = m.ring_a[pos & (kRing - 1)], b1 = m.ring_b[(pos + 8) & (kRing - 1)];
                const uint64_t a2 = m.ring_a[(pos + 16) & (kRing - 1)], b3 = m.ring_b[(pos + 24) & (kRing - 1)];
                uint64_t h1 = mul5add(rotlc<27>(a0), 0x52dce729u);
                uint64_t h2 = mul5add(rotlc<31>(b1) + h1, 0x38495ab5u);
                h1 = mul5add(rotlc<27>(h1 ^ a2) + h2, 0x52dce729u);
                h2 = mul5add(rotlc<31>(h2 ^ b3) + h1, 0x38495ab5u);
                h1 ^= tail_lut[packed_bits(pk, pos + 32u, 63u)];
                h = mm_finish(h1, h2, 35ull);
            }
            __syncwarp();
        } else {
            if (valid) h = murmur_window_generic(reinterpret_cast<const uint8_t *>(s32), pos, k);
        }
        return valid;
    }
};

// tail_lut[c0 | c1 << 2 | c2 << 4] = k1 pre-mix of the 3-byte tail "XYZ" (codes A=0 C=1 T=2 G=3).
__device__ __forceinline__ void init_tail_lut(uint64_t *tail_lut) {
    for (uint32_t i = threadIdx.x; i < 64; i += blockDim.x) {
        const uint64_t t = (uint64_t)((kAsciiLut >> (8 * (i & 3))) & 0xFF) | ((uint64_t)((kAsciiLut >> (8 * ((i >> 2) & 3))) & 0xFF) << 8) |
                           ((uint64_t)((kAsciiLut >> (8 * ((i >> 4) & 3))) & 0xFF) << 16);
        tail_lut[i] = premix_k1(t);
    }
}

// First index in [lo, hi) whose terminal is >= key.
__device__ __forceinline__ uint32_t lower_bound_terms(const uint32_t *__restrict__ terms, uint32_t lo, uint32_t hi, uint32_t key) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(terms + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ QInfo ld_qinfo(const QInfo *qi, uint32_t q) {
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(qi + q));
    return QInfo{v.x, v.y, v.z, v.w};
}

// Lowest common ancestor of pre-order ids u <= v: minimum of (depth << 32 | q) over the Euler-tour
// range between their first occurrences, from the sparse table.  Two dependent round trips.
__device__ __forceinline__ uint64_t lca_depth_node(const DeviceIndex &ix, uint32_t u, uint32_t v) {
    const uint32_t fu = __ldg(&ix.qinfo[u].euler_first), fv = __ldg(&ix.qinfo[v].euler_first);
    const uint32_t j = 31u - __clz(fv - fu + 1u);
    const uint32_t row = j * ix.euler_len;  // the table holds at most 2^27 entries (build_host_index)
    const uint64_t a = __ldg(ix.lca_table + (row + fu)), b = __ldg(ix.lca_table + (row + fv + 1u - (1u << j)));
    return a < b ? a : b;
}

// One-vs-rest decision over `m` children whose vote counters sit in shared memory
// (place_sequence.rs:353-418 proposals, :436-600 decision).  Uniform results in all lanes.
struct Decision {
    uint32_t nprop, n_best, best_ord;
    int32_t best_one, best_rest;
};
__device__ __forceinline__ Decision decide_smem(const uint32_t *cnt, const uint32_t *excl, uint32_t m, uint32_t U, bool ri) {
    const uint32_t lane = lane_id();
    uint32_t ncand = 0;
    for (uint32_t o0 = 0; o0 < m; o0 += 32) {
        const uint32_t o = o0 + lane;
        ncand += __popc(__ballot_sync(kFull, o < m && cnt[o] > 0));
    }
    Decision d{0, 0, 0, 0, 0};
    int32_t best_diff = INT_MIN;
    for (uint32_t o0 = 0; o0 < m; o0 += 32) {
        const uint32_t o = o0 + lane;
        const uint32_t c = o < m ? cnt[o] : 0u, x = o < m ? excl[o] : 0u;
        const int32_t one = (int32_t)((ri && ncand > 1) ? x : c);
        const int32_t rest = ncand > 1 ? (int32_t)(ri ? U - c : U - x) : 0;
        const bool prop = c > 0 && one > rest;
        const uint32_t pm = __ballot_sync(kFull, prop);
        if (pm) {
            d.nprop += __popc(pm);
            const int32_t diff = prop ? one - rest : INT_MIN;
            const int32_t dmax = __reduce_max_sync(kFull, diff);
            const uint32_t eq = __ballot_sync(kFull, prop && diff == dmax);
            if (dmax > best_diff) {
                const int src = __ffs(eq) - 1;
                best_diff = dmax; d.n_best = __popc(eq);
                d.best_ord = __shfl_sync(kFull, o, src);
                d.best_one = __shfl_sync(kFull, one, src);
                d.best_rest = __shfl_sync(kFull, rest, src);
            } else if (dmax == best_diff) {
                d.n_best += __popc(eq);
            }
        }
    }
    return d;
}

// Per-read shared-memory tables (one set per warp, or per CTA for kb-scale reads).
struct ReadTables {
    uint32_t *t1;    // de-duplication set keyed by table slot; later the live-set list (lo / entry, weight)
    uint32_t *t2k;   // histogram keys: node-set record offsets; later `first`
    uint32_t *t2c;   // histogram counts; later `last`
    uint32_t *lst;   // histogram positions of the distinct sets in arrival order; later `hi`
    uint32_t *cnt, *excl;   // vote counters, one per non-leaf child ordinal
    uint32_t *n_sets;       // number of distinct node sets seen
    uint32_t t1_mask, t2_mask, t2_shift;
};

// Adds this pass's hits to the read's tables: de-duplicate by `slot_key` (distinct-hash semantics of
// the reference's HashSets), then add the distinct ones to the node-set histogram with ONE
// shared-memory atomic per group of lanes that hit the same node set (match.any).  Called by all
// 32 lanes; returns the number of distinct new hits of the pass (uniform).
// SHARED == true: several warps fill the tables of one read (CTA-per-read mode): counts are atomic and
// start from zeroed bins.  SHARED == false: the warp owns the tables; a bin's count has one writer per
// pass (the leader of its node set), so plain stores do and the bins need no zeroing.
template <bool SHARED>
__device__ __forceinline__ uint32_t insert_hits(const ReadTables &tb, bool hit, uint32_t slot_key, uint32_t set_off) {
    bool fresh = false;
    if (hit) {
        uint32_t p1 = (slot_key >> 1) & tb.t1_mask;  // bit 0 is the slot within the bucket (mostly 0): not a hash bit
        for (;;) {
            const uint32_t old = atomicCAS(&tb.t1[p1], kEmpty, slot_key);
            if (old == kEmpty) { fresh = true; break; }
            if (old == slot_key) break;  // the same k-mer hash was already counted
            p1 = (p1 + 1) & tb.t1_mask;
        }
    }
    const uint32_t fm = __ballot_sync(kFull, fresh);
    if (fresh) {
        const uint32_t peers = __match_any_sync(fm, set_off);
        if ((uint32_t)(__ffs(peers) - 1) == lane_id()) {
            uint32_t p2 = (set_off * 0x9E3779B1u) >> tb.t2_shift;
            for (;;) {
                const uint32_t old = atomicCAS(&tb.t2k[p2], kEmpty, set_off);
                if constexpr (SHARED) {
                    if (old == kEmpty) tb.lst[atomicAdd(tb.n_sets, 1u)] = p2;
                    if (old == kEmpty || old == set_off) { atomicAdd(&tb.t2c[p2], (uint32_t)__popc(peers)); break; }
                } else {
                    if (old == kEmpty) { tb.lst[atomicAdd(tb.n_sets, 1u)] = p2; tb.t2c[p2] = (uint32_t)__popc(peers); break; }
                    if (old == set_off) { tb.t2c[p2] += (uint32_t)__popc(peers); break; }
                }
                p2 = (p2 + 1) & tb.t2_mask;
            }
        }
    }
    if constexpr (!SHARED) __syncwarp();  // the next pass may elect another lane as the leader of the same bin
    return (uint32_t)__popc(fm);
}

// Everything after the hits of a read are in its tables: restriction to the root, gates, descent,
// and the result record.  One warp; `D` distinct node sets, `n_matched` distinct hits (|M|).
// `trace` (debug export cls_debug_node_counts): every level is evaluated with the vote counters - no LCA
// jump, no two-children shortcut; same outcome by construction - and one row per (level, child with votes)
// is appended to the trace.
template <bool CLOSED>
__device__ __forceinline__ void finish_read(const DeviceIndex &ix, const PlaceParams &pp, const ReadTables &tb,
                                            uint32_t D, uint32_t n_matched, ResultRec *__restrict__ out,
                                            const TraceBuf *trace = nullptr) {
    const uint32_t lane = lane_id();
    const bool tracing = trace != nullptr;
    auto trace_level = [&](uint32_t p, uint32_t m, uint32_t U, int64_t level) {
        const QNode qn = ix.qnodes[p];
        for (uint32_t o = lane; o < m; o += 32) {
            if (tb.cnt[o] == 0) continue;
            const uint32_t at = atomicAdd(trace->n_rows, 1u);
            if (at < trace->cap)
                trace->rows[at] = TraceRow{ix.q_node_id[p], ix.q_node_id[ix.q_child_list[qn.child_first + o]], (uint32_t)level,
                                           tb.cnt[o], tb.excl[o], U};
        }
    };
    uint32_t *t1 = tb.t1, *t2k = tb.t2k, *t2c = tb.t2c, *lst = tb.lst, *cnt = tb.cnt, *excl = tb.excl;
    const bool ri = pp.remove_intersection != 0;
    // ---- live-set list: restrict to sets that contain tree.root.id (M_r, place_sequence.rs:156-166)
    //      CLOSED : t1[2j] = lo, t1[2j+1] = weight, lst[j] = hi (terminal range [lo, hi)),
    //               t2k[j] = terms[lo] ("first"), t2c[j] = terms[hi-1] ("last")
    //      GENERAL: t1[2j] = current mini-tree entry, t1[2j+1] = weight
    for (uint32_t j = lane; j < D; j += 32) {
        const uint32_t p2 = lst[j];
        const uint32_t off = t2k[p2], w = t2c[p2];
        t1[2 * j] = off;
        t1[2 * j + 1] = w;
    }
    __syncwarp();
    uint32_t n_root = 0;
    for (uint32_t j = lane; j < D; j += 32) {
        const uint32_t off = t1[2 * j];
        uint32_t w = t1[2 * j + 1];
        if constexpr (CLOSED) {
            const uint32_t hdr = __ldg(ix.terms + off), last = __ldg(ix.terms + off + 1), first = __ldg(ix.terms + off + 2);
            if (hdr & kTermHasRoot) n_root += w; else w = 0;
            t1[2 * j] = off + 2;
            lst[j] = off + 2 + (hdr & ~kTermHasRoot);
            t2k[j] = first;
            t2c[j] = last;
        } else {
            const SetWord hdr = ix.arena[off];
            if (hdr.x & kSetHasRoot) n_root += w; else w = 0;
            t1[2 * j] = off + 1;
        }
        t1[2 * j + 1] = w;
    }
    n_root = __reduce_add_sync(kFull, n_root);
    __syncwarp();

    // ---- gates (place_sequence.rs:120-139, :156-166, :199-206, :231-254) ---------------
    ResultRec res;
    res.node_id = 0; res.one = 0; res.rest = 0;
    res.n_matched = n_matched; res.n_root_matched = n_root; res.iterations = 0;
    res.status = kUndecided;
    if (n_matched == 0) res.status = CLS_DEV_UNCL_NO_MATCH;
    else if (n_root == 0) res.status = CLS_DEV_UNCL_NO_ROOT;
    else if (ix.root_children_none) res.status = CLS_DEV_ERR_ROOT_NO_CHILDREN;
    else {
        // f64::round (half away from zero) of a non-negative product, without a libdevice call
        const double x = (double)n_matched * pp.min_match_coverage;
        double expected = floor(x);
        if (x - expected >= 0.5) expected += 1.0;
        if ((double)n_root < expected) res.status = CLS_DEV_UNCL_COVERAGE;
    }

    // ---- descent ---------------------------------------------------------------------------
    uint32_t p = 0;  // current parent (dense non-leaf id), root = 0
    int64_t iteration = 0;
    const int64_t max_iter = pp.max_iterations;
    if constexpr (CLOSED) {
        uint32_t depth_p = 0;
        QInfo ip = res.status == kUndecided ? ld_qinfo(ix.qinfo, 0) : QInfo{0, 0, 0, 0};
        while (res.status == kUndecided) {
            // pooled extremes of the live terminals -> every level down to their LCA is unanimous
            uint32_t umin = 0xFFFFFFFFu, vmax = 0, wl = 0;
            for (uint32_t j = lane; j < D; j += 32) {
                const uint32_t w = t1[2 * j + 1];
                if (w == 0) continue;
                umin = min(umin, t2k[j]);
                vmax = max(vmax, t2c[j]);
                wl += w;
            }
            umin = __reduce_min_sync(kFull, umin);
            vmax = __reduce_max_sync(kFull, vmax);
            const uint32_t Wlive = __reduce_add_sync(kFull, wl);
            const uint64_t dn = lca_depth_node(ix, umin, vmax);
            const uint32_t A = (uint32_t)dn, depth_a = (uint32_t)(dn >> 32);
            if (!tracing && depth_a > depth_p) {
                const uint32_t d = depth_a - depth_p;
                if (iteration + (int64_t)d > max_iter) { iteration = (max_iter > 0 ? max_iter : 0) + 1; res.status = CLS_DEV_ERR_MAX_ITERATIONS; break; }
                iteration += d;
                ip = ld_qinfo(ix.qinfo, A);
                if (ip.child_count == 0) {  // update_introspection_node.rs:32-87
                    res.status = CLS_DEV_IDENTITY_FOUND; res.node_id = ix.q_node_id[A];
                    res.one = (int32_t)Wlive; res.rest = 0;
                    break;
                }
                p = A; depth_p = depth_a;
            }
            // ---- evaluate the children of p -------------------------------------------------
            iteration++;
            if (iteration > max_iter) { res.status = CLS_DEV_ERR_MAX_ITERATIONS; break; }
            const uint32_t m = ip.child_count;
            const uint32_t p_end = ip.q_end;
            uint32_t win_q = 0, nprop = 0, n_best = 0;
            int32_t win_one = 0, win_rest = 0;
            QInfo iw{0, 0, 0, 0};
            if (!tracing && m <= 2) {
                // children intervals tile [p+1, p_end): c1 = [p+1, bnd), c2 = [bnd, p_end)
                const QInfo i1 = m ? ld_qinfo(ix.qinfo, p + 1) : QInfo{p_end, 0, 0, 0};
                const uint32_t bnd = i1.q_end;
                uint32_t c1 = 0, c2 = 0, both = 0;
                for (uint32_t j = lane; j < D; j += 32) {
                    const uint32_t w = t1[2 * j + 1];
                    if (w == 0) continue;
                    uint32_t lo = t1[2 * j], first = t2k[j];
                    const uint32_t hi = lst[j];
                    if (first == p) {  // the set ends at p itself for some tip: not a vote for any child
                        ++lo;
                        first = lo < hi ? __ldg(ix.terms + lo) : 0xFFFFFFFFu;
                        t1[2 * j] = lo; t2k[j] = first;
                    }
                    if (lo < hi) {
                        const bool in1 = first < bnd, in2 = t2c[j] >= bnd;
                        c1 += in1 ? w : 0u; c2 += in2 ? w : 0u; both += (in1 && in2) ? w : 0u;
                    }
                }
                c1 = __reduce_add_sync(kFull, c1);
                c2 = __reduce_add_sync(kFull, c2);
                both = __reduce_add_sync(kFull, both);
                const uint32_t U = c1 + c2 - both, x1 = c1 - both, x2 = c2 - both;
                const uint32_t ncand = (c1 > 0) + (c2 > 0);
                const int32_t one1 = (int32_t)((ri && ncand > 1) ? x1 : c1), rest1 = ncand > 1 ? (int32_t)(ri ? U - c1 : U - x1) : 0;
                const int32_t one2 = (int32_t)((ri && ncand > 1) ? x2 : c2), rest2 = ncand > 1 ? (int32_t)(ri ? U - c2 : U - x2) : 0;
                const bool pr1 = c1 > 0 && one1 > rest1, pr2 = c2 > 0 && one2 > rest2;
                nprop = (uint32_t)pr1 + (uint32_t)pr2;
                bool pick2 = pr2 && !pr1;
                n_best = nprop ? 1u : 0u;
                if (pr1 && pr2) {  // provably unreachable; kept for fidelity (:519-599)
                    const int32_t d1 = one1 - rest1, d2 = one2 - rest2;
                    if (d1 == d2) n_best = 2; else pick2 = d2 > d1;
                }
                if (pick2) { win_q = bnd; win_one = one2; win_rest = rest2; if (nprop) iw = ld_qinfo(ix.qinfo, bnd); }
                else { win_q = p + 1; win_one = one1; win_rest = rest1; iw = i1; }
            } else {
                // general fan-out: per-set merge walk of the terminal range against the child
                // intervals, votes in shared-memory counters
                uint32_t u_local = 0;
                for (uint32_t j = lane; j < D; j += 32) {
                    const uint32_t w = t1[2 * j + 1];
                    if (w == 0) continue;
                    uint32_t pos = t1[2 * j];
                    const uint32_t hi = lst[j];
                    if (t2k[j] == p) ++pos;
                    uint32_t npres = 0, last = 0, ord = 0, cend = m ? __ldg(&ix.qinfo[p + 1].q_end) : 0u;
                    while (m && pos < hi) {
                        const uint32_t t = __ldg(ix.terms + pos);
                        while (t >= cend) { cend = __ldg(&ix.qinfo[cend].q_end); ++ord; }
                        atomicAdd(&cnt[ord], w); ++npres; last = ord;
                        ++pos;
                        if (pos < hi && __ldg(ix.terms + pos) < cend) pos = lower_bound_terms(ix.terms, pos, hi, cend);
                    }
                    if (npres) u_local += w;
                    if (npres == 1) atomicAdd(&excl[last], w);
                }
                const uint32_t U = __reduce_add_sync(kFull, u_local);
                __syncwarp();
                if (tracing) trace_level(p, m, U, iteration);
                const Decision dc = decide_smem(cnt, excl, m, U, ri);
                __syncwarp();
                for (uint32_t o = lane; o < m; o += 32) { cnt[o] = 0; excl[o] = 0; }
                __syncwarp();
                nprop = dc.nprop; n_best = dc.n_best; win_one = dc.best_one; win_rest = dc.best_rest;
                win_q = p + 1;
                for (uint32_t o = 0; o < dc.best_ord; ++o) win_q = __ldg(&ix.qinfo[win_q].q_end);
                if (nprop) iw = ld_qinfo(ix.qinfo, win_q);
            }
            if (nprop == 0) {
                if (iteration == 1) res.status = CLS_DEV_UNCL_NO_INTROSPECTION;
                else { res.status = CLS_DEV_MAX_RESOLUTION; res.node_id = ix.q_node_id[p]; }
                break;
            }
            if (n_best != 1) { res.status = CLS_DEV_INCONCLUSIVE; res.node_id = ix.q_node_id[p]; break; }
            if (iw.child_count == 0) {  // update_introspection_node.rs:32-87
                res.status = CLS_DEV_IDENTITY_FOUND; res.node_id = ix.q_node_id[win_q];
                res.one = win_one; res.rest = win_rest;
                break;
            }
            p = win_q; ip = iw; depth_p++;
            const uint32_t win_end = iw.q_end;
            // every live set keeps its terminals inside the winner's interval (or drops out)
            for (uint32_t j = lane; j < D; j += 32) {
                if (t1[2 * j + 1] == 0) continue;
                uint32_t lo = t1[2 * j], hi = lst[j], first = t2k[j], last = t2c[j];
                bool live = lo < hi && last >= win_q && first < win_end;
                if (live && first < win_q) {
                    lo = lower_bound_terms(ix.terms, lo + 1, hi, win_q);
                    first = __ldg(ix.terms + lo);  // lo < hi because last >= win_q
                    live = first < win_end;
                    t1[2 * j] = lo; t2k[j] = first;
                }
                if (live && last >= win_end) {
                    hi = lower_bound_terms(ix.terms, lo + 1, hi - 1, win_end);  // terms[lo] < win_end
                    lst[j] = hi; t2c[j] = __ldg(ix.terms + hi - 1);
                }
                if (!live) t1[2 * j + 1] = 0;
            }
            __syncwarp();
        }
    } else {
        while (res.status == kUndecided) {
            iteration++;
            if (iteration > max_iter) { res.status = CLS_DEV_ERR_MAX_ITERATIONS; break; }
            const QNode qn = ix.qnodes[p];
            const uint32_t m = qn.child_count;
            // votes
            uint32_t u_local = 0;
            for (uint32_t j = lane; j < D; j += 32) {
                const uint32_t w = t1[2 * j + 1];
                if (w == 0) continue;
                const uint32_t cur = t1[2 * j];
                const uint32_t end = cur + ix.arena[cur].y;
                uint32_t npres = 0, last = 0;
                for (uint32_t c = cur + 1; c < end;) {
                    const SetWord e = ix.arena[c];
                    if (e.x & kPresentBit) { last = e.x & ~kPresentBit; atomicAdd(&cnt[last], w); npres++; }
                    c += e.y;
                }
                if (npres) u_local += w;
                if (npres == 1) atomicAdd(&excl[last], w);
            }
            const uint32_t U = __reduce_add_sync(kFull, u_local);
            __syncwarp();
            if (tracing) trace_level(p, m, U, iteration);
            const Decision dc = decide_smem(cnt, excl, m, U, ri);
            __syncwarp();
            for (uint32_t o = lane; o < m; o += 32) { cnt[o] = 0; excl[o] = 0; }
            __syncwarp();
            if (dc.nprop == 0) {
                if (iteration == 1) res.status = CLS_DEV_UNCL_NO_INTROSPECTION;
                else { res.status = CLS_DEV_MAX_RESOLUTION; res.node_id = ix.q_node_id[p]; }
                break;
            }
            if (dc.n_best != 1) {  // several proposals tie on (one - rest): provably unreachable
                res.status = CLS_DEV_INCONCLUSIVE; res.node_id = ix.q_node_id[p];
                break;
            }
            const uint32_t cq = ix.q_child_list[qn.child_first + dc.best_ord];
            if (ix.qnodes[cq].child_count == 0) {  // update_introspection_node.rs:32-87
                res.status = CLS_DEV_IDENTITY_FOUND; res.node_id = ix.q_node_id[cq];
                res.one = dc.best_one; res.rest = dc.best_rest;
                break;
            }
            p = cq;
            // every live set follows the winner (or drops out)
            for (uint32_t j = lane; j < D; j += 32) {
                if (t1[2 * j + 1] == 0) continue;
                const uint32_t cur = t1[2 * j];
                const uint32_t end = cur + ix.arena[cur].y;
                uint32_t next = 0;
                for (uint32_t c = cur + 1; c < end;) {
                    const SetWord e = ix.arena[c];
                    if ((e.x & ~kPresentBit) == dc.best_ord) { next = c; break; }
                    c += e.y;
                }
                if (next) t1[2 * j] = next; else t1[2 * j + 1] = 0;
            }
            __syncwarp();
        }
    }
    res.iterations = (uint32_t)iteration;
    if (lane == 0) *out = res;
}

// ------------------------------------------------------------------------------------------
// finish_read for CLOSED models when the read has at most 32 * SLOTS distinct node sets (97 % of 150 bp
// reads have at most 32, 99.9 % at most 64): lane j keeps sets j, j + 32, ... - its live terminal range [lo, hi), its smallest and largest live
// terminal and its weight - in registers, every vote is one warp reduction, and no loop runs over
// the sets.  Same algorithm and same outcomes as finish_read<true>.
// ------------------------------------------------------------------------------------------
// `set_off[s]` / `weight[s]`: node-set record and number of distinct hits of set lane + 32 s (weight 0 = none);
// `cnt` / `excl`: zeroed shared-memory vote counters of the warp (fan-out beyond two children only).
template <int SLOTS>
__device__ __forceinline__ void finish_read_reg(const DeviceIndex &ix, const PlaceParams &pp, uint32_t *cnt, uint32_t *excl,
                                                const uint32_t (&set_off)[SLOTS], const uint32_t (&weight)[SLOTS],
                                                uint32_t n_matched, ResultRec *__restrict__ out) {
    const uint32_t lane = lane_id();
    const uint32_t *__restrict__ terms = ix.terms;
    const bool ri = pp.remove_intersection != 0;
    // ---- restriction to the sets that contain tree.root.id (M_r, place_sequence.rs:156-166)
    uint32_t lo[SLOTS], hi[SLOTS], first[SLOTS], last[SLOTS], w[SLOTS];
    uint32_t wsum = 0;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        lo[s] = 0; hi[s] = 0; first[s] = 0xFFFFFFFFu; last[s] = 0; w[s] = 0;
        if (weight[s]) {
            const uint32_t off = set_off[s];
            const uint32_t hdr = __ldg(terms + off);
            if (hdr & kTermHasRoot) {
                last[s] = __ldg(terms + off + 1); first[s] = __ldg(terms + off + 2);
                w[s] = weight[s];
                lo[s] = off + 2; hi[s] = lo[s] + (hdr & ~kTermHasRoot);
            }
        }
        wsum += w[s];
    }
    const uint32_t n_root = __reduce_add_sync(kFull, wsum);
    // ---- gates (place_sequence.rs:120-139, :156-166, :199-206, :231-254)
    ResultRec res;
    res.node_id = 0; res.one = 0; res.rest = 0;
    res.n_matched = n_matched; res.n_root_matched = n_root; res.iterations = 0;
    res.status = kUndecided;
    if (n_matched == 0) res.status = CLS_DEV_UNCL_NO_MATCH;
    else if (n_root == 0) res.status = CLS_DEV_UNCL_NO_ROOT;
    else if (ix.root_children_none) res.status = CLS_DEV_ERR_ROOT_NO_CHILDREN;
    else {
        const double x = (double)n_matched * pp.min_match_coverage;  // f64::round, half away from zero
        double expected = floor(x);
        if (x - expected >= 0.5) expected += 1.0;
        if ((double)n_root < expected) res.status = CLS_DEV_UNCL_COVERAGE;
    }
    // ---- descent
    uint32_t p = 0, depth_p = 0;
    int32_t iteration = 0;  // never beyond max_iterations + 1
    const int32_t max_iter = pp.max_iterations;
    QInfo ip = res.status == kUndecided ? ld_qinfo(ix.qinfo, 0) : QInfo{0, 0, 0, 0};
    while (res.status == kUndecided) {
        // pooled extremes of the live terminals -> every level down to their LCA is unanimous
        uint32_t mn = 0xFFFFFFFFu, mx = 0;
#pragma unroll
        for (int s = 0; s < SLOTS; ++s)
            if (w[s]) { mn = min(mn, first[s]); mx = max(mx, last[s]); }
        const uint32_t umin = __reduce_min_sync(kFull, mn), vmax = __reduce_max_sync(kFull, mx);
        const uint64_t dn = lca_depth_node(ix, umin, vmax);
        const uint32_t A = (uint32_t)dn, depth_a = (uint32_t)(dn >> 32);
        if (depth_a > depth_p) {
            const uint32_t d = depth_a - depth_p;
            if ((int64_t)iteration + (int64_t)d > (int64_t)max_iter) { iteration = (max_iter > 0 ? max_iter : 0) + 1; res.status = CLS_DEV_ERR_MAX_ITERATIONS; break; }
            iteration += (int32_t)d;
            ip = ld_qinfo(ix.qinfo, A);
            if (ip.child_count == 0) {  // update_introspection_node.rs:32-87
                uint32_t ws = 0;
#pragma unroll
                for (int s = 0; s < SLOTS; ++s) ws += w[s];
                res.status = CLS_DEV_IDENTITY_FOUND; res.node_id = ix.q_node_id[A];
                res.one = (int32_t)__reduce_add_sync(kFull, ws); res.rest = 0;
                break;
            }
            p = A; depth_p = depth_a;
        }
        // ---- evaluate the children of p
        iteration++;
        if (iteration > max_iter) { res.status = CLS_DEV_ERR_MAX_ITERATIONS; break; }
        const uint32_t m = ip.child_count, p_end = ip.q_end;
        uint32_t win_q = 0, nprop = 0, n_best = 0;
        int32_t win_one = 0, win_rest = 0;
        QInfo iw{0, 0, 0, 0};
        bool has[SLOTS];
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
            if (w[s] && first[s] == p) {  // the set ends at p itself for some tip: that is no vote for any child
                ++lo[s];
                first[s] = lo[s] < hi[s] ? __ldg(terms + lo[s]) : 0xFFFFFFFFu;
            }
            has[s] = w[s] && lo[s] < hi[s];
        }
        if (m <= 2) {
            // children intervals tile [p+1, p_end): c1 = [p+1, bnd), c2 = [bnd, p_end)
            const QInfo i1 = m ? ld_qinfo(ix.qinfo, p + 1) : QInfo{p_end, 0, 0, 0};
            const uint32_t bnd = i1.q_end;
            uint32_t a1 = 0, a2 = 0, ab = 0;
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
                const bool in1 = has[s] && first[s] < bnd, in2 = has[s] && last[s] >= bnd;
                a1 += in1 ? w[s] : 0u; a2 += in2 ? w[s] : 0u; ab += (in1 && in2) ? w[s] : 0u;
            }
            const uint32_t c1 = __reduce_add_sync(kFull, a1), c2 = __reduce_add_sync(kFull, a2);
            const uint32_t both = __reduce_add_sync(kFull, ab);
            const uint32_t U = c1 + c2 - both, x1 = c1 - both, x2 = c2 - both;
            const uint32_t ncand = (c1 > 0) + (c2 > 0);
            const int32_t one1 = (int32_t)((ri && ncand > 1) ? x1 : c1), rest1 = ncand > 1 ? (int32_t)(ri ? U - c1 : U - x1) : 0;
            const int32_t one2 = (int32_t)((ri && ncand > 1) ? x2 : c2), rest2 = ncand > 1 ? (int32_t)(ri ? U - c2 : U - x2) : 0;
            const bool pr1 = c1 > 0 && one1 > rest1, pr2 = c2 > 0 && one2 > rest2;
            nprop = (uint32_t)pr1 + (uint32_t)pr2;
            bool pick2 = pr2 && !pr1;
            n_best = nprop ? 1u : 0u;
            if (pr1 && pr2) {  // provably unreachable; kept for fidelity (:519-599)
                const int32_t d1 = one1 - rest1, d2 = one2 - rest2;
                if (d1 == d2) n_best = 2; else pick2 = d2 > d1;
            }
            if (pick2) { win_q = bnd; win_one = one2; win_rest = rest2; if (nprop) iw = ld_qinfo(ix.qinfo, bnd); }
            else { win_q = p + 1; win_one = one1; win_rest = rest1; iw = i1; }
        } else {
            // general fan-out: every lane merges its terminal ranges against the child intervals,
            // votes in the shared-memory counters
            uint32_t u_local = 0;
#pragma unroll
            for (int s = 0; s < SLOTS; ++s) {
                if (!has[s]) continue;
                uint32_t pos = lo[s], npres = 0, lastc = 0, ord = 0, cend = __ldg(&ix.qinfo[p + 1].q_end);
                while (pos < hi[s]) {
                    const uint32_t t = __ldg(terms + pos);
                    while (t >= cend) { cend = __ldg(&ix.qinfo[cend].q_end); ++ord; }
                    atomicAdd(&cnt[ord], w[s]); ++npres; lastc = ord;
                    ++pos;
                    if (pos < hi[s] && __ldg(terms + pos) < cend) pos = lower_bound_terms(terms, pos, hi[s], cend);
                }
                u_local += w[s];
                if (npres == 1) atomicAdd(&excl[lastc], w[s]);
            }
            const uint32_t U = __reduce_add_sync(kFull, u_local);
            __syncwarp();
            const Decision dc = decide_smem(cnt, excl, m, U, ri);
            __syncwarp();
            for (uint32_t o = lane; o < m; o += 32) { cnt[o] = 0; excl[o] = 0; }
            __syncwarp();
            nprop = dc.nprop; n_best = dc.n_best; win_one = dc.best_one; win_rest = dc.best_rest;
            win_q = p + 1;
            for (uint32_t o = 0; o < dc.best_ord; ++o) win_q = __ldg(&ix.qinfo[win_q].q_end);
            iw = ld_qinfo(ix.qinfo, win_q);
        }
        if (nprop == 0) {
            if (iteration == 1) res.status = CLS_DEV_UNCL_NO_INTROSPECTION;
            else { res.status = CLS_DEV_MAX_RESOLUTION; res.node_id = ix.q_node_id[p]; }
            break;
        }
        if (n_best != 1) { res.status = CLS_DEV_INCONCLUSIVE; res.node_id = ix.q_node_id[p]; break; }
        if (iw.child_count == 0) {  // update_introspection_node.rs:32-87
            res.status = CLS_DEV_IDENTITY_FOUND; res.node_id = ix.q_node_id[win_q];
            res.one = win_one; res.rest = win_rest;
            break;
        }
        p = win_q; ip = iw; depth_p++;
        const uint32_t win_end = iw.q_end;
        // every live set keeps its terminals inside the winner's interval (or drops out)
#pragma unroll
        for (int s = 0; s < SLOTS; ++s) {
            bool live = has[s] && last[s] >= win_q && first[s] < win_end;
            if (live && first[s] < win_q) {
                lo[s] = lower_bound_terms(terms, lo[s] + 1, hi[s], win_q);
                first[s] = __ldg(terms + lo[s]);  // lo < hi because last >= win_q
                live = first[s] < win_end;
            }
            if (live && last[s] >= win_end) {
                hi[s] = lower_bound_terms(terms, lo[s] + 1, hi[s] - 1, win_end);  // terms[lo] < win_end
                last[s] = __ldg(terms + hi[s] - 1);
            }
            if (!live) w[s] = 0;
        }
    }
    res.iterations = (uint32_t)iteration;
    if (lane == 0) *out = res;
}

// The same, fed from the read's shared-memory histogram.
template <int SLOTS>
__device__ __forceinline__ void finish_read_reg(const DeviceIndex &ix, const PlaceParams &pp, const ReadTables &tb,
                                                uint32_t D, uint32_t n_matched, ResultRec *__restrict__ out) {
    uint32_t off[SLOTS], wt[SLOTS];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const uint32_t j = lane_id() + 32u * s;
        off[s] = 0; wt[s] = 0;
        if (j < D) { const uint32_t p2 = tb.lst[j]; off[s] = tb.t2k[p2]; wt[s] = tb.t2c[p2]; }
    }
    finish_read_reg<SLOTS>(ix, pp, tb.cnt, tb.excl, off, wt, n_matched, out);
}

}  // namespace

// ------------------------------------------------------------------------------------------
// Debug/parity kernel: all window hashes of one read, reference order (forward then revcomp).
// One warp; runs the very same decode + hashing code as the placement kernel.
// ------------------------------------------------------------------------------------------
template <int K>
__global__ void hash_only_kernel(const uint32_t *__restrict__ packed, uint32_t len, uint32_t k,
                                 uint64_t *__restrict__ out, uint32_t str_words, uint32_t pk_words) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint64_t tail_lut[64];
    init_tail_lut(tail_lut);
    WarpMem m;
    m.ring_a = reinterpret_cast<uint64_t *>(smem);
    m.ring_b = m.ring_a + kRing;
    m.str_f = smem + 4 * kRing;
    m.str_r = m.str_f + str_words;
    m.pk_f = m.str_r + str_words;
    m.pk_r = m.pk_f + pk_words;
    __syncthreads();
    if (threadIdx.x >= 32) return;
    decode_read(packed, len, m, pk_words);
    __syncwarp();
    WindowHasher<K> wh(m, tail_lut, len, k);
    for (uint32_t strand = 0; strand < 2; ++strand) {
        wh.begin_strand(strand);
        for (uint32_t c = 0; c < wh.n_chunks(); ++c) {
            uint32_t pos;
            uint64_t h;
            if (wh.pass(c, pos, h)) out[(strand ? wh.W : 0u) + pos] = h;
        }
    }
}

// Hand-over to the descent kernels (their own launch, one warp per read): per read of the launch
//     pairs[r * cap + j] = {node-set record offset, distinct hits with that node set}, j < D
//     meta[r] = {n_matched, D};  D = kDone: the read was finished where its histogram was built (D > cap)
// cap = kPairCap for one-warp-per-read launches, kPairCapWide for one-CTA-per-read launches (kb-scale reads
// see a hundred or more distinct node sets).
constexpr uint32_t kPairCap = 64, kPairCapWide = 256, kDone = 0xFFFFFFFFu;
struct ScanOut {
    uint2 *pairs;
    uint2 *meta;
    uint32_t cap;
    // The persistent warps of scan2_kernel and descend_kernel take reads in blocks of kReadBlock from a global counter
    // instead of a static stride: a CTA that becomes resident late (another kernel still holds its SM) or draws cheap
    // reads does not decide when the launch ends (4.48 against 5.07 ms per 1 M reads of config 2, profiles/r2a).
    // counters[0]: scan kernel, [1]: descent kernel, [2]: length of ov_list; zeroed by the launcher.
    uint32_t *counters;
    uint32_t *ov_list;   // reads scan2_kernel could not hand over (too many node sets): finished by scan_kernel afterwards
};
constexpr uint32_t kReadBlock = 2;
// next read of this warp, or >= n_reads when the launch has run out of reads
__device__ __forceinline__ uint32_t next_read(uint32_t *counter, uint32_t &base, uint32_t &used) {
    if (used == kReadBlock) {
        uint32_t b = 0;
        if (lane_id() == 0) b = atomicAdd(counter, kReadBlock);
        base = __shfl_sync(kFull, b, 0);
        used = 0;
    }
    return base + used++;
}

// ------------------------------------------------------------------------------------------
// The placement kernel, persistent CTAs striding over the query range.
//   CTA == false: one WARP per query (short reads: the per-query tables are a few KB)
//   CTA == true : one CTA per query (kb-scale reads): all warps hash / probe / de-duplicate
//                 contiguous chunk ranges of the read into one set of shared tables, warp 0 walks the tree
// ------------------------------------------------------------------------------------------
template <int K, bool CLOSED, bool CTA>
__global__ void __launch_bounds__(CTA ? 512 : 256, CTA ? 2 : 4) place_kernel(DeviceIndex ix, PlaceParams pp,
                                                       const uint32_t *__restrict__ packed,
                                                       const ReadDesc *__restrict__ reads, uint32_t first_read,
                                                       uint32_t n_reads, ResultRec *__restrict__ results,
                                                       PlaceGeom g, ScanOut so, TraceBuf trace,
                                                       const uint8_t *__restrict__ only = nullptr) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint64_t tail_lut[64];
    init_tail_lut(tail_lut);
    const uint32_t lane = lane_id();
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t warps_per_cta = blockDim.x >> 5;
    // layout: [rings of all warps][tables + strings of group 0][... of group 1] ...; a group is one
    // warp (CTA == false) or the whole CTA (CTA == true)
    uint32_t *gbase = smem + 4 * kRing * warps_per_cta + (CTA ? (size_t)0 : (size_t)warp * g.words_per_warp);
    WarpMem wm;
    wm.ring_a = reinterpret_cast<uint64_t *>(smem + 4 * kRing * warp);
    wm.ring_b = wm.ring_a + kRing;
    const uint32_t gtid = CTA ? threadIdx.x : lane, gthreads = CTA ? blockDim.x : 32u;
    auto group_sync = [] { if constexpr (CTA) __syncthreads(); else __syncwarp(); };
    uint32_t *t1 = gbase;                // dedup set keyed by table slot; later the live-set list
    uint32_t *t2k = t1 + g.t1_size;      // histogram keys: node-set record offsets; later `first`
    uint32_t *t2c = t2k + g.t2_size;     // histogram counts; later `last`
    uint32_t *lst = t2c + g.t2_size;     // histogram positions of the distinct sets; later `hi`
    wm.str_f = lst + g.t2_size;
    wm.str_r = wm.str_f + g.str_words;
    wm.pk_f = wm.str_r + g.str_words;
    wm.pk_r = wm.pk_f + g.pk_words;
    uint32_t *cnt = wm.pk_r + g.pk_words;  // vote counters, one per non-leaf child ordinal
    uint32_t *excl = cnt + g.fan_cap;
    uint32_t *n_sets_smem = excl + g.fan_cap;
    uint32_t *n_matched_smem = n_sets_smem + 1;
    const ReadTables tb{t1, t2k, t2c, lst, cnt, excl, n_sets_smem, g.t1_size - 1u, g.t2_size - 1u, 32u - g.t2_log2};
    const uint32_t k = ix.k_size;
    const uint32_t code_mask = ix.m_eff >= 16 ? 0xFFFFFFFFu : ((1u << (2 * ix.m_eff)) - 1u);

    for (uint32_t o = gtid; o < g.fan_cap; o += gthreads) { cnt[o] = 0; excl[o] = 0; }
    __syncthreads();

    const uint32_t gwarp = CTA ? blockIdx.x : blockIdx.x * warps_per_cta + warp;
    const uint32_t gstride = CTA ? gridDim.x : gridDim.x * warps_per_cta;
#pragma unroll 1
    for (uint32_t r = gwarp; r < n_reads; r += gstride) {
        // `only` given (kb-scale reads after scanfrag_kernel + gather_kernel, frag_kernels.cuh): just the reads those two
        // handed back
        if (only && only[r] != 1) continue;   // kRedoPlace
        const ReadDesc rd = reads[first_read + r];
        const uint32_t L = rd.len;
        const uint32_t W = L - k + 1;  // host guarantees L >= k

        // ---- reset per-read tables, decode ------------------------------------------------
        {
            uint4 *z = reinterpret_cast<uint4 *>(t1);
            const uint32_t n4 = (g.t1_size + g.t2_size) >> 2;  // t1 and t2k are contiguous: all kEmpty
            for (uint32_t i = gtid; i < n4; i += gthreads) z[i] = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
            if constexpr (CTA) {  // counts are accumulated atomically by all warps: start from zero
                uint4 *zc = reinterpret_cast<uint4 *>(t2c);
                for (uint32_t i = gtid; i < (g.t2_size >> 2); i += gthreads) zc[i] = make_uint4(0, 0, 0, 0);
            }
            if (gtid == 0) { *n_sets_smem = 0; *n_matched_smem = 0; }
        }
        decode_read(packed + rd.word_off, L, wm, g.pk_words, gtid, gthreads);
        group_sync();

        // ---- hash + probe + dedup + histogram, software pipelined: the bucket of pass i is in
        //      flight while pass i+1 is hashed and pass i-1 is consumed ---------------------------
        // consume(): match the loaded bucket, gate by bucket key, de-duplicate by table slot, and add
        // the distinct hits to the node-set histogram (one shared-memory atomic per group of lanes
        // that hit the same node set, found with match.any).  Called by all 32 lanes.
        auto consume = [=](bool valid, bool rc, uint32_t pos, uint64_t h, uint64_t h0, uint64_t m0, uint64_t h1,
                           uint64_t m1) -> uint32_t {
            uint32_t slot_id = kEmpty, set_off = 0, code = 0;
            if (valid) {
                uint64_t b = h & ix.bucket_mask;
                for (;;) {
                    if (h0 == h && (uint32_t)m0 != kEmpty) { slot_id = (uint32_t)(2 * b); set_off = (uint32_t)m0; code = (uint32_t)(m0 >> 32); break; }
                    if (h1 == h && (uint32_t)m1 != kEmpty) { slot_id = (uint32_t)(2 * b + 1); set_off = (uint32_t)m1; code = (uint32_t)(m1 >> 32); break; }
                    if (!((uint32_t)(m0 >> 32) & kOverflowBit)) break;
                    b = (b + 1) & ix.bucket_mask;
                    ld_bucket(ix.table, b, h0, m0, h1, m1);
                }
            }
            bool hit = slot_id != kEmpty;
            if (hit) {
                // bucket gating: the entry's bucket key must be among the query's prefix keys
                const uint32_t want = code & kCodeMask;
                hit = packed_bits(rc ? wm.pk_r : wm.pk_f, pos, code_mask) == want;
                if (!hit) {  // only possible for models whose bucket keys disagree with their k-mers
                    for (uint32_t p = 0; p < W && !hit; ++p)
                        hit = packed_bits(wm.pk_f, p, code_mask) == want || packed_bits(wm.pk_r, p, code_mask) == want;
                }
            }
            return insert_hits<CTA>(tb, hit, slot_id, set_off);
        };

        uint32_t n_matched = 0;
        {
            WindowHasher<K> wh(wm, tail_lut, L, k);
            const uint32_t n_chunks = wh.n_chunks();
            // this warp's contiguous chunk range [c_lo, c_hi) of each strand (the whole strand when a
            // warp owns the read)
            const uint32_t per = CTA ? (n_chunks + warps_per_cta - 1) / warps_per_cta : n_chunks;
            const uint32_t c_lo = CTA ? min(warp * per, n_chunks) : 0u, c_hi = CTA ? min(c_lo + per, n_chunks) : n_chunks;
#pragma unroll 1
            for (uint32_t strand = 0; strand < 2 && c_lo < c_hi; ++strand) {
                wh.begin_strand(strand, c_lo);
#pragma unroll 1
                for (uint32_t c = c_lo; c < c_hi; ++c) {
                    uint32_t pos;
                    uint64_t h = 0, q0 = 0, qm0 = 0, q1 = 0, qm1 = 0;
                    const bool valid = wh.pass(c, pos, h);
                    if (valid) ld_bucket(ix.table, h & ix.bucket_mask, q0, qm0, q1, qm1);
                    n_matched += consume(valid, strand != 0, pos, h, q0, qm0, q1, qm1);
                }
            }
        }
        if constexpr (CTA) {
            if (lane == 0 && n_matched) atomicAdd(n_matched_smem, n_matched);
            __syncthreads();
            n_matched = *n_matched_smem;
            if (CLOSED && so.pairs && *n_sets_smem <= so.cap) {
                // hand the read over to the descent kernel: one warp walking the tree while seven wait is
                // what made kb-scale reads slow
                const uint32_t D = *n_sets_smem;
                for (uint32_t j = gtid; j < D; j += gthreads) {
                    const uint32_t p2 = lst[j];
                    so.pairs[(size_t)r * so.cap + j] = make_uint2(t2k[p2], t2c[p2]);
                }
                if (gtid == 0) so.meta[r] = make_uint2(n_matched, D);
                __syncthreads();   // the tables are free again for the next read
                continue;
            }
            if (warp != 0) { __syncthreads(); continue; }   // warp 0 finishes the read; see the barrier at the end
            if (so.pairs && lane == 0) so.meta[r] = make_uint2(n_matched, kDone);
        }
        __syncwarp();
        const uint32_t D = *n_sets_smem;

        finish_read<CLOSED>(ix, pp, tb, D, n_matched, results + first_read + r, trace.rows ? &trace : nullptr);
        __syncwarp();
        if constexpr (CTA) __syncthreads();   // the tables are free again for the next read
    }
}

// ------------------------------------------------------------------------------------------
// Short reads, k = 35: the scan kernel (one warp per read: decode, hash, probe, de-duplicate,
// histogram by node set) and the descent kernel (one warp per read as well, its own launch).  The scan
// loop is unrolled over the two halves of the pre-mix ring so that every shared-memory address of a
// pass is a per-lane constant: pass c hashes windows 32c + lane from the pre-mixes at offsets pos,
// pos + 8, pos + 16, pos + 24 and meanwhile pre-mixes offsets 32(c + 1) + lane into the other half.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void premix_store(const uint32_t *w, uint32_t sh8, uint64_t *ra, uint64_t *rb) {
    const uint32_t r0 = w[0], r1 = w[1], r2 = w[2];
    const uint64_t x = pack64(__funnelshift_r(r0, r1, sh8), __funnelshift_r(r1, r2, sh8));
    *ra = premix_k1(x);
    *rb = premix_k2(x);
}

__device__ __forceinline__ uint64_t window_hash35(uint64_t a0, uint64_t b1, uint64_t a2, uint64_t b3, uint64_t tail) {
    uint64_t h1 = mul5add(rotlc<27>(a0), 0x52dce729u);
    uint64_t h2 = mul5add(rotlc<31>(b1) + h1, 0x38495ab5u);
    h1 = mul5add(rotlc<27>(h1 ^ a2) + h2, 0x52dce729u);
    h2 = mul5add(rotlc<31>(h2 ^ b3) + h1, 0x38495ab5u);
    return mm_finish(h1 ^ tail, h2, 35ull);
}

// First-generation scan kernel, descent fused (finish_read*): general (mini-tree) models, callers without hand-over
// scratch, and - with `ov_list` - the reads scan2_kernel left on its overflow list (*ov_count of them).
template <bool CLOSED>
__global__ void __launch_bounds__(256, 4) scan_kernel(DeviceIndex ix, PlaceParams pp, const uint32_t *__restrict__ packed,
                                                      const ReadDesc *__restrict__ reads, uint32_t first_read,
                                                      uint32_t n_reads, ResultRec *__restrict__ results, PlaceGeom g,
                                                      const uint32_t *__restrict__ ov_list, const uint32_t *__restrict__ ov_count) {
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint64_t tail_lut[64];
    init_tail_lut(tail_lut);
    const uint32_t lane = lane_id();
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t warps_per_cta = blockDim.x >> 5;
    uint32_t *gbase = smem + 4 * kRing * warps_per_cta + (size_t)warp * g.words_per_warp;
    uint64_t *ring_a = reinterpret_cast<uint64_t *>(smem + 4 * kRing * warp), *ring_b = ring_a + kRing;
    WarpMem wm;
    wm.ring_a = ring_a; wm.ring_b = ring_b;
    uint32_t *t1 = gbase, *t2k = t1 + g.t1_size, *t2c = t2k + g.t2_size, *lst = t2c + g.t2_size;
    wm.str_f = lst + g.t2_size;
    wm.str_r = wm.str_f + g.str_words;
    wm.pk_f = wm.str_r + g.str_words;
    wm.pk_r = wm.pk_f + g.pk_words;
    uint32_t *cnt = wm.pk_r + g.pk_words, *excl = cnt + g.fan_cap, *n_sets_smem = excl + g.fan_cap;
    const ReadTables tb{t1, t2k, t2c, lst, cnt, excl, n_sets_smem, g.t1_size - 1u, g.t2_size - 1u, 32u - g.t2_log2};
    const uint32_t code_mask = ix.m_eff >= 16 ? 0xFFFFFFFFu : ((1u << (2 * ix.m_eff)) - 1u);
    const uint32_t bmask = (uint32_t)ix.bucket_mask;  // at most 2^30 buckets (cls_index_create)
    // per-lane constants of the hashing loop
    const uint32_t sh8 = (lane & 3u) * 8u, sh2 = (lane & 15u) * 2u;
    uint64_t *const ra0 = ring_a + lane, *const rb0 = ring_b + lane;
    const uint64_t *const rb_o1 = ring_b + ((lane + 40u) & 63u), *const ra_o2 = ring_a + ((lane + 48u) & 63u),
                   *const rb_o3 = ring_b + ((lane + 56u) & 63u);

    for (uint32_t o = lane; o < g.fan_cap; o += 32) { cnt[o] = 0; excl[o] = 0; }
    __syncthreads();

    const uint32_t gwarp = blockIdx.x * warps_per_cta + warp, gstride = gridDim.x * warps_per_cta;
    const uint32_t n_items = ov_list ? *ov_count : n_reads;
#pragma unroll 1
    for (uint32_t item = gwarp; item < n_items; item += gstride) {
        const uint32_t r = ov_list ? ov_list[item] : item;
        const ReadDesc rd = reads[first_read + r];
        const uint32_t L = rd.len;
        const uint32_t W = L - 34u;  // host guarantees L >= k = 35
        {
            uint4 *z = reinterpret_cast<uint4 *>(t1);
            const uint32_t n4 = (g.t1_size + g.t2_size) >> 2;  // t1 and t2k are contiguous: all kEmpty
            for (uint32_t i = lane; i < n4; i += 32) z[i] = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
            if (lane == 0) *n_sets_smem = 0;  // the histogram counts (t2c) are written before they are read
        }
        decode_read(packed + rd.word_off, L, wm, g.pk_words);
        const uint32_t n_chunks = (W + 31u) >> 5;
        uint32_t n_matched = 0;
#pragma unroll 1
        for (uint32_t strand = 0; strand < 2; ++strand) {
            const uint32_t *pk = strand ? wm.pk_r : wm.pk_f;
            const uint32_t *wsrc = (strand ? wm.str_r : wm.str_f) + (lane >> 2);  // + 8 words per 32 offsets
            const uint32_t *pkl = pk + (lane >> 4);                               // + 2 words per 32 bases
            // match the bucket loaded for window `pos` against its hash, gate, and add the hit to the read's tables
            auto consume = [&](uint32_t pos, uint64_t h, uint32_t b, uint64_t h0, uint64_t m0, uint64_t h1, uint64_t m1) {
                const bool valid = pos < W;
                bool e0 = h0 == h && (uint32_t)m0 != kEmpty, e1 = h1 == h && (uint32_t)m1 != kEmpty;
                if (valid && !(e0 || e1) && ((uint32_t)(m0 >> 32) & kOverflowBit)) {  // the bucket overflowed at build time
                    do {
                        b = (b + 1) & bmask;
                        ld_bucket(ix.table, b, h0, m0, h1, m1);
                        e0 = h0 == h && (uint32_t)m0 != kEmpty; e1 = h1 == h && (uint32_t)m1 != kEmpty;
                    } while (!(e0 || e1) && ((uint32_t)(m0 >> 32) & kOverflowBit));
                }
                const uint64_t mm = e0 ? m0 : m1;
                bool hit = valid && (e0 || e1);
                if (hit) {
                    // bucket gating: the entry's bucket key must be among the query's prefix keys
                    const uint32_t want = (uint32_t)(mm >> 32) & kCodeMask;
                    hit = packed_bits(pk, pos, code_mask) == want;
                    if (!hit) {  // only possible for models whose bucket keys disagree with their k-mers
                        for (uint32_t q = 0; q < W && !hit; ++q)
                            hit = packed_bits(wm.pk_f, q, code_mask) == want || packed_bits(wm.pk_r, q, code_mask) == want;
                    }
                }
                n_matched += insert_hits<false>(tb, hit, 2u * b + (e0 ? 0u : 1u), (uint32_t)mm);
            };
            __syncwarp();
            premix_store(wsrc, sh8, ra0, rb0);  // offsets 0..31 -> ring half 0
            // two passes per iteration: the ring loads of both are done first, then the two hash chains
            // run interleaved (independent instruction streams), their two probes are in flight together,
            // and the two results are consumed one after the other
#pragma unroll 1
            for (uint32_t c = 0; c < n_chunks; c += 2) {
                const bool two = c + 1 < n_chunks;  // warp-uniform
                const uint32_t posA = 32u * c + lane, posB = posA + 32u;
                premix_store(wsrc + 8 * (c + 1), sh8, ra0 + 32, rb0 + 32);  // offsets 32(c+1) + lane -> ring half 1
                __syncwarp();
                const uint64_t a0 = ra0[0], b1 = rb0[8], a2 = ra0[16], b3 = rb0[24];
                const uint32_t tiA = __funnelshift_r(pkl[2 * c + 2], pkl[2 * c + 3], sh2) & 63u;
                __syncwarp();
                uint64_t e0 = 0, f1 = 0, e2 = 0, f3 = 0;
                uint32_t tiB = 0;
                if (two) {
                    premix_store(wsrc + 8 * (c + 2), sh8, ra0, rb0);        // offsets 32(c+2) + lane -> ring half 0
                    __syncwarp();
                    e0 = ra0[32]; f1 = *rb_o1; e2 = *ra_o2; f3 = *rb_o3;
                    tiB = __funnelshift_r(pkl[2 * c + 4], pkl[2 * c + 5], sh2) & 63u;
                    __syncwarp();
                }
                const uint64_t hA = window_hash35(a0, b1, a2, b3, tail_lut[tiA]);
                const uint64_t hB = window_hash35(e0, f1, e2, f3, tail_lut[tiB]);
                // lanes past the last window load bucket 0 and ignore it
                const uint32_t bA = posA < W ? (uint32_t)hA & bmask : 0u, bB = (two && posB < W) ? (uint32_t)hB & bmask : 0u;
                uint64_t A0, A1, A2, A3, B0, B1, B2, B3;
                ld_bucket(ix.table, bA, A0, A1, A2, A3);
                ld_bucket(ix.table, bB, B0, B1, B2, B3);
                consume(posA, hA, bA, A0, A1, A2, A3);
                if (two) consume(posB, hB, bB, B0, B1, B2, B3);
            }
        }
        __syncwarp();
        const uint32_t D = *n_sets_smem;
        if (CLOSED && D <= 32) finish_read_reg<1>(ix, pp, tb, D, n_matched, results + first_read + r);
        else if (CLOSED && D <= 64) finish_read_reg<2>(ix, pp, tb, D, n_matched, results + first_read + r);
        else finish_read<CLOSED>(ix, pp, tb, D, n_matched, results + first_read + r);
        __syncwarp();
    }
}

// One warp per read: gates and descent over the {node set, weight} pairs the scan kernel left.
// MAXSLOTS = 2 serves the short-read launches (at most 64 pairs), MAXSLOTS = 8 the kb-scale ones (at most 256).
template <int SLOTS>
__device__ __forceinline__ void descend_from_pairs(const DeviceIndex &ix, const PlaceParams &pp, uint32_t *cnt, uint32_t *excl,
                                                   const uint2 *__restrict__ pr, uint32_t D, uint32_t n_matched,
                                                   ResultRec *__restrict__ out) {
    uint32_t off[SLOTS], wt[SLOTS];
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
        const uint32_t j = lane_id() + 32u * s;
        off[s] = 0; wt[s] = 0;
        if (j < D) { const uint2 v = pr[j]; off[s] = v.x; wt[s] = v.y; }
    }
    finish_read_reg<SLOTS>(ix, pp, cnt, excl, off, wt, n_matched, out);
}

// ------------------------------------------------------------------------------------------
// Several reads per warp: a read with at most G node sets (G = 8 or 16 lanes of a warp: a quarter or a half) leaves most
// lanes of finish_read_reg idle - 62 % of 150-base reads have at most 16 sets.  finish_group runs 32 / G reads side by
// side, one per group of G consecutive lanes: what is warp-uniform there is group-uniform here (held by every lane of the
// group), reductions are butterflies inside the group, and every group carries its own status through a loop that ends
// when all groups are done.  Only two-way levels are handled (the three vote sums travel in one word, 10 bits each, so the
// caller keeps reads of 1 024 hits or more away); a level with a larger fan-out hands the read back (returns true) and
// the caller runs it through finish_read_reg.  Same algorithm, same outcomes (place_sequence.rs:279-601).
// ------------------------------------------------------------------------------------------
template <int G> __device__ __forceinline__ uint32_t group_sum(uint32_t v) {
#pragma unroll
    for (int d = G / 2; d; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
    return v;
}
template <int G> __device__ __forceinline__ uint32_t group_min(uint32_t v) {
#pragma unroll
    for (int d = G / 2; d; d >>= 1) v = min(v, __shfl_xor_sync(kFull, v, d));
    return v;
}
template <int G> __device__ __forceinline__ uint32_t group_max(uint32_t v) {
#pragma unroll
    for (int d = G / 2; d; d >>= 1) v = max(v, __shfl_xor_sync(kFull, v, d));
    return v;
}

constexpr uint32_t kGroupIdle = 0xFFFFFFFEu, kGroupRedo = 0xFFFFFFFDu;

// `have`: this lane's group holds a read; `set_off` / `weight`: the lane's pair of it (weight 0 = none); `n_matched`, `out`:
// group-uniform.  Called by all 32 lanes.
template <int G>
__device__ __forceinline__ bool finish_group(const DeviceIndex &ix, const PlaceParams &pp, bool have, uint32_t set_off, uint32_t weight,
                                             uint32_t n_matched, ResultRec *__restrict__ out) {
    const uint32_t *__restrict__ terms = ix.terms;
    const bool ri = pp.remove_intersection != 0;
    // ---- restriction to the sets that contain tree.root.id (M_r, place_sequence.rs:156-166)
    uint32_t lo = 0, hi = 0, first = 0xFFFFFFFFu, last = 0, w = 0;
    if (have && weight) {
        const uint32_t hdr = __ldg(terms + set_off);
        if (hdr & kTermHasRoot) {
            last = __ldg(terms + set_off + 1); first = __ldg(terms + set_off + 2);
            w = weight;
            lo = set_off + 2; hi = lo + (hdr & ~kTermHasRoot);
        }
    }
    const uint32_t n_root = group_sum<G>(w);
    // ---- gates (place_sequence.rs:120-139, :156-166, :199-206, :231-254)
    uint32_t status = kUndecided, node_q = 0;
    bool has_node = false;
    int32_t one = 0, rest = 0;
    if (!have) status = kGroupIdle;
    else if (n_matched == 0) status = CLS_DEV_UNCL_NO_MATCH;
    else if (n_root == 0) status = CLS_DEV_UNCL_NO_ROOT;
    else if (ix.root_children_none) status = CLS_DEV_ERR_ROOT_NO_CHILDREN;
    else {
        const double x = (double)n_matched * pp.min_match_coverage;  // f64::round, half away from zero
        double expected = floor(x);
        if (x - expected >= 0.5) expected += 1.0;
        if ((double)n_root < expected) status = CLS_DEV_UNCL_COVERAGE;
    }
    // ---- descent
    uint32_t p = 0, depth_p = 0;
    int32_t iteration = 0;  // never beyond max_iterations + 1
    const int32_t max_iter = pp.max_iterations;
    QInfo ip = ld_qinfo(ix.qinfo, 0);
    while (__any_sync(kFull, status == kUndecided)) {
        const bool act = status == kUndecided;
        // pooled extremes of the live terminals -> every level down to their LCA is unanimous
        const uint32_t umin = group_min<G>((act && w) ? first : 0xFFFFFFFFu), vmax = group_max<G>((act && w) ? last : 0u);
        const bool sane = act && umin <= vmax;   // groups that are done (or hold nothing) look up (root, root)
        const uint64_t dn = lca_depth_node(ix, sane ? umin : 0u, sane ? vmax : 0u);
        const uint32_t A = (uint32_t)dn, depth_a = (uint32_t)(dn >> 32);
        bool jump = act && depth_a > depth_p;
        if (jump) {
            const uint32_t d = depth_a - depth_p;
            if ((int64_t)iteration + (int64_t)d > (int64_t)max_iter) { iteration = (max_iter > 0 ? max_iter : 0) + 1; status = CLS_DEV_ERR_MAX_ITERATIONS; jump = false; }
            else { iteration += (int32_t)d; ip = ld_qinfo(ix.qinfo, A); p = A; depth_p = depth_a; }
        }
        const bool ident = jump && ip.child_count == 0;  // update_introspection_node.rs:32-87
        if (__any_sync(kFull, ident)) {
            const uint32_t ws = group_sum<G>(w);
            if (ident) { status = CLS_DEV_IDENTITY_FOUND; node_q = A; has_node = true; one = (int32_t)ws; rest = 0; }
        }
        // ---- evaluate the children of p
        bool ev = status == kUndecided;
        if (ev) {
            iteration++;
            if (iteration > max_iter) { status = CLS_DEV_ERR_MAX_ITERATIONS; ev = false; }
        }
        const uint32_t m = ip.child_count, p_end = ip.q_end;
        if (ev && m > 2) { status = kGroupRedo; ev = false; }
        if (ev && w && first == p) {  // the set ends at p itself for some tip: that is no vote for any child
            ++lo;
            first = lo < hi ? __ldg(terms + lo) : 0xFFFFFFFFu;
        }
        const bool has = ev && w && lo < hi;
        // children intervals tile [p+1, p_end): c1 = [p+1, bnd), c2 = [bnd, p_end)
        QInfo i1{p_end, 0, 0, 0};
        if (ev && m) i1 = ld_qinfo(ix.qinfo, p + 1);
        const uint32_t bnd = i1.q_end;
        const bool in1 = has && first < bnd, in2 = has && last >= bnd;
        const uint32_t tot = group_sum<G>((in1 ? w : 0u) | ((in2 ? w : 0u) << 10) | (((in1 && in2) ? w : 0u) << 20));
        const uint32_t c1 = tot & 1023u, c2 = (tot >> 10) & 1023u, both = tot >> 20;
        const uint32_t U = c1 + c2 - both, x1 = c1 - both, x2 = c2 - both;
        const uint32_t ncand = (c1 > 0) + (c2 > 0);
        const int32_t one1 = (int32_t)((ri && ncand > 1) ? x1 : c1), rest1 = ncand > 1 ? (int32_t)(ri ? U - c1 : U - x1) : 0;
        const int32_t one2 = (int32_t)((ri && ncand > 1) ? x2 : c2), rest2 = ncand > 1 ? (int32_t)(ri ? U - c2 : U - x2) : 0;
        const bool pr1 = c1 > 0 && one1 > rest1, pr2 = c2 > 0 && one2 > rest2;
        const uint32_t nprop = (uint32_t)pr1 + (uint32_t)pr2;
        bool pick2 = pr2 && !pr1;
        uint32_t n_best = nprop ? 1u : 0u;
        if (pr1 && pr2) {  // provably unreachable; kept for fidelity (:519-599)
            const int32_t d1 = one1 - rest1, d2 = one2 - rest2;
            if (d1 == d2) n_best = 2; else pick2 = d2 > d1;
        }
        const uint32_t win_q = pick2 ? bnd : p + 1;
        const int32_t win_one = pick2 ? one2 : one1, win_rest = pick2 ? rest2 : rest1;
        QInfo iw = i1;
        if (ev && pick2 && nprop) iw = ld_qinfo(ix.qinfo, bnd);
        if (ev) {
            if (nprop == 0) {
                if (iteration == 1) status = CLS_DEV_UNCL_NO_INTROSPECTION;
                else { status = CLS_DEV_MAX_RESOLUTION; node_q = p; has_node = true; }
            } else if (n_best != 1) {
                status = CLS_DEV_INCONCLUSIVE; node_q = p; has_node = true;
            } else if (iw.child_count == 0) {  // update_introspection_node.rs:32-87
                status = CLS_DEV_IDENTITY_FOUND; node_q = win_q; has_node = true; one = win_one; rest = win_rest;
            } else {
                p = win_q; ip = iw; depth_p++;
                const uint32_t win_end = iw.q_end;
                // every live set keeps its terminals inside the winner's interval (or drops out)
                bool live = has && last >= win_q && first < win_end;
                if (live && first < win_q) {
                    lo = lower_bound_terms(terms, lo + 1, hi, win_q);
                    first = __ldg(terms + lo);  // lo < hi because last >= win_q
                    live = first < win_end;
                }
                if (live && last >= win_end) {
                    hi = lower_bound_terms(terms, lo + 1, hi - 1, win_end);  // terms[lo] < win_end
                    last = __ldg(terms + hi - 1);
                }
                if (!live) w = 0;
            }
        }
    }
    if (have && status != kGroupRedo && (threadIdx.x & (G - 1)) == 0) {
        ResultRec res;
        res.node_id = has_node ? ix.q_node_id[node_q] : 0;
        res.one = one; res.rest = rest;
        res.n_matched = n_matched; res.n_root_matched = n_root; res.iterations = (uint32_t)iteration;
        res.status = status;
        *out = res;
    }
    return status == kGroupRedo;
}

// (asking ptxas for 8 or 4 resident CTAs per SM changes nothing: 5.08 / 5.07 against 5.07 ms, profiles/r2a)
#define CLS_DESCEND_BOUNDS __launch_bounds__(256)
template <int MAXSLOTS>
__global__ void CLS_DESCEND_BOUNDS descend_kernel(DeviceIndex ix, PlaceParams pp, ScanOut so, uint32_t first_read,
                                                      uint32_t n_reads, ResultRec *__restrict__ results, uint32_t fan_cap) {
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    uint32_t *cnt = smem + (size_t)warp * 2 * fan_cap, *excl = cnt + fan_cap;
    for (uint32_t o = lane; o < fan_cap; o += 32) { cnt[o] = 0; excl[o] = 0; }
    __syncwarp();
    uint32_t dyn_base = 0, dyn_used = kReadBlock;
#pragma unroll 1
    for (;;) {
        const uint32_t r = next_read(so.counters + 1, dyn_base, dyn_used);
        if (r >= n_reads) break;
        const uint2 me = so.meta[r];
        if (me.y == kDone) continue;
        const uint2 *pr = so.pairs + (size_t)r * so.cap;
        ResultRec *out = results + first_read + r;
        if (me.y <= 32) descend_from_pairs<1>(ix, pp, cnt, excl, pr, me.y, me.x, out);
        else if (MAXSLOTS == 2 || me.y <= 64) descend_from_pairs<2>(ix, pp, cnt, excl, pr, me.y, me.x, out);
        else if constexpr (MAXSLOTS > 2) {
            if (me.y <= 128) descend_from_pairs<4>(ix, pp, cnt, excl, pr, me.y, me.x, out);
            else descend_from_pairs<8>(ix, pp, cnt, excl, pr, me.y, me.x, out);
        }
    }
}

namespace {
#include "scan2_kernels.cuh"
#include "frag_kernels.cuh"
#include "giant_kernels.cuh"
}  // namespace

// The descent kernel of the short-read path (at most kPairCap pairs per read).  A warp takes 16 consecutive reads from the
// global counter, sorts them into size classes by their number of pairs and runs four reads of at most 8 pairs, or two
// of at most 16, side by side (finish_group); the others - and whatever finish_group hands back - go one read per warp.
template <int G>
__device__ __forceinline__ uint32_t run_groups(const DeviceIndex &ix, const PlaceParams &pp, const ScanOut &so, uint32_t first_read,
                                               ResultRec *__restrict__ results, uint32_t mask, uint32_t my_r, uint2 my_me) {
    constexpr uint32_t kGroups = 32 / G;
    const uint32_t lane = lane_id(), grp = lane / G, sub = lane & (G - 1);
    uint32_t redo = 0;
    while (mask) {
        // the next (up to) kGroups reads of the class: group g takes the g-th lowest set bit
        uint32_t mine = 0xFFFFFFFFu, picked = 0, rest = mask;
#pragma unroll
        for (uint32_t g = 0; g < kGroups; ++g) {
            if (rest) {
                const uint32_t j = (uint32_t)__ffs(rest) - 1u;
                rest &= rest - 1u;
                picked |= 1u << j;
                if (g == grp) mine = j;
            }
        }
        mask = rest;
        const bool have = mine != 0xFFFFFFFFu;
        const uint32_t src = have ? mine : 0u;
        const uint32_t r = __shfl_sync(kFull, my_r, src), nm = __shfl_sync(kFull, my_me.x, src), D = __shfl_sync(kFull, my_me.y, src);
        uint2 pr = make_uint2(0u, 0u);
        if (have && sub < D) pr = so.pairs[(size_t)r * so.cap + sub];
        const bool again = finish_group<G>(ix, pp, have, pr.x, pr.y, nm, results + first_read + r);
        const uint32_t am = __ballot_sync(kFull, again && sub == 0);   // bit g * G: group g hands its read back
#pragma unroll
        for (uint32_t g = 0; g < kGroups; ++g)
            if ((am >> (g * G)) & 1u) redo |= 1u << __shfl_sync(kFull, mine, g * G);
        (void)picked;
    }
    return redo;
}

__global__ void __launch_bounds__(256) descend16_kernel(DeviceIndex ix, PlaceParams pp, ScanOut so, uint32_t first_read,
                                                        uint32_t n_reads, ResultRec *__restrict__ results, uint32_t fan_cap) {
    extern __shared__ __align__(16) uint32_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    uint32_t *cnt = smem + (size_t)warp * 2 * fan_cap, *excl = cnt + fan_cap;
    for (uint32_t o = lane; o < fan_cap; o += 32) { cnt[o] = 0; excl[o] = 0; }
    __syncwarp();
    // 16 reads per request; 4 once less than one full request per warp is left - in the chunked launches of
    // cls_place_batch a warp only makes three or four requests, and the last round left a quarter of the warps idle
    // (1.37 against 1.12 ms per million reads)
    uint32_t step = 16u;
    const uint32_t all_warps = gridDim.x * (blockDim.x >> 5);
#pragma unroll 1
    for (;;) {
        uint32_t b0 = 0;
        if (lane == 0) b0 = atomicAdd(so.counters + 1, step);
        const uint32_t base = __shfl_sync(kFull, b0, 0);
        if (base >= n_reads) break;
        const uint32_t my_r = base + (lane & 15u);
        uint2 my_me = make_uint2(0u, kDone);
        if (lane < step && my_r < n_reads) my_me = so.meta[my_r];
        if ((uint64_t)base + step + 16ull * all_warps > n_reads) step = 4u;
        const bool todo = lane < 16 && my_me.y != kDone;
        const bool small_ok = todo && my_me.x < 1024u;
        uint32_t m8 = __ballot_sync(kFull, small_ok && my_me.y <= 8u);
        uint32_t m16 = __ballot_sync(kFull, small_ok && my_me.y > 8u && my_me.y <= 16u);
        uint32_t big = __ballot_sync(kFull, todo) & ~(m8 | m16);
        // a lone read of a class is cheaper in the next class up than in a mostly empty group round
        if (__popc(m8) == 1) { m16 |= m8; m8 = 0; }
        if (__popc(m16) == 1) { big |= m16; m16 = 0; }
        big |= run_groups<8>(ix, pp, so, first_read, results, m8, my_r, my_me);
        big |= run_groups<16>(ix, pp, so, first_read, results, m16, my_r, my_me);
        while (big) {
            const uint32_t j = (uint32_t)__ffs(big) - 1u;
            big &= big - 1u;
            const uint32_t r = __shfl_sync(kFull, my_r, j), nm = __shfl_sync(kFull, my_me.x, j), D = __shfl_sync(kFull, my_me.y, j);
            const uint2 *pr = so.pairs + (size_t)r * so.cap;
            if (D <= 32) descend_from_pairs<1>(ix, pp, cnt, excl, pr, D, nm, results + first_read + r);
            else descend_from_pairs<2>(ix, pp, cnt, excl, pr, D, nm, results + first_read + r);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Host launchers
// ------------------------------------------------------------------------------------------
static inline uint32_t ceil_log2(uint32_t x) {
    uint32_t l = 0;
    while ((1u << l) < x) ++l;
    return l;
}

PlaceGeom make_place_geom(uint32_t max_len, uint32_t k, uint32_t max_fanout) {
    PlaceGeom g{};
    g.max_len = max_len;
    const uint32_t H = max_len >= k ? 2 * (max_len - k + 1) : 2;
    g.str_words = ((max_len + 15u) / 16u) * 4u + 4u;  // decoded in 16-base groups, + over-read pad
    g.pk_words = (((max_len + 15u) / 16u) + 4u + 3u) & ~3u;
    g.t1_log2 = ceil_log2(H * 2 < 64 ? 64 : H * 2);
    g.t2_log2 = ceil_log2(H + 1 < 32 ? 32 : H + 1);
    g.t1_size = 1u << g.t1_log2;
    g.t2_size = 1u << g.t2_log2;
    g.fan_cap = max_fanout < 1 ? 1 : max_fanout;
    // tables + strings of one group (a warp or a CTA); the pre-mix rings (4 * kRing words per warp) come on top
    g.words_per_warp = g.t1_size + 3 * g.t2_size + 2 * g.str_words + 2 * g.pk_words + 2 * g.fan_cap + 2;
    g.words_per_warp = (g.words_per_warp + 3u) & ~3u;
    g.cta_per_read = (size_t)(g.words_per_warp + 4 * kRing) * 4 > 12 * 1024 ? 1u : 0u;  // reads beyond ~300 bp
    return g;
}

static inline ScanOut no_scan_out() {
    ScanOut so{};
    so.pairs = nullptr; so.meta = nullptr; so.cap = 0; so.counters = nullptr; so.ov_list = nullptr;
    return so;
}
// hand-over scratch of a launch: pairs[n_reads][cap], meta[n_reads], 16 counters, ov_list[n_reads]
static inline size_t scratch_bytes_for(uint32_t n_reads, uint32_t cap) { return (size_t)n_reads * ((size_t)cap * 8 + 8 + 4) + 256 + 64; }
static inline ScanOut carve_scratch(void *scratch, uint32_t n_reads, uint32_t cap) {
    char *base = reinterpret_cast<char *>(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    ScanOut so;
    so.pairs = reinterpret_cast<uint2 *>(base);
    so.meta = so.pairs + (size_t)n_reads * cap;
    so.cap = cap;
    so.counters = reinterpret_cast<uint32_t *>(so.meta + n_reads);
    so.ov_list = so.counters + 16;
    return so;
}
// The descent kernels run persistent CTAs: exactly as many as are resident at once (a larger grid would run a second,
// mostly empty wave).  descend16_kernel after the short-read scan (at most kPairCap pairs per read) ...
static cudaError_t launch_descend16(const DeviceIndex &ix, const PlaceParams &pp, const ScanOut &so, uint32_t first_read,
                                    uint32_t n_reads, ResultRec *results, uint32_t fan_cap, int sm_count, cudaStream_t stream) {
    const size_t dsmem = (size_t)2 * fan_cap * 4 * 8;
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, descend16_kernel, 256, dsmem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    const uint32_t dgrid = std::min<uint32_t>((uint32_t)(sm_count * occ), (n_reads + 127) / 128);
    descend16_kernel<<<dgrid, 256, dsmem, stream>>>(ix, pp, so, first_read, n_reads, results, fan_cap);
    return cudaGetLastError();
}
// ... and descend_kernel<8> after the kb-scale scan (at most kPairCapWide pairs per read)
static cudaError_t launch_descend8(const DeviceIndex &ix, const PlaceParams &pp, const ScanOut &so, uint32_t first_read,
                                   uint32_t n_reads, ResultRec *results, uint32_t fan_cap, int sm_count, cudaStream_t stream) {
    const size_t dsmem = (size_t)2 * fan_cap * 4 * 8;
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, descend_kernel<8>, 256, dsmem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    uint32_t dgrid = (uint32_t)(sm_count * occ);
    const uint32_t need = (n_reads + 7) / 8;
    if (dgrid > need) dgrid = need;
    descend_kernel<8><<<dgrid, 256, dsmem, stream>>>(ix, pp, so, first_read, n_reads, results, fan_cap);
    return cudaGetLastError();
}

// ---- kb-scale reads, k = 35, closed models: scanfrag_kernel hashes and probes (frag_kernels.cuh), the placement kernel takes
//      it from there.  The hits of one WAVE of reads live behind the hand-over scratch: 8 bytes per window and strand.
constexpr size_t kFragWaveBytes = (size_t)1 << 30;
static inline uint32_t frag_hit_stride(const PlaceGeom &g) { return 2u * (g.max_len - 34u); }
static inline uint32_t frag_wave_reads(uint32_t n_reads, const PlaceGeom &g) {
    const size_t per = (size_t)frag_hit_stride(g) * 8 + 1;
    return (uint32_t)std::min<size_t>(n_reads, std::max<size_t>(1, kFragWaveBytes / per));
}
static inline size_t frag_scratch_bytes(uint32_t n_reads, const PlaceGeom &g) {
    return (size_t)frag_wave_reads(n_reads, g) * ((size_t)frag_hit_stride(g) * 8 + 1) + 512;
}

template <int K, bool CLOSED, bool CTA>
static cudaError_t launch_place_t(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed,
                                  const ReadDesc *reads, uint32_t first_read, uint32_t n_reads,
                                  ResultRec *results, const PlaceGeom &g, int sm_count, cudaStream_t stream,
                                  void *scratch = nullptr, size_t scratch_bytes = 0, uint32_t *n_launches = nullptr,
                                  TraceBuf trace = TraceBuf{nullptr, nullptr, 0}) {
    const size_t ring = (size_t)4 * kRing * 4, group = (size_t)g.words_per_warp * 4;
    int warps = 8;
    size_t smem;
    if (CTA) {
        // the tables of a kb-scale read leave room for two CTAs per SM: sixteen warps each keep the SM busy
        warps = 16;
        if (group + ring * warps > 113 * 1024) warps = 8;
        smem = group + ring * warps;
    } else {
        while (warps > 1 && (group + ring) * warps > 200 * 1024) warps >>= 1;
        smem = (group + ring) * warps;
    }
    if (smem > 226 * 1024) return cudaErrorInvalidConfiguration;
    // always the same (maximal) opt-in size: concurrent callers with different geometries must not
    // lower each other's limit between this call and the launch
    cudaError_t e = cudaFuncSetAttribute(place_kernel<K, CLOSED, CTA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, place_kernel<K, CLOSED, CTA>, warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    uint32_t grid = (uint32_t)(sm_count * occ);
    const uint32_t need = CTA ? n_reads : (n_reads + warps - 1) / warps;
    if (grid > need) grid = need;
    if (grid == 0) return cudaSuccess;
    // kb-scale reads of closed models: the histogram goes to the wide descent kernel when the caller gave scratch
    const bool split = CTA && CLOSED && scratch && scratch_bytes >= scratch_bytes_for(n_reads, kPairCapWide) &&
                       (size_t)2 * g.fan_cap * 4 * 8 <= 48 * 1024;
    ScanOut so = no_scan_out();
    if (split) {
        so = carve_scratch(scratch, n_reads, kPairCapWide);
        if ((e = cudaMemsetAsync(so.counters, 0, 64, stream)) != cudaSuccess) return e;
    }
    bool two_phase = false;
    if constexpr (K == 35 && CLOSED && CTA) {
        const size_t pair_b = (scratch_bytes_for(n_reads, kPairCapWide) + 255) & ~(size_t)255;
        two_phase = split && !trace.rows && scratch_bytes >= pair_b + frag_scratch_bytes(n_reads, g);
        if (two_phase) {
            char *base = reinterpret_cast<char *>(((uintptr_t)scratch + 255) & ~(uintptr_t)255) + pair_b;
            const uint32_t wave = frag_wave_reads(n_reads, g), stride = frag_hit_stride(g);
            uint32_t *counter = reinterpret_cast<uint32_t *>(base);
            uint2 *hits = reinterpret_cast<uint2 *>(base + 256);
            uint8_t *redo = reinterpret_cast<uint8_t *>(hits + (size_t)wave * stride);
            const uint32_t frags = (g.max_len - 34u + kFragWindows - 1u) / kFragWindows;
            const size_t fsmem = (size_t)Scan2Layout<4>::kBytes * 8;
            if ((e = cudaFuncSetAttribute(scanfrag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem)) != cudaSuccess) return e;
            int focc = 0;
            if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&focc, scanfrag_kernel, 256, fsmem)) != cudaSuccess) return e;
            if (focc < 1) focc = 1;
            for (uint32_t a = 0; a < n_reads; a += wave) {
                const uint32_t n = std::min(wave, n_reads - a);
                if ((e = cudaMemsetAsync(counter, 0, 4, stream)) != cudaSuccess) return e;
                if ((e = cudaMemsetAsync(redo, 0, n, stream)) != cudaSuccess) return e;
                const uint64_t units = (uint64_t)n * frags;
                const uint32_t fgrid = (uint32_t)std::min<uint64_t>((uint64_t)sm_count * focc, (units + 7) / 8);
                scanfrag_kernel<<<fgrid, 256, fsmem, stream>>>(ix, packed, reads, first_read + a, n, frags, hits, stride, redo, counter);
                if ((e = cudaGetLastError()) != cudaSuccess) return e;
                ScanOut sa = so;
                sa.pairs = so.pairs + (size_t)a * so.cap;
                sa.meta = so.meta + a;
                int gocc = 0;
                if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&gocc, gather_kernel, 256, 0)) != cudaSuccess) return e;
                gather_kernel<<<std::min<uint32_t>((uint32_t)(sm_count * std::max(gocc, 1)), n), 256, 0, stream>>>(reads, first_read + a, n, hits, stride,
                                                                                                                redo, sa);
                if ((e = cudaGetLastError()) != cudaSuccess) return e;
                // reads with more node-set records than the descent kernel holds in registers: walked from shared memory
                const size_t wsmem = (size_t)kWideWarps * (5u * kGListCap + 2u * g.fan_cap) * 4;
                if ((e = cudaFuncSetAttribute(descend_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem)) != cudaSuccess) return e;
                if ((e = cudaMemsetAsync(counter, 0, 4, stream)) != cudaSuccess) return e;
                descend_wide_kernel<<<std::min<uint32_t>((uint32_t)(2 * sm_count), (n + 127) / 128), 32 * kWideWarps, wsmem, stream>>>(
                    ix, pp, first_read + a, n, hits, stride, redo, results, g.fan_cap, counter);
                if ((e = cudaGetLastError()) != cudaSuccess) return e;
                // the reads the kernels handed back (foreign bucket keys, a table that filled up): hashed again, as ever
                const uint32_t pgrid = std::min<uint32_t>((uint32_t)(sm_count * occ), n);
                place_kernel<K, CLOSED, CTA><<<pgrid, warps * 32, smem, stream>>>(ix, pp, packed, reads, first_read + a, n, results, g, sa, trace, redo);
                if ((e = cudaGetLastError()) != cudaSuccess) return e;
                if (n_launches) *n_launches += 4;
            }
        }
    }
    if (!two_phase) {
        place_kernel<K, CLOSED, CTA><<<grid, warps * 32, smem, stream>>>(ix, pp, packed, reads, first_read, n_reads, results, g, so, trace);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        if (n_launches) ++*n_launches;
    }
    if (split) {
        if ((e = launch_descend8(ix, pp, so, first_read, n_reads, results, g.fan_cap, sm_count, stream)) != cudaSuccess) return e;
        if (n_launches) ++*n_launches;
    }
    return cudaSuccess;
}

template <int K, bool CLOSED>
static cudaError_t launch_place_m(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed,
                                  const ReadDesc *reads, uint32_t first_read, uint32_t n_reads,
                                  ResultRec *results, const PlaceGeom &g, int sm_count, cudaStream_t stream,
                                  void *scratch, size_t scratch_bytes, uint32_t *n_launches) {
    return g.cta_per_read ? launch_place_t<K, CLOSED, true>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, scratch, scratch_bytes, n_launches)
                          : launch_place_t<K, CLOSED, false>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, nullptr, 0, n_launches);
}

// ---- reads whose tables exceed the shared memory of an SM: tables in global memory (giant_kernels.cuh) ----
static inline bool needs_giant(const PlaceGeom &g) {
    return g.cta_per_read && (size_t)g.words_per_warp * 4 + (size_t)4 * kRing * 4 * 8 > (size_t)226 * 1024;
}
constexpr size_t kGiantWaveBytes = (size_t)1 << 30;   // arenas of one wave of giant reads
static inline size_t giant_scratch_bytes(uint32_t n_reads, const PlaceGeom &g) {
    const size_t per = (size_t)g.words_per_warp * 4;
    const size_t wave = std::max<size_t>(1, kGiantWaveBytes / per);
    return std::min<size_t>(n_reads, wave) * per + 256;
}

template <int K>
static cudaError_t launch_giant(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads,
                                uint32_t first_read, uint32_t n_reads, ResultRec *results, const PlaceGeom &g, int sm_count,
                                cudaStream_t stream, void *scratch, size_t scratch_bytes, uint32_t *n_launches) {
    const size_t per = (size_t)g.words_per_warp * 4;
    uint32_t *arenas = reinterpret_cast<uint32_t *>(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    if (!scratch || scratch_bytes < per + 256) return cudaErrorMemoryAllocation;
    const uint32_t wave = (uint32_t)std::min<size_t>(n_reads, (scratch_bytes - 256) / per);
    const uint32_t W = g.max_len - ix.k_size + 1, chunks = 2 * ((W + 31u) / 32u);
    for (uint32_t a = 0; a < n_reads; a += wave) {
        const uint32_t n = std::min(wave, n_reads - a);
        // blocks per read: enough warps for its chunks, and about four blocks per SM over the wave
        uint32_t bx = std::max<uint32_t>(1u, std::min<uint32_t>((chunks + 63u) / 64u, std::max<uint32_t>(1u, (uint32_t)(4 * sm_count) / n)));
        const uint32_t bp = std::max<uint32_t>(1u, std::min<uint32_t>((g.words_per_warp + 256u * 64u - 1u) / (256u * 64u), std::max<uint32_t>(1u, (uint32_t)(8 * sm_count) / n)));
        giant_prepare_kernel<<<dim3(bp, n), 256, 0, stream>>>(packed, reads, first_read + a, g, arenas);
        giant_scan_kernel<K><<<dim3(bx, n), 256, 0, stream>>>(ix, reads, first_read + a, g, arenas);
        if (ix.closed) giant_finish_kernel<true><<<n, 32, 0, stream>>>(ix, pp, first_read + a, results, g, arenas);
        else giant_finish_kernel<false><<<n, 32, 0, stream>>>(ix, pp, first_read + a, results, g, arenas);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        if (n_launches) *n_launches += 3;
    }
    return cudaSuccess;
}

// ---- short reads, k = 35: scan kernel (+ descent kernel when the caller provides the hand-over scratch) ----
size_t place_scratch_bytes(uint32_t n_reads, uint32_t max_len, uint32_t k, uint32_t max_fanout) {
    if (max_len < k || n_reads == 0) return 0;
    const PlaceGeom g = make_place_geom(max_len, k, max_fanout);
    if (needs_giant(g)) return giant_scratch_bytes(n_reads, g);
    if (g.cta_per_read) {
        const size_t pair_b = (scratch_bytes_for(n_reads, kPairCapWide) + 255) & ~(size_t)255;
        return k == 35 ? pair_b + frag_scratch_bytes(n_reads, g) : pair_b;
    }
    return k == 35 ? scratch_bytes_for(n_reads, kPairCap) : 0;
}

template <bool CLOSED>
static cudaError_t launch_scan_old(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed,
                                   const ReadDesc *reads, uint32_t first_read, uint32_t n_reads, ResultRec *results,
                                   const PlaceGeom &g, int sm_count, cudaStream_t stream, const uint32_t *ov_list,
                                   const uint32_t *ov_count, uint32_t *n_launches) {
    const size_t ring = (size_t)4 * kRing * 4, group = (size_t)g.words_per_warp * 4;
    int warps = 8;
    while (warps > 1 && (group + ring) * warps > 200 * 1024) warps >>= 1;
    const size_t smem = (group + ring) * warps;
    if (smem > 226 * 1024) return cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(scan_kernel<CLOSED>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, scan_kernel<CLOSED>, warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    uint32_t grid = (uint32_t)(sm_count * occ);
    const uint32_t need = (n_reads + warps - 1) / warps;
    if (grid > need) grid = need;
    if (ov_list && grid > (uint32_t)sm_count) grid = (uint32_t)sm_count;  // the overflow list is short (its length is known on the device only)
    scan_kernel<CLOSED><<<grid, warps * 32, smem, stream>>>(ix, pp, packed, reads, first_read, n_reads, results, g, ov_list, ov_count);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (n_launches) ++*n_launches;
    return cudaSuccess;
}

template <int PPS, int MINB>
static cudaError_t launch_scan2(const DeviceIndex &ix, const uint32_t *packed, const ReadDesc *reads, uint32_t first_read,
                                uint32_t n_reads, const ScanOut &so, int sm_count, cudaStream_t stream) {
    const size_t smem = (size_t)Scan2Layout<PPS>::kBytes * 8;
    cudaError_t e = cudaFuncSetAttribute(scan2_kernel<PPS, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, scan2_kernel<PPS, MINB>, 256, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    uint32_t grid = (uint32_t)(sm_count * occ);
    const uint32_t need = (n_reads + 8 * kScanBlock - 1) / (8 * kScanBlock);
    if (grid > need) grid = need;
    scan2_kernel<PPS, MINB><<<grid, 256, smem, stream>>>(ix, packed, reads, first_read, n_reads, so);
    return cudaGetLastError();
}

// Short reads, k = 35.  Closed models with hand-over scratch: scan2_kernel -> descend_kernel -> scan_kernel over the
// (mostly empty) overflow list.  Otherwise the first-generation kernel with the descent fused.
template <bool CLOSED>
static cudaError_t launch_scan_t(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed,
                                 const ReadDesc *reads, uint32_t first_read, uint32_t n_reads, ResultRec *results,
                                 const PlaceGeom &g, int sm_count, cudaStream_t stream, void *scratch, size_t scratch_bytes,
                                 uint32_t *n_launches) {
    const bool split = CLOSED && scratch && scratch_bytes >= scratch_bytes_for(n_reads, kPairCap) &&
                       (size_t)2 * g.fan_cap * 4 * 8 <= 48 * 1024 && g.max_len <= Scan2Layout<8>::kMaxLen;
    if (!split) return launch_scan_old<CLOSED>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, nullptr, nullptr, n_launches);
    const ScanOut so = carve_scratch(scratch, n_reads, kPairCap);
    cudaError_t e = cudaMemsetAsync(so.counters, 0, 64, stream);
    if (e != cudaSuccess) return e;
    // a table well inside the 126 MB L2 wants registers, one that lives in HBM wants warps (scan2_kernels.cuh)
    const bool l2_resident = (ix.bucket_mask + 1) * sizeof(Slot) * 2 <= ((size_t)96 << 20);
    if (g.max_len > Scan2Layout<4>::kMaxLen) e = launch_scan2<8, 4>(ix, packed, reads, first_read, n_reads, so, sm_count, stream);
    else if (l2_resident) e = launch_scan2<4, 4>(ix, packed, reads, first_read, n_reads, so, sm_count, stream);
    else e = launch_scan2<4, 5>(ix, packed, reads, first_read, n_reads, so, sm_count, stream);
    if (e != cudaSuccess) return e;
    if (n_launches) ++*n_launches;
    if ((e = launch_descend16(ix, pp, so, first_read, n_reads, results, g.fan_cap, sm_count, stream)) != cudaSuccess) return e;
    if (n_launches) ++*n_launches;
    return launch_scan_old<true>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, so.ov_list, so.counters + 2, n_launches);
}

cudaError_t launch_place(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed,
                         const ReadDesc *reads, uint32_t first_read, uint32_t n_reads, ResultRec *results,
                         const PlaceGeom &g, int sm_count, cudaStream_t stream, void *scratch, size_t scratch_bytes,
                         uint32_t *n_launches) {
    if (n_reads == 0) return cudaSuccess;
    if (needs_giant(g))
        return ix.k_size == 35 ? launch_giant<35>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, scratch, scratch_bytes, n_launches)
                               : launch_giant<0>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, scratch, scratch_bytes, n_launches);
    if (ix.k_size == 35 && !g.cta_per_read) {
        return ix.closed ? launch_scan_t<true>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, scratch, scratch_bytes, n_launches)
                         : launch_scan_t<false>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, nullptr, 0, n_launches);
    }
    if (ix.k_size == 35) {
        return ix.closed ? launch_place_t<35, true, true>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, scratch, scratch_bytes, n_launches)
                         : launch_place_t<35, false, true>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, nullptr, 0, n_launches);
    }
    return ix.closed ? launch_place_m<0, true>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, scratch, scratch_bytes, n_launches)
                     : launch_place_m<0, false>(ix, pp, packed, reads, first_read, n_reads, results, g, sm_count, stream, nullptr, 0, n_launches);
}

// Debug export: place ONE read with the level-by-level walk and record the vote counters of every level.
cudaError_t launch_trace(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads,
                         ResultRec *results, const PlaceGeom &g, int sm_count, cudaStream_t stream, TraceBuf trace) {
    if (ix.k_size == 35) {
        if (g.cta_per_read)
            return ix.closed ? launch_place_t<35, true, true>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace)
                             : launch_place_t<35, false, true>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace);
        return ix.closed ? launch_place_t<35, true, false>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace)
                         : launch_place_t<35, false, false>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace);
    }
    if (g.cta_per_read)
        return ix.closed ? launch_place_t<0, true, true>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace)
                         : launch_place_t<0, false, true>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace);
    return ix.closed ? launch_place_t<0, true, false>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace)
                     : launch_place_t<0, false, false>(ix, pp, packed, reads, 0, 1, results, g, sm_count, stream, nullptr, 0, nullptr, trace);
}

cudaError_t launch_hash_only(const uint32_t *packed, uint32_t len, uint32_t k, uint64_t *out, cudaStream_t stream) {
    const uint32_t str_words = ((len + 15u) / 16u) * 4u + 4u + (k + 3) / 4;
    const uint32_t pk_words = (((len + 15u) / 16u) + 4u + 3u) & ~3u;
    const size_t smem = (size_t)(4 * kRing + 2 * str_words + 2 * pk_words) * 4;
    if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
    cudaError_t e;
    if (k == 35) {
        e = cudaFuncSetAttribute(hash_only_kernel<35>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        hash_only_kernel<35><<<1, 64, smem, stream>>>(packed, len, k, out, str_words, pk_words);
    } else {
        e = cudaFuncSetAttribute(hash_only_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        hash_only_kernel<0><<<1, 64, smem, stream>>>(packed, len, k, out, str_words, pk_words);
    }
    return cudaGetLastError();
}

#include "routed_kernels.cuh"

}  // namespace cls
