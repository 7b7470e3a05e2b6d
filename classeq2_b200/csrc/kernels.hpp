// Launch interface of the sm_100a kernels (kernels.cu), used by the C-ABI layer (capi_internal.hpp).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/classeq_b200.h"
#include "device_types.hpp"

namespace cls {

// device-side status values are the ABI's cls_status values
constexpr uint32_t CLS_DEV_UNCL_NO_MATCH = CLS_STATUS_UNCL_NO_MATCH;
constexpr uint32_t CLS_DEV_UNCL_NO_ROOT = CLS_STATUS_UNCL_NO_ROOT;
constexpr uint32_t CLS_DEV_UNCL_COVERAGE = CLS_STATUS_UNCL_COVERAGE;
constexpr uint32_t CLS_DEV_UNCL_NO_INTROSPECTION = CLS_STATUS_UNCL_NO_INTROSPECTION;
constexpr uint32_t CLS_DEV_MAX_RESOLUTION = CLS_STATUS_MAX_RESOLUTION;
constexpr uint32_t CLS_DEV_IDENTITY_FOUND = CLS_STATUS_IDENTITY_FOUND;
constexpr uint32_t CLS_DEV_INCONCLUSIVE = CLS_STATUS_INCONCLUSIVE;
constexpr uint32_t CLS_DEV_ERR_MAX_ITERATIONS = CLS_STATUS_ERR_MAX_ITERATIONS;
constexpr uint32_t CLS_DEV_ERR_ROOT_NO_CHILDREN = CLS_STATUS_ERR_ROOT_NO_CHILDREN;

// Per-warp shared-memory geometry of one launch (all reads of a launch share it; the host
// groups reads into length classes so that short reads do not pay for long ones).
struct PlaceGeom {
    uint32_t str_words;       // 32-bit words per decoded strand string
    uint32_t pk_words;        // 32-bit words per 2-bit packed strand (zero padded)
    uint32_t t1_size, t1_log2;  // hit de-duplication set (u32 slots), power of two >= 2 * max hits
    uint32_t t2_size, t2_log2;  // node-set histogram (keys + counts), power of two > max hits
    uint32_t fan_cap;         // vote counters per warp (max non-leaf fan-out of the tree)
    uint32_t words_per_warp;  // tables + strings of one group (warp or CTA), without the pre-mix rings
    uint32_t cta_per_read;    // 1: one CTA per read (long reads), 0: one warp per read
    uint32_t max_len;         // longest read of the launch (bases)
};

PlaceGeom make_place_geom(uint32_t max_len, uint32_t k, uint32_t max_fanout);

// One row of the debug trace (cls_debug_node_counts): the vote counters of one child at one level.
struct TraceRow {
    uint64_t parent_id, child_id;
    uint32_t level, cnt, excl, u;
};
struct TraceBuf {
    TraceRow *rows;
    uint32_t *n_rows;
    uint32_t cap;
};
cudaError_t launch_trace(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads,
                         ResultRec *results, const PlaceGeom &g, int sm_count, cudaStream_t stream, TraceBuf trace);

// Scratch the short-read path (k = 35, closed models) wants for a launch over `n_reads` reads: the scan
// kernel hands every read's {node set, weight} pairs to a separate descent kernel through it.  0 when that
// path does not apply.  Without (enough) scratch the scan warps run the descent themselves.
// Reads whose per-read tables exceed the shared memory of an SM (beyond ~4 kb at k = 35) keep their tables in this
// scratch instead (giant_kernels.cuh): it is then REQUIRED, and sized for one wave of such reads.
size_t place_scratch_bytes(uint32_t n_reads, uint32_t max_len, uint32_t k, uint32_t max_fanout);

// Places reads [first_read, first_read + n_reads) of a length class.  `n_launches` (optional) is
// incremented once per kernel launched.
cudaError_t launch_place(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed,
                         const ReadDesc *reads, uint32_t first_read, uint32_t n_reads, ResultRec *results,
                         const PlaceGeom &g, int sm_count, cudaStream_t stream, void *scratch, size_t scratch_bytes,
                         uint32_t *n_launches);

// ---- hash-sharded index (routed_kernels.cuh) ------------------------------------------------------
constexpr uint32_t kMaxShards = 8;
constexpr uint32_t kProbeReplyBytes = 12;
cudaError_t launch_route(uint32_t k, const uint32_t *packed, const ReadDesc *reads, uint32_t first_read, uint32_t n_reads,
                         const PlaceGeom &g, uint32_t n_shards, uint64_t seg_cap, uint64_t *const *seg_ptrs,
                         uint16_t *slot_win, uint2 *runs, unsigned long long *cursor, uint32_t *overflow, int sm_count, cudaStream_t stream);
cudaError_t launch_shard_probe(const DeviceIndex &ix, uint32_t shard, const uint64_t *hashes, uint64_t n, void *replies,
                               cudaStream_t stream);
// The same over a segment of `seg_cap` slots whose count is read on the device: min(*d_count, seg_cap) hashes.
cudaError_t launch_shard_probe_counted(const DeviceIndex &ix, uint32_t shard, const uint64_t *hashes, uint64_t seg_cap,
                                       const unsigned long long *d_count, void *replies, int sm_count, cudaStream_t stream);
cudaError_t launch_place_routed(const DeviceIndex &ix, const PlaceParams &pp, const uint32_t *packed, const ReadDesc *reads,
                                uint32_t first_read, uint32_t n_reads, ResultRec *results, const PlaceGeom &g,
                                uint32_t n_shards, uint64_t seg_cap, const uint2 *runs, const uint16_t *slot_win, const void *replies,
                                int sm_count, cudaStream_t stream, void *scratch, size_t scratch_bytes);

// 2-bit packing on the device (pack_kernels.cu): ASCII bases of reads [first, first + count) -> packed words at their
// descriptors' word offsets; bad[j] = 1 for a read with a byte other than A/C/G/T (either case).
cudaError_t launch_ascii_pack(const uint8_t *ascii, const uint64_t *src_off, const ReadDesc *descs, uint32_t first, uint32_t count,
                              uint32_t max_len, uint32_t *words, uint8_t *bad, cudaStream_t stream);

cudaError_t launch_hash_only(const uint32_t *packed, uint32_t len, uint32_t k, uint64_t *out, cudaStream_t stream);

}  // namespace cls
