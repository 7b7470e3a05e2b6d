/*
 * classeq_b200.h - C ABI of the B200-native placement path of classeq.
 *
 * This is the drop-in boundary for ONE path of the reference
 * (LepistaBioinformatics/classeq2, v0.10.0): everything that happens inside
 *   core/src/use_cases/place_sequences/place_sequence.rs:42-602   (place_sequence)
 * for every query of a batch, i.e. what the closure at
 *   core/src/use_cases/place_sequences/mod.rs:151-159
 * computes.  The reference has no FFI layer of its own (pure safe Rust); the
 * entry points below are what a Rust `extern "C"` block would bind (see
 * INTEGRATION.md for the binding and for the call-site patch).
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every host buffer, the
 *     library owns device memory behind the opaque handles;
 *   - every function returns 0 (CLS_OK) or a negative cls_error code and never
 *     throws/aborts across the ABI; the text of the last error of the calling
 *     thread is available from cls_last_error();
 *   - per-query failures (reference: `Err(MappedErrors)` -> a line in
 *     `<out>.error`, mod.rs:160-169) are per-query STATUS values, not call errors;
 *   - there is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with CLS_ERR_CUDA.
 */
#ifndef CLASSEQ_B200_H
#define CLASSEQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLS_ABI_VERSION 2

typedef enum cls_error {
    CLS_OK = 0,
    CLS_ERR_INVALID_ARGUMENT = -1, /* NULL pointer, inconsistent sizes, malformed view            */
    CLS_ERR_CUDA = -2,             /* CUDA runtime/driver failure (incl. "no device")              */
    CLS_ERR_UNSUPPORTED = -3,      /* model outside the supported envelope (see cls_index_create) */
    CLS_ERR_OUT_OF_MEMORY = -4,
    CLS_ERR_NCCL = -5
} cls_error;

/* Node kinds: clade.rs:5-16 (serde UPPERCASE "ROOT" | "NODE" | "LEAF"). */
enum { CLS_KIND_ROOT = 0, CLS_KIND_NODE = 1, CLS_KIND_LEAF = 2 };

/* cls_model_view.flags */
enum {
    /* tree.root.children is `None` (place_sequence.rs:199-206 -> Err for every query
     * that survives the coverage gate).  `Some(vec![])` is expressed by an empty
     * child range instead. */
    CLS_MODEL_ROOT_CHILDREN_NONE = 1u,
    /* Testing knob: serialise node sets as general "mini-tree" records even when every set is
     * upward closed (the library picks the faster terminal-list records for such models; both
     * give identical results - see DESIGN.md "node-set records"). */
    CLS_MODEL_FORCE_GENERAL_SETS = 2u
};

/*
 * Borrowed, flat view of the reference's model types, built by the caller right
 * after `load_database` (ports/cli/src/cmds/place_sequences.rs:135,
 * ports/watcher/src/cmds/watch_dir/mod.rs:355):
 *
 *   Tree.root / Clade      core/src/domain/dtos/tree.rs:9-52, clade.rs:18-38
 *   Tree.kmers_map         core/src/domain/dtos/kmers_map.rs:77-87
 *                          map: MinimizerKey(u64) -> MinimizerValue(HashMap<u64 hash, HashSet<u64 node id>>)
 *
 * Nodes are listed in any order with node 0 == tree.root; `child_idx` holds node
 * INDICES (not ids) in the order of `Clade.children`.  Each (bucket key, hash)
 * pair of the two-level map is one entry; its node set is `set_node_ids[set_off[s]
 * .. set_off[s+1])` with s = entry_set[i] (several entries may share one set; a
 * caller that does not de-duplicate passes entry_set[i] = i).  Node sets hold the
 * reference's sparse u64 node IDS; ids that do not occur in the tree are legal
 * and ignored, exactly as the reference never consults them.
 */
typedef struct cls_model_view {
    uint32_t k_size;                /* KmersMap.k_size  (kmers_map.rs:79)                */
    uint32_t m_size;                /* KmersMap.m_size  (kmers_map.rs:83)                */
    uint32_t flags;
    uint32_t reserved;
    uint64_t n_nodes;
    const uint64_t *node_id;        /* [n_nodes]   Clade.id                              */
    const uint8_t *node_kind;       /* [n_nodes]   CLS_KIND_*  (Clade.kind; is_leaf() is by kind, clade.rs:166-172) */
    const uint64_t *child_off;      /* [n_nodes+1] CSR over child_idx                    */
    const uint64_t *child_idx;      /* [child_off[n_nodes]] node indices                 */
    uint64_t n_entries;
    const uint64_t *entry_bucket;   /* [n_entries] MinimizerKey.0                        */
    const uint64_t *entry_hash;     /* [n_entries] k-mer hash (murmur3_x64_128(.., 0).0) */
    const uint64_t *entry_set;      /* [n_entries] index into set_off                    */
    uint64_t n_sets;
    const uint64_t *set_off;        /* [n_sets+1]                                        */
    const uint64_t *set_node_ids;   /* [set_off[n_sets]] node ids                        */
} cls_model_view;

/*
 * A batch of queries as the reference's FASTA reader hands them to
 * place_sequence (file_or_stdin.rs:76-116 after sequence.rs:47-56): bodies are
 * ASCII, already filtered to A/C/G/T.  Lower-case a/c/g/t is accepted and
 * upper-cased (kmers_map.rs:410, :431-443).  Any other byte makes that one query
 * CLS_STATUS_ERR_INVALID_BASE (the reference would panic, kmers_map.rs:440).
 * Query i is bases[offsets[i] .. offsets[i+1]).
 */
typedef struct cls_batch {
    uint64_t n_queries;
    const uint8_t *bases;
    const uint64_t *offsets;        /* [n_queries+1], non-decreasing */
} cls_batch;

/* Knobs of place_sequence (place_sequence.rs:46-48, :64-75); same meaning as the
 * CLI's -i / -m / -r (ports/cli/src/cmds/place_sequences.rs:18-82).  The Option<>
 * defaults are applied by cls_params_default(). */
typedef struct cls_params {
    int32_t max_iterations;         /* default 1000                                    */
    uint32_t remove_intersection;   /* default 0 (false)                               */
    double min_match_coverage;      /* default 0.7; clamped to [0,1] by the library    */
} cls_params;

/*
 * Per-query outcome.  Strings of the reference are reconstructed by the host
 * from (status, node_id, n_root_matched) - see INTEGRATION.md.
 */
typedef enum cls_status {
    CLS_STATUS_ERR_TOO_SHORT = 0,      /* Err("The sequence does not contain enough kmers.")  place_sequence.rs:98-102 */
    CLS_STATUS_UNCL_NO_MATCH = 1,      /* Unclassifiable("Query sequence {header:?} may not be related to the phylogeny") :130-139 */
    CLS_STATUS_UNCL_NO_ROOT = 2,       /* Unclassifiable("Query sequence has no overlapping kmers with the reference tree") :156-166 */
    CLS_STATUS_UNCL_COVERAGE = 3,      /* Unclassifiable("Insufficient kmers coverage: {n_root_matched}") :241-254 */
    CLS_STATUS_UNCL_NO_INTROSPECTION = 4, /* Unclassifiable("Tree introspection not possible. ...") :446-454 */
    CLS_STATUS_MAX_RESOLUTION = 5,     /* MaxResolutionReached(node_id, "LCA Accepted") :456-465 */
    CLS_STATUS_IDENTITY_FOUND = 6,     /* IdentityFound(AdherenceTest{clade: node_id, one, rest}) update_introspection_node.rs:32-87 */
    CLS_STATUS_INCONCLUSIVE = 7,       /* Inconclusive(.., "Multiple proposals") :584-598 (provably unreachable; node_id = parent) */
    CLS_STATUS_ERR_MAX_ITERATIONS = 8, /* Err("The maximum number of iterations has been reached.") :295-301 */
    CLS_STATUS_ERR_ROOT_NO_CHILDREN = 9, /* Err("The root node does not have children. This is unexpected.") :199-206 */
    CLS_STATUS_ERR_INVALID_BASE = 10   /* non-ACGT byte in the body (reference: panic) */
} cls_status;

/* Caller-allocated result arrays, each of length n_queries.  `one`/`rest` are the
 * AdherenceTest fields (adherence_test.rs:6-17, i32); the three counters are the
 * values the reference records on its tracing span (place_sequence.rs:90-182). */
typedef struct cls_result {
    uint8_t *status;          /* cls_status                                               */
    uint64_t *node_id;        /* Clade.id of the placement (IDENTITY_FOUND, MAX_RESOLUTION, INCONCLUSIVE), else 0 */
    int32_t *one;             /* IDENTITY_FOUND only, else 0                              */
    int32_t *rest;            /* IDENTITY_FOUND only, else 0                              */
    uint32_t *n_query_kmers;  /* query.kmers.count        = 2*(L-k+1), 0 if L < k         */
    uint32_t *n_matched;      /* query.kmers.treeMatches  = |M|                           */
    uint32_t *n_root_matched; /* subject.kmers.queryMatches = |M_r|                       */
    uint32_t *iterations;     /* descent levels entered                                   */
} cls_result;

/* Device-side timing of the last cls_place_batch / cls_place_resident call on a
 * handle (CUDA events on the library's stream); the analogue of the reference's
 * PlacementTime (place_sequences/mod.rs:30-34) at batch granularity. */
typedef struct cls_timing {
    double pack_ms;    /* host 2-bit packing + length ordering   */
    double h2d_ms;     /* pinned host -> device copies            */
    double kernel_ms;  /* placement kernel(s)                     */
    double d2h_ms;     /* result records device -> host           */
    double total_ms;   /* wall clock of the call                  */
    uint64_t kernel_launches;
    uint64_t h2d_bytes;      /* bytes copied host -> device by the call (ABI version 2)                     */
    uint64_t d2h_bytes;      /* bytes copied device -> host by the call                                      */
    uint32_t pack_on_device; /* 0: bases packed to 2 bit on the host; 1: on the device, ASCII staged through pinned memory; */
    uint32_t reserved;       /* 2: on the device, ASCII copied straight from pinned caller memory; 3: mixed (cls_set_pack_mode) */
} cls_timing;

typedef struct cls_index cls_index;                 /* a model resident on one GPU            */
typedef struct cls_resident_batch cls_resident_batch; /* a packed query batch resident in HBM  */

int cls_abi_version(void);
const char *cls_last_error(void);                   /* thread-local, never NULL               */
void cls_params_default(cls_params *p);

/* Number of CUDA devices visible (>= 0) or a negative cls_error. */
int cls_device_count(void);

/*
 * Serialise the model to the GPU (once per model; the hook is right after
 * `load_database`).  Builds the open-addressed k-mer table, the de-duplicated
 * node-set records and the flattened tree, and uploads them to `device`.
 * CLS_ERR_UNSUPPORTED is returned - never a silently different answer - for:
 *   m_size > 12; k_size == 0; duplicated Clade ids; the same k-mer hash stored
 *   under two different bucket keys (a cross-bucket 64-bit collision,
 *   p ~ n^2 / 2^65); more than 2^24 nodes.
 */
int cls_index_create(const cls_model_view *model, int device, cls_index **out);
void cls_index_destroy(cls_index *index);

/*
 * ONE handle over several GPUs of the box, for callers that are a single process fanning out internally - the
 * reference's CLI, API and watcher (ports/cli/src/cmds/place_sequences.rs:125-156,
 * ports/watcher/src/cmds/watch_dir/mod.rs:480-490; the worker pool of place_sequences/mod.rs:123-126).  The
 * index is built once on the host and replicated on every listed device; cls_place_batch and
 * cls_place_sequences cut each batch into one contiguous part per replica (equal shares of the bases) and run the
 * parts side by side, one host thread + stream set per replica, all sharing the library's one host pool; results
 * are identical to the single-device call.  Every other call on such a handle (resident batches, FASTA ingest,
 * debug exports) works on its first device.
 *   cls_index_create_multi    `device_mask` bit d = CUDA device d; 0 = every visible device
 *   cls_index_create_devices  an explicit list; a device may be listed more than once (several replicas and
 *                             pipelines on one GPU)
 */
int cls_index_create_multi(const cls_model_view *model, uint64_t device_mask, cls_index **out);
int cls_index_create_devices(const cls_model_view *model, uint32_t n_devices, const int *devices, cls_index **out);

/* Introspection of a created index (all sizes in elements unless stated). */
typedef struct cls_index_info {
    uint32_t k_size, m_size;
    uint64_t n_entries;        /* entries uploaded (entries in unreachable buckets are dropped) */
    uint64_t n_buckets;        /* 32-byte buckets of two 16-byte slots                           */
    uint64_t table_bytes;
    uint64_t n_distinct_sets;
    uint64_t set_arena_bytes;
    uint64_t n_nonleaf_nodes;
    uint32_t max_nonleaf_fanout;
    int32_t device;
    uint32_t closed_sets;      /* 1: terminal-list records + LCA jumps; 0: general mini-tree records */
    uint32_t n_devices;        /* 1, or the number of replicas behind a multi-device handle (`device` = the first) */
} cls_index_info;
int cls_index_get_info(const cls_index *index, cls_index_info *info);

/*
 * The hot path, host buffers in / host buffers out: pack to 2 bit, order by
 * length, copy to the device, place, copy the result records back.  Callable
 * concurrently from several host threads on the same handle (each call takes a
 * private stream + workspace).  Replaces the body of the `par_bridge` closure's
 * call to place_sequence (mod.rs:123-159) for the whole batch.
 */
int cls_place_batch(cls_index *index, const cls_batch *batch, const cls_params *params,
                    cls_result *result);

/*
 * The same path split at the PCIe boundary, for callers (and benchmarks) that
 * keep the packed batch resident in HBM: upload once, place many times.
 * `stream` is a cudaStream_t (or NULL for the library's own stream);
 * cls_place_resident only enqueues work, cls_resident_fetch synchronises the
 * stream and scatters the result records into `result`.
 */
int cls_batch_upload(cls_index *index, const cls_batch *batch, cls_resident_batch **out);
int cls_place_resident(cls_index *index, cls_resident_batch *rb, const cls_params *params,
                       void *stream);
int cls_resident_fetch(cls_index *index, cls_resident_batch *rb, void *stream, cls_result *result);
void cls_resident_destroy(cls_resident_batch *rb);
/* Bytes the resident batch occupies in HBM (packed bases + descriptors + result records). */
uint64_t cls_resident_bytes(const cls_resident_batch *rb);

int cls_get_timing(const cls_index *index, cls_timing *out);

/*
 * Where cls_place_batch packs the query bases to 2 bit: 1 = on the host (AVX-512 / AVX2 packer on the library's host
 * pool; 38 bytes per 150-base read cross PCIe), 2 = on the device (the ASCII bases cross PCIe as they are - straight
 * from `batch->bases` when that memory is pinned, cudaHostAlloc / cudaHostRegister, else through a pinned staging
 * ring), 3 = mixed (batches of short reads: the chunks of a call are dealt to both in the ratio that lets the host
 * cores and the copy engine finish together; other batches: as 2), 0 = automatic: on the host with sixteen cores or
 * more per GPU in use, else on the device.  Process-wide; overrides the CLS_PACK=host|device|mixed environment variable.
 * Results are identical in every mode.  Returns the previous mode, or a negative cls_error.  The reference has no
 * counterpart: its reader hands place_sequence a String (place_sequences/mod.rs:118-159).
 */
int cls_set_pack_mode(int mode);

/*
 * FASTA ingest on the device: the raw bytes of a (multi-)FASTA file go to the GPU, which classifies
 * every byte (header line / sequence line), upper-cases, keeps A/C/G/T only - everything else is
 * deleted and the flanks joined (sequence.rs:47-56) - and packs the records to 2 bit; the record rules
 * of the reference's reader (file_or_stdin.rs:76-116: '>' lines start records and lose every '>',
 * empty lines are skipped, "\n" and "\r\n" terminate lines, a trailing record without sequence is
 * dropped while a mid-file one is kept, a record whose header text is empty is never sent and stops the
 * reader at the next header line if it had sequence, sequence before the first header stops it at once)
 * are applied to the per-line facts on the host.  The result is a resident batch exactly as
 * cls_batch_upload would have built from the reader's records (use cls_place_resident /
 * cls_resident_fetch; results come in record order), plus where every record's header sits in `text`:
 * header = text[header_begin + .. header_end) minus every '>'.  The arrays live in the batch and are
 * freed with it.  CLS_ERR_UNSUPPORTED: the text holds a byte >= 0x80 (Rust's to_uppercase() is
 * Unicode-aware; use the host reader, cls_filter_sequence, for such files).
 */
typedef struct cls_fasta_records {
    uint64_t n_records;
    const uint64_t *header_begin;   /* byte offset of the header line (its '>')                       */
    const uint64_t *header_end;     /* one past the header line's content ("\n" / "\r\n" excluded)   */
    const uint32_t *length;         /* filtered sequence length in bases                              */
} cls_fasta_records;
int cls_fasta_upload(cls_index *index, const uint8_t *text, uint64_t n_bytes, cls_resident_batch **out,
                     cls_fasta_records *records);

/*
 * FASTQ queries.  The reference reads only FASTA; these rules make a FASTQ file and its FASTA rendering (">" + title,
 * then the sequence line) place identically, for titles that are not empty and hold no '>', and a last record with at
 * least one base.  Lines end at "\n"; a "\r" right before the "\n" belongs to the terminator; the last line may lack one.
 * A record is exactly four lines (wrapped multi-line FASTQ is malformed):
 *   1. the title line starts with '@'; the header is the rest of the line, byte for byte (one '@' removed, nothing else);
 *   2. the sequence line, filtered as a FASTA sequence line: ASCII letters upper-cased, A/C/G/T kept, every other byte
 *      (N, IUPAC codes, '.', '-', bytes >= 0x80) deleted and the flanks joined;
 *   3. the separator line starts with '+'; the rest of it is ignored;
 *   4. the quality line has as many bytes as the sequence line (terminator excluded); its content is not used.
 * Every well-formed record is sent, also one whose filtered sequence is empty or shorter than k (it becomes
 * CLS_STATUS_ERR_TOO_SHORT) and one whose title is '@' alone (empty header).  Blank lines may follow the last record only.
 * A malformed file is refused as a whole with CLS_ERR_INVALID_ARGUMENT, nothing placed or written, and cls_last_error()
 * names the first bad record ("malformed FASTQ record <1-based number>: <reason>"): a title line without '@', a separator
 * line without '+', a quality length that differs from the sequence length, a blank line among the records, a truncated
 * last record, a title that is not valid UTF-8 (headers are written as UTF-8 text).
 *
 * cls_fastq_upload: FASTQ ingest on the device, as cls_fasta_upload: the resident batch cls_batch_upload would have built
 * from cls_fastq_read's records, in record order; header = text[header_begin .. header_end) as it is (header_begin is one
 * past the '@').  Works on the first device of a multi-device or sharded handle.  Texts of 4 GiB or more are
 * CLS_ERR_UNSUPPORTED.
 */
int cls_fastq_upload(cls_index *index, const uint8_t *text, uint64_t n_bytes, cls_resident_batch **out,
                     cls_fasta_records *records);

/*
 * Hash-sharded index (config 5 of BASELINE.json; SURVEY.md section 8e).  The k-mer table is split over up
 * to 8 GPUs by `owner = (hash >> 61) % n_shards`; node-set records and the tree are replicated.
 * The reference has no counterpart (its index is one in-memory HashMap, kmers_map.rs:77-87): these
 * calls split cls_place_resident at the two points where query k-mers cross NVLink, so that the
 * caller's collective (NCCL all-to-all on the device buffers) sits between them:
 *
 *   home  GPU  cls_route_hashes   hash every window, append it to its owner's segment
 *                                 d_send[o * seg_cap .. + counts_out[o])  (uint64 hashes);
 *                                 d_slot_win[slot] = window (strand * W + pos) behind that slot of d_send
 *                                 (uint16, n_shards * seg_cap entries); the hashes of one read form one
 *                                 contiguous run per owner (the run table stays inside `rb`)
 *   all-to-all of the segments (hashes travel to their owners)
 *   owner GPU  cls_shard_probe    one cls_probe_reply (12 bytes) per received hash, same order
 *   all-to-all back, into a reply buffer laid out exactly like d_send
 *   home  GPU  cls_place_routed   gating, distinct-hash counting, descent; results as cls_place_resident
 *
 * All d_* pointers are device memory owned by the caller.  cls_route_hashes synchronises `stream`
 * (the counts are needed on the host for the exchange); the other two only enqueue.
 * CLS_ERR_OUT_OF_MEMORY from cls_route_hashes means seg_cap was too small for some owner.
 * Reads longer than 161 bases (beyond the one-warp-per-read geometry) are CLS_ERR_UNSUPPORTED on this path.
 */
typedef struct cls_probe_reply {
    uint32_t set_off;   /* node-set record of the hit, 0xFFFFFFFF = not in the index       */
    uint32_t slot;      /* globally unique id of the table slot (distinct-hash counting)   */
    uint32_t code;      /* 2-bit prefix code of the entry's bucket key (gated at home)     */
} cls_probe_reply;
int cls_index_create_shard(const cls_model_view *model, int device, uint32_t shard, uint32_t n_shards,
                           cls_index **out);
int cls_routed_windows(cls_index *index, cls_resident_batch *rb, uint64_t *n_windows);
int cls_route_hashes(cls_index *index, cls_resident_batch *rb, uint32_t n_shards, uint64_t seg_cap,
                     void *d_send, void *d_slot_win, uint64_t *counts_out, void *stream);
int cls_shard_probe(cls_index *index, const void *d_hashes, uint64_t n, void *d_replies, void *stream);

/*
 * The same pipeline with the exchange FUSED into the kernels over NVLink peer memory (no collective
 * moves the payload).  Every rank owns an inbox (n_shards segments of seg_cap hashes) and a reply box
 * (n_shards segments of seg_cap replies) allocated with cls_peer_alloc, publishes their CUDA IPC
 * handles, and maps its peers' with cls_peer_open.  Then
 *   cls_route_hashes_p2p   d_segments[o] = owner o's inbox + my_rank * seg_cap (a peer pointer):
 *                          the route kernel stores every hash straight into its owner's memory;
 *   (counts all-to-all, 8 integers - also the point after which the inboxes are complete)
 *   cls_shard_probe        once per sender s: hashes = my inbox + s * seg_cap, replies = sender s's
 *                          reply box + my_rank * seg_cap (a peer pointer): the probe kernel stores
 *                          every reply straight into the memory of the GPU that asked;
 *   (barrier)  cls_place_routed on the local reply box.
 */
/*
 * The same hash-sharded index behind ONE handle of ONE process - the reference's CLI and watcher are single processes
 * (ports/cli/src/cmds/place_sequences.rs:125-156): shard s (entries with (hash >> 61) % n_shards == s) on devices[s], the
 * node-set records and the tree on every listed device.  1 <= n_shards <= 8; a device may be listed more than once
 * (several shards on one GPU).  Peer access is enabled between every pair of distinct listed devices; a pair that
 * cannot reach each other is CLS_ERR_UNSUPPORTED (there is no staged copy path).  On such a handle:
 *   cls_place_batch      cuts the batch into one part per shard (equal shares of the bases; part s is placed at its
 *                        HOME, devices[s]) and runs sub-batches of at most 2^19 reads per home, each as route -> probe ->
 *                        place on one stream per shard, chained by events across devices: every home stores every hash
 *                        straight into its owner's inbox (a peer store), every owner answers straight into the sender's
 *                        reply box, every home places once every owner has answered.  The host waits once per
 *                        sub-batch.  Exchange buffers are allocated once and grow with the sub-batch: at 2^19 reads of 150
 *                        bases (k = 35) on eight shards, 3.1 GB per GPU.  A segment that overflows (a low-complexity read
 *                        sends all its windows to one owner) runs that sub-batch again with an exact bound.
 *                        cls_place_sequences goes through it.
 *   cls_batch_upload, cls_fasta_upload, cls_resident_fetch   work on the first shard's device;
 *   cls_place_resident   routes the resident batch from there to every owner, and WAITS for the placement;
 *   cls_index_get_info   n_devices = n_shards, device = devices[0], n_entries / n_buckets / table_bytes summed;
 *   cls_get_timing, cls_index_destroy as usual.
 * Reads longer than 161 bases make the call CLS_ERR_UNSUPPORTED before anything runs.  The routed calls above and
 * cls_debug_node_counts refuse the handle (CLS_ERR_INVALID_ARGUMENT).  Calls on one sharded handle from several host
 * threads are correct and run one at a time.  Results are identical to those of a replicated index.
 */
int cls_index_create_sharded(const cls_model_view *model, uint32_t n_shards, const int *devices, cls_index **out);
int cls_route_hashes_p2p(cls_index *index, cls_resident_batch *rb, uint32_t n_shards, uint64_t seg_cap,
                         void *const *d_segments, void *d_slot_win, uint64_t *counts_out, void *stream);
int cls_peer_alloc(int device, uint64_t bytes, void **d_ptr, uint8_t ipc_handle[64]);
int cls_peer_open(int device, const uint8_t ipc_handle[64], void **d_ptr);
int cls_peer_close(int device, void *d_ptr);
int cls_peer_free(int device, void *d_ptr);
int cls_place_routed(cls_index *index, cls_resident_batch *rb, const void *d_replies, const void *d_slot_win,
                     uint32_t n_shards, uint64_t seg_cap, const cls_params *params, void *stream);

/*
 * Parity/debug exports.
 *
 * cls_debug_kmer_hashes: run the extraction + hashing kernel alone on one query
 * and return, in the reference's order (all forward windows, then all windows of
 * the reverse complement: kmers_map.rs:387-395), the 2*(L-k+1) values
 * murmurhash3_x64_128(window, 0).0.  `*n_out` receives the count; at most `cap`
 * values are written.  Does not need an index.
 *
 * cls_debug_host_murmur3_x64_128_h1: the host-side hash used while building the
 * index (bucket keys of all 4^m prefixes); exported so tests can pin it to the
 * reference's known answers without a GPU.
 */
int cls_debug_kmer_hashes(int device, uint32_t k_size, const uint8_t *bases, uint64_t len,
                          uint64_t *out_hashes, uint64_t cap, uint64_t *n_out);

/*
 * cls_debug_node_counts: per-node hit counts of ONE query, level by level (SURVEY.md section 8b).  The query
 * is placed with a walk that evaluates every level with the vote counters (no shortcut of any kind; the
 * outcome is the production path's - tests hold the two equal) and returns one row per evaluated level
 * and non-leaf child c of the current node with at least one vote:
 *   cnt  = |K(c)|, the matched distinct hashes whose node set contains c      (place_sequence.rs:319-333)
 *   excl = hashes whose node set contains c and no other non-leaf child of the current node
 *   u    = hashes whose node set contains any non-leaf child of the current node
 * from which the reference's (one, rest) follow: default one = cnt, rest = u - excl; remove_intersection
 * one = excl, rest = u - cnt; a single child with votes: (cnt, 0)              (place_sequence.rs:353-418)
 * Rows are sorted by (level, child id); `*n_rows` receives the number of rows the walk produced (it may
 * exceed `cap`).  `result` (optional, arrays of length 1) receives the placement.
 */
typedef struct cls_level_count {
    uint64_t parent_id, child_id;
    uint32_t level, cnt, excl, u;
} cls_level_count;
int cls_debug_node_counts(cls_index *index, const uint8_t *bases, uint64_t len, const cls_params *params,
                          cls_level_count *rows, uint64_t cap, uint64_t *n_rows, cls_result *result);
uint64_t cls_debug_host_murmur3_x64_128_h1(const uint8_t *data, uint64_t len, uint64_t seed);

/*
 * cls_debug_pack_read: the host-side 2-bit packer used by cls_place_batch / cls_batch_upload
 * (code = (ascii >> 1) & 3 -> A=0 C=1 T=2 G=3, 16 bases per 32-bit word, base j in bits 2j..2j+1).
 * Writes ceil(len / 16) words (at most cap_words).  Returns 1 if every byte was A/C/G/T (either
 * case), 0 if a byte was invalid, negative on bad arguments.  `variant` picks the body: 0 = the one the
 * library picked at run time (AVX-512, else AVX2+BMI2, else portable), 1 = portable SWAR, 2 = AVX2+BMI2,
 * 3 = AVX-512 (CLS_ERR_UNSUPPORTED if this CPU cannot run it); tests hold them all equal.
 */
int cls_debug_pack_read(const uint8_t *bases, uint64_t len, uint32_t *words_out, uint64_t cap_words, int variant);

/*
 * Native writer of the reference's result records (no GPU needed): what `place_sequences` appends to
 * `<out>.yaml|.jsonl` and `<out>.error` for every query (place_sequences/mod.rs:160-249), from the cls_result arrays
 * of a batch, the query headers and the serde fields of the tree's clades (clade.rs:18-38):
 *   Err statuses            -> the error text, appended to `err_text`
 *   Unclassifiable          -> {query, code}                                   (placement omitted, mod.rs:174-177)
 *   MaxResolutionReached    -> {query, code, annotations?, placement: <clade id>}
 *   IdentityFound           -> {query, code, annotations?, placement: {clade: <full Clade incl. children>, one, rest}}
 * `annotations` = the tree's annotations whose clade lies on the path to the root of the placement clade
 * (clade.rs:95-125), sorted by clade (mod.rs:180-224); every annotation is handed over ALREADY RENDERED, once per
 * tree, as the YAML list item ("- clade: 45\n  meta:\n  - !Taxid 1452\n") and as the JSON object.
 * format 0: serde_yaml documents ("---\n" + block style), 1: serde_json lines.  Nodes come parents first (pre-order
 * as a flattening of Tree.root produces it; node 0 = root) and the child lists must form a tree, else
 * CLS_ERR_INVALID_ARGUMENT.  NaN support / length = None; parent_id < 0 = None.
 * The two texts are malloc'ed by the library: release them with cls_text_free.
 */
typedef struct cls_record_tree {
    uint64_t n_nodes;
    const uint64_t *node_id;         /* Clade.id                                            */
    const int64_t *parent_id;        /* Clade.parent, -1 = None                             */
    const uint8_t *node_kind;        /* CLS_KIND_*                                          */
    const uint8_t *children_some;    /* Clade.children is Some(..) (possibly empty)         */
    const double *support;           /* NaN = None                                          */
    const double *length;            /* NaN = None                                          */
    const uint8_t *has_name;         /* Clade.name is Some                                  */
    const uint64_t *name_off;        /* [n_nodes+1] byte offsets into names                 */
    const char *names;               /* UTF-8, not terminated                               */
    const uint64_t *child_off;       /* [n_nodes+1] CSR over child_idx, as in cls_model_view */
    const uint64_t *child_idx;
    uint32_t has_annotations;        /* Tree.annotations is Some                            */
    uint32_t reserved;
    uint64_t n_annotations;
    const uint64_t *ann_clade;       /* [n_annotations] Annotation.clade                    */
    const uint64_t *ann_yaml_off;    /* [n_annotations+1] into ann_yaml                     */
    const char *ann_yaml;
    const uint64_t *ann_json_off;    /* [n_annotations+1] into ann_json                     */
    const char *ann_json;
} cls_record_tree;
int cls_records_render(const cls_record_tree *tree, uint64_t n_queries, const uint64_t *header_off, const char *headers,
                       const cls_result *result, uint32_t format, char **out_text, uint64_t *out_len, char **err_text,
                       uint64_t *err_len);
void cls_text_free(char *text);

/*
 * The reference's FASTA reader on the host (file_or_stdin.rs:76-116 with the filter of sequence.rs:47-56), for texts
 * the device ingest does not take (bytes >= 0x80, streams) and for callers that want the batch in host memory: the
 * records the reader sends, as a cls_batch-shaped pair (bases, offsets) plus where every header line sits in `text`
 * (header = text[header_begin .. header_end) minus every '>').  Same record rules as cls_fasta_upload.  The arrays
 * live in the handle: release it with cls_fasta_text_destroy.
 */
typedef struct cls_fasta_text cls_fasta_text;
typedef struct cls_fasta_host_records {
    uint64_t n_records;
    const uint64_t *header_begin;
    const uint64_t *header_end;
    const uint64_t *offsets;        /* [n_records+1] into bases */
    const uint8_t *bases;           /* filtered, upper-cased A/C/G/T */
} cls_fasta_host_records;
int cls_fasta_read(const uint8_t *text, uint64_t n_bytes, cls_fasta_text **out, cls_fasta_host_records *records);
void cls_fasta_text_destroy(cls_fasta_text *t);
/* The FASTQ reader on the host (rules above cls_fastq_upload): header = text[header_begin .. header_end) as it is.  The
 * handle is released with cls_fasta_text_destroy. */
int cls_fastq_read(const uint8_t *text, uint64_t n_bytes, cls_fasta_text **out, cls_fasta_host_records *records);

/*
 * `place_sequences` as the reference spells it (core/src/use_cases/place_sequences/mod.rs:43-53): a query FASTA (path,
 * NULL or "-" for stdin), an output path, the knobs -> `<out>.yaml|.jsonl` and `<out>.error`.
 *   cls_place_sequences    the whole use-case in one call: open, cls_place_batch per 2^20 queries, write, close
 *   cls_sequences_open     path handling of mod.rs:73-106 (extension replaced by the format's, parent directory created,
 *                          an existing result file removed if `overwrite`, else CLS_ERR_INVALID_ARGUMENT with the
 *                          reference's message) + the reader (:118-119); `batch` receives a borrowed view of the records
 *   cls_sequences_write    appends the records / error texts of the next `n` results (in record order) to the two files
 * The split exists for callers that place on their own schedule (several GPUs, resident batches) and for tests.
 * `format` is 0 (yaml) or 1 (jsonl), ORed with CLS_QUERY_FASTQ to read the query as FASTQ (cls_fastq_read; its headers
 * are written as they are, while FASTA headers lose every '>').  A malformed FASTQ query is CLS_ERR_INVALID_ARGUMENT
 * before either file is created.
 */
#define CLS_QUERY_FASTQ 0x100u
typedef struct cls_sequences cls_sequences;
int cls_sequences_open(const char *query_path, const char *out_file, uint32_t format, uint32_t overwrite,
                       cls_sequences **out, cls_batch *batch);
int cls_sequences_write(cls_sequences *s, const cls_record_tree *tree, uint64_t n, const cls_result *result);
void cls_sequences_close(cls_sequences *s);
int cls_place_sequences(cls_index *index, const cls_record_tree *tree, const char *query_path, const char *out_file,
                        const cls_params *params, uint32_t format, uint32_t overwrite, uint64_t *n_placed);

/*
 * cls_debug_plan_batch: the host-side planner of cls_place_batch / cls_batch_upload on its own (no GPU needed):
 * queries shorter than k get their status on the host (pre_status[i] = CLS_STATUS_ERR_TOO_SHORT, else 0xFF), the
 * others are grouped into LENGTH CLASSES - all reads of a class share one per-read table geometry; longest class
 * first; input order is kept inside a class - and laid out back to back at word boundaries: perm[j] = caller index
 * of the j-th read on the device (n_device of them), word_off[j] = its first packed word (word_off[n_device] =
 * n_words), classes[c] = {first device position, count, longest read}.  Any output pointer may be NULL.
 */
typedef struct cls_plan_class {
    uint32_t first, count, max_len;
} cls_plan_class;
int cls_debug_plan_batch(uint32_t k_size, const cls_batch *batch, uint8_t *pre_status, uint32_t *perm, uint32_t *word_off,
                         cls_plan_class *classes, uint32_t cap_classes, uint32_t *n_classes, uint32_t *n_device, uint64_t *n_words);

/*
 * cls_debug_plan_fast: the JUST-IN-TIME plan cls_place_batch uses for batches of short reads (every read has k .. 162
 * bases: the device order is the input order and nothing is decided on the host), run chunk by chunk over the whole
 * batch (`chunk_reads` per step) without a GPU.  *n_planned = reads planned before the first chunk holding a read that
 * does not qualify (cls_place_batch then starts over with the general plan of cls_debug_plan_batch) - the whole
 * batch when all qualify; word_off[j] (n_planned + 1 entries), lens[j], src_off[j] (where read j starts in
 * batch->bases, relative to the first read) for the planned reads; *max_len = their longest.  Output pointers other
 * than n_planned may be NULL.
 */
int cls_debug_plan_fast(uint32_t k_size, const cls_batch *batch, uint64_t chunk_reads, uint32_t *word_off, uint32_t *lens,
                        uint64_t *src_off, uint32_t *max_len, uint64_t *n_planned);

/*
 * Host helpers mirroring the reference's input side (no GPU needed).
 *
 * cls_filter_sequence: SequenceBody::remove_non_iupac_from_sequence
 * (sequence.rs:47-56) for one line of UTF-8 text: upper-case, keep A/C/G/T.
 * Writes at most `cap` bytes to `out`, returns the filtered length.
 */
uint64_t cls_filter_sequence(const uint8_t *line, uint64_t len, uint8_t *out, uint64_t cap);

/*
 * Host-side model builder (no GPU needed): the k-mer -> node-set map that the reference's
 * `map_kmers_to_tree` (core/src/use_cases/build_database/mod.rs:26-181) produces for a tree and
 * a list of (tip, sequence) pairs.  The call indexes EXACTLY the pairs it is given: which sequence
 * goes with which tip is the caller's decision, and it matters - the reference's MSA loop pairs
 * header i with the sequence of record i-1, gives the first header no k-mers and drops the last
 * sequence (mod.rs:93-116), so a database that must equal a reference-built one has to be fed those
 * pairs (the host mirror does so by default: classeq2_b200/build.py:map_kmers_to_tree(pairing=
 * "reference"), build_loop_records; pairing="own" gives every tip its own sequence).
 * For every tip, every window of the sequence and of its reverse complement
 * (kmers_map.rs:375-398) is hashed; the node set of a (bucket key, hash) entry is the union of
 * the root->tip id paths (both ends included, clade.rs:127-156) of the tips containing it.
 * Only the tree part of `tree` is read (k_size/m_size/nodes/children); `tip_node[i]` is the node
 * index of the tip whose sequence is bases[offsets[i] .. offsets[i+1]) (ASCII, A/C/G/T only).
 * cls_built_model_view fills `out` with the tree pointers of `tree` (borrowed from the caller)
 * plus entry/set arrays owned by the handle; it stays valid until cls_built_model_destroy.
 */
typedef struct cls_built_model cls_built_model;
int cls_model_build(const cls_model_view *tree, uint64_t n_tips, const uint64_t *tip_node,
                    const uint8_t *bases, const uint64_t *offsets, cls_built_model **out);
int cls_built_model_view(const cls_built_model *bm, const cls_model_view *tree, cls_model_view *out);
void cls_built_model_destroy(cls_built_model *bm);

/*
 * The same builder on the GPU (SURVEY.md section 8f, row 4: `build-db`, map_kmers_to_tree,
 * build_database/mod.rs:26-181).  Same arguments, same pairing of tips and sequences, and the same result
 * as cls_model_build: entries in (hash, bucket key) order, node sets numbered in order of their first
 * entry; only the order of the ids inside one node set differs (a set has no order: the reference keeps
 * HashSets, kmers_map.rs:16-17).  Every window of both strands is hashed by one kernel, the occurrences are
 * radix-sorted, entries / tip lists / node sets come from flag scans; the tree (parents, depths) is the only
 * thing prepared on the host.  No CPU fallback: CLS_ERR_CUDA without a device.  CLS_ERR_UNSUPPORTED: more
 * than 2^31 - 1 k-mer occurrences in one call, a sequence longer than 4 GiB, k_size beyond 100 KiB.
 */
int cls_model_build_device(const cls_model_view *tree, uint64_t n_tips, const uint64_t *tip_node,
                           const uint8_t *bases, const uint64_t *offsets, int device, cls_built_model **out);

#ifdef __cplusplus
}
#endif
#endif /* CLASSEQ_B200_H */
