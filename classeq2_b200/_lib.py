"""ctypes binding of ``libclasseq_b200.so`` (the C ABI declared in ``include/classeq_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (``make -C classeq2_b200/csrc``).
There is deliberately no fallback of any kind: if the shared object is missing the import of
this module raises, and if no CUDA device is usable every compute call returns
``CLS_ERR_CUDA`` which :func:`check` turns into :class:`ClsError`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CLASSEQ_B200_LIB selects another build of the same library (to compare two builds)
LIB_PATH = os.environ.get("CLASSEQ_B200_LIB") or os.path.join(_HERE, "libclasseq_b200.so")

CLS_OK = 0
CLS_ERR_INVALID_ARGUMENT = -1
CLS_ERR_CUDA = -2
CLS_ERR_UNSUPPORTED = -3
CLS_ERR_OUT_OF_MEMORY = -4
CLS_ERR_NCCL = -5

QUERY_FASTQ = 0x100   # CLS_QUERY_FASTQ: ORed into the format of cls_sequences_open / cls_place_sequences

KIND_ROOT, KIND_NODE, KIND_LEAF = 0, 1, 2
MODEL_ROOT_CHILDREN_NONE = 1
MODEL_FORCE_GENERAL_SETS = 2

(STATUS_ERR_TOO_SHORT, STATUS_UNCL_NO_MATCH, STATUS_UNCL_NO_ROOT, STATUS_UNCL_COVERAGE,
 STATUS_UNCL_NO_INTROSPECTION, STATUS_MAX_RESOLUTION, STATUS_IDENTITY_FOUND, STATUS_INCONCLUSIVE,
 STATUS_ERR_MAX_ITERATIONS, STATUS_ERR_ROOT_NO_CHILDREN, STATUS_ERR_INVALID_BASE) = range(11)

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
u64p = C.POINTER(C.c_uint64)


class ModelView(C.Structure):
    _fields_ = [
        ("k_size", C.c_uint32), ("m_size", C.c_uint32), ("flags", C.c_uint32), ("reserved", C.c_uint32),
        ("n_nodes", C.c_uint64), ("node_id", u64p), ("node_kind", u8p), ("child_off", u64p), ("child_idx", u64p),
        ("n_entries", C.c_uint64), ("entry_bucket", u64p), ("entry_hash", u64p), ("entry_set", u64p),
        ("n_sets", C.c_uint64), ("set_off", u64p), ("set_node_ids", u64p),
    ]


class Batch(C.Structure):
    _fields_ = [("n_queries", C.c_uint64), ("bases", u8p), ("offsets", u64p)]


class Params(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("remove_intersection", C.c_uint32),
                ("min_match_coverage", C.c_double)]


class Result(C.Structure):
    _fields_ = [("status", u8p), ("node_id", u64p), ("one", i32p), ("rest", i32p),
                ("n_query_kmers", u32p), ("n_matched", u32p), ("n_root_matched", u32p), ("iterations", u32p)]


class Timing(C.Structure):
    _fields_ = [("pack_ms", C.c_double), ("h2d_ms", C.c_double), ("kernel_ms", C.c_double),
                ("d2h_ms", C.c_double), ("total_ms", C.c_double), ("kernel_launches", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("pack_on_device", C.c_uint32), ("reserved", C.c_uint32)]


class IndexInfo(C.Structure):
    _fields_ = [("k_size", C.c_uint32), ("m_size", C.c_uint32), ("n_entries", C.c_uint64),
                ("n_buckets", C.c_uint64), ("table_bytes", C.c_uint64), ("n_distinct_sets", C.c_uint64),
                ("set_arena_bytes", C.c_uint64), ("n_nonleaf_nodes", C.c_uint64),
                ("max_nonleaf_fanout", C.c_uint32), ("device", C.c_int32),
                ("closed_sets", C.c_uint32), ("n_devices", C.c_uint32)]


class FastaRecords(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("header_begin", u64p), ("header_end", u64p), ("length", u32p)]


class LevelCount(C.Structure):
    _fields_ = [("parent_id", C.c_uint64), ("child_id", C.c_uint64), ("level", C.c_uint32), ("cnt", C.c_uint32),
                ("excl", C.c_uint32), ("u", C.c_uint32)]


class PlanClass(C.Structure):
    _fields_ = [("first", C.c_uint32), ("count", C.c_uint32), ("max_len", C.c_uint32)]


class RecordTree(C.Structure):
    _fields_ = [("n_nodes", C.c_uint64), ("node_id", u64p), ("parent_id", C.POINTER(C.c_int64)), ("node_kind", u8p),
                ("children_some", u8p), ("support", C.POINTER(C.c_double)), ("length", C.POINTER(C.c_double)),
                ("has_name", u8p), ("name_off", u64p), ("names", C.c_char_p), ("child_off", u64p), ("child_idx", u64p),
                ("has_annotations", C.c_uint32), ("reserved", C.c_uint32), ("n_annotations", C.c_uint64),
                ("ann_clade", u64p), ("ann_yaml_off", u64p), ("ann_yaml", C.c_char_p), ("ann_json_off", u64p),
                ("ann_json", C.c_char_p)]


class FastaHostRecords(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("header_begin", u64p), ("header_end", u64p), ("offsets", u64p), ("bases", u8p)]


class ClsError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"classeq_b200 error {code}: {message}")
        self.code = code
        self.message = message


# name -> (restype, argtypes); every symbol include/classeq_b200.h declares
PROTOTYPES = {
    "cls_abi_version": (C.c_int, []),
    "cls_last_error": (C.c_char_p, []),
    "cls_params_default": (None, [C.POINTER(Params)]),
    "cls_device_count": (C.c_int, []),
    "cls_index_create": (C.c_int, [C.POINTER(ModelView), C.c_int, C.POINTER(C.c_void_p)]),
    "cls_index_destroy": (None, [C.c_void_p]),
    "cls_index_get_info": (C.c_int, [C.c_void_p, C.POINTER(IndexInfo)]),
    "cls_place_batch": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(Params), C.POINTER(Result)]),
    "cls_batch_upload": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.POINTER(C.c_void_p)]),
    "cls_place_resident": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p]),
    "cls_resident_fetch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Result)]),
    "cls_resident_destroy": (None, [C.c_void_p]),
    "cls_resident_bytes": (C.c_uint64, [C.c_void_p]),
    "cls_get_timing": (C.c_int, [C.c_void_p, C.POINTER(Timing)]),
    "cls_set_pack_mode": (C.c_int, [C.c_int]),
    "cls_fasta_upload": (C.c_int, [C.c_void_p, u8p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(FastaRecords)]),
    "cls_fastq_upload": (C.c_int, [C.c_void_p, u8p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(FastaRecords)]),
    "cls_index_create_shard": (C.c_int, [C.POINTER(ModelView), C.c_int, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "cls_index_create_multi": (C.c_int, [C.POINTER(ModelView), C.c_uint64, C.POINTER(C.c_void_p)]),
    "cls_index_create_devices": (C.c_int, [C.POINTER(ModelView), C.c_uint32, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]),
    "cls_index_create_sharded": (C.c_int, [C.POINTER(ModelView), C.c_uint32, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]),
    "cls_routed_windows": (C.c_int, [C.c_void_p, C.c_void_p, u64p]),
    "cls_route_hashes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, u64p, C.c_void_p]),
    "cls_shard_probe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "cls_route_hashes_p2p": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(C.c_void_p), C.c_void_p, u64p, C.c_void_p]),
    "cls_peer_alloc": (C.c_int, [C.c_int, C.c_uint64, C.POINTER(C.c_void_p), u8p]),
    "cls_peer_open": (C.c_int, [C.c_int, u8p, C.POINTER(C.c_void_p)]),
    "cls_peer_close": (C.c_int, [C.c_int, C.c_void_p]),
    "cls_peer_free": (C.c_int, [C.c_int, C.c_void_p]),
    "cls_place_routed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.POINTER(Params), C.c_void_p]),
    "cls_debug_kmer_hashes": (C.c_int, [C.c_int, C.c_uint32, u8p, C.c_uint64, u64p, C.c_uint64, u64p]),
    "cls_debug_node_counts": (C.c_int, [C.c_void_p, u8p, C.c_uint64, C.POINTER(Params), C.POINTER(LevelCount), C.c_uint64, u64p,
                                        C.POINTER(Result)]),
    "cls_debug_host_murmur3_x64_128_h1": (C.c_uint64, [u8p, C.c_uint64, C.c_uint64]),
    "cls_records_render": (C.c_int, [C.POINTER(RecordTree), C.c_uint64, u64p, C.c_char_p, C.POINTER(Result), C.c_uint32,
                                     C.POINTER(C.c_void_p), u64p, C.POINTER(C.c_void_p), u64p]),
    "cls_text_free": (None, [C.c_void_p]),
    "cls_fasta_read": (C.c_int, [u8p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(FastaHostRecords)]),
    "cls_fasta_text_destroy": (None, [C.c_void_p]),
    "cls_fastq_read": (C.c_int, [u8p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(FastaHostRecords)]),
    "cls_sequences_open": (C.c_int, [C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(Batch)]),
    "cls_sequences_write": (C.c_int, [C.c_void_p, C.POINTER(RecordTree), C.c_uint64, C.POINTER(Result)]),
    "cls_sequences_close": (None, [C.c_void_p]),
    "cls_place_sequences": (C.c_int, [C.c_void_p, C.POINTER(RecordTree), C.c_char_p, C.c_char_p, C.POINTER(Params), C.c_uint32,
                                      C.c_uint32, u64p]),
    "cls_debug_plan_fast": (C.c_int, [C.c_uint32, C.POINTER(Batch), C.c_uint64, u32p, u32p, u64p, u32p, u64p]),
    "cls_debug_plan_batch": (C.c_int, [C.c_uint32, C.POINTER(Batch), u8p, u32p, u32p, C.POINTER(PlanClass), C.c_uint32, u32p, u32p, u64p]),
    "cls_debug_pack_read": (C.c_int, [u8p, C.c_uint64, u32p, C.c_uint64, C.c_int]),
    "cls_filter_sequence": (C.c_uint64, [u8p, C.c_uint64, u8p, C.c_uint64]),
    "cls_model_build": (C.c_int, [C.POINTER(ModelView), C.c_uint64, u64p, u8p, u64p, C.POINTER(C.c_void_p)]),
    "cls_model_build_device": (C.c_int, [C.POINTER(ModelView), C.c_uint64, u64p, u8p, u64p, C.c_int, C.POINTER(C.c_void_p)]),
    "cls_built_model_view": (C.c_int, [C.c_void_p, C.POINTER(ModelView), C.POINTER(ModelView)]),
    "cls_built_model_destroy": (None, [C.c_void_p]),
}


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C classeq2_b200/csrc`). classeq2_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def last_error() -> str:
    return (lib.cls_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> int:
    if rc < 0:
        raise ClsError(rc, last_error())
    return rc
