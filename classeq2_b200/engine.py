"""Thin object layer over the C ABI: a model resident on one GPU and batched placement calls.

All compute happens in ``libclasseq_b200.so`` (hand-written sm_100a kernels); this module only
marshals numpy buffers.  Reference call being replaced for a whole batch at once:
``place_sequence`` (core/src/use_cases/place_sequences/place_sequence.rs:42-602) as invoked by the
``par_bridge`` closure of ``place_sequences`` (place_sequences/mod.rs:123-159).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib
from .model import FlatModel, Tree, _ptr

RESULT_DTYPES = (("status", np.uint8), ("node_id", np.uint64), ("one", np.int32), ("rest", np.int32),
                 ("n_query_kmers", np.uint32), ("n_matched", np.uint32), ("n_root_matched", np.uint32),
                 ("iterations", np.uint32))


@dataclass
class PlaceParams:
    """place_sequence.rs:46-48 - ``None`` means the reference's default (:64-75)."""
    max_iterations: Optional[int] = None
    min_match_coverage: Optional[float] = None
    remove_intersection: Optional[bool] = None

    def to_c(self) -> _lib.Params:
        p = _lib.Params()
        _lib.lib.cls_params_default(C.byref(p))
        if self.max_iterations is not None:
            p.max_iterations = int(self.max_iterations)
        if self.min_match_coverage is not None:
            p.min_match_coverage = float(self.min_match_coverage)
        if self.remove_intersection is not None:
            p.remove_intersection = 1 if self.remove_intersection else 0
        return p


class BatchResult:
    """Struct-of-arrays result of a batch (one element per query, caller order)."""

    def __init__(self, n: int):
        self.n = n
        for name, dt in RESULT_DTYPES:
            setattr(self, name, np.zeros(n, dtype=dt))

    def to_c(self) -> _lib.Result:
        r = _lib.Result()
        r.status = _ptr(self.status, _lib.u8p)
        r.node_id = _ptr(self.node_id, _lib.u64p)
        r.one = _ptr(self.one, _lib.i32p)
        r.rest = _ptr(self.rest, _lib.i32p)
        r.n_query_kmers = _ptr(self.n_query_kmers, _lib.u32p)
        r.n_matched = _ptr(self.n_matched, _lib.u32p)
        r.n_root_matched = _ptr(self.n_root_matched, _lib.u32p)
        r.iterations = _ptr(self.iterations, _lib.u32p)
        return r

    def row(self, i: int) -> dict:
        return {name: getattr(self, name)[i].item() for name, _ in RESULT_DTYPES}


def make_batch(seqs: Union[Sequence[Union[str, bytes]], Tuple[np.ndarray, np.ndarray]]):
    """(bases uint8[], offsets uint64[n+1]) from a list of strings, or pass such a pair through."""
    if isinstance(seqs, tuple) and len(seqs) == 2 and isinstance(seqs[0], np.ndarray):
        bases = np.ascontiguousarray(seqs[0], dtype=np.uint8)
        offsets = np.ascontiguousarray(seqs[1], dtype=np.uint64)
        return bases, offsets
    bs = [s.encode("utf-8") if isinstance(s, str) else bytes(s) for s in seqs]
    offsets = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        offsets[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    bases = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if bs else np.zeros(0, np.uint8)
    return bases, offsets


def _c_batch(bases: np.ndarray, offsets: np.ndarray) -> _lib.Batch:
    b = _lib.Batch()
    b.n_queries = len(offsets) - 1
    b.bases = _ptr(bases, _lib.u8p)
    b.offsets = _ptr(offsets, _lib.u64p)
    return b


class Index:
    """A model serialised to one GPU (``cls_index_create``): upload once per model."""

    def __init__(self, model: Union[FlatModel, Tree, "_lib.ModelView"], device: int = 0, keepalive=None,
                 shard: int = 0, n_shards: int = 1, devices=None, device_mask: Optional[int] = None, sharded_devices=None):
        """``n_shards > 1``: this handle holds the k-mer table entries with ``(hash >> 61) % n_shards ==
        shard`` only (``cls_index_create_shard``); such a handle serves the routed calls of
        :mod:`classeq2_b200.parallel` and refuses ``place_batch``.

        ``devices`` (a list of CUDA devices, repeats allowed) or ``device_mask`` (bit d = device d, 0 = all visible):
        ONE handle over several GPUs (``cls_index_create_devices`` / ``cls_index_create_multi``): the index is
        replicated, ``place_batch`` cuts every batch into one part per replica and runs them side by side.

        ``sharded_devices`` (a list of 1 to 8 CUDA devices, repeats allowed): ONE handle over a HASH-SHARDED index
        (``cls_index_create_sharded``): shard s of the k-mer table on ``sharded_devices[s]``, k-mers routed between the
        devices inside the library.  ``place_batch``, ``upload``, ``upload_fasta`` and :func:`place_sequences` work on it,
        for reads of up to 161 bases."""
        if isinstance(model, Tree):
            model = FlatModel.from_tree(model)
        view = model.view if hasattr(model, "view") else model
        self._keep = (model, keepalive)
        self._h = C.c_void_p()
        if sharded_devices is not None:
            devs = (C.c_int * len(sharded_devices))(*[int(d) for d in sharded_devices])
            _lib.check(_lib.lib.cls_index_create_sharded(C.byref(view), len(sharded_devices), devs, C.byref(self._h)))
            device = sharded_devices[0] if len(sharded_devices) else 0
        elif devices is not None:
            devs = (C.c_int * len(devices))(*[int(d) for d in devices])
            _lib.check(_lib.lib.cls_index_create_devices(C.byref(view), len(devices), devs, C.byref(self._h)))
            device = devices[0] if len(devices) else 0
        elif device_mask is not None:
            _lib.check(_lib.lib.cls_index_create_multi(C.byref(view), int(device_mask), C.byref(self._h)))
            device = self.info()["device"]
        else:
            _lib.check(_lib.lib.cls_index_create_shard(C.byref(view), int(device), int(shard), int(n_shards), C.byref(self._h)))
        self.device = int(device)
        self.shard, self.n_shards = int(shard), int(n_shards)

    def info(self) -> dict:
        inf = _lib.IndexInfo()
        _lib.check(_lib.lib.cls_index_get_info(self._h, C.byref(inf)))
        return {f: getattr(inf, f) for f, _ in inf._fields_}

    def place_batch(self, seqs, params: Optional[PlaceParams] = None) -> BatchResult:
        """Host buffers in, host buffers out (``cls_place_batch``)."""
        bases, offsets = make_batch(seqs)
        res = BatchResult(len(offsets) - 1)
        cb, cp, cr = _c_batch(bases, offsets), (params or PlaceParams()).to_c(), res.to_c()
        _lib.check(_lib.lib.cls_place_batch(self._h, C.byref(cb), C.byref(cp), C.byref(cr)))
        return res

    def place_batch_into(self, bases: np.ndarray, offsets: np.ndarray, res: BatchResult,
                         params: Optional[PlaceParams] = None) -> None:
        """Same as :meth:`place_batch` without any allocation on the Python side (benchmarks)."""
        cb, cp, cr = _c_batch(bases, offsets), (params or PlaceParams()).to_c(), res.to_c()
        _lib.check(_lib.lib.cls_place_batch(self._h, C.byref(cb), C.byref(cp), C.byref(cr)))

    def upload(self, seqs) -> "ResidentBatch":
        return ResidentBatch(self, seqs)

    def upload_fasta(self, text: Union[bytes, bytearray, memoryview, np.ndarray]):
        """``cls_fasta_upload``: parse, filter and pack a FASTA text ON THE DEVICE.  Returns ``(batch, headers,
        lengths)``: a :class:`ResidentBatch` holding the records the reference's reader would send, their
        headers (every '>' removed) and filtered lengths."""
        return self._upload_text(text, _lib.lib.cls_fasta_upload, lambda h: h.replace(b">", b"").decode("utf-8", "replace"))

    def upload_fastq(self, text: Union[bytes, bytearray, memoryview, np.ndarray]):
        """``cls_fastq_upload``: parse, check, filter and pack a FASTQ text ON THE DEVICE (rules: ``include/classeq_b200.h``).
        Returns ``(batch, headers, lengths)`` as :meth:`upload_fasta`, the headers as they stand after the '@'.  A malformed
        text raises :class:`ClsError` (``CLS_ERR_INVALID_ARGUMENT``) naming its first bad record."""
        return self._upload_text(text, _lib.lib.cls_fastq_upload, lambda h: h.decode("utf-8"))

    def _upload_text(self, text, upload, header):
        arr = np.frombuffer(text, dtype=np.uint8) if not isinstance(text, np.ndarray) else np.ascontiguousarray(text, dtype=np.uint8)
        if arr.size == 0:
            arr = np.zeros(1, np.uint8)
            n_bytes = 0
        else:
            n_bytes = arr.size
        h = C.c_void_p()
        rec = _lib.FastaRecords()
        _lib.check(upload(self._h, arr.ctypes.data_as(_lib.u8p), n_bytes, C.byref(h), C.byref(rec)))
        n = int(rec.n_records)
        hb = np.ctypeslib.as_array(rec.header_begin, shape=(n,)).copy() if n else np.zeros(0, np.uint64)
        he = np.ctypeslib.as_array(rec.header_end, shape=(n,)).copy() if n else np.zeros(0, np.uint64)
        ln = np.ctypeslib.as_array(rec.length, shape=(n,)).copy() if n else np.zeros(0, np.uint32)
        raw = arr.tobytes() if n else b""
        headers = [header(raw[int(a):int(b)]) for a, b in zip(hb, he)]
        return ResidentBatch._from_handle(self, h, n), headers, ln

    def debug_node_counts(self, seq, params: Optional[PlaceParams] = None, cap: int = 1 << 16):
        """``cls_debug_node_counts``: (rows, result) for one query; rows are dicts with parent_id, child_id, level,
        cnt, excl, u, sorted by (level, child id)."""
        b = seq.encode() if isinstance(seq, str) else bytes(seq)
        arr = np.frombuffer(b, dtype=np.uint8).copy() if b else np.zeros(1, np.uint8)
        rows = (_lib.LevelCount * cap)()
        n = C.c_uint64()
        res = BatchResult(1)
        cp, cr = (params or PlaceParams()).to_c(), res.to_c()
        _lib.check(_lib.lib.cls_debug_node_counts(self._h, _ptr(arr, _lib.u8p), len(b), C.byref(cp), rows, cap, C.byref(n), C.byref(cr)))
        if n.value > cap:
            raise RuntimeError(f"trace has {n.value} rows, cap is {cap}")
        out = [{f: getattr(rows[i], f) for f, _ in _lib.LevelCount._fields_} for i in range(n.value)]
        return out, res

    def shard_probe(self, d_hashes: int, n: int, d_replies: int, stream: int = 0) -> None:
        """``cls_shard_probe``: answer ``n`` received hashes (device pointers) from this shard of the table."""
        _lib.check(_lib.lib.cls_shard_probe(self._h, C.c_void_p(d_hashes), int(n), C.c_void_p(d_replies), C.c_void_p(stream)))

    def timing(self) -> dict:
        t = _lib.Timing()
        _lib.check(_lib.lib.cls_get_timing(self._h, C.byref(t)))
        return {f: getattr(t, f) for f, _ in t._fields_}

    def close(self):
        if self._h:
            _lib.lib.cls_index_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ResidentBatch:
    """A packed query batch resident in HBM (``cls_batch_upload``): upload once, place many times."""

    def __init__(self, index: Index, seqs):
        self.index = index
        bases, offsets = make_batch(seqs)
        self.n = len(offsets) - 1
        self._h = C.c_void_p()
        cb = _c_batch(bases, offsets)
        _lib.check(_lib.lib.cls_batch_upload(index._h, C.byref(cb), C.byref(self._h)))

    @classmethod
    def _from_handle(cls, index: "Index", handle, n: int) -> "ResidentBatch":
        rb = cls.__new__(cls)
        rb.index, rb.n, rb._h = index, n, handle
        return rb

    def place(self, params: Optional[PlaceParams] = None, stream: int = 0) -> None:
        """Enqueue the placement kernels on ``stream`` (a ``cudaStream_t`` as int); asynchronous."""
        cp = (params or PlaceParams()).to_c()
        _lib.check(_lib.lib.cls_place_resident(self.index._h, self._h, C.byref(cp), C.c_void_p(stream)))

    def fetch(self, stream: int = 0) -> BatchResult:
        res = BatchResult(self.n)
        cr = res.to_c()
        _lib.check(_lib.lib.cls_resident_fetch(self.index._h, self._h, C.c_void_p(stream), C.byref(cr)))
        return res

    def nbytes(self) -> int:
        return int(_lib.lib.cls_resident_bytes(self._h))

    # ---- hash-sharded index: the three device stages around the two all-to-alls --------------------
    def routed_windows(self) -> int:
        """Number of k-mer windows (2 * (L - k + 1) summed over the reads on the device)."""
        n = C.c_uint64()
        _lib.check(_lib.lib.cls_routed_windows(self.index._h, self._h, C.byref(n)))
        return int(n.value)

    def route_hashes(self, n_shards: int, seg_cap: int, d_send: int, d_slot_win: int, stream: int = 0) -> np.ndarray:
        """``cls_route_hashes``: fills the caller's device buffers (raw pointers) and returns the number
        of hashes routed to every owner."""
        counts = np.zeros(8, dtype=np.uint64)
        _lib.check(_lib.lib.cls_route_hashes(self.index._h, self._h, int(n_shards), int(seg_cap), C.c_void_p(d_send),
                                             C.c_void_p(d_slot_win), _ptr(counts, _lib.u64p), C.c_void_p(stream)))
        return counts[:n_shards].copy()

    def route_hashes_p2p(self, n_shards: int, seg_cap: int, seg_ptrs, d_slot_win: int, stream: int = 0) -> np.ndarray:
        """``cls_route_hashes_p2p``: ``seg_ptrs[o]`` is where owner ``o`` keeps the hashes of THIS rank (a
        peer pointer into its inbox); the route kernel stores there directly over NVLink."""
        counts = np.zeros(8, dtype=np.uint64)
        arr = (C.c_void_p * 8)(*[C.c_void_p(int(p)) for p in seg_ptrs] + [None] * (8 - len(seg_ptrs)))
        _lib.check(_lib.lib.cls_route_hashes_p2p(self.index._h, self._h, int(n_shards), int(seg_cap), arr,
                                                 C.c_void_p(d_slot_win), _ptr(counts, _lib.u64p), C.c_void_p(stream)))
        return counts[:n_shards].copy()

    def place_routed(self, d_replies: int, d_slot_win: int, n_shards: int, seg_cap: int,
                     params: Optional[PlaceParams] = None, stream: int = 0) -> None:
        cp = (params or PlaceParams()).to_c()
        _lib.check(_lib.lib.cls_place_routed(self.index._h, self._h, C.c_void_p(d_replies), C.c_void_p(d_slot_win),
                                             int(n_shards), int(seg_cap), C.byref(cp), C.c_void_p(stream)))

    def close(self):
        if self._h:
            _lib.lib.cls_resident_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def debug_kmer_hashes(seq: Union[str, bytes], k_size: int, device: int = 0) -> np.ndarray:
    """All window hashes of one query in the reference's order (``cls_debug_kmer_hashes``)."""
    b = seq.encode() if isinstance(seq, str) else bytes(seq)
    arr = np.frombuffer(b, dtype=np.uint8).copy() if b else np.zeros(0, np.uint8)
    cap = max(0, 2 * (len(b) - k_size + 1))
    out = np.zeros(max(cap, 1), dtype=np.uint64)
    n = C.c_uint64()
    _lib.check(_lib.lib.cls_debug_kmer_hashes(int(device), int(k_size), _ptr(arr, _lib.u8p), len(b),
                                              _ptr(out, _lib.u64p), cap, C.byref(n)))
    return out[: n.value]


def host_murmur3_h1(data: bytes, seed: int = 0) -> int:
    arr = np.frombuffer(data, dtype=np.uint8).copy() if data else np.zeros(1, np.uint8)
    return int(_lib.lib.cls_debug_host_murmur3_x64_128_h1(_ptr(arr, _lib.u8p), len(data), seed))


def filter_sequence(line: Union[str, bytes]) -> str:
    """``SequenceBody::remove_non_iupac_from_sequence`` (sequence.rs:47-56) via the C ABI."""
    b = line.encode("utf-8") if isinstance(line, str) else bytes(line)
    arr = np.frombuffer(b, dtype=np.uint8).copy() if b else np.zeros(1, np.uint8)
    out = np.zeros(max(len(b), 1), dtype=np.uint8)
    n = _lib.lib.cls_filter_sequence(_ptr(arr, _lib.u8p), len(b), _ptr(out, _lib.u8p), len(out))
    return out[:n].tobytes().decode("ascii")
