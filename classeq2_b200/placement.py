"""Host-side mirror of the reference's ``place_sequences`` use-case around the GPU path.

Reference (paths relative to its checkout):

* ``place_sequences``                 core/src/use_cases/place_sequences/mod.rs:43-270
* FASTA reader + ACGT filter          core/src/domain/dtos/file_or_stdin.rs:76-116, sequence.rs:47-56
* ``PlacementStatus`` / response      core/src/domain/dtos/placement_response.rs:7-94,
                                      adherence_test.rs:6-17, annotation.rs:3-34
* annotation join                     mod.rs:180-224, clade.rs:95-125
* ``load_database``                   ports/lib/src/functions/load_database.rs:9-53

Same argument meaning, same output files (``<out>.yaml|.jsonl`` and ``<out>.error``), same record
shape and strings.  The per-query algorithm (the body of the ``par_bridge`` closure's call to
``place_sequence``, mod.rs:151-159) runs on the GPU through ``cls_place_batch``; this module only
parses and batches; the records are serialised by the library's native writer (``cls_records_render``) or, as a
cross-check, by the emitters below.  Records are written in input order (the reference's order is the
nondeterministic completion order of its rayon tasks - compare outputs as maps keyed by query).
"""
from __future__ import annotations

import ctypes as C
import ctypes.util
import io
import json
import os
import sys
import time
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Tuple, Union

import numpy as np

from . import _lib
from .engine import BatchResult, Index, PlaceParams, filter_sequence
from .model import Clade, FlatModel, Tree

ERR_TOO_SHORT = "The sequence does not contain enough kmers."                       # place_sequence.rs:98-102
ERR_MAX_ITER = "The maximum number of iterations has been reached."                 # :295-301
ERR_ROOT_NO_CHILDREN = "The root node does not have children. This is unexpected."  # :199-206
ERR_INVALID_BASE = "Invalid character in sequence"                                  # kmers_map.rs:440 (a panic there)
MSG_NO_ROOT = "Query sequence has no overlapping kmers with the reference tree"     # :156-166
MSG_NO_INTROSPECTION = ("Tree introspection not possible. Query sequence has no overlapping kmers "
                        "with the reference tree")                                  # :446-454


# --------------------------------------------------------------------------------------------------
# FASTA reading (file_or_stdin.rs:76-116)
# --------------------------------------------------------------------------------------------------
def read_fasta_text(text: str) -> List[Tuple[str, str]]:
    """The (header, body) records the reference's reader sends down its channel, in order.
    Per line: skip if empty; a line starting with '>' starts a record (ALL '>' removed from the
    header); other lines are upper-cased and filtered to A/C/G/T (``cls_filter_sequence``) and
    appended.  A trailing record with an empty body is dropped, a mid-file one is kept (it then
    fails with "not enough kmers").  A sequence line before any header aborts the read; the caller
    ignores that error (mod.rs:119) and places what was sent so far."""
    out: List[Tuple[str, str]] = []
    header, parts = "", []
    lines = text.split("\n")
    terminated = [True] * len(lines)
    terminated[-1] = False          # what follows the last "\n" (possibly nothing) has no terminator
    if lines and lines[-1] == "":
        lines.pop()
    for line, term in zip(lines, terminated):
        if term and line.endswith("\r"):   # BufRead::lines strips "\n" and then one "\r": only "\r\n" is a terminator
            line = line[:-1]
        if line == "":
            continue
        if line.startswith(">"):
            if header != "":
                out.append((header, "".join(parts)))
                parts = []
            elif parts:
                return out
            header = line.replace(">", "")
        else:
            f = filter_sequence(line)
            if f:
                parts.append(f)
    if header != "" and parts:
        out.append((header, "".join(parts)))
    return out


def read_fasta_native(data: Union[bytes, bytearray, memoryview, str]) -> Tuple[List[str], np.ndarray, np.ndarray]:
    """``cls_fasta_read``: the same reader in the library (C++, one pass over the bytes).  Returns ``(headers, bases,
    offsets)`` - the records :func:`read_fasta_text` would return, the sequences as one ``cls_batch``-shaped pair."""
    raw = data.encode("utf-8") if isinstance(data, str) else bytes(data)
    arr = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    h, rec = C.c_void_p(), _lib.FastaHostRecords()
    _lib.check(_lib.lib.cls_fasta_read(arr.ctypes.data_as(_lib.u8p), len(raw), C.byref(h), C.byref(rec)))
    try:
        n = int(rec.n_records)
        offsets = np.ctypeslib.as_array(rec.offsets, shape=(n + 1,)).copy()
        total = int(offsets[-1])
        bases = np.ctypeslib.as_array(rec.bases, shape=(max(total, 1),))[:total].copy()
        hb = np.ctypeslib.as_array(rec.header_begin, shape=(n,)).tolist() if n else []
        he = np.ctypeslib.as_array(rec.header_end, shape=(n,)).tolist() if n else []
    finally:
        _lib.lib.cls_fasta_text_destroy(h)
    headers = [raw[a:b].replace(b">", b"").decode("utf-8") for a, b in zip(hb, he)]
    return headers, bases, offsets


def read_fasta(query: Union[str, os.PathLike, io.TextIOBase]) -> List[Tuple[str, str]]:
    """``FileOrStdin``: a path, ``"-"`` for stdin, or an open text stream."""
    if hasattr(query, "read"):
        return read_fasta_text(query.read())
    if str(query) == "-":
        return read_fasta_text(sys.stdin.read())
    with open(query, "r", encoding="utf-8", newline="") as f:   # no newline translation: "\r" alone is not a line break
        return read_fasta_text(f.read())


# --------------------------------------------------------------------------------------------------
# FASTQ reading (the rules are stated in include/classeq_b200.h, above cls_fastq_upload)
# --------------------------------------------------------------------------------------------------
FASTQ_REASONS = {
    1: "blank line inside the records",
    2: "title line does not start with '@'",
    3: "truncated record (fewer than four lines)",
    4: "separator line does not start with '+'",
    5: "quality length differs from sequence length",
    6: "title is not valid UTF-8",
}
_FASTQ_KEEP = bytes(range(256)).translate(bytes.maketrans(b"acgt", b"ACGT"))   # ASCII upper-casing of a/c/g/t
_FASTQ_DROP = bytes(c for c in range(256) if c not in b"ACGTacgt")


def read_fastq_text(data: Union[bytes, bytearray, memoryview, str]) -> List[Tuple[str, str]]:
    """The (header, sequence) records of a FASTQ text, in order: four lines per record, the header is the title line
    after its '@', the sequence line keeps its A/C/G/T bytes (either case) and loses every other byte.  A malformed text
    raises :class:`ClsError` (``CLS_ERR_INVALID_ARGUMENT``) with the message ``cls_fastq_read`` gives for it."""
    raw = data.encode("utf-8") if isinstance(data, str) else bytes(data)
    lines = raw.split(b"\n")
    terminated = [True] * len(lines)
    terminated[-1] = False          # what follows the last "\n" (possibly nothing) has no terminator
    if lines[-1] == b"":
        lines.pop()
        terminated.pop()
    lines = [ln[:-1] if term and ln.endswith(b"\r") else ln for ln, term in zip(lines, terminated)]
    last = max((i for i, ln in enumerate(lines) if ln), default=-1)     # blank lines may only follow the last record
    out: List[Tuple[str, str]] = []
    for r in range(last // 4 + 1 if last >= 0 else 0):
        def bad(code: int):
            return _lib.ClsError(_lib.CLS_ERR_INVALID_ARGUMENT, f"malformed FASTQ record {r + 1}: {FASTQ_REASONS[code]}")
        title = lines[4 * r]
        if not title:
            raise bad(1)
        if not title.startswith(b"@"):
            raise bad(2)
        if 4 * r + 3 >= len(lines):
            raise bad(3)
        seq, sep, qual = lines[4 * r + 1: 4 * r + 4]
        if not sep.startswith(b"+"):
            raise bad(4)
        if len(qual) != len(seq):
            raise bad(5)
        try:
            header = title[1:].decode("utf-8")
        except UnicodeDecodeError:
            raise bad(6) from None
        out.append((header, seq.translate(_FASTQ_KEEP, _FASTQ_DROP).decode("ascii")))
    return out


def read_fastq_native(data: Union[bytes, bytearray, memoryview, str]) -> Tuple[List[str], np.ndarray, np.ndarray]:
    """``cls_fastq_read``: the FASTQ reader in the library.  Returns ``(headers, bases, offsets)`` as
    :func:`read_fasta_native` - the records :func:`read_fastq_text` returns."""
    raw = data.encode("utf-8") if isinstance(data, str) else bytes(data)
    arr = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(1, np.uint8)
    h, rec = C.c_void_p(), _lib.FastaHostRecords()
    _lib.check(_lib.lib.cls_fastq_read(arr.ctypes.data_as(_lib.u8p), len(raw), C.byref(h), C.byref(rec)))
    try:
        n = int(rec.n_records)
        offsets = np.ctypeslib.as_array(rec.offsets, shape=(n + 1,)).copy()
        total = int(offsets[-1])
        bases = np.ctypeslib.as_array(rec.bases, shape=(max(total, 1),))[:total].copy()
        hb = np.ctypeslib.as_array(rec.header_begin, shape=(n,)).tolist() if n else []
        he = np.ctypeslib.as_array(rec.header_end, shape=(n,)).tolist() if n else []
    finally:
        _lib.lib.cls_fasta_text_destroy(h)
    headers = [raw[a:b].decode("utf-8") for a, b in zip(hb, he)]
    return headers, bases, offsets


def read_fastq(query: Union[str, os.PathLike, io.IOBase]) -> List[Tuple[str, str]]:
    """:func:`read_fastq_text` on a path, ``"-"`` for stdin, or an open stream."""
    if hasattr(query, "read"):
        return read_fastq_text(query.read())
    if str(query) == "-":
        return read_fastq_text(sys.stdin.buffer.read())
    with open(query, "rb") as f:
        return read_fastq_text(f.read())


# --------------------------------------------------------------------------------------------------
# serde-compatible emitters (serde_yaml 0.9 / serde_json 1.0 with ryu float formatting)
# --------------------------------------------------------------------------------------------------
def ryu_float(x: float) -> str:
    """f64 formatting of serde_yaml / serde_json (the ``ryu`` crate): shortest round-trip digits,
    decimal notation for 1e-5 <= |x| < 1e16, exponent form ``1e-6`` / ``1.5e16`` outside, and a
    trailing ``.0`` on integral values in decimal notation."""
    if x != x:
        return ".nan"
    if x in (float("inf"), float("-inf")):
        return ".inf" if x > 0 else "-.inf"
    if x == 0:
        return "-0.0" if str(x).startswith("-") else "0.0"
    sign = "-" if x < 0 else ""
    r = repr(abs(x))
    mant, _, exp = r.partition("e")
    ip, _, fp = mant.partition(".")
    if fp == "0":
        fp = ""
    digits = (ip + fp).lstrip("0")
    # decimal exponent of the first digit: value = 0.d1d2... * 10^kk
    kk = (len(ip) if ip != "0" else -(len(fp) - len(fp.lstrip("0")))) + (int(exp) if exp else 0)
    digits = digits.rstrip("0") or "0"
    n = len(digits)
    if 0 < kk <= 16:
        if n <= kk:
            return sign + digits + "0" * (kk - n) + ".0"
        return sign + digits[:kk] + "." + digits[kk:]
    if -5 < kk <= 0:
        return sign + "0." + "0" * (-kk) + digits
    e = kk - 1
    return sign + (digits if n == 1 else digits[0] + "." + digits[1:]) + "e" + str(e)


class Tag:
    """One ``annotation.rs`` ``Tag`` (externally tagged enum: YAML ``!Taxid 1452``, JSON ``{"Taxid":1452}``)."""
    __slots__ = ("name", "value")

    def __init__(self, name: str, value):
        self.name, self.value = name, value

    def __eq__(self, o):
        return isinstance(o, Tag) and (self.name, self.value) == (o.name, o.value)

    def __repr__(self):
        return f"Tag({self.name!r}, {self.value!r})"


_YAML_SPECIAL_FIRST = set("-?:,[]{}#&*!|>'\"%@`")


_F64 = None


def _serde_yaml_reads_it_as_another_type(s: str) -> bool:
    """serde_yaml 0.9 (``ser.rs`` ``serialize_str`` -> ``de.rs`` ``visit_untagged_scalar``; the crate is not vendored in the
    reference tree, this restates its published source): a string that would read back as null, a boolean, an integer or
    a finite float under the YAML 1.2 core schema - or as digits with a leading zero - is emitted single-quoted; for
    everything else the style is libyaml's choice."""
    global _F64
    import math
    import re
    if _F64 is None:
        _F64 = re.compile(r"[+-]?(\d+\.?\d*|\.\d+)([eE][+-]?\d+)?\Z")
    if s in ("", "null", "Null", "NULL", "~", "true", "True", "TRUE", "false", "False", "FALSE"):
        return True
    if not s.isascii():
        return False
    body = s[1:] if s[0] in "+-" else s
    if body[:2] in ("0x", "0o", "0b"):                      # parse_unsigned_int / parse_negative_int
        digits = {"0x": "0123456789abcdefABCDEF", "0o": "01234567", "0b": "01"}[body[:2]]
        rest = body[2:]
        if rest and all(c in digits for c in rest) and int(rest, {"0x": 16, "0o": 8, "0b": 2}[body[:2]]) < 2 ** 128:
            return True
    if body.isdigit():                                      # an integer, or digits_but_not_number (a leading zero)
        return True
    unpositive = s
    if s[0] == "+":
        unpositive = s[1:]
        if unpositive[:1] in ("+", "-"):
            return False
    if unpositive in (".inf", ".Inf", ".INF") or s in ("-.inf", "-.Inf", "-.INF", ".nan", ".NaN", ".NAN"):
        return True
    return bool(_F64.match(unpositive)) and math.isfinite(float(unpositive))        # str::parse::<f64>() and is_finite()


def _yaml_plain_ok(s: str) -> bool:
    """Whether the string goes out as a plain scalar: serde_yaml leaves the style to libyaml (see above) and libyaml's
    ``yaml_emitter_analyze_scalar`` allows a plain scalar in block context."""
    if _serde_yaml_reads_it_as_another_type(s):
        return False
    if s[0] == " " or s[-1] == " " or s.startswith(("---", "...")):   # libyaml: 0x20 only; document markers
        return False
    if s[0] in _YAML_SPECIAL_FIRST and not (s[0] in "-?:" and len(s) > 1 and s[1] not in " \t"):
        return False
    if ": " in s or " #" in s or s.endswith(":") or any(_yaml_special(ord(c)) for c in s):
        return False
    return True


_YAML_ESCAPES = {"\0": "\\0", "\a": "\\a", "\b": "\\b", "\t": "\\t", "\n": "\\n", "\v": "\\v", "\f": "\\f", "\r": "\\r",
                 "\x1b": "\\e", '"': '\\"', "\\": "\\\\", "\x85": "\\N", "\u2028": "\\L", "\u2029": "\\P"}


def _yaml_special(o: int) -> bool:
    """Outside libyaml's printable set (IS_PRINTABLE: 0x0A, 0x20-0x7E, 0x85, 0xA0-0xD7FF, 0xE000-0xFFFD without the BOM);
    0x85 and the Unicode line separators count as breaks, which a quoted one-line scalar cannot hold unescaped either."""
    return o < 0x20 or o == 0x7F or 0x80 <= o <= 0x9F or o in (0x2028, 0x2029, 0xFEFF) or 0xD800 <= o <= 0xDFFF or o >= 0xFFFE


def _yaml_scalar(v, indent: int) -> str:
    if v is None:
        return "null"
    if isinstance(v, bool):
        return "true" if v else "false"
    if isinstance(v, int):
        return str(v)
    if isinstance(v, float):
        return ryu_float(v)
    s = str(v)
    if "\n" in s:  # literal block scalar, serde_yaml's choice for multi-line strings
        body = s[:-1] if s.endswith("\n") else s
        chomp = "" if s.endswith("\n") else "-"
        pad = " " * indent
        return "|" + chomp + "\n" + "\n".join((pad + ln) if ln else "" for ln in body.split("\n"))
    if _yaml_plain_ok(s):
        return s
    # libyaml's choice when a plain scalar is not allowed: single quotes ('' for an apostrophe) unless the text holds a
    # character outside its printable set - then double quotes with its escapes (yaml_emitter_select_scalar_style)
    if not any(_yaml_special(ord(ch)) for ch in s):
        return "'" + s.replace("'", "''") + "'"
    out = ['"']
    for ch in s:
        o = ord(ch)
        if ch in _YAML_ESCAPES:
            out.append(_YAML_ESCAPES[ch])
        elif not _yaml_special(o):
            out.append(ch)
        elif o <= 0xFF:
            out.append("\\x%02X" % o)
        elif o <= 0xFFFF:
            out.append("\\u%04X" % o)
        else:
            out.append("\\U%08X" % o)
    out.append('"')
    return "".join(out)


def yaml_dump(obj, indent: int = 0) -> str:
    """serde_yaml-style block emission of dicts / lists / scalars / ``Tag``s (no document marker)."""
    out: List[str] = []
    _yaml_emit(obj, indent, out, first_prefix=None)
    return "\n".join(out) + "\n"


def _yaml_emit(obj, indent: int, out: List[str], first_prefix: Optional[str]):
    pad = " " * indent

    def line(prefix_pad, text):
        out.append(prefix_pad + text)

    if isinstance(obj, dict):
        first = True
        for k, v in obj.items():
            pp = first_prefix if (first and first_prefix is not None) else pad
            first = False
            key = _yaml_scalar(k, indent)
            if isinstance(v, dict) and v:
                line(pp, f"{key}:")
                _yaml_emit(v, indent + 2, out, None)
            elif isinstance(v, list) and v:
                line(pp, f"{key}:")
                _yaml_emit(v, indent, out, None)        # serde_yaml does not indent sequences in maps
            elif isinstance(v, Tag):
                line(pp, f"{key}: !{v.name} {_yaml_scalar(v.value, indent + 2)}")
            else:
                sv = "{}" if isinstance(v, dict) else "[]" if isinstance(v, list) else _yaml_scalar(v, indent + 2)
                line(pp, f"{key}: {sv}")
    elif isinstance(obj, list):
        for item in obj:
            if isinstance(item, (dict, list)) and item:
                _yaml_emit(item, indent + 2, out, first_prefix=pad + "- ")
            elif isinstance(item, Tag):
                line(pad, f"- !{item.name} {_yaml_scalar(item.value, indent + 2)}")
            else:
                line(pad, "- " + _yaml_scalar(item, indent + 2))
    else:
        line(pad if first_prefix is None else first_prefix, _yaml_scalar(obj, indent))


def json_dump(obj) -> str:
    """serde_json compact form (no spaces, ryu floats, externally tagged ``Tag``s)."""
    if isinstance(obj, Tag):
        return "{" + json.dumps(obj.name) + ":" + json_dump(obj.value) + "}"
    if isinstance(obj, dict):
        return "{" + ",".join(json.dumps(str(k), ensure_ascii=False) + ":" + json_dump(v) for k, v in obj.items()) + "}"
    if isinstance(obj, list):
        return "[" + ",".join(json_dump(v) for v in obj) + "]"
    if isinstance(obj, bool) or obj is None or isinstance(obj, int):
        return json.dumps(obj)
    if isinstance(obj, float):
        return ryu_float(obj) if obj == obj and abs(obj) != float("inf") else "null"
    return json.dumps(str(obj), ensure_ascii=False)


def load_annotations(path_or_text: Union[str, os.PathLike]) -> List[dict]:
    """Annotations YAML (``-a`` of ``cls place``, ports/cli/src/cmds/place_sequences.rs:137-144):
    a list of ``{clade: u32, meta?: [Tag]}`` with YAML-tagged enum values."""
    import yaml

    class L(yaml.SafeLoader):
        pass

    def tag(loader, suffix, node):
        v = loader.construct_scalar(node)
        return Tag(suffix, int(v) if suffix == "Taxid" else v)

    L.add_multi_constructor("!", tag)
    text = path_or_text
    if os.path.exists(str(path_or_text)):
        with open(path_or_text, "r", encoding="utf-8") as f:
            text = f.read()
    data = yaml.load(text, Loader=L) or []
    return [{"clade": int(a["clade"]), **({"meta": a["meta"]} if a.get("meta") is not None else {})} for a in data]


# --------------------------------------------------------------------------------------------------
# Result records (mod.rs:170-239, placement_response.rs:30-94)
# --------------------------------------------------------------------------------------------------
def rust_debug_str(s: str) -> str:
    """``format!("{:?}", s)`` of a Rust ``String``."""
    out = ['"']
    for ch in s:
        o = ord(ch)
        if ch == '"':
            out.append('\\"')
        elif ch == "\\":
            out.append("\\\\")
        elif ch == "\n":
            out.append("\\n")
        elif ch == "\r":
            out.append("\\r")
        elif ch == "\t":
            out.append("\\t")
        elif ch == "\0":
            out.append("\\0")
        elif o < 0x20 or o == 0x7F:
            out.append("\\u{%x}" % o)
        else:
            out.append(ch)
    out.append('"')
    return "".join(out)


def status_code(status: int, header: str, n_root_matched: int) -> Tuple[Optional[str], Optional[str]]:
    """(code string of an ``Ok`` placement, error string of an ``Err``) for a ``cls_status``."""
    S = _lib
    if status == S.STATUS_ERR_TOO_SHORT:
        return None, ERR_TOO_SHORT
    if status == S.STATUS_ERR_MAX_ITERATIONS:
        return None, ERR_MAX_ITER
    if status == S.STATUS_ERR_ROOT_NO_CHILDREN:
        return None, ERR_ROOT_NO_CHILDREN
    if status == S.STATUS_ERR_INVALID_BASE:
        return None, ERR_INVALID_BASE
    if status == S.STATUS_UNCL_NO_MATCH:
        return f"Unclassifiable: Query sequence SequenceHeader({rust_debug_str(header)}) may not be related to the phylogeny", None
    if status == S.STATUS_UNCL_NO_ROOT:
        return f"Unclassifiable: {MSG_NO_ROOT}", None
    if status == S.STATUS_UNCL_COVERAGE:
        return f"Unclassifiable: Insufficient kmers coverage: {n_root_matched}", None
    if status == S.STATUS_UNCL_NO_INTROSPECTION:
        return f"Unclassifiable: {MSG_NO_INTROSPECTION}", None
    if status == S.STATUS_MAX_RESOLUTION:
        return "MaxResolutionReached: LCA Accepted", None
    if status == S.STATUS_IDENTITY_FOUND:
        return "IdentityFound", None
    if status == S.STATUS_INCONCLUSIVE:
        return "Inconclusive: Multiple proposals", None
    raise ValueError(f"unknown status {status}")


class _TreeLookup:
    """id -> Clade and id -> path-to-root ids (clade.rs:95-125), built once per tree."""

    def __init__(self, tree: Tree):
        self.by_id: Dict[int, Clade] = {}
        self.parent: Dict[int, Optional[int]] = {}
        stack = [(tree.root, None)]
        while stack:
            c, p = stack.pop()
            if c.id not in self.by_id:          # get_node_by_id returns the first pre-order match
                self.by_id[c.id] = c
                self.parent[c.id] = c.parent
            for ch in reversed(c.children or []):
                stack.append((ch, c.id))

    def path_to_root(self, clade_id: int) -> set:
        path, cur, hops = set(), clade_id, 0
        while cur is not None and cur in self.by_id and hops <= len(self.by_id):
            path.add(cur)
            p = self.parent[cur]
            if p is not None:
                path.add(p)
            cur, hops = p, hops + 1
        return path


def placement_response(header: str, row: dict, tree: Tree, lookup: Optional[_TreeLookup] = None) -> Tuple[Optional[dict], Optional[str]]:
    """(``PlacementResponse`` as an ordered dict, error text).  Field order: query, code,
    annotations?, placement? (placement_response.rs:61-72); ``placement`` is the full AdherenceTest
    for IdentityFound, the bare clade id for MaxResolutionReached, the code string for Inconclusive,
    and omitted for Unclassifiable (mod.rs:174-177)."""
    code, err = status_code(row["status"], header, row["n_root_matched"])
    if err is not None:
        return None, err
    lookup = lookup or _TreeLookup(tree)
    o: dict = {"query": header, "code": code}
    placement, clade_id = None, None
    st = row["status"]
    if st == _lib.STATUS_IDENTITY_FOUND:
        clade_id = int(row["node_id"])
        placement = {"clade": lookup.by_id[clade_id].to_obj(), "one": int(row["one"]), "rest": int(row["rest"])}
    elif st == _lib.STATUS_MAX_RESOLUTION:
        clade_id = int(row["node_id"])
        placement = clade_id
    elif st == _lib.STATUS_INCONCLUSIVE:
        placement = code
    if tree.annotations is not None and clade_id is not None:  # mod.rs:180-224
        path = lookup.path_to_root(clade_id) if clade_id in lookup.by_id else set()
        recs = [a for a in tree.annotations if int(a["clade"]) in path]
        if recs:
            o["annotations"] = sorted(recs, key=lambda a: int(a["clade"]))
    if placement is not None:
        o["placement"] = placement
    return o, None


class RecordTree:
    """The serde fields of every clade of a tree (+ its annotations, rendered once) as the flat arrays of
    ``cls_record_tree``: what the library's native record writer ``cls_records_render`` needs."""

    def __init__(self, tree: Tree):
        clades, node_id, node_kind, child_off, child_idx = FlatModel.tree_arrays(tree.root)
        n = len(clades)
        nan = float("nan")
        self.node_id, self.node_kind = node_id, node_kind
        self.child_off, self.child_idx = child_off, (child_idx if len(child_idx) else np.zeros(1, np.uint64))
        self.parent_id = np.array([-1 if c.parent is None else c.parent for c in clades], np.int64)
        self.children_some = np.array([c.children is not None for c in clades], np.uint8)
        self.support = np.array([nan if c.support is None else c.support for c in clades], np.float64)
        self.length = np.array([nan if c.length is None else c.length for c in clades], np.float64)
        self.has_name = np.array([c.name is not None for c in clades], np.uint8)
        names = [(c.name or "").encode("utf-8") for c in clades]
        self.name_off = np.zeros(n + 1, np.uint64)
        self.name_off[1:] = np.cumsum([len(x) for x in names])
        self.names = b"".join(names)
        ann = tree.annotations or []
        ys = [yaml_dump([a]).encode("utf-8") for a in ann]
        js = [json_dump(a).encode("utf-8") for a in ann]
        self.ann_clade = np.array([int(a["clade"]) for a in ann] or [0], np.uint64)
        self.ann_yaml_off, self.ann_json_off = np.zeros(len(ann) + 1, np.uint64), np.zeros(len(ann) + 1, np.uint64)
        if ann:
            self.ann_yaml_off[1:] = np.cumsum([len(x) for x in ys])
            self.ann_json_off[1:] = np.cumsum([len(x) for x in js])
        self.ann_yaml, self.ann_json = b"".join(ys), b"".join(js)
        v = self.view = _lib.RecordTree()
        v.n_nodes = n
        v.node_id, v.node_kind = _p(self.node_id, _lib.u64p), _p(self.node_kind, _lib.u8p)
        v.parent_id = self.parent_id.ctypes.data_as(C.POINTER(C.c_int64))
        v.children_some, v.has_name = _p(self.children_some, _lib.u8p), _p(self.has_name, _lib.u8p)
        v.support = self.support.ctypes.data_as(C.POINTER(C.c_double))
        v.length = self.length.ctypes.data_as(C.POINTER(C.c_double))
        v.name_off, v.names = _p(self.name_off, _lib.u64p), self.names
        v.child_off, v.child_idx = _p(self.child_off, _lib.u64p), _p(self.child_idx, _lib.u64p)
        v.has_annotations = 0 if tree.annotations is None else 1
        v.n_annotations = len(ann)
        v.ann_clade = _p(self.ann_clade, _lib.u64p)
        v.ann_yaml_off, v.ann_yaml = _p(self.ann_yaml_off, _lib.u64p), self.ann_yaml
        v.ann_json_off, v.ann_json = _p(self.ann_json_off, _lib.u64p), self.ann_json


def _p(a: np.ndarray, typ):
    return a.ctypes.data_as(typ)


def render_records(headers: List[str], res: BatchResult, rtree: RecordTree, output_format: str = "yaml") -> Tuple[bytes, bytes]:
    """``cls_records_render``: the bytes the reference appends to ``<out>.yaml|.jsonl`` and to ``<out>.error`` for a
    batch, written by the library (multi-threaded C++) - byte-identical to :func:`placement_response` +
    :func:`yaml_dump` / :func:`json_dump` record by record."""
    return _render(headers, res, rtree, output_format, None, None)


def _render(headers: List[str], res: BatchResult, rtree: RecordTree, output_format: str, fo, fe):
    """``cls_records_render``; the two texts go straight from the library's buffers to the files ``fo`` / ``fe`` (no
    copy through ``bytes``: a batch of a million records can be gigabytes of YAML), or come back as ``bytes``."""
    hb = [h.encode("utf-8") for h in headers]
    off = np.zeros(len(hb) + 1, np.uint64)
    if hb:
        off[1:] = np.cumsum([len(x) for x in hb])
    text = b"".join(hb)
    out, err = C.c_void_p(), C.c_void_p()
    n_out, n_err = C.c_uint64(), C.c_uint64()
    cr = res.to_c()
    _lib.check(_lib.lib.cls_records_render(C.byref(rtree.view), len(hb), _p(off, _lib.u64p), text, C.byref(cr),
                                           0 if output_format == "yaml" else 1, C.byref(out), C.byref(n_out),
                                           C.byref(err), C.byref(n_err)))
    try:
        if fo is None:
            return _c_text(out, n_out.value), _c_text(err, n_err.value)
        for f, ptr, n in ((fo, out, n_out.value), (fe, err, n_err.value)):
            if n:
                f.write(memoryview((C.c_ubyte * n).from_address(ptr.value)))
        return None
    finally:
        _lib.lib.cls_text_free(out)
        _lib.lib.cls_text_free(err)


_C_TEXT_PIECE = 1 << 30


def _c_text(ptr, n: int) -> bytes:
    """``n`` bytes at ``ptr`` as ``bytes``.  ``ctypes.string_at`` takes a C ``int`` size: beyond 2 GiB it silently
    wraps (a million IdentityFound records near the root of a tree are several GB of YAML), so big texts are copied
    in pieces."""
    if not n:
        return b""
    if n <= _C_TEXT_PIECE:
        return C.string_at(ptr, n)
    base = ptr.value if isinstance(ptr, C.c_void_p) else int(ptr)
    return b"".join(C.string_at(base + a, min(_C_TEXT_PIECE, n - a)) for a in range(0, n, _C_TEXT_PIECE))


@dataclass
class PlacementTime:
    """place_sequences/mod.rs:30-34 - at batch granularity the per-sequence time is the batch's
    device+host time divided by the batch size."""
    sequence: str
    milliseconds_time: float


# --------------------------------------------------------------------------------------------------
# load_database (ports/lib/src/functions/load_database.rs:9-53)
# --------------------------------------------------------------------------------------------------
def _zstd_decompress(data: bytes) -> Optional[bytes]:
    name = ctypes.util.find_library("zstd") or "libzstd.so.1"
    try:
        z = C.CDLL(name)
    except OSError:
        return None
    z.ZSTD_getFrameContentSize.restype = C.c_ulonglong
    z.ZSTD_getFrameContentSize.argtypes = [C.c_char_p, C.c_size_t]
    z.ZSTD_decompress.restype = C.c_size_t
    z.ZSTD_decompress.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]
    z.ZSTD_isError.restype = C.c_uint
    z.ZSTD_isError.argtypes = [C.c_size_t]
    z.ZSTD_createDStream.restype = C.c_void_p
    z.ZSTD_freeDStream.argtypes = [C.c_void_p]
    z.ZSTD_decompressStream.restype = C.c_size_t

    class Buf(C.Structure):
        _fields_ = [("p", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]

    z.ZSTD_decompressStream.argtypes = [C.c_void_p, C.POINTER(Buf), C.POINTER(Buf)]
    size = z.ZSTD_getFrameContentSize(data, len(data))
    if size == 2**64 - 2:       # ZSTD_CONTENTSIZE_ERROR: not a zstd frame
        return None
    if size != 2**64 - 1:       # known size
        out = C.create_string_buffer(int(size) or 1)
        n = z.ZSTD_decompress(out, int(size) or 1, data, len(data))
        return None if z.ZSTD_isError(n) else out.raw[:n]
    # unknown size (streamed encoder, as the reference's `zstd::Encoder` writes): stream it
    ds = z.ZSTD_createDStream()
    src = C.create_string_buffer(data, len(data))
    chunk = C.create_string_buffer(1 << 20)
    ib = Buf(C.cast(src, C.c_void_p), len(data), 0)
    parts = []
    try:
        while ib.pos < ib.size:
            ob = Buf(C.cast(chunk, C.c_void_p), len(chunk), 0)
            r = z.ZSTD_decompressStream(ds, C.byref(ob), C.byref(ib))
            if z.ZSTD_isError(r):
                return None
            parts.append(chunk.raw[:ob.pos])
            if r == 0 and ib.pos >= ib.size:
                break
    finally:
        z.ZSTD_freeDStream(ds)
    return b"".join(parts)


def load_database(path: Union[str, os.PathLike]) -> Tree:
    """Try zstd -> YAML first, then plain YAML (load_database.rs:9-53); JSON is a YAML subset."""
    import yaml
    with open(path, "rb") as f:
        raw = f.read()
    text = _zstd_decompress(raw)
    if text is None:
        text = raw
    loader = getattr(yaml, "CSafeLoader", yaml.SafeLoader)
    obj = yaml.load(text.decode("utf-8"), Loader=loader)
    return Tree.from_obj(obj)


def _zstd_compress(data: bytes, level: int = 0) -> bytes:
    name = ctypes.util.find_library("zstd") or "libzstd.so.1"
    z = C.CDLL(name)
    z.ZSTD_compressBound.restype = C.c_size_t
    z.ZSTD_compressBound.argtypes = [C.c_size_t]
    z.ZSTD_compress.restype = C.c_size_t
    z.ZSTD_compress.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int]
    z.ZSTD_isError.restype = C.c_uint
    z.ZSTD_isError.argtypes = [C.c_size_t]
    cap = z.ZSTD_compressBound(len(data))
    buf = C.create_string_buffer(cap)
    n = z.ZSTD_compress(buf, cap, data, len(data), level)
    if z.ZSTD_isError(n):
        raise OSError("ZSTD_compress failed")
    return buf.raw[:n]


def save_database(tree: Tree, path: Union[str, os.PathLike], compress: bool = True) -> str:
    """What ``build-db`` writes (ports/cli/src/cmds/build_db.rs:67-75): the serde_yaml text of the ``Tree`` inside a
    zstd frame (level 0), extension forced to ``.cls``; ``compress=False`` writes the plain YAML under the given name.
    Returns the path written.  ``load_database`` reads both back."""
    text = yaml_dump(tree.to_obj()).encode("utf-8")
    if compress:
        root, _ = os.path.splitext(os.fspath(path))     # PathBuf::set_extension("cls")
        out = root + ".cls"
        data = _zstd_compress(text, 0)
    else:
        out, data = os.fspath(path), text
    with open(out, "wb") as f:
        f.write(data)
    return out


# --------------------------------------------------------------------------------------------------
# place_sequences (mod.rs:43-270)
# --------------------------------------------------------------------------------------------------
def place_sequences(query_sequence, tree: Tree, out_file: Union[str, os.PathLike],
                    max_iterations: Optional[int] = None, min_match_coverage: Optional[float] = None,
                    overwrite: bool = False, output_format: str = "yaml",
                    remove_intersection: Optional[bool] = None, *, index: Optional[Index] = None,
                    device: int = 0, batch_size: int = 1 << 20, ingest: str = "host",
                    writer: str = "native", reader: str = "native", query_format: str = "fasta") -> List[PlacementTime]:
    """Place every sequence of a FASTA input on ``tree`` and append one record per query to
    ``<out_file>.yaml|.jsonl`` (errors to ``<out_file>.error``), as the reference does.

    ``index`` may carry an already uploaded model (``cls_index_create`` once per model - the hook is
    right after ``load_database``); otherwise the model is uploaded for this call.
    ``ingest="device"`` parses, filters and packs the FASTA text on the GPU (``cls_fasta_upload``; file paths
    only, ASCII only) instead of with the host reader; the records and results are identical.
    ``writer="native"`` (default) serialises the records in the library (``cls_records_render``, multi-threaded C++);
    ``writer="python"`` uses this module's emitters - the two write byte-identical files (tests/test_record_writer.py).
    ``reader="native"`` (default, host ingest) parses the FASTA text in the library (``cls_fasta_read``); ``"python"``
    uses :func:`read_fasta_text` - the same records (tests/test_fasta_reader.py).
    ``query_format="fastq"`` reads the query as FASTQ (rules: ``include/classeq_b200.h``) with every ingest and reader:
    ``cls_fastq_upload``, ``cls_fastq_read`` or :func:`read_fastq_text`.  A malformed FASTQ raises :class:`ClsError`
    before either file is created.
    """
    if writer not in ("native", "python") or reader not in ("native", "python"):
        raise ValueError("writer / reader must be 'native' or 'python'")
    if query_format not in ("fasta", "fastq"):
        raise ValueError("query_format must be 'fasta' or 'fastq'")
    fastq = query_format == "fastq"
    if ingest not in ("host", "device"):
        raise ValueError("ingest must be 'host' or 'device'")
    if output_format not in ("yaml", "jsonl"):
        raise ValueError("output_format must be 'yaml' or 'jsonl'")           # output_format.rs
    base = os.fspath(out_file)
    root, _ext = os.path.splitext(base)                                       # PathBuf::set_extension
    out_path, err_path = f"{root}.{output_format}", f"{root}.error"
    out_dir = os.path.dirname(out_path)
    if out_dir and not os.path.exists(out_dir):
        try:
            os.mkdir(out_dir)                                                # create_dir, error ignored (:92-94)
        except OSError:
            pass
    if os.path.exists(out_path):
        if not overwrite:
            raise FileExistsError(f"Could not overwrite existing file {rust_debug_str(out_path)} when overwrite "
                                  "option is `false`.")                         # :96-101
        os.remove(out_path)

    own_index = index is None
    if own_index:
        index = Index(tree, device=device)
    device_batch = host_bases = host_offsets = None
    if ingest == "device":
        if hasattr(query_sequence, "read") or str(query_sequence) == "-":
            raise ValueError("ingest='device' reads a file path")
        try:
            with open(query_sequence, "rb") as f:
                raw = f.read()
        except OSError:
            raw = b""                                                          # nothing placed, no error (see below)
        try:
            device_batch, headers, _ = index.upload_fastq(raw) if fastq else index.upload_fasta(raw)
        except BaseException:
            if own_index:
                index.close()
            raise
        records = [(h, None) for h in headers]
        batch_size = max(len(records), 1)
    elif reader == "native":
        if hasattr(query_sequence, "read"):
            raw = query_sequence.read()
        elif str(query_sequence) == "-":
            raw = sys.stdin.buffer.read()
        else:
            try:
                with open(query_sequence, "rb") as f:
                    raw = f.read()
            except OSError:
                # a query that cannot be opened or read is not an error of the use-case: the reference drops the reader's
                # Result (`let _ = query_sequence.sequence_content_by_channel(sender)`, mod.rs:119), has created both files
                # by then (:111-115) and returns Ok with nothing placed - as cls_sequences_open does
                raw = b""
        try:
            headers, host_bases, host_offsets = read_fastq_native(raw) if fastq else read_fasta_native(raw)
        except BaseException:
            if own_index:
                index.close()
            raise
        records = [(h, None) for h in headers]
    else:
        try:
            records = read_fastq(query_sequence) if fastq else read_fasta(query_sequence)
        except OSError:
            records = []
        except BaseException:
            if own_index:
                index.close()
            raise
    lookup = _TreeLookup(tree) if writer == "python" else None
    rtree = RecordTree(tree) if writer == "native" else None
    params = PlaceParams(max_iterations, min_match_coverage, remove_intersection)
    times: List[PlacementTime] = []
    try:
        with open(out_path, "ab") as fo, open(err_path, "ab") as fe:
            for a in range(0, len(records), batch_size):
                chunk = records[a:a + batch_size]
                t0 = time.perf_counter()
                if device_batch is not None:
                    device_batch.place(params)
                    res = device_batch.fetch()
                elif host_offsets is not None:
                    off = host_offsets[a:a + len(chunk) + 1]
                    res = index.place_batch((host_bases[int(off[0]):int(off[-1])], off - off[0]), params)
                else:
                    res = index.place_batch([s for _, s in chunk], params)
                per_seq_ms = (time.perf_counter() - t0) * 1e3 / max(len(chunk), 1)
                if rtree is not None:
                    _render([h for h, _ in chunk], res, rtree, output_format, fo, fe)
                    times.extend(PlacementTime(header, per_seq_ms) for header, _ in chunk)
                    continue
                else:
                    buf_o, buf_e = [], []
                    for i, (header, _) in enumerate(chunk):
                        obj, err = placement_response(header, res.row(i), tree, lookup)
                        if err is not None:
                            buf_e.append(err)                                # err.to_string() (:160-169)
                        elif output_format == "yaml":
                            buf_o.append("---\n" + yaml_dump(obj))
                        else:
                            buf_o.append(json_dump(obj) + "\n")
                        times.append(PlacementTime(header, per_seq_ms))
                    text_o, text_e = "".join(buf_o).encode("utf-8"), "".join(buf_e).encode("utf-8")
                fo.write(text_o)
                fe.write(text_e)
    finally:
        if device_batch is not None:
            device_batch.close()
        if own_index:
            index.close()
    return times


def place_sequences_native(query_sequence: Union[str, os.PathLike], tree: Tree, out_file: Union[str, os.PathLike],
                           max_iterations: Optional[int] = None, min_match_coverage: Optional[float] = None,
                           overwrite: bool = False, output_format: str = "yaml",
                           remove_intersection: Optional[bool] = None, *, index: Optional[Index] = None, device: int = 0,
                           query_format: str = "fasta") -> int:
    """The whole use-case in ONE library call (``cls_place_sequences``): path handling, FASTA or FASTQ reader, placement on
    the GPU and record writer all run in the library; this wrapper only flattens the tree.  Same arguments as
    :func:`place_sequences` (a path or ``"-"`` for stdin), same files.  Returns the number of records placed."""
    if output_format not in ("yaml", "jsonl"):
        raise ValueError("output_format must be 'yaml' or 'jsonl'")
    if query_format not in ("fasta", "fastq"):
        raise ValueError("query_format must be 'fasta' or 'fastq'")
    fmt = (0 if output_format == "yaml" else 1) | (_lib.QUERY_FASTQ if query_format == "fastq" else 0)
    own_index = index is None
    if own_index:
        index = Index(tree, device=device)
    try:
        rtree = RecordTree(tree)
        params = PlaceParams(max_iterations, min_match_coverage, remove_intersection).to_c()
        n = C.c_uint64()
        rc = _lib.lib.cls_place_sequences(index._h, C.byref(rtree.view), os.fspath(query_sequence).encode(), os.fspath(out_file).encode(),
                                          C.byref(params), fmt, 1 if overwrite else 0, C.byref(n))
        if rc == _lib.CLS_ERR_INVALID_ARGUMENT and _lib.last_error().startswith("Could not overwrite existing file"):
            raise FileExistsError(_lib.last_error())
        _lib.check(rc)
        return int(n.value)
    finally:
        if own_index:
            index.close()
