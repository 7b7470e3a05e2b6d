"""FASTQ queries: the Python mirror of the rules (read_fastq_text), the host reader (cls_fastq_read) and the device ingest
(cls_fastq_upload) give the same records, or refuse a malformed text at the same first bad record; a FASTQ file places
exactly as its FASTA rendering does, through every ingest and both public calls."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import CAPI_HOST_SOURCES, CSRC

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")

S = b"ACGTTGCAAGCTTGCATGCCTGCAGGTCGACTCTAGAGGATCCCCGGGTACCGAGCTCGAATTC"


def rec(title: bytes, seq: bytes, eol: bytes = b"\n", sep: bytes = b"+", qual: bytes = None) -> bytes:
    return b"@" + title + eol + seq + eol + sep + eol + (b"I" * len(seq) if qual is None else qual) + eol


EDGE_CASES = [
    b"", b"\n", b"\n\n\r\n",
    rec(b"a", S), rec(b"a", S)[:-1],                                          # no final newline
    rec(b"a", S) + b"\n\n\r\n\n",                                             # trailing blank lines
    rec(b"a", S, b"\r\n") + rec(b"b", S.lower(), b"\r\n"),                     # CRLF
    rec(b"a", S, qual=b"@" + b"I" * (len(S) - 1)) + rec(b"b", S, qual=b"+" * len(S)),   # quality lines starting with '@' / '+'
    rec(b"x>y@z >", S) + rec(b"", S) + rec(b"@@", S),                          # '>' and '@' in titles, '@' alone
    rec(b"mixed", b"acgtNNRYK..--" + bytes([0xC3, 0xA9, 0xFF]) + b"ACgt" + S), # lower case, N, IUPAC, bytes >= 0x80
    rec(b"empty", b"") + rec(b"short", S[:20]) + rec(b"k", S[:35]) + rec(b"last", b""),   # empty and short sequences
    rec(b"long", (S * 160)[:10000]),                                          # a 10 kb read
    rec(b"sep", S, sep=b"+sep text"),
    rec(b"u\xc3\xa9\xe2\x82\xac", S),                                         # UTF-8 title
    rec(b"cr_at_eof", S)[:-1] + b"\r",                                        # "\r" without "\n" is quality content: malformed
]

MALFORMED = [   # (text, 1-based first bad record, reason code)
    (rec(b"a", S) + b"\n" + rec(b"b", S), 2, 1),
    (rec(b"a", S) + b">b\n" + S + b"\n+\n" + b"I" * len(S) + b"\n", 2, 2),
    (rec(b"a", S) + b"@b\nACGT\n", 2, 3),
    (rec(b"a", S) + b"@b\nACGT\n+\n", 2, 3),
    (rec(b"a", S) + b"@b\n", 2, 3),
    (rec(b"a", S) + rec(b"b", S, sep=b"-"), 2, 4),
    (rec(b"a", S) + rec(b"b", S, qual=b"II"), 2, 5),
    (rec(b"a", S) + rec(b"b", S, qual=b"I" * (len(S) - 1) + b"\rI"), 2, 5),   # a '\r' inside the line is content
    (rec(b"a", S) + rec(b"b\xff", S) + rec(b"c", S, sep=b"-"), 2, 6),
    (rec(b"a\xc3", S), 1, 6),
    (rec(b"a", S)[:-1] + b"\r", 1, 5),
    (rec(b"a", S) + b"\n\n" + b"x\n", 2, 1),
    (rec(b"a", S + b"\n" + S), 1, 4),                                         # wrapped (multi-line) FASTQ
    (b"ACGT\n", 1, 2),
]


def random_fastq(rng, n_reads, lens, bases, offsets, eol=b"\n", junk=True):
    """A FASTQ text of the given reads plus the records a reader must give for it (titles and filtered sequences)."""
    parts, want = [], []
    junk_bytes = list(b"NnRYKM-.*") + [0xC3, 0xA9, 0xFF]
    for i in range(n_reads):
        s = bases[int(offsets[i]):int(offsets[i + 1])].tobytes()
        if rng.random() < 0.3:
            s = s.lower()
        line = bytearray(s)
        if junk and rng.random() < 0.3:
            for p in sorted(rng.integers(0, len(line) + 1, int(rng.integers(1, 5))).tolist(), reverse=True):
                line[p:p] = bytes(rng.choice(junk_bytes, int(rng.integers(1, 4))).tolist())
        title = f"r{i} len={len(s)}".encode() + (b" @x>y" if rng.random() < 0.1 else b"")
        qual = bytes(rng.integers(33, 75, len(line), dtype=np.uint8).tolist())
        if rng.random() < 0.05 and qual:
            qual = b"@" + qual[1:]
        parts.append(b"@" + title + eol + bytes(line) + eol + b"+" + eol + qual + eol)
        want.append((title.decode(), s.upper().decode()))
    return b"".join(parts), want


# ---- host readers, no GPU ----------------------------------------------------------------------------------------------
def _host_agree(text: bytes):
    from classeq2_b200 import _lib
    from classeq2_b200.placement import read_fastq_native, read_fastq_text
    try:
        want = read_fastq_text(text)
    except _lib.ClsError as e:
        with pytest.raises(_lib.ClsError) as got:
            read_fastq_native(text)
        assert got.value.code == _lib.CLS_ERR_INVALID_ARGUMENT and got.value.message == e.message, (text[:200], e.message)
        return None
    headers, bases, offsets = read_fastq_native(text)
    assert headers == [h for h, _ in want], text[:200]
    seqs = [bases[int(offsets[i]):int(offsets[i + 1])].tobytes().decode() for i in range(len(headers))]
    assert seqs == [s for _, s in want], text[:200]
    return want


def test_mirror_and_host_reader_agree_on_edge_cases():
    for t in EDGE_CASES:
        _host_agree(t)
    from classeq2_b200.placement import read_fastq_text
    assert [h for h, _ in read_fastq_text(EDGE_CASES[8])] == ["x>y@z >", "", "@@"]
    assert read_fastq_text(EDGE_CASES[9])[0][1] == "ACGTACGT" + S.decode()
    assert [len(s) for _, s in read_fastq_text(EDGE_CASES[10])] == [0, 20, 35, 0]
    assert read_fastq_text(EDGE_CASES[13])[0][0] == "ué€"


def test_malformed_texts_name_the_first_bad_record():
    from classeq2_b200 import _lib
    from classeq2_b200.placement import FASTQ_REASONS, read_fastq_native, read_fastq_text
    for text, record, code in MALFORMED:
        for reader in (read_fastq_text, read_fastq_native):
            with pytest.raises(_lib.ClsError) as e:
                reader(text)
            assert e.value.code == _lib.CLS_ERR_INVALID_ARGUMENT
            assert e.value.message == f"malformed FASTQ record {record}: {FASTQ_REASONS[code]}", (text, e.value.message)


@pytest.mark.parametrize("chunk", [None, "1", "7", "64"])
def test_host_reader_over_chunk_boundaries(monkeypatch, chunk):
    """Small CLS_FASTA_CHUNK: the chunks start inside records, on every line of them, and every rule falls on a boundary."""
    if chunk:
        monkeypatch.setenv("CLS_FASTA_CHUNK", chunk)
    for t in EDGE_CASES:
        _host_agree(t)
    for text, record, _ in MALFORMED:
        _host_agree(text)
    rng = np.random.default_rng(5)
    for _ in range(20):
        parts = [EDGE_CASES[int(i)] for i in rng.integers(3, 14, 6) if EDGE_CASES[int(i)].endswith(b"\n")]
        _host_agree(b"".join(parts))
        bad = MALFORMED[int(rng.integers(0, len(MALFORMED)))][0]
        _host_agree(b"".join(parts) + bad)


@pytest.mark.parametrize("seed", range(6))
def test_random_texts_host(seed):
    rng = np.random.default_rng(300 + seed)
    n = int(rng.integers(1, 300))
    lens = rng.integers(0, 400, n)
    bases = np.frombuffer(bytes(rng.choice(list(b"ACGT"), int(lens.sum())).tolist()), np.uint8)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    text, want = random_fastq(rng, n, lens, bases, offsets, b"\r\n" if seed % 2 else b"\n")
    assert _host_agree(text) == want


@pytest.mark.parametrize("seed", range(6))
def test_fastq_equals_its_fasta_rendering_on_the_host_readers(seed):
    """Titles non-empty and free of '>', the last record with at least one base: the FASTQ reader and the FASTA reader
    on the rendering (">" + title, the sequence line) give the same records."""
    from classeq2_b200.placement import read_fasta_native, read_fasta_text, read_fastq_native, read_fastq_text
    rng = np.random.default_rng(40 + seed)
    n = int(rng.integers(1, 200))
    lens = rng.integers(0, 300, n)
    lens[-1] = max(int(lens[-1]), 1)
    bases = np.frombuffer(bytes(rng.choice(list(b"ACGTacgtNn-"), int(lens.sum())).tolist()), np.uint8)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    eol = b"\r\n" if seed % 3 == 1 else b"\n"
    fq, fa = [], []
    for i in range(n):
        title = f"q{i} some@text".encode()
        seq = bases[int(offsets[i]):int(offsets[i + 1])].tobytes()
        if not any(c in b"ACGTacgt" for c in seq) and i == n - 1:
            seq += b"A"
        fq.append(b"@" + title + eol + seq + eol + b"+" + eol + b"#" * len(seq) + eol)
        fa.append(b">" + title + eol + seq + eol)
    fq, fa = b"".join(fq), b"".join(fa)
    h1, b1, o1 = read_fastq_native(fq)
    h2, b2, o2 = read_fasta_native(fa)
    assert h1 == h2 and o1.tolist() == o2.tolist() and b1.tobytes() == b2.tobytes()
    assert read_fastq_text(fq) == read_fasta_text(fa.decode())


def test_query_format_is_checked(tmp_path):
    import classeq2_b200 as cq
    with pytest.raises(ValueError):
        cq.place_sequences(str(tmp_path / "q"), None, tmp_path / "r", query_format="sam")
    with pytest.raises(ValueError):
        cq.place_sequences_native(str(tmp_path / "q"), None, tmp_path / "r", query_format="fq")


def test_sequences_open_with_fastq_flag(tmp_path):
    """cls_sequences_open reads the query as FASTQ with CLS_QUERY_FASTQ, keeps titles as they are, refuses other bits and
    creates no file for a malformed query.  (Host only: the reader and the path handling.)"""
    import ctypes as C
    from classeq2_b200 import _lib
    q = tmp_path / "q.fq"
    q.write_bytes(rec(b"a>b", S) + rec(b"c", S[:10]))
    h, batch = C.c_void_p(), _lib.Batch()
    out = str(tmp_path / "o" / "res")
    assert _lib.lib.cls_sequences_open(str(q).encode(), out.encode(), _lib.QUERY_FASTQ | 1, 0, C.byref(h), C.byref(batch)) == 0
    try:
        assert batch.n_queries == 2 and [batch.offsets[i] for i in range(3)] == [0, len(S), len(S) + 10]
        assert os.path.exists(out + ".jsonl") and os.path.exists(out + ".error")
    finally:
        _lib.lib.cls_sequences_close(h)
    for bad_format in (2, 0x200, 0x101 | 0x400):
        assert _lib.lib.cls_sequences_open(str(q).encode(), out.encode(), bad_format, 1, C.byref(h), C.byref(batch)) == _lib.CLS_ERR_INVALID_ARGUMENT
    q.write_bytes(rec(b"a", S) + b"@b\nAC\n+\nI\n")
    out2 = str(tmp_path / "p" / "res")
    assert _lib.lib.cls_sequences_open(str(q).encode(), out2.encode(), _lib.QUERY_FASTQ, 0, C.byref(h), C.byref(batch)) == _lib.CLS_ERR_INVALID_ARGUMENT
    assert _lib.last_error() == "malformed FASTQ record 2: quality length differs from sequence length"
    assert not os.path.exists(out2 + ".yaml") and not os.path.exists(out2 + ".error")


# ---- the host side of cls_fastq_upload against a fake CUDA runtime, under ASan + UBSan ---------------------------------
def test_fastq_upload_host_side_under_asan(tmp_path):
    """The C ABI's host sources and fastq_ingest.cpp compiled with g++ against tests/native/fakecuda, the FASTQ kernels restated as serial walks
    (tests/native/fake_fastq_kernels.cpp): cls_fastq_upload's host side (record count, first bad record, UTF-8 titles,
    lengths, planning, packing) gives cls_fastq_read's records and, through the oracle, the same placements."""
    if shutil.which("g++") is None:
        pytest.skip("needs g++")
    native = os.path.join(HERE, "native")
    orc, exe = str(tmp_path / "oracle.o"), str(tmp_path / "fastq_fake")
    # the oracle is the checker: compiled once, without a sanitizer (its allocations would dominate the run under one)
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-c", os.path.join(ROOT, "oracle", "classeq_oracle.cpp"), "-o", orc],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    san = ["-fsanitize=address,undefined", "-fno-sanitize-recover=undefined"]
    srcs = CAPI_HOST_SOURCES + [os.path.join(CSRC, "fastq_ingest.cpp")] + \
           [os.path.join(native, f) for f in ("fastq_fake_main.cpp", "fake_kernels.cpp", "fake_fastq_kernels.cpp")]
    r = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-pthread", *san, "-I", os.path.join(native, "fakecuda"), *srcs, orc, "-o", exe],
                       capture_output=True, text=True)
    assert "error:" not in r.stderr and "undefined reference" not in r.stderr, r.stderr[-3000:]   # a real build error is a failure
    if r.returncode != 0:
        pytest.skip(f"cannot build with the sanitizers here: {r.stderr[-300:]}")
    p = subprocess.run([exe], capture_output=True, text=True, timeout=1200)
    assert "ERROR: AddressSanitizer" not in p.stderr and "runtime error" not in p.stderr, p.stderr[:4000]
    assert p.returncode == 0 and p.stdout.startswith("bad=0 "), (p.returncode, p.stdout, p.stderr[-2000:])


# ---- the device ingest (-m gpu) ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def setup():
    import classeq2_b200 as cq
    from classeq2_b200 import synth
    sm = synth.make_model(80, 400, 55)
    ix = cq.Index(sm.flat, device=0)
    yield cq, sm, ix
    ix.close()


PARAMS = [dict(), dict(min_match_coverage=0.3, remove_intersection=True), dict(max_iterations=3, min_match_coverage=0.9)]


def _device_check(cq, ix, text: bytes, params=PARAMS[:1]):
    """cls_fastq_upload == the host readers: records, header slices, lengths, placements; or the same refusal."""
    from classeq2_b200 import _lib
    want = _host_agree(text)
    if want is None:
        from classeq2_b200.placement import read_fastq_native
        with pytest.raises(_lib.ClsError) as host:
            read_fastq_native(text)
        with pytest.raises(_lib.ClsError) as dev:
            ix.upload_fastq(text)
        assert dev.value.code == _lib.CLS_ERR_INVALID_ARGUMENT and dev.value.message == host.value.message, text[:200]
        return 0
    rb, headers, lengths = ix.upload_fastq(text)
    try:
        assert headers == [h for h, _ in want], (text[:200], headers[:5], want[:5])
        assert lengths.tolist() == [len(s) for _, s in want]
        for kw in params:
            p = cq.PlaceParams(**kw)
            rb.place(p)
            got = rb.fetch()
            ref = ix.place_batch([s for _, s in want], p)
            for f, _ in cq.engine.RESULT_DTYPES:
                assert (getattr(got, f) == getattr(ref, f)).all(), (f, kw, text[:200])
    finally:
        rb.close()
    return len(want)


@pytest.mark.gpu
def test_device_edge_cases_and_malformed(setup):
    cq, sm, ix = setup
    assert sum(_device_check(cq, ix, t, PARAMS) for t in EDGE_CASES) > 15
    for text, _, _ in MALFORMED:
        _device_check(cq, ix, text)
    for i in range(len(MALFORMED)):   # a bad record after many good ones, and several bad ones: the first one is named
        text = b"".join(rec(f"g{j}".encode(), S) for j in range(300)) + MALFORMED[i][0] + MALFORMED[(i + 3) % len(MALFORMED)][0]
        _device_check(cq, ix, text)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_device_random_texts(setup, seed):
    cq, sm, ix = setup
    from classeq2_b200 import synth
    rng = np.random.default_rng(700 + seed)
    n = int(rng.integers(1, 500))
    lens = rng.integers(20, 700 if seed % 3 else 3500, n)
    bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, n, lens, 11 + seed)
    eol = b"\r\n" if seed % 4 == 1 else b"\n"
    text, want = random_fastq(rng, n, lens, bases, offsets, eol)
    if seed % 5 == 0:
        text = text[:-len(eol)]                 # no terminator after the last line
    assert _device_check(cq, ix, text, PARAMS) == n


@pytest.mark.gpu
def test_device_records_across_tile_edges(setup):
    """Padding before a block of short records moves every record and line boundary over every offset around the 4 KiB
    tile edges (and the 16-byte thread chunks inside them)."""
    cq, sm, ix = setup
    body = b"".join(rec(f"t{j}".encode(), S[: 3 + j % 11]) for j in range(40))
    for pad in range(0, 72):
        lead = rec(b"pad", b"A" * (4096 - 40 - pad)) if pad % 2 else rec(b"p" * (4000 - pad), b"AC")
        _device_check(cq, ix, lead + body)
        bad = lead + body[: len(body) // 2] + b"@x\nAC\n+\nI\n" + body
        _device_check(cq, ix, bad)


@pytest.mark.gpu
def test_colletotrichum_as_fastq_places_like_place_batch(setup, col_flat, col_queries):
    import classeq2_b200 as cq
    ix = cq.Index(col_flat, device=0)
    try:
        text = b"".join(rec(h.encode(), s.encode()) for h, s in col_queries)
        assert _device_check(cq, ix, text, PARAMS) == len(col_queries)
    finally:
        ix.close()


def _fastq_and_fasta(tmp_path, col_queries):
    fq, fa = tmp_path / "q.fastq", tmp_path / "q.fasta"
    rng = np.random.default_rng(3)
    fq.write_bytes(b"".join(rec(h.encode(), s.encode(), qual=bytes(rng.integers(33, 75, len(s), dtype=np.uint8).tolist()))
                            for h, s in col_queries))
    fa.write_bytes(b"".join(b">" + h.encode() + b"\n" + s.encode() + b"\n" for h, s in col_queries))
    return str(fq), str(fa)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["yaml", "jsonl"])
def test_place_sequences_fastq_writes_the_fasta_files(tmp_path, col_tree, col_flat, col_queries, fmt):
    """place_sequences on a FASTQ - host ingest with both readers, device ingest, and place_sequences_native - writes
    files byte-identical to each other and to place_sequences on the FASTA rendering."""
    import classeq2_b200 as cq
    tree = cq.Tree.from_obj(col_tree.to_obj())
    fq, fa = _fastq_and_fasta(tmp_path, col_queries)
    ix = cq.Index(col_flat, device=0)
    try:
        runs = {
            "fasta": lambda o: cq.place_sequences(fa, tree, o, output_format=fmt, index=ix),
            "host": lambda o: cq.place_sequences(fq, tree, o, output_format=fmt, index=ix, query_format="fastq"),
            "python": lambda o: cq.place_sequences(fq, tree, o, output_format=fmt, index=ix, query_format="fastq", reader="python"),
            "device": lambda o: cq.place_sequences(fq, tree, o, output_format=fmt, index=ix, query_format="fastq", ingest="device"),
            "native": lambda o: cq.place_sequences_native(fq, tree, o, output_format=fmt, index=ix, query_format="fastq"),
        }
        files = {}
        for name, run in runs.items():
            run(tmp_path / name / "r")
            files[name] = ((tmp_path / name / f"r.{fmt}").read_bytes(), (tmp_path / name / "r.error").read_bytes())
        assert len(files["fasta"][0]) > 10000
        for name in runs:
            assert files[name] == files["fasta"], name
        # a malformed FASTQ: refused by every path, nothing written
        bad = tmp_path / "bad.fastq"
        bad.write_bytes(open(fq, "rb").read() + b"@tail\nACGT\n+\nII\n")
        n_rec = len(col_queries) + 1
        for name, run in [("host", lambda o: cq.place_sequences(str(bad), tree, o, output_format=fmt, index=ix, query_format="fastq")),
                          ("python", lambda o: cq.place_sequences(str(bad), tree, o, output_format=fmt, index=ix, query_format="fastq", reader="python")),
                          ("device", lambda o: cq.place_sequences(str(bad), tree, o, output_format=fmt, index=ix, query_format="fastq", ingest="device")),
                          ("native", lambda o: cq.place_sequences_native(str(bad), tree, o, output_format=fmt, index=ix, query_format="fastq"))]:
            with pytest.raises(cq._lib.ClsError) as e:
                run(tmp_path / ("bad_" + name) / "r")
            assert e.value.message == f"malformed FASTQ record {n_rec}: quality length differs from sequence length", name
            assert not (tmp_path / ("bad_" + name) / f"r.{fmt}").exists() and not (tmp_path / ("bad_" + name) / "r.error").exists()
    finally:
        ix.close()


@pytest.mark.gpu
def test_multi_device_and_sharded_handles(setup):
    """cls_fastq_upload on a multi-device handle and on a sharded handle (two shards on device 0): the records and the
    results of a single-device index.  (Reads of up to 161 bases: what the sharded handle places.)"""
    cq, sm, ref = setup
    from classeq2_b200 import synth
    rng = np.random.default_rng(17)
    n = 3000
    lens = rng.integers(20, 162, n)
    bases, offsets, _ = synth.make_reads(sm.ref_codes, sm.ref_lens, n, lens, 23)
    text, _ = random_fastq(rng, n, lens, bases, offsets)
    others = [cq.Index(sm.flat, devices=[0, 0]), cq.Index(sm.flat, sharded_devices=[0, 0])]
    try:
        rb, h0, l0 = ref.upload_fastq(text)
        rb.place()
        want = rb.fetch()
        rb.close()
        for ix in others:
            rb, h, ln = ix.upload_fastq(text)
            try:
                assert h == h0 and ln.tolist() == l0.tolist()
                rb.place()
                got = rb.fetch()
                for f, _ in cq.engine.RESULT_DTYPES:
                    assert (getattr(got, f) == getattr(want, f)).all(), f
            finally:
                rb.close()
    finally:
        for ix in others:
            ix.close()
