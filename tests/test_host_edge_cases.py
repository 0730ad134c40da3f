"""Host-side edge cases around the device path (CPU tier): CR-only line ends in the record-table sizing, and PE chunk
cuts whose two files are not at the same read when the buffer fills up."""
import ctypes as C

import numpy as np
import pytest

import binfile_helpers as BF
from fastore_b200 import _native as N
from fastore_b200 import synth


def test_record_table_capacity_counts_lone_cr_line_ends():
    """SkipLine (FastqParser.cpp:46-68) takes a lone CR as a line end, so fsh_max_records has to count it: a CR-only
    FASTQ must parse completely instead of stopping with FSH_STOP_CAPACITY after two records."""
    cfg = synth.synth_config(500, 60, seed=31)
    t1, _, r1, _ = synth.generate(cfg, threads=1)
    cr = np.frombuffer(t1.tobytes().replace(b"\n", b"\r"), dtype=np.uint8).copy()
    lib = N.host_lib()
    assert lib.fsh_max_records(N.np_ptr(cr), cr.size) >= 500
    recs, st = synth.parse_chunk(cr, keep_headers=True, keep_comments=True, quality_method=0)
    assert len(recs) == 500 and st.stop_reason == 0
    assert np.array_equal(recs["seq_len"], r1["seq_len"]) and np.array_equal(recs["seq_off"], r1["seq_off"])
    # mixed: CRLF everywhere still counts one line end per line
    crlf = np.frombuffer(t1.tobytes().replace(b"\n", b"\r\n"), dtype=np.uint8).copy()
    assert lib.fsh_max_records(N.np_ptr(crlf), crlf.size) == 500 + 2
    recs, st = synth.parse_chunk(crlf, keep_headers=True, keep_comments=True, quality_method=0)
    assert len(recs) == 500 and st.stop_reason == 0


@pytest.mark.skipif(not BF.have_ref_tools(), reason="oracle/_ref tools not built (no /root/reference here)")
def test_pe_chunks_stay_paired_when_the_cut_points_differ(tmp_path):
    """Mate files whose records differ in size (longer titles in file 2) reach the cut window at different reads.  The
    reference's re-synchronisation (FastqStream.cpp:166-189) advances its read-id counter once per skipped *line*, so it
    skips 4x too far in one file and then 12x in the other and pairs the wrong mates for the rest of the chunk (its
    ASSERT(rid_1 == rid_2) is compiled out).  Our reader deliberately does the arithmetic per *record*: chunks always hold
    the same reads in both files.  Checked by decoding our bin files with the reference's own decoder: every pair comes
    back with its own mate."""
    files = BF.write_fastq(tmp_path, "in", 16000, 100, True, 240)
    recs2 = BF.fastq_records(files[1])
    with open(files[1], "wb") as f:                      # mate 2 gets a comment: every record of file 2 is 24 bytes longer
        for t, s, q in recs2:
            f.write(t + b" mate=2 lane=7 tile=1234\n" + s + b"\n+\n" + q + b"\n")
    flags = dict(paired=True, b=2)
    sizes = BF.host_chain(files, tmp_path / "ours", flags, BF.oracle_producer)
    assert len(sizes) >= 3
    outs = [tmp_path / "dec_1.fastq", tmp_path / "dec_2.fastq"]
    BF.decode_with_reference(tmp_path / "ours", outs, True)
    want = sorted((a[1], a[2], b[1], b[2]) for a, b in zip(BF.fastq_records(files[0]), recs2))
    got = sorted((a[1], a[2], b[1], b[2]) for a, b in zip(BF.fastq_records(outs[0]), BF.fastq_records(outs[1])))
    assert got == want


def _parse(text, validate, **kw):
    lib = N.host_lib()
    cap = int(lib.fsh_max_records(N.np_ptr(text), text.size))
    recs = np.zeros(cap, dtype=N.RECORD_DTYPE)
    st = N.FshParseStats()
    rc = lib.fsh_parse_chunk_ex(N.np_ptr(text), text.size, int(kw.get("keep_headers", True)), int(kw.get("keep_comments", True)), 33, 0, validate,
                                N.np_ptr(recs), cap, C.byref(st))
    return rc, recs[: st.n_records].copy(), st


def test_memchr_line_scanner_follows_skipline():
    """fsh_parse_chunk_ex finds line ends with memchr; it has to give what SkipLine (FastqParser.cpp:46-68) gives byte by byte:
    LF, CRLF and lone-CR line ends, a CR in the middle of a line, a chunk without a final line end, a record cut short."""
    cfg = synth.synth_config(300, 80, seed=41, header_comments=True)
    t1, _, r1, _ = synth.generate(cfg, threads=1)
    raw = t1.tobytes()
    lines = raw.split(b"\n")
    mixed = b""
    for i, ln in enumerate(lines[:-1]):                       # every record with a different kind of line end
        mixed += ln + (b"\n", b"\r\n", b"\r")[(i // 4) % 3]
    variants = {"lf": raw, "crlf": raw.replace(b"\n", b"\r\n"), "cr": raw.replace(b"\n", b"\r"), "mixed": mixed, "no_final_eol": raw[:-1],
                "cut_short": raw[: len(raw) // 2], "cr_inside_title": raw.replace(b" len=", b"\rlen=", 3)}
    for name, txt in variants.items():
        text = np.frombuffer(txt, dtype=np.uint8).copy()
        rc0, a, st0 = _parse(text, 1)
        # the byte-wise reference of this test: SkipLine restated in Python
        pos, want = 0, []
        def skip():
            nonlocal pos
            n0 = pos
            while pos < len(txt) and txt[pos] not in (10, 13):
                pos += 1
            ln = pos - n0
            if pos < len(txt):
                pos += 2 if (txt[pos] == 13 and pos + 1 < len(txt) and txt[pos + 1] == 10) else 1
            return n0, ln
        while pos < len(txt):
            h, hl = skip()
            if hl == 0 or txt[h] != ord("@"):
                break
            s_, sl = skip()
            _, pl = skip()
            if pl == 0:
                break
            q, ql = skip()
            if ql != sl:
                break
            want.append((h, s_, q, sl, hl))
        got = [(int(r["head_off"]), int(r["seq_off"]), int(r["qua_off"]), int(r["seq_len"]), int(r["head_len"])) for r in a]
        assert got == want, name
        rc1, b, st1 = _parse(text, 0)
        assert np.array_equal(a, b) and st0.consumed_bytes == st1.consumed_bytes and st0.stop_reason == st1.stop_reason, name
    # the byte-level contract check is what validate_bytes switches
    bad = np.frombuffer(raw.replace(b"A", b"a", 1), dtype=np.uint8).copy()
    assert _parse(bad, 1)[0] == N.FSB_ERR_INPUT and _parse(bad, 0)[0] == N.FSB_OK


def test_title_statistics_merged_per_chunk_equal_the_reference(tmp_path):
    """The CLI's parser threads gather the header-field statistics per chunk (fsh_titles) and the writer merges them in chunk
    order; the footer must be the one the reference writes from its record-by-record statistics."""
    files = BF.write_fastq(tmp_path, "in", 16000, 100, True, 250, header_comments=True)
    flags = dict(paired=True, b=2)
    BF.host_chain(files, tmp_path / "ours", flags, BF.oracle_producer, merge_titles=True)
    BF.assert_reference_files(tmp_path / "ours", files, flags, "title_statistics", tmp_path)


def test_large_requests_read_as_slices_reassemble_the_file(tmp_path):
    """The chunk reader serves requests of 32 MB and more on regular files as four positioned reads side by side
    (bin_io.cpp: MultiFile::read_current); smaller ones go through fread.  Either way the chunks, put back together with the
    line ends the cutter drops between them, are the file -- also across the seam between two input files."""
    lib = N.host_lib()
    lib.fsh_reader_open.restype = C.c_void_p
    lib.fsh_reader_open.argtypes = [C.POINTER(C.c_char_p), C.c_uint32, C.POINTER(C.c_char_p), C.c_uint32, C.c_uint64]
    lib.fsh_reader_next.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_uint64)]
    lib.fsh_reader_close.argtypes = [C.c_void_p]
    cfg = synth.synth_config(330000, 100, seed=77)                    # 71 MB
    text, _, _, _ = synth.generate(cfg, threads=4)
    raw = text.tobytes()
    cut = raw.find(b"\n@", len(raw) // 3) + 1                         # two input files, split at a record boundary
    paths = [tmp_path / "a.fastq", tmp_path / "b.fastq"]
    paths[0].write_bytes(raw[:cut]); paths[1].write_bytes(raw[cut:])
    for block in (40 << 20, 12 << 20):                                # sliced reads / plain reads
        files = (C.c_char_p * 2)(str(paths[0]).encode(), str(paths[1]).encode())
        r = lib.fsh_reader_open(files, 2, None, 0, block)
        assert r
        buf = np.empty(block + 64, dtype=np.uint8)
        size = C.c_uint64()
        chunks = []
        while lib.fsh_reader_next(r, buf.ctypes.data, C.byref(size), None, None) > 0 and size.value:
            chunks.append(buf[: size.value].tobytes())
        lib.fsh_reader_close(r)
        assert len(chunks) >= 2
        assert b"\n".join(chunks) + b"\n" == raw, f"block {block >> 20} MB"
