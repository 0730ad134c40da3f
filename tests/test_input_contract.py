"""The device's input check (fsb_stage, DESIGN §2) against a plain statement of the input contract, byte by byte and entry
by entry.  Two kernels decide whether a batch is inside the contract (stage.cuh):

  * stage_stats_kernel checks the record table: read length 1..255, every view inside its chunk's text, equal PE mate lengths;
  * validate_text_kernel (FSB_OPT_VALIDATE, on by default) checks the bytes behind the table: sequence symbols A C G T N,
    quality bytes in [offset, offset + 64) -- or >= offset in the 1-bit mode --, 7-bit characters in the kept title after '@'.

A byte the check wrongly accepts is coded by K1 as some symbol, silently; so every test here counts rejections as well as
acceptances.  The CPU tier runs the kernel's per-mate check (stage_core.cuh, through tests/emul) at every byte value, span
position, alignment and quality offset; the GPU tier plants bad bytes and bad table entries in whole batches and compares
the library's count, lowest record and chunk with the Python count."""
import ctypes as C
import re

import numpy as np
import pytest

from fastore_b200 import _native as N
from test_kernel_core_on_cpu import emul  # noqa: F401  (fixture: the kernels' per-thread cores built for the host)

SEQ, QUA, TITLE = 0, 1, 2
KIND_NAME = {SEQ: "sequence", QUA: "quality", TITLE: "title"}


# ---- the contract, one byte at a time (the rules of csrc/host/fastq_parser.cpp) --------------------------------------------
def valid_bytes(kind, offset=33, need_range=True):
    """Boolean table over the 256 byte values: which are inside the contract for a byte of this kind."""
    v = np.arange(256)
    if kind == SEQ:
        return np.isin(v, np.frombuffer(b"ACGTN", dtype=np.uint8))
    if kind == TITLE:
        return v < 128
    q = v - offset
    return ((q >= 0) & (q < 64)) if need_range else (q >= 0)


QUA8 = np.array([0] * 2 + [1] * 8 + [2] * 10 + [3] * 5 + [4] * 5 + [5] * 5 + [6] * 5 + [7] * 24, dtype=np.uint32)   # quaToIdx_8bin


def coded(q_bits, words, offset, threshold):
    """What the port codes four quality bytes as (oracle/fastore_oracle.c, store_next_record), packed the way quality4<Q>
    returns them: the byte at the top of the word first."""
    out = np.zeros(words.size, dtype=np.uint32)
    for j in range(4):
        c = ((words >> np.uint32(24 - 8 * j)) & np.uint32(0xFF)).astype(np.int64) - offset
        if q_bits == 6:
            sym, width = c & 63, 6
        elif q_bits == 3:
            sym, width = QUA8[c & 63], 3
        else:
            sym, width = (c >= threshold), 1
        out = (out << np.uint32(width)) | sym.astype(np.uint32)
    return out


# ---- the emulated check --------------------------------------------------------------------------------------------------
def _bind(lib):
    lib.emul_check_spans.restype = None
    lib.emul_check_spans.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_void_p]
    lib.emul_quality4.restype = None
    lib.emul_quality4.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
    return lib


def emul_check(lib, buf, spans, offset=33, need_range=True):
    """validate_text_kernel's per-mate check of every (offset, length, kind) span of buf: True where it passes."""
    spans = np.ascontiguousarray(spans, dtype=np.int32)
    ok = np.zeros(len(spans), dtype=np.uint8)
    _bind(lib).emul_check_spans(N.np_ptr(buf), buf.size, N.np_ptr(spans), len(spans), offset, int(need_range), N.np_ptr(ok))
    return ok.astype(bool)


def byte_pools(table):
    """(valid, invalid) byte values; where every value is valid (the 1-bit mode at offset 0) the invalid pool is the valid one."""
    good, bad = np.nonzero(table)[0].astype(np.uint8), np.nonzero(~table)[0].astype(np.uint8)
    return good, (bad if bad.size else good)


def planted(kind, table, cases, rng):
    """One span per case (align, length, pos, value): its own 16-byte aligned region, the span at `align` inside it, filled
    with random valid bytes except `value` at `pos` (pos < 0: nothing planted).  Every byte of the region outside the span --
    the rest of its first and last piece and one piece more -- is invalid, so a check that looks past the span rejects.
    Returns (buffer, spans, contract verdict per span, the case of each span).  Cases of one (align, length) are laid out together as a 2-D array."""
    good, bad = byte_pools(table)
    cases = np.asarray(cases, dtype=np.int64).reshape(-1, 4)
    parts, spans, want, keys, base = [], [], [], [], 0
    for (a, L) in sorted(set(map(tuple, cases[:, :2].tolist()))):
        sel = cases[(cases[:, 0] == a) & (cases[:, 1] == L)]
        R = ((a + L + 15) // 16) * 16 + 16
        blk = bad[rng.integers(0, bad.size, (len(sel), R))]
        blk[:, a: a + L] = good[rng.integers(0, good.size, (len(sel), L))]
        hit = sel[:, 2] >= 0
        rows = np.nonzero(hit)[0]
        blk[rows, a + sel[hit, 2]] = sel[hit, 3]
        parts.append(blk.ravel())
        spans.append(np.stack([base + R * np.arange(len(sel)) + a, np.full(len(sel), L), np.full(len(sel), kind)], axis=1))
        want.append(np.where(hit, table[sel[:, 3] & 0xFF], True))
        keys.append(sel)
        base += R * len(sel)
    return np.concatenate(parts), np.concatenate(spans), np.concatenate(want), np.concatenate(keys)


def assert_check(lib, kind, table, cases, rng, what, offset=33, need_range=True):
    buf, spans, want, key = planted(kind, table, cases, rng)
    got = emul_check(lib, buf, spans, offset, need_range)
    bad = np.nonzero(got != want)[0]
    if bad.size:
        a, L, pos, value = key[bad[0]]
        raise AssertionError(f"{what}: {KIND_NAME[kind]} span of {L} bytes at alignment {a}, byte {value:#04x} at {pos}: check says "
                             f"{'ok' if got[bad[0]] else 'bad'}, the contract {'ok' if want[bad[0]] else 'bad'} ({bad.size} of {len(want)} spans differ)")


LENGTHS = tuple(range(1, 18)) + (31, 32, 33, 239, 240, 241, 254, 255)
TITLE_LENGTHS = (0,) + tuple(range(1, 18)) + (31, 32, 33, 239, 240, 241, 254)          # after the '@' of a title of at most 255 bytes
PIECE_BYTES = (0, 3, 4, 15)                                                               # and byte 16 = byte 0 of the next piece
PIECES = (0, 1, 15, 16)                                                                   # piece 16: the 17th, spans over 240 bytes


def positions(a, L):
    """Span positions of the first and last byte, and of bytes 0, 3, 4, 15 of pieces 0, 1, 15 and 16 (counted from the
    aligned start)."""
    p = {0, L - 1} | {16 * pc + r - a for pc in PIECES for r in PIECE_BYTES}
    return sorted(x for x in p if 0 <= x < L)


def every_value_cases(lengths):
    cases = []
    for L in lengths:
        for a in range(16):
            if L == 0:
                cases.append((a, 0, -1, 0))
            for pos in positions(a, L):
                cases.extend((a, L, pos, v) for v in range(256))
    return cases


MODES = [(SEQ, 33, True), (QUA, 33, True), (QUA, 33, False), (TITLE, 33, True)]
MODE_IDS = ["sequence", "quality_range", "quality_1bit", "title"]


# ---- CPU tier ------------------------------------------------------------------------------------------------------------------
def test_planted_spans_hold_what_they_say():
    """The builder: spans valid but for the planted byte, every byte around them invalid."""
    rng = np.random.default_rng(0)
    table = valid_bytes(SEQ)
    cases = [(a, L, pos, v) for a, L, pos, v in ((0, 1, 0, 65), (15, 255, 254, 0), (3, 33, 16, 0x43), (7, 17, -1, 0))]
    buf, spans, want, key = planted(SEQ, table, cases, rng)
    for (o, L, _), w, (a, _, pos, v) in zip(spans, want, key):
        assert o % 16 == a
        span = buf[o: o + L]
        inside = np.delete(span, pos) if pos >= 0 else span
        assert table[inside].all() and w == (pos < 0 or table[v])
        assert pos < 0 or span[pos] == v
        assert not table[buf[o - a: o]].any() and not table[buf[o + L: o - a + ((a + L + 15) // 16) * 16 + 16]].any()


@pytest.mark.parametrize("kind,offset,need_range", MODES, ids=MODE_IDS)
def test_every_byte_value_at_every_position(emul, kind, offset, need_range):
    """Each of the 256 values at the first and last byte of the span, at bytes 0, 3, 4, 15 of the first, second, 16th and
    17th aligned piece, at every one of the 16 start alignments and every span length around the piece edges (titles: 0..254
    bytes after the '@').  The rest of the span holds random valid bytes, everything beside it invalid bytes."""
    rng = np.random.default_rng(100 + kind + 2 * need_range)
    cases = every_value_cases(TITLE_LENGTHS if kind == TITLE else LENGTHS)
    assert_check(emul, kind, valid_bytes(kind, offset, need_range), cases, rng, "every value", offset, need_range)


@pytest.mark.parametrize("kind,offset,need_range", MODES + [(QUA, 0, True), (QUA, 127, True), (QUA, 0, False), (QUA, 127, False)],
                         ids=MODE_IDS + ["quality_range_off0", "quality_range_off127", "quality_1bit_off0", "quality_1bit_off127"])
def test_all_pairs_of_adjacent_bytes(emul, kind, offset, need_range):
    """All 65 536 value pairs in two neighbouring bytes -- inside one word (bytes 1, 2) and across a word boundary (bytes 3,
    4) -- of a whole piece and of a span that covers its pieces only in part: a borrow, carry or shift that leaks from one
    byte into the next changes a verdict here."""
    table = valid_bytes(kind, offset, need_range)
    rng = np.random.default_rng(7)
    v1, v2 = np.divmod(np.arange(65536), 256)
    for a, L, p in ((0, 16, 1), (0, 16, 3), (1, 14, 0), (1, 14, 2), (0, 32, 15)):
        good, bad = byte_pools(table)
        R = ((a + L + 15) // 16) * 16 + 16
        blk = bad[rng.integers(0, bad.size, (65536, R))]
        blk[:, a: a + L] = good[rng.integers(0, good.size, (65536, L))]
        blk[:, a + p], blk[:, a + p + 1] = v1, v2
        spans = np.stack([R * np.arange(65536) + a, np.full(65536, L), np.full(65536, kind)], axis=1)
        got = emul_check(emul, blk.ravel(), spans, offset, need_range)
        want = table[v1] & table[v2]
        bad_at = np.nonzero(got != want)[0]
        assert bad_at.size == 0, (f"{KIND_NAME[kind]} at offset {offset}, span {L} at alignment {a}, bytes {p}, {p + 1} = "
                                  f"{v1[bad_at[0]]:#04x} {v2[bad_at[0]]:#04x}: check {'ok' if got[bad_at[0]] else 'bad'} ({bad_at.size} pairs differ)")


@pytest.mark.parametrize("need_range", [True, False], ids=["range", "1bit"])
def test_quality_check_at_every_offset(emul, need_range):
    """The quality predicate at every offset 0..127 the contract allows, for all 256 byte values, at every position of a word
    and every start alignment."""
    rng = np.random.default_rng(11)
    for offset in range(128):
        table = valid_bytes(QUA, offset, need_range)
        cases = [(v % 16, 20, (v * 7) % 20, v) for v in range(256)] + [(v % 16, 5, v % 5, v) for v in range(256)]
        assert_check(emul, QUA, table, cases, rng, f"offset {offset}", offset, need_range)


def quality_words(values, rng, n_random=4000):
    """Words of in-range quality bytes: every value at every byte of a word, and random words."""
    n = values.size
    idx = np.stack([(np.arange(n) + 17 * j) % n for j in range(4)], axis=1)
    idx = np.concatenate([idx, rng.integers(0, n, (n_random, 4))])
    b = values[idx].astype(np.uint32)
    return b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16) | (b[:, 3] << 24)


def emul_quality4(lib, q_bits, words, offset, threshold):
    out = np.zeros(words.size, dtype=np.uint32)
    _bind(lib).emul_quality4(q_bits, N.np_ptr(words), words.size, offset, threshold, N.np_ptr(out))
    return out


def test_quality_coding_at_every_offset(emul):
    """quality4<6>, <3> and <1> -- K1's coding of four quality bytes -- at every offset 0..127 against (q - offset) coded the
    way the port codes it, over every in-range byte; the 1-bit mode at thresholds 0, 1, 20, 62 and 63."""
    rng = np.random.default_rng(12)
    for offset in range(128):
        for q_bits, thresholds in ((6, (0,)), (3, (0,)), (1, (0, 1, 20, 62, 63))):
            values = np.arange(offset, offset + 64 if q_bits != 1 else 256)
            words = quality_words(values, rng, 1000)
            for thr in thresholds:
                got, want = emul_quality4(emul, q_bits, words, offset, thr), coded(q_bits, words, offset, thr)
                bad = np.nonzero(got != want)[0]
                assert bad.size == 0, f"quality4<{q_bits}> at offset {offset}, threshold {thr}: word {words[bad[0]]:#010x} -> {got[bad[0]]:#x}, port {want[bad[0]]:#x}"


def test_offsets_above_127_break_the_check_and_the_coding(emul):
    """Why fsb_create refuses quality_offset > 127.  The check keeps only seven bits of the offset: at offset 200 it rejects
    every valid byte of the 6-bit modes and takes bytes below the offset in the 1-bit mode.  The 6- and 3-bit coding forms
    (q | 128) - offset per byte, which borrows from the byte above once q | 128 is below the offset (offsets above 128); in the
    last word of a read such bytes are the ones behind it (the line end), and the read's last symbols are miscoded."""
    rng = np.random.default_rng(13)
    cases = [(v % 16, 20, (v * 7) % 20, v) for v in range(256)]
    for offset in (128, 200, 255):
        for need_range in (True, False):
            buf, spans, want, key = planted(QUA, valid_bytes(QUA, offset, need_range), cases, rng)
            assert (emul_check(emul, buf, spans, offset, need_range) != want).any(), f"offset {offset}"
    # the read's last two quality bytes on top of the word, then '\n' and the next line's first byte ('@')
    for offset in (160, 200):
        q = np.array([offset + 5, offset + 40], dtype=np.uint32)
        word = np.array([(q[0] << 24) | (q[1] << 16) | (10 << 8) | 64], dtype=np.uint32)
        for q_bits in (6, 3):
            assert (emul_quality4(emul, q_bits, word, offset, 0) >> np.uint32(2 * q_bits)) != (coded(q_bits, word, offset, 0) >> np.uint32(2 * q_bits)), \
                f"quality4<{q_bits}> at offset {offset}"
        # at offsets the contract allows the same word codes right
        ok = np.array([((offset - 100 + 5) << 24) | ((offset - 100 + 40) << 16) | (10 << 8) | 64], dtype=np.uint32)
        for q_bits in (6, 3):
            assert emul_quality4(emul, q_bits, ok, offset - 100, 0) == coded(q_bits, ok, offset - 100, 0)


# ---- GPU tier ------------------------------------------------------------------------------------------------------------------
# Batches are built directly as FASTQ text with a uniform record layout, so that every byte of every record has a known
# place.  The library reports the lowest rejected record, its chunk and the number of rejected mates (bytes) or records (table):
# all three are compared with the Python count.
FSB_OPT_VALIDATE = 3
PRINTABLE = np.arange(32, 127, dtype=np.uint8)


def fastq_block(n, L, H, rng, offset=33, need_range=True):
    """n records of L bases under H-byte titles ('@' and printable characters), LF line ends, qualities valid at the offset.
    Returns (text, record table)."""
    S = H + 1 + L + 3 + L + 1
    t = np.empty((n, S), dtype=np.uint8)
    t[:, 0] = ord("@")
    t[:, 1:H] = PRINTABLE[rng.integers(0, PRINTABLE.size, (n, H - 1))]
    t[:, H] = 10
    t[:, H + 1: H + 1 + L] = np.frombuffer(b"ACGTN", dtype=np.uint8)[rng.integers(0, 5, (n, L))]
    t[:, H + 1 + L: H + L + 4] = np.frombuffer(b"\n+\n", dtype=np.uint8)
    t[:, H + L + 4: H + 2 * L + 4] = rng.integers(offset, offset + 64 if need_range else 256, (n, L), dtype=np.int64).clip(0, 255)
    t[:, -1] = 10
    recs = np.zeros(n, dtype=N.RECORD_DTYPE)
    base = S * np.arange(n)
    recs["head_off"], recs["seq_off"], recs["qua_off"] = base, base + H + 1, base + H + L + 4
    recs["seq_len"], recs["head_len"] = L, H
    return t.ravel(), recs


def span_ok(text, off, length, table, block=8192):
    """True per span whose bytes are all valid (table over the 256 values), spans of any length."""
    out = np.ones(off.size, dtype=bool)
    cols = np.arange(max(1, int(length.max(initial=0))))
    for s in range(0, off.size, block):
        o, m = off[s: s + block].astype(np.int64), length[s: s + block].astype(np.int64)
        inside = cols[None, :] < m[:, None]
        idx = np.where(inside, o[:, None] + cols[None, :], 0)
        out[s: s + block] = (table[text[idx]] | ~inside).all(axis=1)
    return out


def contract(params, chunks_data):
    """The contract over a batch, chunk by chunk: per record, whether its table entry violates stage_stats_kernel's rule, and
    how many of its mates hold a byte outside the contract (FSB_OPT_VALIDATE).  chunks_data: [(text1, recs1, text2, recs2)]."""
    pe = bool(params.paired_end)
    need_range = params.quality_method != N.FSB_QUA_BINARY
    out = []
    for t1, r1, t2, r2 in chunks_data:
        L = r1["seq_len"].astype(np.int64)
        ts0 = t1.size
        tbad = ~((L >= 1) & (L <= 255) & (r1["seq_off"] + L <= ts0) & (r1["qua_off"] + L <= ts0) & (r1["head_off"].astype(np.int64) + r1["head_len"] <= ts0))
        if pe:
            L2 = r2["seq_len"].astype(np.int64)
            tbad |= ~((L2 == L) & (r2["seq_off"] + L2 <= t2.size) & (r2["qua_off"] + L2 <= t2.size))
        nbad = np.zeros(len(r1), dtype=np.int64)
        for m, (t, r) in enumerate(((t1, r1), (t2, r2)) if pe else ((t1, r1),)):
            ok = ~tbad
            i = np.nonzero(ok)[0]
            good = span_ok(t, r["seq_off"][i], r["seq_len"][i], valid_bytes(SEQ))
            good &= span_ok(t, r["qua_off"][i], r["seq_len"][i], valid_bytes(QUA, params.quality_offset, need_range))
            if m == 0 and params.reads_have_headers:
                good &= span_ok(t, r["head_off"][i] + 1, np.maximum(r["head_len"][i].astype(np.int64) - 1, 0), valid_bytes(TITLE))
            nbad[i] += ~good
        out.append((tbad, nbad))
    return out


def expected_message(verdicts, chunk0=0):
    """(record, chunk, count, 'record' | 'mate') the library must report, or None."""
    for what, col in (("record", 0), ("mate", 1)):
        total = sum(int((v[col] > 0).sum() if col == 0 else v[col].sum()) for v in verdicts)
        if total:
            for ci, v in enumerate(verdicts):
                bad = np.nonzero(v[col] > 0)[0]
                if bad.size:
                    return int(bad[0]), chunk0 + ci, total, what
    return None


MESSAGE = re.compile(r"record (\d+) of chunk (\d+) .*; (\d+) such (record|mate)\(s\)")


def device_message(call):
    from fastore_b200.binner import FastoreError
    try:
        call()
    except FastoreError as e:
        m = MESSAGE.search(str(e))
        assert m, str(e)
        return int(m[1]), int(m[2]), int(m[3]), m[4]
    return None


def make_chunks(chunks_data):
    return [N.make_chunk(t1, r1, t2, r2) for t1, r1, t2, r2 in chunks_data]


def bisect_disagreement(g, params, base, plants, apply):
    """A batch whose verdict disagrees with the contract: halve its planted bytes until one plant alone disagrees, and name it."""
    while len(plants) > 1:
        for half in (plants[: len(plants) // 2], plants[len(plants) // 2:]):
            data = apply(base, half)
            if device_message(lambda: g.stage(make_chunks(data))) != expected_message(contract(params, data)):
                plants = half
                break
        else:
            return "the halves agree on their own (the disagreement needs bytes of both)"
    data = apply(base, plants)
    return f"plant {plants[0]}: device {device_message(lambda: g.stage(make_chunks(data)))}, contract {expected_message(contract(params, data))}"


def assert_verdict(g, params, base, plants, apply, what, chunk0=0):
    data = apply(base, plants)
    want = expected_message(contract(params, data), chunk0)
    got = device_message(lambda: g.stage(make_chunks(data)))
    if got != want:
        raise AssertionError(f"{what}: device {got}, contract {want}; " + (bisect_disagreement(g, params, base, plants, apply) if plants else ""))
    return want


def plant_bytes(base, plants):
    """plants: (chunk, mate, record, field, pos, value) -> copies of the texts with the bytes written."""
    out = []
    for ci, (t1, r1, t2, r2) in enumerate(base):
        texts = [t1.copy(), t2.copy() if t2 is not None else None]
        for c, m, i, field, pos, value in plants:
            if c == ci:
                texts[m][int((r1 if m == 0 else r2)[field][i]) + pos] = value
        out.append((texts[0], r1, texts[1], r2))
    return out


def clean_batch_equals_the_port(g, params):
    """After a rejection the context still bins a clean batch like the port."""
    import oracle_helpers as O
    from test_gpu_parity import gpu_block_dict
    rng = np.random.default_rng(1)
    t1, r1 = fastq_block(300, 90, 30, rng, params.quality_offset, params.quality_method != N.FSB_QUA_BINARY)
    t2, r2 = fastq_block(300, 90, 30, rng, params.quality_offset, params.quality_method != N.FSB_QUA_BINARY) if params.paired_end else (None, None)
    ch = N.make_chunk(t1, r1, t2, r2)
    O.assert_blocks_equal(gpu_block_dict(g.bin_chunks([ch])[0]), O.bin_chunk("orc", params, ch), "clean batch after a rejection")


BYTE_MODES = [(N.FSB_QUA_NONE, off) for off in (0, 33, 64, 100, 127)] + [(N.FSB_QUA_BINARY, off) for off in (33, 64, 127)]


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["se", "pe"])
@pytest.mark.parametrize("method,offset", BYTE_MODES, ids=[f"m{m}_off{o}" for m, o in BYTE_MODES])
def test_device_check_every_byte_value(method, offset, paired):
    """All 256 values at the first, 16th, 17th, 241st and last byte of 255-base sequences and qualities and of 255-byte titles,
    one planted byte per record, in a batch of 50 000 records: the check's grid covers 37 888 mates a round, so the records
    past 40 000 are checked in a later round.  Mate 2's title is not kept, so bytes planted there must be accepted."""
    from fastore_b200.binner import GpuBinner
    params = N.make_params(signature_len=8, skip_zone_len=0, paired_end=paired, quality_method=method, quality_offset=offset)
    need_range = method != N.FSB_QUA_BINARY
    rng = np.random.default_rng(offset + 1000 * paired + 7 * method)
    n, L, H = 50000, 255, 255
    t1, r1 = fastq_block(n, L, H, rng, offset, need_range)
    t2, r2 = fastq_block(n, L, H, rng, offset, need_range) if paired else (None, None)
    base = [(t1, r1, t2, r2)]
    plants = [(0, m, None, field, pos, v) for m in ((0, 1) if paired else (0,)) for field in ("seq_off", "qua_off", "head_off")
              for pos in ((0, 15, 16, 240, 254) if field != "head_off" else (1, 15, 16, 240, 254)) for v in range(256)]
    recs = rng.permutation(n)[: len(plants)]
    plants = [(c, m, int(i), f, p, v) for (c, m, _, f, p, v), i in zip(plants, recs)]
    tables = {"seq_off": valid_bytes(SEQ), "qua_off": valid_bytes(QUA, offset, need_range), "head_off": valid_bytes(TITLE)}
    bad = [p for p in plants if not tables[p[3]][p[5]] and not (p[1] == 1 and p[3] == "head_off")]
    good = [p for p in plants if p not in set(bad)]
    with GpuBinner(params, per_read=True) as g:
        assert assert_verdict(g, params, base, good, plant_bytes, "valid bytes") is None
        want = assert_verdict(g, params, base, bad, plant_bytes, "invalid bytes")
        assert want[2] == len(bad) and want[3] == "mate"
        late = [p for p in bad if p[2] >= 40000]
        assert len(late) > 100 and assert_verdict(g, params, base, late, plant_bytes, "invalid bytes past the first round")[0] >= 40000
        clean_batch_equals_the_port(g, params)


def many_chunks(rng, n_chunks=256, paired=False):
    return [(*fastq_block(int(n), 100, 24 + ci % 9, rng), *(fastq_block(int(n), 100, 24, rng) if paired else (None, None)))
            for ci, n in enumerate(rng.integers(20, 60, n_chunks))]


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["se", "pe"])
def test_device_check_in_every_chunk_of_a_full_batch(paired):
    """A batch of 256 chunks at k = 8, the most a batch takes: bad bytes in the first, a middle and the last chunk, one chunk at
    a time and all three together, with record tables and handed over as text alone (parsed on the device)."""
    from fastore_b200.binner import GpuBinner
    params = N.make_params(signature_len=8, skip_zone_len=0, paired_end=paired)
    rng = np.random.default_rng(256 + paired)
    base = many_chunks(rng, 256, paired)
    sets = [[(ci, m, 7, "seq_off", 50, ord("a")), (ci, 0, 3, "qua_off", 99, 32)] for ci, m in ((0, 0), (128, 1 if paired else 0), (255, 0))]
    with GpuBinner(params) as g:
        assert assert_verdict(g, params, base, [], plant_bytes, "clean") is None
        for plants in sets + [sum(sets, [])]:
            want = assert_verdict(g, params, base, plants, plant_bytes, f"chunks {sorted({p[0] for p in plants})}")
            assert want[:2] == (3, plants[0][0]) and want[2] == len(plants)
            data = plant_bytes(base, plants)
            text_only = [N.make_chunk(t1, None, t2, None) for t1, _, t2, _ in data]
            assert device_message(lambda: g.stage(text_only)) == want, "text alone"
        clean_batch_equals_the_port(g, params)


def edit(base, edits):
    """edits: (chunk, mate, record, field, value) -> copies of the tables with the entries written; field "len" is the read
    length of both mates (only the length is wrong), "seq_len" that of one mate."""
    out = []
    for ci, (t1, r1, t2, r2) in enumerate(base):
        r = [r1.copy(), r2.copy() if r2 is not None else None]
        for c, m, i, field, value in edits:
            if c == ci:
                for mm in ((0, 1) if field == "len" else (m,)):
                    if r[mm] is not None:
                        r[mm]["seq_len" if field == "len" else field][i] = value
        out.append((t1, r[0], t2, r[1]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["se", "pe"])
def test_device_table_check_at_its_edges(paired):
    """stage_stats_kernel's rule against its Python statement: views ending exactly at the end of the text and one byte
    past it, read lengths 0, 1, 255, 256 and 65 535, mate lengths 1 apart, mate-2 views at the end of a mate-2 text longer or
    shorter than mate 1's, and in a batch of unequal chunks views that fit a neighbouring chunk but not their own (and the
    other way round), which a wrong chunk look-up would judge by the neighbour's size.  The texts end in bytes that are valid
    as bases, qualities and title characters alike, so that an accepted view is accepted by the byte check too."""
    from fastore_b200.binner import GpuBinner
    params = N.make_params(signature_len=8, skip_zone_len=0, paired_end=paired)
    rng = np.random.default_rng(3 + paired)
    tail = lambda k: np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, k)]
    small, big = [], []
    for n, extra in ((40, 300), (400, 600), (30, 300)):
        t1, r1 = fastq_block(n, 100, 20, rng)
        t2, r2 = fastq_block(n, 100, 20, rng) if paired else (None, None)
        t1 = np.concatenate([t1, tail(extra)])
        if paired:
            t2 = np.concatenate([t2, tail(extra + 77)])                       # mate 2's text is longer
        (small if n < 100 else big).append((t1, r1, t2, r2))
    one = [small[0]]
    ts0 = one[0][0].size
    cases = [[(0, 0, 5, "seq_off", ts0 - 100)], [(0, 0, 5, "seq_off", ts0 - 99)], [(0, 0, 6, "qua_off", ts0 - 100)], [(0, 0, 6, "qua_off", ts0 - 99)],
             [(0, 0, 7, "head_off", ts0 - 20)], [(0, 0, 7, "head_off", ts0 - 19)]]
    cases += [[(0, 0, 9, "len", L)] for L in (0, 1, 255, 256, 65535)]
    if paired:
        ts1 = one[0][2].size
        cases += [[(0, 1, 11, "seq_len", 99)], [(0, 1, 11, "seq_len", 101)], [(0, 0, 11, "seq_len", 99)],
                  [(0, 1, 12, "seq_off", ts1 - 100)], [(0, 1, 12, "seq_off", ts1 - 99)], [(0, 1, 13, "qua_off", ts1 - 100)], [(0, 1, 13, "qua_off", ts1 - 99)],
                  [(0, 0, 14, "seq_off", ts1 - 100)]]                        # fits mate 2's longer text, not mate 1's
    batch = [small[0], big[0], small[1]]
    tb = [c[0].size for c in batch]
    neighbour = [[(2, 0, 4, "seq_off", tb[1] - 100)], [(1, 0, 4, "seq_off", tb[1] - 100)], [(0, 0, 4, "qua_off", tb[1] - 100)],
                 [(1, 0, 30, "seq_off", tb[1] - 100), (2, 0, 2, "qua_off", tb[2] - 100)]]
    if paired:
        neighbour += [[(2, 1, 4, "seq_off", batch[1][2].size - 100)], [(1, 1, 4, "qua_off", batch[1][2].size - 100)]]
    with GpuBinner(params) as g:
        for base, edits_list in ((one, cases), (batch, neighbour)):
            for edits in edits_list:
                data = edit(base, edits)
                want = expected_message(contract(params, data))
                assert device_message(lambda: g.stage(make_chunks(data))) == want, f"{edits}: contract {want}"
                if want is not None:
                    clean_batch_equals_the_port(g, params)
        # the cases really are on both sides of each edge
        verdicts = [expected_message(contract(params, edit(one, e))) for e in cases]
        assert sum(v is None for v in verdicts) >= 4 and sum(v is not None and v[3] == "record" for v in verdicts) >= 6


ACCEPT_MODES = [(m, 0) for m in (N.FSB_QUA_NONE, N.FSB_QUA_8BIN, N.FSB_QUA_QVZ)] + [(N.FSB_QUA_BINARY, thr) for thr in (0, 63)]


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["se", "pe"])
@pytest.mark.parametrize("offset", [0, 1, 100, 127])
def test_every_in_range_quality_byte_codes_like_the_port(offset, paired):
    """Acceptance: every quality byte inside the contract at offsets 0, 1, 100 and 127 -- at 100 and 127 the 6- and 3-bit
    modes take bytes of 128 and more -- is taken and coded like the port, for methods 0, 2 and 3 and the 1-bit mode at
    thresholds 0 and 63."""
    from fastore_b200.binner import GpuBinner
    from test_envelope import assert_matches, generated, qual_index, quals
    t1, t2, r1, r2 = generated(3000, 151, 8100 + offset + paired, paired, min_len=40, nrich=0.05)
    for method, thr in ACCEPT_MODES:
        params = N.make_params(signature_len=8, skip_zone_len=2, paired_end=paired, quality_method=method, quality_offset=offset, binary_threshold=thr)
        hi = offset + 63 if method != N.FSB_QUA_BINARY else 0xFF
        rng = np.random.default_rng(offset)
        a, b = t1.copy(), (t2.copy() if paired else None)
        for t, r in ((a, r1), (b, r2)):
            if t is not None:
                quals(t, r, offset, hi, rng)
        assert np.unique(a[qual_index(r1)]).size == hi - offset + 1
        ch = N.make_chunk(a, r1, b, r2)
        import oracle_helpers as O
        with GpuBinner(params, per_read=True) as g:
            assert_matches(g.bin_chunks([ch])[0], O.bin_chunk("orc", params, ch), params, ch, f"offset {offset}, method {method}, threshold {thr}")


@pytest.mark.gpu
@pytest.mark.parametrize("text_only", [False, True], ids=["tables", "text"])
def test_pipelined_rejections_name_the_callers_chunk(text_only):
    """fsb_bin_chunks cuts the caller's chunk list into sub-batches (here one chunk each); a rejection names the chunk by its
    index in the caller's list: a bad byte in chunk 4, then a bad table entry (with text alone: a read of 256 bases) in
    chunk 5."""
    from fastore_b200.binner import GpuBinner
    params = N.make_params(signature_len=8, skip_zone_len=0, paired_end=False)
    rng = np.random.default_rng(45)
    base = many_chunks(rng, 7)
    bad_byte = plant_bytes(base, [(4, 0, 9, "seq_off", 17, 0xC1)])
    if text_only:
        t_long, _ = fastq_block(1, 256, 24, rng)
        t5 = base[5][0]
        bad_table = list(base)
        bad_table[5] = (np.concatenate([t5, t_long]), None, None, None)
        to_chunks = lambda data: [N.make_chunk(t1, None) for t1, _, _, _ in data]
        want_table = (len(base[5][1]), 5)
    else:
        bad_table = edit(base, [(5, 0, 11, "seq_off", base[5][0].size)])
        to_chunks = make_chunks
        want_table = (11, 5)
    with GpuBinner(params, sub_batch_records=1) as g:
        assert device_message(lambda: g.bin_chunks(to_chunks(bad_byte))) == (9, 4, 1, "mate")
        from fastore_b200.binner import FastoreError
        with pytest.raises(FastoreError) as e:
            g.bin_chunks(to_chunks(bad_table))
        m = re.search(r"record (\d+) of chunk (\d+)", str(e.value))
        assert m and (int(m[1]), int(m[2])) == want_table, str(e.value)
        clean_batch_equals_the_port(g, params)


@pytest.mark.gpu
def test_quality_offset_above_127_is_refused():
    """The byte check and the quality coding are defined for offsets 0..127 (see test_offsets_above_127_break_the_check_and_the_coding)."""
    from fastore_b200.binner import GpuBinner, FastoreError
    for offset in (128, 255):
        with pytest.raises(FastoreError, match=r"fsb_create failed \(1\)"):
            GpuBinner(N.make_params(quality_offset=offset))
    with GpuBinner(N.make_params(quality_offset=127)) as g:
        clean_batch_equals_the_port(g, g.params)
