"""The device path at the edges of its accepted input that the parity cases (tests/cases.py) and the synthetic generator never
reach, compared bit for bit with the C port -- streams, descriptors, per-read signature and info -- and with the compiled
reference where it is built:

  * read lengths on both sides of every 32-base word, so that every instance of K1 and of the rebin scan runs
    (NW = ceil(max_len / 32) = 1..8, each with its own window size, shared-memory plan, slot geometry and K4 staging);
  * signature lengths 3..15, with no signature bits cut off and with all but one cut off.  k = 14 and 15 are the only lengths
    whose sort takes four radix passes (keys of 2k + 1 = 29 and 31 bits) and whose keys leave room for only 8 and 2 chunks
    in one batch: fsb_bin_chunks cuts longer chunk lists there and fsb_stage refuses them;
  * titles of 1..255 bytes, and the largest slot the input contract allows (PE 255 bp, 6-bit quality, 255-byte titles);
  * the whole quality alphabet of every method at offsets 33 and 64, and bytes up to 0xFF in the 1-bit mode;
  * the general layout kernels for batches of one read length (FSB_OPT_FUSED_LAYOUT 0) and the sort whose first pass K1
    counts (FSB_OPT_FUSED_HIST 1).

The CPU tier runs the per-thread cores of the kernels (tests/emul) over the same inputs, so that a failure on the GPU narrows
to the code only the device runs: shared-memory plans, cp.async gathers, K4 staging, the sort and the cutting of batches."""
import ctypes as C

import numpy as np
import pytest

import oracle_helpers as O
from cases import STRESS
from fastore_b200 import _native as N
from fastore_b200 import synth
from test_gpu_parity import gpu_block_dict
from test_kernel_core_on_cpu import emul  # noqa: F401  (fixture: the kernels' per-thread cores built for the host)
from test_rebin_signature import a_signature_of

FSB_OPT_FUSED_LAYOUT, FSB_OPT_FUSED_HIST = 9, 12        # include/fastore_b200.h


# ---- input builders ----------------------------------------------------------------------------------------------------------
def qual_index(recs):
    """Text positions of every quality byte of a record table."""
    lens = recs["seq_len"].astype(np.int64)
    return np.repeat(recs["qua_off"].astype(np.int64) - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))


def quals(text, recs, lo, hi, rng):
    """Overwrite the quality span of every record with bytes uniform over [lo, hi], in place: the record table stays valid."""
    idx = qual_index(recs)
    text[idx] = rng.integers(lo, hi, idx.size, dtype=np.uint8, endpoint=True)


PRINTABLE = np.arange(32, 127, dtype=np.uint8)           # space and the printable 7-bit characters


def titles(n, lo, hi, rng):
    """n title lines of lo..hi bytes: '@', then printable 7-bit characters and spaces."""
    return [b"@" + PRINTABLE[rng.integers(0, PRINTABLE.size, int(m) - 1)].tobytes() for m in rng.integers(lo, hi, n, endpoint=True)]


def fastq(seqs, qualities, heads) -> np.ndarray:
    """FASTQ text of records given as byte strings (titles with their '@'), LF line ends."""
    return np.frombuffer(b"".join(b"%s\n%s\n+\n%s\n" % r for r in zip(heads, seqs, qualities)), dtype=np.uint8).copy()


def spans(text, recs, field):
    raw = text.tobytes()
    return [raw[o: o + m] for o, m in zip(recs[field].tolist(), recs["seq_len"].tolist())]


def retitled(inp, lo, hi, seed):
    """A generated input's reads and qualities under new titles of lo..hi bytes, written out and read back by the host parser."""
    rng = np.random.default_rng(seed)
    out = {}
    for m, (t, r) in enumerate(((inp[0], inp[2]), (inp[1], inp[3]))):
        if t is None:
            out[m] = (None, None)
            continue
        text = fastq(spans(t, r, "seq_off"), spans(t, r, "qua_off"), titles(len(r), lo, hi, rng))
        recs, _ = synth.parse_chunk(text)
        assert len(recs) == len(r)
        out[m] = (text, recs)
    return out[0][0], out[1][0], out[0][1], out[1][1]


def generated(n, L, seed, paired=False, **kw):
    return synth.generate(synth.synth_config(n, L, paired=paired, seed=seed, **kw), threads=4)


def tag(pe):
    return "pe" if pe else "se"


# ---- the cases: synthetic input, binning parameters, then optional new titles (lo, hi) and qualities (lo, hi, shift) -------------
LENGTHS = (31, 32, 33, 64, 65, 70, 96, 97, 128, 160, 161, 170, 192, 193, 200, 224, 225)
KS = (3, 5, 7, 9, 11, 14, 15)
CASES = {}
for L in LENGTHS:                  # one length per batch: the one-scan layout
    for pe in (False, True):
        CASES[f"len{L}_{tag(pe)}"] = dict(gen=dict(n=2500, L=L, seed=4000 + 2 * L + pe, paired=pe, **STRESS),
                                          params=dict(signature_len=8, skip_zone_len=3, paired_end=pe))
for L in (70, 192, 224):           # longest read in NW 3, 6, 7, lengths differ: the general layout kernels
    for pe in (False, True):
        CASES[f"mixed{L}_{tag(pe)}"] = dict(gen=dict(n=3000, L=L, min_len=L // 3, seed=4600 + 2 * L + pe, paired=pe, **STRESS),
                                            params=dict(signature_len=8, skip_zone_len=0, paired_end=pe))
for k in KS:
    for cut in (0, 2 * k - 1):
        for pe in (False, True):
            CASES[f"k{k}_cut{cut}_{tag(pe)}"] = dict(gen=dict(n=3000, L=min(255, 60 + 13 * k), min_len=1, seed=5000 + 100 * k + 2 * cut + pe, paired=pe, **STRESS),
                                                     params=dict(signature_len=k, skip_zone_len=1 + k % 5, cutoff_bits=cut, paired_end=pe))
for k, pe in ((14, False), (15, True)):
    # big bins: the in-bin (input) order must survive all four passes, and the N-bin (the key's top bit) must come last
    CASES[f"k{k}_genome_{tag(pe)}"] = dict(gen=dict(n=20000, L=100, seed=6000 + k, paired=pe, genome_len=3000, sub_rate=0.0, alln=0.01),
                                           params=dict(signature_len=k, skip_zone_len=2, paired_end=pe))
    # every pass over many sort tiles
    CASES[f"k{k}_200k_{tag(pe)}"] = dict(gen=dict(n=200000, L=150 if pe else 100, min_len=40 if pe else 0, seed=6100 + k, paired=pe, **STRESS),
                                         params=dict(signature_len=k, skip_zone_len=2, paired_end=pe))
for pe in (False, True):
    # the largest slot: K1 fits the fewest warps, and the persistent K1 and K4 go round their loops
    CASES[f"slot_max_{tag(pe)}"] = dict(gen=dict(n=150000, L=255, seed=6200 + pe, paired=pe, **STRESS),
                                        params=dict(signature_len=10, skip_zone_len=0, paired_end=pe),
                                        titles=(240, 255), quals=(33, 96, 0), split=2)
    CASES[f"titles_{tag(pe)}"] = dict(gen=dict(n=4000, L=151, min_len=30, seed=6300 + pe, paired=pe, **STRESS),
                                      params=dict(signature_len=8, skip_zone_len=0, paired_end=pe), titles=(1, 255))
for pe in (False, True):
    for off in (33, 64):
        # offset 64 codes the same Phred values as offset 33: the same bytes shifted by 31
        for m in (N.FSB_QUA_NONE, N.FSB_QUA_8BIN, N.FSB_QUA_QVZ):
            CASES[f"qual_m{m}_off{off}_{tag(pe)}"] = dict(gen=dict(n=3000, L=151, min_len=40, seed=6400 + 10 * m + pe, paired=pe, **STRESS),
                                                          params=dict(signature_len=8, skip_zone_len=2, paired_end=pe, quality_method=m, quality_offset=off),
                                                          quals=(33, 96, off - 33))
        # the 1-bit mode takes every byte from the offset up
        for thr in (0, 20, 63):
            CASES[f"qual_bin_thr{thr}_off{off}_{tag(pe)}"] = dict(gen=dict(n=3000, L=151, min_len=40, seed=6500 + thr + pe, paired=pe, **STRESS),
                                                                  params=dict(signature_len=8, skip_zone_len=2, paired_end=pe, quality_method=N.FSB_QUA_BINARY,
                                                                              quality_offset=off, binary_threshold=thr),
                                                                  quals=(off, 0xFF, 0))


def build(name, cap=None):
    """(params, (text1, text2, records1, records2)) of a case; `cap` limits its record count."""
    spec = CASES[name]
    g = dict(spec["gen"])
    n, L, seed = g.pop("n"), g.pop("L"), g["seed"]
    inp = generated(min(n, cap or n), L, **g)
    if "titles" in spec:
        inp = retitled(inp, *spec["titles"], seed=seed)
    if "quals" in spec:
        lo, hi, shift = spec["quals"]
        rng = np.random.default_rng(seed)
        for t, r in ((inp[0], inp[2]), (inp[1], inp[3])):
            if t is not None:
                quals(t, r, lo, hi, rng)
                t[qual_index(r)] += shift
    return N.make_params(**spec["params"]), inp


def chunk_of(inp):
    return N.make_chunk(inp[0], inp[2], inp[1], inp[3])


def batch_of(inp):
    """Three chunks: the input's last record alone, the input, and every few records of it in reverse order -- the same
    reads, so the batch keeps the input's read lengths, titles and K1 instance.  Returns (chunks, tables to keep alive)."""
    t1, t2, r1, r2 = inp
    step = max(3, len(r1) // 1500)
    keep = []

    def part(sl):
        a, b = r1[sl].copy(), (r2[sl].copy() if r2 is not None else None)
        keep.append((a, b))
        return N.make_chunk(t1, a, t2, b)
    return [part(slice(-1, None)), chunk_of(inp), part(slice(None, None, -step))], keep


def assert_matches(got, want, params, chunk, what):
    """A device block against the port's block of the same chunk (and against the compiled reference where it is built)."""
    O.assert_blocks_equal(gpu_block_dict(got), want, f"{what} (gpu vs port)")
    if O.have_reference():
        O.assert_blocks_equal(gpu_block_dict(got), O.bin_chunk("ref", params, chunk), f"{what} (gpu vs compiled reference)")


def set_option(g, option, value):
    g._check(g._lib.fsb_set_option(g._ctx, option, value))


# ---- CPU tier: the builders, and the kernels' per-thread cores on every case ---------------------------------------------------
def test_builders_write_what_they_are_given():
    rng = np.random.default_rng(1)
    heads = titles(3000, 1, 255, rng)
    assert {len(h) for h in heads} == set(range(1, 256))
    seqs = [b"ACGTN"[i % 5: i % 5 + 1] * (1 + i % 255) for i in range(3000)]
    qs = [bytes([33 + (i % 64)]) * len(s) for i, s in enumerate(seqs)]
    text = fastq(seqs, qs, heads)
    recs, st = synth.parse_chunk(text)
    assert st.n_records == 3000 and st.consumed_bytes == text.size
    assert set((recs["head_off"] % 16).tolist()) == set(range(16))          # title starts at every offset mod 16
    raw = text.tobytes()
    assert spans(text, recs, "seq_off") == seqs and spans(text, recs, "qua_off") == qs
    assert [raw[o: o + m] for o, m in zip(recs["head_off"].tolist(), recs["head_len"].tolist())] == heads
    # quals: every quality byte over the whole range, nothing else touched
    before = text.copy()
    quals(text, recs, 64, 0xFF, rng)
    idx = qual_index(recs)
    outside = np.ones(text.size, dtype=bool)
    outside[idx] = False
    assert np.array_equal(text[outside], before[outside])
    assert text[idx].min() == 64 and text[idx].max() == 0xFF and np.unique(text[idx]).size == 0xFF - 64 + 1
    assert np.array_equal(synth.parse_chunk(text, quality_method=N.FSB_QUA_BINARY, quality_offset=64)[0], recs)
    # the largest slot really is the largest: 255 bases and 255-byte titles
    params, inp = build("slot_max_pe", cap=3000)
    assert int(inp[2]["head_len"].max()) == 255 and int(inp[2]["seq_len"].min()) == 255 == int(inp[3]["seq_len"].max())
    assert not params.signature_mask_cutoff_bits and params.quality_method == N.FSB_QUA_NONE


@pytest.mark.parametrize("m", [N.FSB_QUA_NONE, N.FSB_QUA_8BIN, N.FSB_QUA_QVZ])
def test_offset_64_inputs_code_like_offset_33(m):
    """The offset-64 cases are the offset-33 cases with every quality byte moved up by 31: the port codes both alike, over the
    whole alphabet."""
    p33, a = build(f"qual_m{m}_off33_pe")
    p64, b = build(f"qual_m{m}_off64_pe")
    for t, r in ((a[0], a[2]), (a[1], a[3])):
        assert np.unique(t[qual_index(r)]).size == 64
    O.assert_blocks_equal(O.bin_chunk("orc", p64, chunk_of(b)), O.bin_chunk("orc", p33, chunk_of(a)), f"method {m}: offset 64 vs 33")


@pytest.mark.parametrize("name", list(CASES))
def test_kernel_cores_match_the_port(emul, name):
    """K1's signature core, the K1 / K4 packing cores and the one-scan layout, one "thread" after the other on the host
    (inputs above 20000 records are cut to that here)."""
    params, inp = build(name, cap=20000)
    chunk = chunk_of(inp)
    want = O.bin_chunk("orc", params, chunk)
    n = int(chunk.n_records)
    sig, info = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
    assert emul.emul_signatures(C.byref(params), C.byref(chunk), N.np_ptr(sig), N.np_ptr(info)) == N.FSB_OK
    for what, got, ref in (("signature", sig, want["read_signature"]), ("info", info, want["read_info"])):
        bad = np.nonzero(got != ref)[0]
        assert bad.size == 0, f"{name}: {what} of read {bad[0]}: {got[bad[0]]:#x} vs {ref[bad[0]]:#x} ({bad.size} differ)"
    emul.emul_pack.restype = C.c_int
    emul.emul_pack.argtypes = [C.POINTER(N.FsbParams), C.POINTER(N.FsbChunk)] + [C.c_void_p] * 5
    bufs = [np.zeros(want[s].size + 64, dtype=np.uint8) for s in ("meta", "dna", "qua", "head")]
    sizes = np.zeros(4, dtype=np.uint64)
    assert emul.emul_pack(C.byref(params), C.byref(chunk), *[N.np_ptr(b) for b in bufs], N.np_ptr(sizes)) == N.FSB_OK
    for k, s in enumerate(("meta", "dna", "qua", "head")):
        assert int(sizes[k]) == want[s].size, f"{name}: stream {s} size {int(sizes[k])} vs {want[s].size}"
        bad = np.nonzero(bufs[k][: want[s].size] != want[s])[0]
        assert bad.size == 0, f"{name}: stream {s} differs at byte {bad[0]} of {want[s].size} ({bad.size} bytes differ)"
    emul.emul_layout_fused.restype = C.c_long
    emul.emul_layout_fused.argtypes = [C.POINTER(N.FsbParams), C.POINTER(N.FsbChunk), C.c_uint32, C.c_uint32]
    uniform = all(r is None or (r["seq_len"] == inp[2]["seq_len"][0]).all() for r in (inp[2], inp[3]))
    for per_thread, threads in ((32, 128), (3, 5), (1, 7)):
        bad = emul.emul_layout_fused(C.byref(params), C.byref(chunk), per_thread, threads)
        assert bad == (0 if uniform else -1), f"{name}: one-scan layout, {per_thread} x {threads}: {bad}"


REBIN = [(k, L) for k in (14, 15) for L in (70, 200, 224)]


def rebin_input(k, L):
    params = N.make_params(signature_len=k, skip_zone_len=3)
    text, _, recs, _ = generated(1500, L, 7000 + 10 * k + L, **STRESS)
    return params, text, recs, (a_signature_of(params, text, recs, 3), 0), (2, 1 << k, 4 ** k)


@pytest.mark.parametrize("k,L", REBIN)
def test_rebin_core_matches_the_port(emul, k, L):
    params, text, recs, curs, parities = rebin_input(k, L)
    emul.emul_new_minimizers.restype = C.c_int
    emul.emul_new_minimizers.argtypes = [C.POINTER(N.FsbParams), C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    for cur in curs:
        for parity in parities:
            want = O.new_minimizers_port(params, text, recs, cur, parity)
            sig, info = np.zeros(len(recs), dtype=np.uint32), np.zeros(len(recs), dtype=np.uint32)
            assert emul.emul_new_minimizers(C.byref(params), N.np_ptr(text), text.size, N.np_ptr(recs), len(recs), cur, parity, N.np_ptr(sig), N.np_ptr(info)) == 0
            assert np.array_equal(sig, want[0]), f"cur {cur} parity {parity}: signature of read {int(np.nonzero(sig != want[0])[0][0])}"
            assert np.array_equal(info, want[1]), f"cur {cur} parity {parity}: info of read {int(np.nonzero(info != want[1])[0][0])}"


# ---- GPU tier ----------------------------------------------------------------------------------------------------------------
def run_case(name, options=()):
    """The case as one chunk (fsb_bin_chunks), then inside a batch of three chunks (fsb_bin_chunks, and stage / run / fetch
    with the case's run split)."""
    from fastore_b200.binner import GpuBinner
    params, inp = build(name)
    chunks, keep = batch_of(inp)
    want = [O.bin_chunk("orc", params, ch) for ch in chunks]
    split = CASES[name].get("split")
    with GpuBinner(params, per_read=True) as g:
        for opt, value in options:
            set_option(g, opt, value)
        assert_matches(g.bin_chunks([chunks[1]])[0], want[1], params, chunks[1], f"{name}, one chunk")
        for ci, blk in enumerate(g.bin_chunks(chunks)):
            assert_matches(blk, want[ci], params, chunks[ci], f"{name}, chunk {ci} of 3")
        if split:
            g.set_run_split(split)
            g.stage(chunks)
            g.run()
            for ci, blk in enumerate(g.fetch()):
                assert_matches(blk, want[ci], params, chunks[ci], f"{name}, chunk {ci} of 3, run split {split}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_case_matches_the_port(name):
    run_case(name)


OPTION_CASES = ["len33_se", "len224_pe", "mixed192_pe", "k14_genome_se", "k15_genome_pe", "k15_cut0_pe", "qual_m2_off64_pe"]


@pytest.mark.gpu
@pytest.mark.parametrize("option,value", [(FSB_OPT_FUSED_LAYOUT, 0), (FSB_OPT_FUSED_HIST, 1)], ids=["general_layout", "fused_hist"])
@pytest.mark.parametrize("name", OPTION_CASES)
def test_options_give_the_same_blocks(name, option, value):
    run_case(name, [(option, value)])


def limit_chunks(k, n_chunks):
    """Small chunks at signature length k (the longest list fsb_bin_chunks' default sub-batch size would not cut)."""
    pe = k == 15
    params = N.make_params(signature_len=k, skip_zone_len=2, paired_end=pe)
    keep = [generated(400 + 250 * ci, 120, 7500 + 20 * k + ci, pe, min_len=1, **STRESS) for ci in range(n_chunks)]
    return params, [chunk_of(t) for t in keep], keep


MAX_CHUNKS = {14: 8, 15: 2}          # 2^(32 - key bits) chunk indices fit in a 32-bit sort key


@pytest.mark.gpu
@pytest.mark.parametrize("k,n_chunks", [(14, 11), (15, 5)])
def test_bin_chunks_cuts_at_the_chunk_limit_of_the_key(k, n_chunks):
    from fastore_b200.binner import GpuBinner
    params, chunks, keep = limit_chunks(k, n_chunks)
    assert sum(int(ch.n_records) for ch in chunks) < 400000 and n_chunks > MAX_CHUNKS[k]
    with GpuBinner(params, per_read=True) as g:
        got = g.bin_chunks(chunks)
    for ci, ch in enumerate(chunks):
        assert_matches(got[ci], O.bin_chunk("orc", params, ch), params, ch, f"k {k}, chunk {ci} of {n_chunks}")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [14, 15])
def test_stage_takes_exactly_the_chunk_limit_of_the_key(k):
    """The top chunk index sets the key's top bit at k = 15; one chunk more is refused and leaves the context usable."""
    from fastore_b200.binner import GpuBinner, FastoreError
    params, chunks, keep = limit_chunks(k, MAX_CHUNKS[k] + 1)
    want = [O.bin_chunk("orc", params, ch) for ch in chunks]
    with GpuBinner(params, per_read=True) as g:
        for attempt in range(2):
            g.stage(chunks[attempt: attempt + MAX_CHUNKS[k]])
            g.run()
            for ci, blk in enumerate(g.fetch()):
                assert_matches(blk, want[attempt + ci], params, chunks[attempt + ci], f"k {k}, attempt {attempt}, chunk {ci}")
            if attempt == 0:
                with pytest.raises(FastoreError, match="too many chunks"):
                    g.stage(chunks)


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True])
def test_device_byte_check_at_offset_64(paired):
    """FSB_OPT_VALIDATE at quality offset 64: the 6-bit modes take [64, 127], the 1-bit mode every byte from 64 up; what is
    taken is coded like the port codes it."""
    from fastore_b200.binner import GpuBinner, FastoreError
    t1, t2, r1, r2 = generated(700, 100, 64, paired, nrich=0.05)
    rng = np.random.default_rng(64)
    for t, r in ((t1, r1), (t2, r2)):
        if t is not None:
            quals(t, r, 64, 127, rng)
    six = N.make_params(signature_len=8, skip_zone_len=0, paired_end=paired, quality_offset=64)
    one = N.make_params(signature_len=8, skip_zone_len=0, paired_end=paired, quality_method=N.FSB_QUA_BINARY, quality_offset=64)
    at = int(r1["qua_off"][123]) + 50
    with GpuBinner(six, per_read=True) as g, GpuBinner(one, per_read=True) as gb:
        for gpu, params, refused, taken in ((g, six, (63, 128, 0xFF), (127, 64)), (gb, one, (63, 33), (128, 0xFF, 64))):
            for value in refused:
                t = t1.copy()
                t[at] = value
                with pytest.raises(FastoreError, match="outside the input contract"):
                    gpu.bin_chunks([N.make_chunk(t, r1, t2, r2)])
            for value in taken:
                t = t1.copy()
                t[at] = value
                ch = N.make_chunk(t, r1, t2, r2)
                assert_matches(gpu.bin_chunks([ch])[0], O.bin_chunk("orc", params, ch), params, ch, f"byte {value}, method {params.quality_method}")


@pytest.mark.gpu
@pytest.mark.parametrize("k,L", REBIN)
def test_rebin_kernel_matches_the_port(k, L):
    from fastore_b200.binner import GpuBinner
    params, text, recs, curs, parities = rebin_input(k, L)
    raw = text.tobytes()
    with GpuBinner(params) as g:
        for cur in curs:
            for parity in parities:
                want = O.new_minimizers_port(params, text, recs, cur, parity)
                sig, info = g.find_new_minimizers(text, recs, cur, parity)
                assert np.array_equal(sig, want[0]), f"cur {cur} parity {parity}: signature of read {int(np.nonzero(sig != want[0])[0][0])}"
                assert np.array_equal(info, want[1]), f"cur {cur} parity {parity}: info of read {int(np.nonzero(info != want[1])[0][0])}"
                if O.REBIN_REF_LIB.exists():
                    for i, r in enumerate(recs):
                        seq = raw[int(r["seq_off"]): int(r["seq_off"]) + int(r["seq_len"])]
                        s, p, rev = O.find_new_minimizer("ref", params, seq, cur, parity)
                        assert (sig[i], info[i]) == (s, p | (N.FSB_INFO_REVERSE if rev else 0)), f"cur {cur} parity {parity}: read {i} vs the reference"
