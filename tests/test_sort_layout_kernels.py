"""The kernels between K1 and K4 on their own: the exclusive scans, the stable radix sort of one sub-batch and the one-scan
layout (scan_sort.cuh, layout_fused.cuh), each driven through the host function run_sub uses, at the tile, warp and block
edges where their index arithmetic goes wrong.  The end-to-end suite reaches them only through whole blocks, where a fault
shows up as one wrong stream byte far from its cause; here a mismatch names the first index and its tile, warp and block.

References: np.cumsum for the scans, a stable argsort for the sort, and for the layout emul_layout_tables (tests/emul), a
sequential walk over the sorted records that the CPU tier pins to the plain walk of the layout scan and to the C port.
The GPU tier builds tests/gpu_harness/sort_layout.cu with the product's nvcc flags."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_helpers as O
from cases import CASES, make_case
from fastore_b200 import _native as N
from fastore_b200 import build as B
from fastore_b200 import synth
from test_kernel_core_on_cpu import emul  # noqa: F401  (fixture)

ROOT = Path(__file__).resolve().parent.parent
HARNESS_SRC = ROOT / "tests" / "gpu_harness" / "sort_layout.cu"
HARNESS_LIB = ROOT / "tests" / "gpu_harness" / "_build" / "libsort_layout.so"
FILL32 = 0xA5A5A5A5
FILL64 = 0xA5A5A5A5A5A5A5A5
P = C.c_void_p
U64 = C.c_uint64


def _emul_layout_api(lib):
    lib.emul_sorted_case.restype = C.c_long
    lib.emul_sorted_case.argtypes = [C.POINTER(N.FsbParams), C.POINTER(N.FsbChunk), U64, P, P]
    lib.emul_plain_walk.restype = U64
    lib.emul_plain_walk.argtypes = [C.POINTER(N.FsbParams), P, P, U64, C.c_uint32, P, P]
    lib.emul_layout_tables.restype = U64
    lib.emul_layout_tables.argtypes = [C.POINTER(N.FsbParams), P, P, U64, C.c_uint32, C.c_uint32, P, P, P, P, P, P, P]
    return lib


def where(i):
    """The tile, warp and block a record index falls in, for both the sort (4096-key tiles) and the layout (32-record K4
    tiles, 1024-record warps, 4096-record blocks)."""
    return f"index {i}: 32-tile {i // 32} (+{i % 32}), warp {i // 1024} (+{i % 1024}), block {i // 4096} (+{i % 4096})"


def assert_equal(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    bad = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
    if bad.size:
        i = int(bad[0])
        row = i // int(np.prod(got.shape[1:])) if got.ndim > 1 else i
        raise AssertionError(f"{what}: {bad.size} differ; first at flat {i} ({where(row)}): {got.reshape(-1)[i]!r} vs {want.reshape(-1)[i]!r}")


# ---- the layout: keys, cards and the reference walk ------------------------------------------------------------------

def card_make(rec, info, len_a, len_b, head):
    """core.cuh: card_make, vectorised."""
    rec, info = rec.astype(np.uint64), info.astype(np.uint64)
    return ((rec << np.uint64(36)) | (np.uint64(head & 0xFF) << np.uint64(28)) | (np.uint64(len_b & 0xFF) << np.uint64(20))
            | (np.uint64(len_a & 0xFF) << np.uint64(12)) | ((info & np.uint64(0xFF)) << np.uint64(4)) | ((info >> np.uint64(16)) & np.uint64(0xF)))


def layout_reference(emul_lib, params, keys, cards, ulen, n_chunks):
    n = keys.size
    tiles = (n + 31) // 32
    nbins = int(np.count_nonzero(np.diff(keys.astype(np.int64)))) + 1
    ref = dict(loc=np.zeros(4 * n, np.uint32), binfo=np.zeros(n, np.uint32), tbase=np.zeros(4 * (tiles + 1), np.uint64),
               desc=np.zeros(nbins, N.BIN_DESC_DTYPE), chunk_start=np.full(5 * (n_chunks + 1), FILL64, np.uint64), nb=np.zeros(1, np.uint32))
    cleared = np.zeros(4 * (tiles + 1), np.uint64)
    m = emul_lib.emul_layout_tables(C.byref(params), N.np_ptr(keys), N.np_ptr(cards), n, ulen, n_chunks,
                                    *[N.np_ptr(ref[k]) for k in ("loc", "binfo", "tbase", "desc", "chunk_start", "nb")], N.np_ptr(cleared))
    ref["cleared"] = cleared[:m]
    return ref


# ---- CPU tier: the reference walk against the layout scan's plain walk and against the port ----------------------------

UNIFORM = [c[0] for c in CASES if "min_len" not in c[1]]


@pytest.mark.parametrize("name", UNIFORM)
def test_layout_tables_walk_matches_the_plain_walk(emul, name):
    """emul_layout_tables' positions (loc re-based on tbase) and descriptors equal the plain walk that
    test_one_scan_layout_matches_the_sequential_walk pins the layout scan to, on the case split into two chunks."""
    lib = _emul_layout_api(emul)
    params, chunk, _ = make_case(name)
    n = int(chunk.n_records)
    keys, cards = np.zeros(n, np.uint32), np.zeros(n, np.uint64)
    ulen = lib.emul_sorted_case(C.byref(params), C.byref(chunk), n // 2, N.np_ptr(keys), N.np_ptr(cards))
    assert ulen > 0
    at = np.zeros(4 * n, np.uint64)
    desc = np.zeros(n, N.BIN_DESC_DTYPE)
    nb = lib.emul_plain_walk(C.byref(params), N.np_ptr(keys), N.np_ptr(cards), n, ulen, N.np_ptr(at), N.np_ptr(desc))
    ref = layout_reference(lib, params, keys, cards, ulen, 2)
    assert int(ref["nb"][0]) == nb
    assert_equal(ref["desc"], desc[:nb], f"{name}: descriptors")
    tb = ref["tbase"].reshape(-1, 4)
    for k in range(4 if params.reads_have_headers else 3):
        b0 = tb[np.arange(n) // 32, k]
        got = ref["loc"][k * n:(k + 1) * n].astype(np.uint64) - (b0 & np.uint64(127)) + b0
        assert_equal(got, at[k * n:(k + 1) * n], f"{name}: stream {k} positions")
    opens = np.r_[True, keys[1:] != keys[:-1]]
    assert_equal(ref["binfo"] >> 16 & 1, opens.astype(np.uint32), f"{name}: bin starts")
    # the end entry: the bins and every stream's bytes; chunk 1 starts at the bin of its first key, after chunk 0's bytes
    cs = ref["chunk_start"].reshape(-1, 5)
    sizes = [desc[f"{s}_size"][:nb].astype(np.int64) for s in ("meta", "dna", "qua", "head")]
    assert cs[2, 0] == nb and [int(cs[2, 1 + k]) for k in range(4)] == [int(s.sum()) for s in sizes]
    b1 = int(np.count_nonzero(opens[:int(np.searchsorted(keys, 1 << (2 * params.signature_len + 1)))]))
    if b1 < nb:
        assert cs[1, 0] == b1 and [int(cs[1, 1 + k]) for k in range(4)] == [int(s[:b1].sum()) for s in sizes]


@pytest.mark.parametrize("name", UNIFORM)
def test_layout_tables_match_the_port(emul, name):
    """On the case as one chunk, emul_layout_tables' descriptors and stream sizes equal the C port's block."""
    lib = _emul_layout_api(emul)
    params, chunk, _ = make_case(name)
    want = O.bin_chunk("orc", params, chunk)
    n = int(chunk.n_records)
    keys, cards = np.zeros(n, np.uint32), np.zeros(n, np.uint64)
    ulen = lib.emul_sorted_case(C.byref(params), C.byref(chunk), n, N.np_ptr(keys), N.np_ptr(cards))
    ref = layout_reference(lib, params, keys, cards, ulen, 1)
    assert_equal(ref["desc"], want["bins"], f"{name}: descriptors")
    end = ref["chunk_start"].reshape(-1, 5)[1]
    for k, s in enumerate(("meta", "dna", "qua", "head")):
        assert int(end[1 + k]) == want[s].size, f"{name}: stream {s} size {int(end[1 + k])} vs {want[s].size}"


# ---- GPU tier ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def harness():
    deps = [HARNESS_SRC, *(ROOT / "fastore_b200" / "csrc").glob("*.cuh"), ROOT / "include" / "fastore_b200.h"]
    if not HARNESS_LIB.exists() or any(d.stat().st_mtime > HARNESS_LIB.stat().st_mtime for d in deps):
        HARNESS_LIB.parent.mkdir(exist_ok=True)
        # built under a name of its own, then renamed: a concurrent run never loads a half-written library
        tmp = HARNESS_LIB.with_name(f"{HARNESS_LIB.name}.{os.getpid()}.tmp")
        subprocess.run([B.NVCC, *B.NVCC_FLAGS, "-shared", "-o", str(tmp), str(HARNESS_SRC), "-lcudart"], check=True)
        os.replace(tmp, HARNESS_LIB)
    lib = C.CDLL(str(HARNESS_LIB))
    for f in ("h_scan_u32_u32", "h_scan_u32_u64", "h_scan4_u32_u64", "h_scan4_u64_u64"):
        getattr(lib, f).restype = C.c_int
        getattr(lib, f).argtypes = [P, U64, P]
    lib.h_sort.restype = C.c_int
    lib.h_sort.argtypes = [P, P, U64, P, C.c_uint32, C.c_int, C.c_int, P, P, P]
    lib.h_layout.restype = C.c_int
    lib.h_layout.argtypes = [C.POINTER(N.FsbParams), P, P, U64, C.c_uint32, P, C.c_uint32, P, P, P, P, P, P, P, P, P]
    return lib


# ---- scans ----

SCAN_N = [0, 1, 15, 16, 17, 4095, 4096, 4097, 1024 * 4096, 1024 * 4096 + 1, 3 * 1024 * 4096 + 5]


def scan_inputs(n, dtype, out_bits, rng):
    """all zero, all one, all 0xFFFFFFFF (into 64 bits only) and random, with the sum below 2^out_bits"""
    yield "zero", np.zeros(n, dtype)
    yield "one", np.ones(n, dtype)
    if out_bits == 64:
        yield "ffffffff", np.full(n, 0xFFFFFFFF, dtype)
    top = min((1 << out_bits) // max(n, 1), 1 << (8 * np.dtype(dtype).itemsize)) - 1
    yield "random", rng.integers(0, top, n, dtype=np.uint64, endpoint=True).astype(dtype)


def scan_want(v):
    w = np.zeros(v.size + 1, np.uint64)
    np.cumsum(v, dtype=np.uint64, out=w[1:])
    return w


def scan_check(got, want, what):
    bad = np.flatnonzero(got != want)
    if bad.size:
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.size} differ; first out[{i}] (scan tile {i // 4096}, tile-sum block {i // (4096 * 1024)}): "
                             f"{int(got[i]):#x} vs {int(want[i]):#x}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", SCAN_N)
@pytest.mark.parametrize("kind", ["u32_u32", "u32_u64"])
def test_exclusive_scan(harness, kind, n):
    out_t = np.uint32 if kind == "u32_u32" else np.uint64
    rng = np.random.default_rng(n + 7)
    for name, v in scan_inputs(n, np.uint32, 32 if out_t is np.uint32 else 64, rng):
        out = np.full(n + 1, FILL64, np.uint64).astype(out_t)
        assert getattr(harness, f"h_scan_{kind}")(N.np_ptr(v), n, N.np_ptr(out)) == 0
        scan_check(out.astype(np.uint64), scan_want(v), f"exclusive_scan {kind} n={n} {name}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", SCAN_N)
@pytest.mark.parametrize("kind", ["u32_u64", "u64_u64"])
def test_exclusive_scan4(harness, kind, n):
    in_t = np.uint32 if kind == "u32_u64" else np.uint64
    rng = np.random.default_rng(n + 11)
    for name, _ in scan_inputs(0, in_t, 64, rng):
        # four different arrays: the pattern, then three random ones
        arrays = [v for nm, v in scan_inputs(n, in_t, 64, rng) if nm == name] + [rng.integers(0, (1 << 32) - 1, n, dtype=np.uint64).astype(in_t) for _ in range(3)]
        v = np.concatenate(arrays) if n else np.zeros(0, in_t)
        out = np.full(4 * (n + 1), FILL64, np.uint64)
        assert getattr(harness, f"h_scan4_{kind}")(N.np_ptr(v), n, N.np_ptr(out)) == 0
        for k in range(4):
            scan_check(out[k * (n + 1):(k + 1) * (n + 1)], scan_want(arrays[k]), f"exclusive_scan4 {kind} n={n} {name} array {k}")


# ---- sort ----

CHUNK_SIZES = [0, 1, 2, 3, 4, 5, 31, 32, 33, 4095, 4096, 4097, 8191, 8192, 8193]


def sort_plan(bits):
    passes = (bits + 8) // 9
    base, rem = divmod(bits, passes)
    return [base + (1 if p >= passes - rem else 0) for p in range(passes)]


def sig_pattern(kind, m, bits, rng):
    """one chunk's signatures (bits wide) of a pattern"""
    top = (1 << bits) - 1
    widths = sort_plan(bits)
    if kind == "zero":
        return np.zeros(m, np.uint32)
    if kind == "ones":
        return np.full(m, top, np.uint32)
    if kind == "nbin":
        return np.full(m, 1 << (bits - 1), np.uint32)
    if kind == "two":
        a, b = rng.integers(0, top, 2, endpoint=True)
        return np.where(np.arange(m) % 2 == 0, a, b).astype(np.uint32)
    if kind == "descending":
        return np.sort(rng.integers(0, top, m, endpoint=True))[::-1].astype(np.uint32)
    if kind == "uniform":
        return rng.integers(0, top, m, endpoint=True).astype(np.uint32)
    if kind == "zipf":
        return (rng.zipf(1.2, m) - 1).clip(0, top).astype(np.uint32)
    # "digitP" / "everyP": only pass P's digit varies (random / every value once, in random order), the other bits fixed
    p = int(kind[-1]) % len(widths)
    shift, w = sum(widths[:p]), widths[p]
    base = int(rng.integers(0, top, endpoint=True)) & ~(((1 << w) - 1) << shift)
    d = rng.integers(0, 1 << w, m) if kind.startswith("digit") else np.resize(rng.permutation(1 << w), m)
    return (base | (d.astype(np.int64) << shift)).astype(np.uint32)


SIG_PATTERNS = ["zero", "ones", "nbin", "two", "descending", "uniform", "zipf"] + [f"{k}{p}" for k in ("digit", "every") for p in range(4)]


def sort_batches(bits, rng):
    """Batches (chunk sizes, patterns, signatures): every pattern of SIG_PATTERNS on every chunk size of CHUNK_SIZES, the sizes
    in one of three orders per pattern so that chunks start at every residue mod 4; a batch has at most as many chunks as the
    key leaves room for."""
    max_chunks = min(1 << (32 - bits), 16)
    orders = [CHUNK_SIZES, CHUNK_SIZES[::-1], [int(s) for s in rng.permutation(CHUNK_SIZES)]]
    for p, kind in enumerate(SIG_PATTERNS):
        sizes = orders[p % len(orders)]
        for c0 in range(0, len(sizes), max_chunks):
            group = [int(s) for s in sizes[c0:c0 + max_chunks]]
            yield group, [kind] * len(group), [sig_pattern(kind, m, bits, rng) for m in group]
    # the key's chunk limit: the last chunk index with every signature bit set (0xFFFFFFFF at 31 bits)
    yield [5, 33], ["two", "ones"], [sig_pattern("two", 5, bits, rng), sig_pattern("ones", 33, bits, rng)]


def run_sort(harness, sizes, sigs, bits, fused, rng, what):
    """one sub-batch whose chunks take the top chunk indices of the key; returns the starts of the non-empty chunks"""
    max_chunks = 1 << (32 - bits)
    first = np.zeros(len(sizes) + 1, np.uint64)
    first[1:] = np.cumsum(sizes)
    n = int(first[-1])
    chunk = np.repeat(np.arange(max_chunks - len(sizes), max_chunks, dtype=np.uint64), sizes)
    keys = ((chunk << np.uint64(bits)) | np.concatenate(sigs).astype(np.uint64)).astype(np.uint32)
    cards = (np.arange(n, dtype=np.uint64) << np.uint64(36)) | rng.integers(0, 1 << 36, n, dtype=np.uint64)
    got_k, got_c = np.full(n, FILL32, np.uint32), np.full(n, FILL64, np.uint64)
    nt = U64()
    assert harness.h_sort(N.np_ptr(keys), N.np_ptr(cards), n, N.np_ptr(first), len(sizes), bits, int(fused), N.np_ptr(got_k), N.np_ptr(got_c), C.byref(nt)) == 0
    assert nt.value == sum((s + 4095) // 4096 for s in sizes), what
    order = np.argsort(keys, kind="stable")
    for arr, want, nm in ((got_k, keys[order], "key"), (got_c, cards[order], "card")):
        bad = np.flatnonzero(arr != want)
        if bad.size:
            i = int(bad[0])
            c = int(np.searchsorted(first, i, side="right")) - 1
            r = i - int(first[c])
            raise AssertionError(f"{what}: {bad.size} {nm}s differ; first at {i}: chunk {c} (size {sizes[c]}, starts at {int(first[c])}, "
                                 f"mod 4 = {int(first[c]) % 4}), record {r} of it: sort tile {r // 4096} (+{r % 4096}), strip {r % 4096 // 32}; "
                                 f"{int(arr[i]):#x} vs {int(want[i]):#x}")
    return {int(first[c]) % 4 for c in range(len(sizes)) if sizes[c]}


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["hist", "fusedhist"])
@pytest.mark.parametrize("bits", [2 * k + 1 for k in range(3, 16)])
def test_sort_sub_batch(harness, bits, fused):
    """Every key width 7..31 (1 to 4 passes, digits of 5 to 9 bits), chunk sizes around the strip and tile edges starting at
    every residue mod 4, and the patterns of SIG_PATTERNS, against a stable argsort of keys and unique cards."""
    rng = np.random.default_rng(bits * 2 + fused)
    residues, covered = set(), set()
    for b, (sizes, kinds, sigs) in enumerate(sort_batches(bits, rng)):
        residues |= run_sort(harness, sizes, sigs, bits, fused, rng, f"bits {bits} fused {fused} batch {b} sizes {sizes} patterns {kinds}")
        covered |= set(zip(kinds, sizes))
    assert residues == {0, 1, 2, 3}
    assert covered >= {(k, m) for k in SIG_PATTERNS for m in CHUNK_SIZES}


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["hist", "fusedhist"])
def test_sort_count_table_beyond_1024_scan_tiles(harness, fused):
    """36 M keys at 27 bits: a 512-digit pass over 8790 sort tiles has a count table of 4.5 M entries, more than 1024 scan
    tiles, so the scan of the tile sums carries from one round of 1024 to the next."""
    bits, n = 27, 36_000_000
    assert (n + 4095) // 4096 * 512 > 1024 * 4096
    rng = np.random.default_rng(27)
    run_sort(harness, [n], [rng.integers(0, 1 << bits, n, dtype=np.uint32)], bits, fused, rng, f"36 M keys fused {fused}")


# ---- layout ----

LAYOUT_N = [1, 2, 3, 31, 32, 33, 1023, 1024, 1025, 3073, 4095, 4096, 4097, 1 << 20, (1 << 20) + 1, 3 * (1 << 20) + 3]
LAYOUT_K = 11                  # 4^11 signatures: a bin per record up to 4 M records; 9 chunk bits
# (paired, titles kept, uniform length); the 1-bit quality mode throughout, the fewest quality bits a record can have
LAYOUT_PARAMS = [(pe, heads, L) for pe in (False, True) for heads in (True, False) for L in (1, 100, 255)]
BIN_PATTERNS = ["one_bin", "bin_per_record", "bins_31", "bins_32", "bins_33", "tile_offsets", "warp_block_edges", "nbin", "same_sig_across_chunks"]


def chunk_layouts(n):
    """chunk sizes summing to n: one chunk, empty chunks first / in the middle / consecutive / last"""
    a, b = n // 3, n - n // 3
    yield [n]
    yield [0, 0, a, 0, 0, b, 0]
    yield [0, n] if n < 2 else [a, 0, b, 0, 0]


def bin_sizes(kind, m, rng):
    if m == 0:
        return []
    if kind == "one_bin" or kind == "nbin":
        return [m]
    if kind == "bin_per_record":
        return [1] * m
    if kind.startswith("bins_"):
        w = int(kind[5:])
        return [w] * (m // w) + ([m % w] if m % w else [])
    if kind == "tile_offsets":             # starts at offsets 0, 1, ..., 31 of successive tiles (33 = 32 + 1), then short ones
        sizes = [33] * min(m // 33, 32)
        rest = m - sum(sizes)
        while rest:
            s = min(rest, int(rng.integers(1, 8)))
            sizes.append(s)
            rest -= s
        return sizes
    if kind == "warp_block_edges":         # long bins that run over warp (1024) and block (4096) edges
        sizes, rest = [], m
        while rest:
            s = min(rest, int(rng.choice([1000, 1023, 1025, 3000, 4097, 5000])))
            sizes.append(s)
            rest -= s
        return sizes
    return [m]


def layout_keys(kind, chunks, bits, nbin_only, rng):
    nbin = 1 << (bits - 1)
    keys, last = [], None
    for c, m in enumerate(chunks):
        sizes = bin_sizes(kind if not nbin_only else "one_bin", m, rng)
        nb = len(sizes)
        if nbin_only or kind == "nbin":
            sigs = [nbin] * nb
        elif kind == "same_sig_across_chunks" and last is not None:
            sigs = [last] * nb
        else:
            step = max(1, (nbin - 1) // max(nb, 1))
            sigs = list(np.arange(nb, dtype=np.int64) * step + rng.integers(0, step, nb))
            if nb > 1 and kind in ("warp_block_edges", "tile_offsets"):
                sigs[-1] = nbin                # the N-bin closes the chunk
        if nb:
            last = int(sigs[-1]) if sigs[-1] != nbin else int(sigs[0])
        keys.append((np.uint64(c) << np.uint64(bits)) | np.repeat(np.asarray(sigs, np.uint64), sizes))
    return np.concatenate(keys).astype(np.uint32)


_pools = {}


def card_pool(emul_lib, pe, heads, L):
    """cards of 4096 records that emul_signatures has run on (lengths, info, title lengths)"""
    key = (pe, heads, L)
    if key not in _pools:
        params = layout_params(pe, heads)
        cfg = synth.synth_config(4096, L, paired=pe, seed=300 + L + 2 * pe + heads, header_comments=heads, nrich=0.05)
        t1, t2, r1, r2 = synth.generate(cfg, threads=4)
        if not heads:
            r1 = r1.copy(); r1["head_len"] = 0
        chunk = N.make_chunk(t1, r1, t2, r2)
        sig, info = np.zeros(4096, np.uint32), np.zeros(4096, np.uint32)
        assert emul_lib.emul_signatures(C.byref(params), C.byref(chunk), N.np_ptr(sig), N.np_ptr(info)) == N.FSB_OK
        _pools[key] = (info, r1["seq_len"].astype(np.uint64), (r2["seq_len"] if pe else np.zeros(4096)).astype(np.uint64),
                       np.minimum(r1["head_len"], 255).astype(np.uint64))
    return _pools[key]


def layout_params(pe, heads):
    return N.make_params(signature_len=LAYOUT_K, skip_zone_len=0, paired_end=pe, quality_method=N.FSB_QUA_BINARY, reads_have_headers=heads)


def run_layout(harness, emul_lib, pe, heads, L, n, kind, chunks, rng):
    what = f"layout {'PE' if pe else 'SE'} titles {'kept' if heads else 'dropped'} L={L} n={n} {kind} chunks {chunks}"
    params = layout_params(pe, heads)
    bits = 2 * LAYOUT_K + 1
    keys = layout_keys(kind, chunks, bits, L <= LAYOUT_K, rng)
    info, la, lb, hl = card_pool(emul_lib, pe, heads, L)
    pick = rng.integers(0, 4096, n)
    cards = card_make(np.arange(n, dtype=np.uint64), info[pick], la[pick], lb[pick], hl[pick])
    nch = len(chunks)
    first = np.zeros(nch + 1, np.uint64)
    first[1:] = np.cumsum(chunks)
    ref = layout_reference(emul_lib, params, keys, cards, L, nch)
    tiles = (n + 31) // 32
    end = ref["tbase"][4 * tiles:]
    words = np.array([(int(e) + 31) // 32 for e in end], np.uint64)
    got = dict(loc=np.zeros(4 * n, np.uint32), binfo=np.zeros(n, np.uint32), tbase=np.zeros(4 * (tiles + 1), np.uint64),
               desc=np.zeros(ref["desc"].size, N.BIN_DESC_DTYPE), chunk_start=np.zeros(5 * (nch + 1), np.uint64), nb=np.zeros(1, np.uint32),
               summary=np.zeros(12 * nch, np.uint64), streams=np.zeros(int(words.sum()), np.uint32))
    rc = harness.h_layout(C.byref(params), N.np_ptr(keys), N.np_ptr(cards), n, L, N.np_ptr(first), nch, N.np_ptr(words),
                          *[N.np_ptr(got[k]) for k in ("loc", "binfo", "tbase", "desc", "chunk_start", "nb", "summary", "streams")])
    assert rc == 0, f"{what}: CUDA error {rc}"
    assert int(got["nb"][0]) == int(ref["nb"][0]), f"{what}: {int(got['nb'][0])} bins vs {int(ref['nb'][0])}"
    for k in range(4):
        assert_equal(got["loc"][k * n:(k + 1) * n], ref["loc"][k * n:(k + 1) * n], f"{what}: loc[{k}]")
    assert_equal(got["binfo"], ref["binfo"], f"{what}: binfo")
    tb_got, tb_ref = got["tbase"].reshape(-1, 4), ref["tbase"].reshape(-1, 4)
    bad = np.flatnonzero((tb_got != tb_ref).any(axis=1))
    assert bad.size == 0, f"{what}: tbase of tile {bad[0]} (of {tiles}; {where(int(bad[0]) * 32)}): {tb_got[bad[0]]} vs {tb_ref[bad[0]]}"
    if ref["desc"].size:
        bad = np.flatnonzero(got["desc"] != ref["desc"])
        assert bad.size == 0, f"{what}: descriptor of bin {bad[0]}: {got['desc'][bad[0]]} vs {ref['desc'][bad[0]]}"
    assert_equal(got["chunk_start"].reshape(-1, 5), ref["chunk_start"].reshape(-1, 5), f"{what}: chunk starts (rows: chunks)")
    # the streams: only the words two K4 tiles share are cleared; everything else keeps the fill
    want = np.full(int(words.sum()), FILL32, np.uint32)
    base = np.r_[0, np.cumsum(words)].astype(np.int64)
    kk = (ref["cleared"] >> np.uint64(60)).astype(np.int64)
    want[base[kk] + (ref["cleared"] & np.uint64((1 << 60) - 1)).astype(np.int64)] = 0
    for k in range(4):
        assert_equal(got["streams"][base[k]:base[k + 1]], want[base[k]:base[k + 1]], f"{what}: stream {k} words (index = word)")
    # chunk summaries: a chunk without records takes the start of the next one that has some
    cs = ref["chunk_start"].reshape(-1, 5).astype(np.int64)
    nxt = list(range(nch + 1))
    for c in range(nch - 1, -1, -1):
        nxt[c] = c if chunks[c] else nxt[c + 1]
    starts = [int(cs[nxt[c], 0]) for c in range(nch + 1)]
    summ = got["summary"].reshape(-1, 12).astype(np.int64)
    for c in range(nch):
        s0, s1 = cs[nxt[c]], cs[nxt[c + 1]]
        d = ref["desc"][starts[c]:starts[c + 1]]
        want_s = [s0[0], s1[0] - s0[0], *s0[1:], *(s1[1:] - s0[1:]), int(d["raw_dna_size"].sum()), int(d["raw_head_size"].sum())]
        assert list(summ[c]) == [int(x) for x in want_s], f"{what}: summary of chunk {c}: {list(summ[c])} vs {want_s}"


def layout_cases():
    for n in LAYOUT_N:
        for pe, heads, L in LAYOUT_PARAMS:
            if n >= 1 << 20 and (pe, heads, L) not in ((True, True, 100), (False, False, 255)):
                continue                   # the largest batches with two parameter sets
            yield pytest.param(n, pe, heads, L, id=f"n{n}-{'pe' if pe else 'se'}-{'heads' if heads else 'noheads'}-L{L}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,pe,heads,L", list(layout_cases()))
def test_fused_layout(harness, emul, n, pe, heads, L):
    """Every bin pattern over three chunk layouts against emul_layout_tables: loc, binfo, tbase, descriptors, chunk starts,
    the bin count, the chunk summaries and exactly which stream words are cleared."""
    emul_lib = _emul_layout_api(emul)
    rng = np.random.default_rng(n * 31 + L + 2 * pe + heads)
    # reads no longer than a signature all lie in the N-bin: one bin per chunk, whatever the pattern
    for kind in (BIN_PATTERNS if L > LAYOUT_K else ["nbin"]):
        for chunks in chunk_layouts(n):
            run_layout(harness, emul_lib, pe, heads, L, n, kind, chunks, rng)
