"""Helpers for whole-bin-file parity (Mode A / Mode C of SURVEY.md 8c): run the reference tools from
oracle/_ref, parse / mask .bmeta, and drive the host reader -> parser -> [block producer] -> writer
chain from Python (the block producer is the oracle in the CPU tier, the CLI uses the GPU)."""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import subprocess
from pathlib import Path

import numpy as np

import oracle_helpers as O
from fastore_b200 import _native as N
from fastore_b200 import synth

ROOT = Path(__file__).resolve().parent.parent
REF_DIR = ROOT / "oracle" / "_ref"
CLI = ROOT / "fastore_b200" / "fastore_bin_b200"
GOLDEN_FILES = ROOT / "tests" / "golden" / "bin_files.json"

# never-initialised bytes of the 88-byte BinModuleConfig dump in the footer (SURVEY.md 8c): struct padding,
# qvzOpts.uncompressed and the two char* of qv_options_t
PARAM_MASK = [3] + list(range(18, 24)) + list(range(26, 32)) + [34] + list(range(36, 56)) + list(range(65, 72)) + [85, 86, 87]


def have_ref_tools() -> bool:
    return (REF_DIR / "fastore_bin").exists()


def write_fastq(tmp: Path, name: str, n: int, L: int, paired: bool, seed: int, **kw):
    cfg = synth.synth_config(n, L, paired=paired, seed=seed, **kw)
    t1, t2, _, _ = synth.generate(cfg, threads=4, with_tables=False)
    f1 = tmp / f"{name}_1.fastq"
    f1.write_bytes(t1.tobytes())
    files = [f1]
    if paired:
        f2 = tmp / f"{name}_2.fastq"
        f2.write_bytes(t2.tobytes())
        files.append(f2)
    return files


def flags_to_args(flags: dict) -> list[str]:
    a = []
    if flags.get("paired"): a.append("-z")
    if flags.get("headers", True): a.append("-H")
    if not flags.get("comments", True): a.append("-C")
    a += [f"-q{flags.get('q', 0)}", f"-p{flags.get('k', 8)}", f"-s{flags.get('s', 0)}", f"-b{flags.get('b', 2)}"]
    if "w" in flags: a.append(f"-w{flags['w']}")
    return a


def run_reference_bin(files, out_prefix: Path, flags: dict, threads: int = 1):
    cmd = [str(REF_DIR / "fastore_bin"), "e", "-i" + " ".join(str(f) for f in files), f"-o{out_prefix}", f"-t{threads}"] + flags_to_args(flags)
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)


def run_cli(files, out_prefix: Path, flags: dict, gpus: int = 1, workers: int | None = None, per_call: int | None = None, device_parse: bool = False):
    cmd = [str(CLI), "e", "-i" + " ".join(str(f) for f in files), f"-o{out_prefix}", f"-G{gpus}"] + flags_to_args(flags)
    if workers is not None: cmd.append(f"-W{workers}")
    if per_call is not None: cmd.append(f"-K{per_call}")
    if device_parse: cmd.append("-D")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r


def make_config(flags: dict) -> N.FshBinConfig:
    cfg = N.FshBinConfig()
    cfg.params = N.make_params(signature_len=flags.get("k", 8), skip_zone_len=flags.get("s", 0), paired_end=flags.get("paired", False),
                               quality_method=flags.get("q", 0), binary_threshold=flags.get("w", 20), reads_have_headers=flags.get("headers", True))
    cfg.min_block_bin_size = 8
    cfg.keep_comments = 1 if flags.get("comments", True) else 0
    cfg.verbose = 0
    cfg.fastq_block_size = flags.get("b", 2) << 20
    return cfg


def host_chain(files, out_prefix: Path, flags: dict, producer, merge_titles: bool = False):
    """reader -> parser -> producer(params, chunk) -> writer, chunk by chunk, like the -t1 loop of BinModule.cpp:124-167.
    merge_titles: gather the title statistics per chunk (fsh_titles) and merge them, the way the CLI's parser threads do."""
    lib = N.host_lib()
    cfg = make_config(flags)
    paired = bool(flags.get("paired"))
    half = len(files) // 2 if paired else len(files)
    a1 = (C.c_char_p * half)(*[str(f).encode() for f in files[:half]])
    a2 = (C.c_char_p * max(1, len(files) - half))(*[str(f).encode() for f in files[half:]] or [b""])
    rd = lib.fsh_reader_open(a1, half, a2, len(files) - half if paired else 0, cfg.fastq_block_size)
    assert rd, lib.fsh_last_error()
    wr = lib.fsh_writer_open(str(out_prefix).encode(), C.byref(cfg))
    assert wr, lib.fsh_last_error()
    b1 = np.zeros(cfg.fastq_block_size + 64, dtype=np.uint8)
    b2 = np.zeros(cfg.fastq_block_size + 64, dtype=np.uint8) if paired else None
    s1, s2 = C.c_uint64(), C.c_uint64()
    sizes = []
    while lib.fsh_reader_next(rd, N.np_ptr(b1), C.byref(s1), N.np_ptr(b2) if paired else None, C.byref(s2)) == 1:
        t1 = b1[: s1.value]
        r1, _ = synth.parse_chunk(t1, keep_headers=flags.get("headers", True), keep_comments=flags.get("comments", True), quality_method=flags.get("q", 0))
        t2 = r2 = None
        if paired:
            t2 = b2[: s2.value]
            r2, _ = synth.parse_chunk(t2, keep_headers=flags.get("headers", True), keep_comments=flags.get("comments", True), quality_method=flags.get("q", 0))
            n = min(len(r1), len(r2)); r1, r2 = r1[:n].copy(), r2[:n].copy()
        sizes.append((int(s1.value), int(s2.value), len(r1)))
        if len(r1) == 0:
            continue
        chunk = N.make_chunk(t1, r1, t2, r2)
        blk, keep = producer(cfg.params, chunk)
        if merge_titles:
            tt = lib.fsh_titles_new()
            assert lib.fsh_titles_add(tt, N.np_ptr(t1), N.np_ptr(r1), len(r1)) == 0
            if paired:
                assert lib.fsh_titles_add(tt, N.np_ptr(t2), N.np_ptr(r2), len(r2)) == 0
            assert lib.fsh_titles_consistent(tt) == 1
            assert lib.fsh_writer_merge_titles(wr, tt) == 0, lib.fsh_last_error()
            lib.fsh_titles_free(tt)
        else:
            assert lib.fsh_writer_add_titles(wr, N.np_ptr(t1), N.np_ptr(r1), len(r1)) == 0
            if paired:
                assert lib.fsh_writer_add_titles(wr, N.np_ptr(t2), N.np_ptr(r2), len(r2)) == 0
        assert lib.fsh_writer_add_block(wr, C.byref(blk)) == 0, lib.fsh_last_error()
        del keep
    lib.fsh_reader_close(rd)
    assert lib.fsh_writer_close(wr) == 0, lib.fsh_last_error()
    return sizes


def oracle_producer(params, chunk):
    """fsb_block over the oracle's output (CPU tier: checks the host code around the device path)."""
    d = O.bin_chunk("orc", params, chunk)
    b = N.FsbBlock()
    for name in ("meta", "dna", "qua", "head"):
        setattr(b, name, N.np_ptr(d[name]) if d[name].size else None)
        setattr(b, name + "_size", d[name].size)
    b.raw_dna_size, b.raw_head_size = d["raw_dna_size"], d["raw_head_size"]
    b.bins = N.np_ptr(d["bins"])
    b.n_bins = d["bins"].shape[0]
    b.n_records = d["n_records"]
    return b, d


def assert_bin_files_equal(a: Path, b: Path, headers: bool):
    for ext in (".bdna", ".bqua") + ((".bhead",) if headers else ()):
        x, y = Path(str(a) + ext).read_bytes(), Path(str(b) + ext).read_bytes()
        assert x == y, f"{ext}: sizes {len(x)} vs {len(y)}"
    x, y = bytearray(Path(str(a) + ".bmeta").read_bytes()), bytearray(Path(str(b) + ".bmeta").read_bytes())
    assert len(x) == len(y), f".bmeta sizes {len(x)} vs {len(y)}"
    foot = int.from_bytes(x[0:8], "little")
    assert foot == int.from_bytes(y[0:8], "little")
    for i in PARAM_MASK:
        x[foot + i] = 0; y[foot + i] = 0
    if x != y:
        i = next(k for k in range(len(x)) if x[k] != y[k])
        raise AssertionError(f".bmeta differs at byte {i} (footer starts at {foot}, params end at {foot + 88}): {x[i]} vs {y[i]}")


def bin_file_digests(prefix: Path, headers: bool) -> dict:
    """SHA-256 of each bin file, the .bmeta with the never-initialised parameter bytes of its footer zeroed."""
    out = {ext: hashlib.sha256(Path(str(prefix) + ext).read_bytes()).hexdigest() for ext in (".bdna", ".bqua") + ((".bhead",) if headers else ())}
    x = bytearray(Path(str(prefix) + ".bmeta").read_bytes())
    foot = int.from_bytes(x[0:8], "little")
    for i in PARAM_MASK:
        x[foot + i] = 0
    out[".bmeta"] = hashlib.sha256(x).hexdigest()
    return out


def assert_reference_files(ours: Path, files, flags: dict, key: str, tmp: Path):
    """Our bin files against what the reference's `fastore_bin e -t1` writes for the same input files: the reference itself
    where oracle/_ref is built, its stored digests (tests/golden/bin_files.json, key `key`) elsewhere."""
    headers = flags.get("headers", True)
    if have_ref_tools():
        run_reference_bin(files, tmp / "ref", flags)
        assert_bin_files_equal(ours, tmp / "ref", headers)
        return
    want = json.loads(GOLDEN_FILES.read_text())[key]
    assert [hashlib.sha256(Path(f).read_bytes()).hexdigest() for f in files] == want["input_sha256"], \
        f"{key}: the synthetic generator wrote other input files than the golden digests were taken from"
    got = bin_file_digests(ours, headers)
    for ext, digest in want["files"].items():
        assert got[ext] == digest, f"{key}: {ext} differs from the reference's file"


def decode_with_reference(prefix: Path, out_files, paired: bool):
    """reference `fastore_bin d`: an independent reader of our bin files (Mode C)."""
    cmd = [str(REF_DIR / "fastore_bin"), "d", f"-i{prefix}", "-o" + " ".join(str(f) for f in out_files), "-t1"] + (["-z"] if paired else [])
    subprocess.run(cmd, check=True, capture_output=True, timeout=600)


def downstream_roundtrip(prefix: Path, work: Path, paired: bool, rebin: bool):
    """The reference's own consumers of a bin file (scripts/fastore_compress.sh): [fastore_rebin e -p2 ->] fastore_pack e ->
    fastore_pack d.  Returns the decoded FASTQ paths."""
    pe = ["-z"] if paired else []
    src = prefix
    if rebin:
        subprocess.run([str(REF_DIR / "fastore_rebin"), "e", f"-i{src}", f"-o{work}/rebin2", "-t1", "-r", "-w1024", "-W1024", "-p2"] + pe,
                       check=True, capture_output=True, timeout=900)
        src = work / "rebin2"
        pack = ["-r", "-f256", "-c10", "-d8", "-w1024", "-W1024"]
    else:
        pack = ["-f256", "-c10", "-d8", "-w256", "-W256"]
    subprocess.run([str(REF_DIR / "fastore_pack"), "e", f"-i{src}", f"-o{work}/packed", "-t1"] + pack + pe, check=True, capture_output=True, timeout=900)
    outs = [work / "unpacked_1.fastq"] + ([work / "unpacked_2.fastq"] if paired else [])
    subprocess.run([str(REF_DIR / "fastore_pack"), "d", f"-i{work}/packed", "-o" + " ".join(str(o) for o in outs), "-t1"] + pe,
                   check=True, capture_output=True, timeout=900)
    return outs


def fastq_records(path: Path):
    lines = path.read_bytes().split(b"\n")
    if lines and lines[-1] == b"": lines.pop()
    return [(lines[i], lines[i + 1], lines[i + 3]) for i in range(0, len(lines) - 3, 4)]
