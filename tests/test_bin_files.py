"""Whole-file parity of the host code around the device path (chunk reader, parser, header
statistics, bin-file writer) against the reference's own `fastore_bin e -t1` (SURVEY.md 8c, Mode A),
and consumability of our files by the reference's decoder (Mode C).  CPU tier: the blocks come from
the oracle, so only the host code is under test.  The GPU tier runs the real CLI."""
import pytest

import binfile_helpers as BF

needs_ref_tools = pytest.mark.skipif(not BF.have_ref_tools(), reason="the reference's decoder and downstream tools (oracle/_ref) are not built")

CASES = [
    ("se100_multichunk", dict(n=30000, L=100, paired=False, seed=201), dict(b=2)),
    ("pe150_multichunk", dict(n=22000, L=150, paired=True, seed=202), dict(paired=True, b=2)),
    ("pe100_fast_s10_reduced", dict(n=9000, L=100, paired=True, seed=203, header_comments=True), dict(paired=True, s=10, q=2, comments=False, b=2)),
    ("se250_p12_max_noheads", dict(n=6000, L=250, paired=False, seed=204, nrich=0.1, lowcomplex=0.1), dict(k=12, s=10, q=1, headers=False, b=2)),
    ("se_crlf", dict(n=12000, L=100, paired=False, seed=205, crlf=True), dict(b=2)),
]


@pytest.mark.parametrize("name,gen,flags", CASES, ids=[c[0] for c in CASES])
def test_host_chain_reproduces_reference_files(tmp_path, name, gen, flags):
    files = BF.write_fastq(tmp_path, name, gen["n"], gen["L"], gen["paired"], gen["seed"], **{k: v for k, v in gen.items() if k not in ("n", "L", "paired", "seed")})
    sizes = BF.host_chain(files, tmp_path / "ours", flags, BF.oracle_producer)
    assert len(sizes) >= (2 if "multichunk" in name else 1)
    BF.assert_reference_files(tmp_path / "ours", files, flags, name, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("name,gen,flags", CASES, ids=[c[0] for c in CASES])
def test_cli_reproduces_reference_files(tmp_path, name, gen, flags):
    assert BF.CLI.exists(), "fastore_bin_b200 is not built"
    files = BF.write_fastq(tmp_path, name, gen["n"], gen["L"], gen["paired"], gen["seed"], **{k: v for k, v in gen.items() if k not in ("n", "L", "paired", "seed")})
    BF.run_cli(files, tmp_path / "ours", flags)
    BF.assert_reference_files(tmp_path / "ours", files, flags, name, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("name,gen,flags", CASES, ids=[c[0] for c in CASES])
def test_cli_with_device_side_parse_reproduces_reference_files(tmp_path, name, gen, flags):
    """-D: the chunks go to the library as text alone and are parsed on the GPU (parse.cuh); the tables come back for the title
    statistics.  Same files as `fastore_bin e -t1`, CRLF and -C included."""
    files = BF.write_fastq(tmp_path, name, gen["n"], gen["L"], gen["paired"], gen["seed"], **{k: v for k, v in gen.items() if k not in ("n", "L", "paired", "seed")})
    BF.run_cli(files, tmp_path / "ours", flags, device_parse=True, per_call=3)
    BF.assert_reference_files(tmp_path / "ours", files, flags, name, tmp_path)


@needs_ref_tools
@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True])
def test_reference_decoder_reads_our_files(tmp_path, paired):
    """Mode C: the reference's `fastore_bin d` reconstructs the input records from the CLI's bin files."""
    files = BF.write_fastq(tmp_path, "in", 15000, 100, paired, 210 + int(paired), nrich=0.05)
    flags = dict(paired=paired, b=2)
    BF.run_cli(files, tmp_path / "ours", flags)
    outs = [tmp_path / "dec_1.fastq"] + ([tmp_path / "dec_2.fastq"] if paired else [])
    BF.decode_with_reference(tmp_path / "ours", outs, paired)
    for src, dec in zip(files, outs):
        assert sorted(BF.fastq_records(src)) == sorted(BF.fastq_records(dec))


@pytest.mark.gpu
@pytest.mark.parametrize("workers,per_call", [(2, 1), (3, 4)])
def test_cli_with_many_workers_is_byte_identical(tmp_path, workers, per_call):
    """Chunk i -> worker i mod (G * W) with an ordered writer turn: the files depend neither on the number of GPUs nor
    on the workers per GPU nor on how many chunks one fsb_bin_chunks call takes.  Runs on every device the box has and
    with at least two workers (contexts) on each, so the N>1 dispatch is exercised on a 1-GPU box too."""
    from fastore_b200 import _native as N
    G = N.cuda_lib().fsb_device_count()
    assert G >= 1
    files = BF.write_fastq(tmp_path, "mg", 60000, 150, True, 220)
    flags = dict(paired=True, b=2)
    BF.run_cli(files, tmp_path / "ours", flags, gpus=G, workers=workers, per_call=per_call)
    BF.assert_reference_files(tmp_path / "ours", files, flags, "many_workers", tmp_path)


DOWNSTREAM = [("se_c0_pack", False, False, dict(s=10, b=2)), ("pe_c1_rebin_pack", True, True, dict(paired=True, b=2)),
              ("se_c1_rebin_pack", False, True, dict(b=2))]


@needs_ref_tools
@pytest.mark.parametrize("name,paired,rebin,flags", DOWNSTREAM, ids=[d[0] for d in DOWNSTREAM])
def test_reference_rebin_and_pack_consume_host_chain_files(tmp_path, name, paired, rebin, flags):
    """Mode C, downstream tools: fastore_rebin e -p2 -> fastore_pack e -> fastore_pack d (the reference's own pipeline,
    scripts/fastore_compress.sh) accept the files of our writer and give back the input record multiset.  CPU tier: blocks
    from the oracle, so the host writer is what is under test."""
    files = BF.write_fastq(tmp_path, "in", 9000, 100, paired, 230 + int(paired), nrich=0.03)
    BF.host_chain(files, tmp_path / "ours", flags, BF.oracle_producer)
    outs = BF.downstream_roundtrip(tmp_path / "ours", tmp_path, paired, rebin)
    for src, dec in zip(files, outs):
        assert sorted(BF.fastq_records(src)) == sorted(BF.fastq_records(dec))


@needs_ref_tools
@pytest.mark.gpu
@pytest.mark.parametrize("name,paired,rebin,flags", DOWNSTREAM, ids=[d[0] for d in DOWNSTREAM])
def test_reference_rebin_and_pack_consume_cli_files(tmp_path, name, paired, rebin, flags):
    """The same with the bin files of the real CLI (GPU path): what north_star asks -- fastore_rebin and fastore_pack
    consume our output unchanged (RebinModule.cpp:32, BinFile.cpp:592-628)."""
    files = BF.write_fastq(tmp_path, "in", 9000, 100, paired, 230 + int(paired), nrich=0.03)
    BF.run_cli(files, tmp_path / "ours", flags)
    outs = BF.downstream_roundtrip(tmp_path / "ours", tmp_path, paired, rebin)
    for src, dec in zip(files, outs):
        assert sorted(BF.fastq_records(src)) == sorted(BF.fastq_records(dec))
