#!/usr/bin/env python
"""Generates tests/golden/golden.json (+ small .npz with full outputs) from the COMPILED REFERENCE
(oracle/_ref/libfastore_ref.so: the reference's own Categorize + PackToBins objects), and
tests/golden/bin_files.json from the reference's own `fastore_bin e -t1`.  Run where oracle/_ref is
built (FASTORE_REFERENCE=<reference sources> python -m fastore_b200.build):

    python tests/golden/make_golden.py

The reference ships no golden vectors of its own (SURVEY.md section 4); these pin the oracle port and
the CUDA path on boxes where the reference cannot be compiled.  Inputs are regenerated from seeds by
the C++ generator; their digest is stored too, so a generator change is detected, not mis-attributed."""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

import oracle_helpers as O  # noqa: E402
from cases import CASES, make_case  # noqa: E402

FULL = ("se_single_record", "pe_three_records")          # tiny cases stored byte for byte


def digest(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def block_digests(d: dict) -> dict:
    out = {s: {"size": int(d[s].size), "sha256": digest(d[s])} for s in ("meta", "dna", "qua", "head")}
    out["bins"] = {"count": int(d["bins"].shape[0]), "sha256": digest(d["bins"])}
    out["read_signature"] = digest(d["read_signature"])
    out["read_info"] = digest(d["read_info"])
    out["raw_dna_size"], out["raw_head_size"], out["n_records"] = int(d["raw_dna_size"]), int(d["raw_head_size"]), int(d["n_records"])
    return out


def bin_file_cases():
    """(key, synthetic input, fastore_bin flags) of every whole-file comparison: tests/test_bin_files.py's CASES, plus the inputs
    of test_cli_with_many_workers_is_byte_identical and test_title_statistics_merged_per_chunk_equal_the_reference."""
    from test_bin_files import CASES as FILE_CASES
    return list(FILE_CASES) + [("many_workers", dict(n=60000, L=150, paired=True, seed=220), dict(paired=True, b=2)),
                               ("title_statistics", dict(n=16000, L=100, paired=True, seed=250, header_comments=True), dict(paired=True, b=2))]


def bin_file_golden(tmp: Path) -> dict:
    """Digests of the input files and of what the reference's `fastore_bin e -t1` writes for them (tests/golden/bin_files.json)."""
    import binfile_helpers as BF
    assert BF.have_ref_tools(), "oracle/_ref/fastore_bin is not built"
    out = {}
    for key, gen, flags in bin_file_cases():
        files = BF.write_fastq(tmp, key, gen["n"], gen["L"], gen["paired"], gen["seed"], **{k: v for k, v in gen.items() if k not in ("n", "L", "paired", "seed")})
        BF.run_reference_bin(files, tmp / key, flags)
        out[key] = {"input_sha256": [digest(np.fromfile(f, dtype=np.uint8)) for f in files],
                    "files": BF.bin_file_digests(tmp / key, flags.get("headers", True))}
    return out


def main():
    assert O.have_reference(), "oracle/_ref is not built"
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        files = bin_file_golden(Path(tmp))
    (HERE / "bin_files.json").write_text(json.dumps(files, indent=1, sort_keys=True) + "\n")
    golden = {}
    for name, _, _ in CASES:
        params, chunk, keep = make_case(name)
        d = O.bin_chunk("ref", params, chunk)
        t1, t2 = keep[0], keep[1]
        golden[name] = {"input_sha256": [digest(t1)] + ([digest(t2)] if t2 is not None else []), "block": block_digests(d)}
        if name in FULL:
            np.savez_compressed(HERE / f"{name}.npz", **{k: d[k] for k in ("meta", "dna", "qua", "head", "bins", "read_signature", "read_info")})
    (HERE / "golden.json").write_text(json.dumps(golden, indent=1, sort_keys=True) + "\n")
    print(f"wrote {len(golden)} cases")


if __name__ == "__main__":
    main()
