#!/usr/bin/env python
"""bench.py -- reads/s of the fastore_bin categorise + scatter path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --config c1|c2|c3|c4r|c4m|c5 ...         (the other BASELINE configs; lines kept under profiles/)
    python bench.py ... --dump-outputs DIR                   (also writes the last timed step's output as DIR/*.npy)

A "step" is one pass of the hot path (K1 ingest -> stable sort -> layout scan -> K4 place) over one batch of
synthetic FASTQ chunks.  Workload (SURVEY.md 8d):

  N = 1   BASELINE configs[1]: 10 M synthetic 150 bp pairs, lossless binning parameters (-z -H -q0 -p8 -s0), cut
          into the chunks the reference's `-b256` chunk cutter produces;
  N > 1   BASELINE configs[2]: 100 M such pairs as eight 12.5 M-pair shards (seeds 1030..1037) spread over the N
          ranks -- a fixed total ("scaling": "strong"); chunks are independent units, there is no collective on the
          data path.

  value     whole-job reads/s with the chunks already resident in HBM (kernels only -- RESIDENT: no copies, no host
            parsing --, CUDA events on the library's stream, max over ranks);
  e2e       the same metric through the C ABI call fsb_bin_chunks with HOST buffers: pinned chunk text + record
            tables host->device, kernels, packed streams + descriptors device->host, every step (pipelined); its
            h2d_ms / d2h_ms / kernel_ms are the three legs timed one at a time (fsb_stage, fsb_run, fsb_fetch);
  roofline  algorithmic bytes (SURVEY 8d: every input byte the path consumes + every output byte it produces, counted
            exactly by the library) / CUDA-event duration vs MEASURED_PEAKS.json -- for the dominant kernel as the
            contract defines it (`frac`), for that kernel against the bytes it moves itself (`kernel_own_frac`) and
            for the whole path (`whole_path_frac`, the only one whose numerator and denominator cover the same work);
  parity    after the timed regions every rank checks whole chunks of its shard, as the resident run produced them,
            bit for bit against the compiled reference (oracle/_ref; the C port where it is not built); a mismatch
            fails the run;
  cpu_baseline  the compiled reference's Categorize + PackToBins (oracle/_ref) timed on the host cores on a bounded
            sample of the same workload (rank 0, N=1 only).

The oracle libraries are loaded only for the parity check, the cpu_baseline leg and --impl reference.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True       # the tree may be read-only; the benchmark leaves nothing in it

METRIC = "reads_per_sec_binned"
UNIT = "reads/s"
PE_CUT_WINDOW = 1 << 20      # FastqStream.h:142: the PE chunk cutter backs off 1 MiB
SE_CUT_WINDOW = 1 << 13      # FastqStream.h:99

# BASELINE.json configs (SURVEY.md 8d).  `n` counts records: reads (SE) or pairs (PE).
WORKLOADS = {
    "c1": dict(desc="BASELINE configs[0]: 1M synthetic 100 bp single-end reads, lossless profile (-H -q0 -p8 -s0), -b16 chunking",
               n=1_000_000, L=100, paired=False, seed=101, block_mib=16, synth={}, params=dict(signature_len=8, skip_zone_len=0)),
    "c2": dict(desc="BASELINE configs[1]: 10M synthetic 150 bp paired-end reads (pairs), lossless binning params (-z -H -q0 -p8 -s0), -b256 chunking",
               n=10_000_000, L=150, paired=True, seed=102, block_mib=256, synth={}, params=dict(signature_len=8, skip_zone_len=0, paired_end=True)),
    "c3": dict(desc="BASELINE configs[2]: 100M synthetic 150 bp paired-end reads (pairs) as eight 12.5M-pair shards (seeds 1030-1037) sharded "
                    "across the GPUs, lossless binning params (-z -H -q0 -p8 -s0), -b256 chunking",
               n=100_000_000, L=150, paired=True, seed=1030, shards=8, block_mib=256, synth={}, params=dict(signature_len=8, skip_zone_len=0, paired_end=True)),
    "c4r": dict(desc="BASELINE configs[3], reduced profile: 2M synthetic 250 bp single-end reads, -H -C -q2 -p12 -s10, -b256 chunking",
                n=2_000_000, L=250, paired=False, seed=104, block_mib=256, synth=dict(header_comments=True), keep_comments=False,
                params=dict(signature_len=12, skip_zone_len=10, quality_method=2)),
    "c4m": dict(desc="BASELINE configs[3], max profile: 2M synthetic 250 bp paired-end reads (pairs), -z -q1 -p12 -s10 (no headers), -b256 chunking",
                n=2_000_000, L=250, paired=True, seed=104, block_mib=256, synth={},
                params=dict(signature_len=12, skip_zone_len=10, paired_end=True, quality_method=1, reads_have_headers=False)),
    "c5": dict(desc="BASELINE configs[4]: 2M synthetic 150 bp pairs, 10% N-rich (10-60% N), 10% low-complexity, 1% all-N, directed tie set, "
                    "lossless binning params (-z -H -q0 -p8 -s0), -b256 chunking",
               n=2_000_000, L=150, paired=True, seed=105, block_mib=256, synth=dict(nrich=0.10, lowcomplex=0.10, alln=0.01, tie=0.01),
               params=dict(signature_len=8, skip_zone_len=0, paired_end=True)),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampling of SM clocks and throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._th = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    f = [x.strip() for x in out.split(",")]
                    self.samples.append((float(f[1]), float(f[2]), f[4], f[5], f[6], f[7]))
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._th:
            self._th.join(timeout=10)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": sorted(reasons), "samples": len(sm)}


def pinned_alloc_factory(lib, keep):
    """numpy uint8 arrays over cudaHostAlloc'd memory (freed at exit)."""
    def alloc(nbytes):
        p = lib.fsb_host_alloc(max(int(nbytes), 1))
        if not p:
            raise MemoryError("fsb_host_alloc failed")
        keep.append(p)
        buf = (C.c_uint8 * int(nbytes)).from_address(p)
        return np.frombuffer(buf, dtype=np.uint8)
    return alloc


def pinned_records(lib, keep, recs):
    from fastore_b200 import _native as N
    raw = pinned_alloc_factory(lib, keep)(recs.nbytes)
    out = raw.view(N.RECORD_DTYPE)
    out[:] = recs
    return out


def make_params(w):
    from fastore_b200 import _native as N
    return N.make_params(quality_offset=33, **w["params"])


def rank_shards(w, rank: int, world: int, total: int | None):
    """[(seed, first_index, n_records)] of this rank.  Sharded workloads (c3) spread their shards round-robin over the
    ranks; the others give every rank its own range of the same stream (rank r: records [r n, (r + 1) n))."""
    n = int(total) if total else int(w["n"])
    if "shards" in w:
        S = w["shards"]
        per = n // S
        return [(w["seed"] + s, 0, per) for s in range(S) if s % world == rank]
    return [(w["seed"], rank * n, n)]


def workload_chunks(w, shards, pinned: bool, lib=None, keep=None, threads=None, limit_records=None):
    """The rank's records as a list of chunks cut like `-b<block>` cuts the input (FastqStream.cpp:44-228): every chunk
    but the last of a shard holds the records that fit in (block - window) bytes of (mate-1) text."""
    from fastore_b200 import _native as N
    from fastore_b200 import synth
    window = PE_CUT_WINDOW if w["paired"] else SE_CUT_WINDOW
    chunks, keepalive = [], []
    alloc = pinned_alloc_factory(lib, keep) if pinned else None
    keep_comments = w.get("keep_comments", True)
    headers = bool(w["params"].get("reads_have_headers", True))
    for seed, first, n_shard in shards:
        if limit_records is not None:
            n_shard = min(n_shard, limit_records)
        probe = synth.synth_config(1, w["L"], paired=w["paired"], seed=seed, first_index=first + n_shard - 1, **w["synth"])
        b1, b2 = C.c_uint64(), C.c_uint64()
        N.host_lib().fsh_synth_size(C.byref(probe), C.byref(b1), C.byref(b2))
        per_chunk = max(1, ((w["block_mib"] << 20) - window) // int(b1.value))      # widest title of the shard
        done = 0
        while done < n_shard:
            n = min(per_chunk, n_shard - done)
            cfg = synth.synth_config(n, w["L"], paired=w["paired"], seed=seed, first_index=first + done, **w["synth"])
            t1, t2, r1, r2 = synth.generate(cfg, threads=threads, out=alloc)
            if not keep_comments or not headers:
                # -C cuts the title at the first space, without -H no title is kept: the host parser's table
                r1, _ = synth.parse_chunk(t1, keep_headers=headers, keep_comments=keep_comments, quality_method=w["params"].get("quality_method", 0))
                if t2 is not None:
                    r2, _ = synth.parse_chunk(t2, keep_headers=headers, keep_comments=keep_comments, quality_method=w["params"].get("quality_method", 0))
            if pinned:
                r1 = pinned_records(lib, keep, r1)
                r2 = pinned_records(lib, keep, r2) if r2 is not None else None
            keepalive.append((t1, t2, r1, r2))
            chunks.append(N.make_chunk(t1, r1, t2, r2))
            done += n
    return chunks, keepalive


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def config_dict(w, name, n_gpus, n_rank, n_chunks, total):
    mates = 2 if w["paired"] else 1
    p = w["params"]
    return {"workload": w["desc"], "config": name, "records_total": int(total), "reads_total": int(total) * mates,
            "records_per_gpu": int(n_rank), "reads_per_gpu": int(n_rank) * mates, "read_len": w["L"], "paired": w["paired"],
            "chunks_per_gpu": n_chunks, "signature_len": p.get("signature_len", 8), "skip_zone_len": p.get("skip_zone_len", 0),
            "quality_mode": f"q{p.get('quality_method', 0)}", "headers": bool(p.get("reads_have_headers", True)),
            "sharding": f"{n_gpus} rank(s), whole chunks per rank, no data-path collective",
            "l2_policy": "inputs and outputs per step exceed the 126 MB L2 many times over; no flush needed"}


# -------------------------------------------------------------------------------------------------
def oracle():
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle_helpers as O
    return O


def cpu_sample(chunks, threads, target_s=12.0):
    """A bounded sample for the CPU legs: the first `n` records of chunk 0, split across `threads` workers like `-t N`."""
    from fastore_b200 import _native as N
    ch0 = chunks[0]
    n = int(min(ch0.n_records, max(20000, 50_000 * threads * target_s / 12.0 * 3)))
    sample = N.FsbChunk()
    C.memmove(C.byref(sample), C.byref(ch0), C.sizeof(N.FsbChunk))
    sample.n_records = n
    return sample, n


def run_reference_arm(args, w, name):
    """--impl reference: the reference's own CPU implementation of the path (Categorize + PackToBins, compiled from
    /root/reference into oracle/_ref) on all host cores, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from fastore_b200 import build
    build.build_host()
    O = oracle()
    if not O.PORT_LIB.exists() and not O.have_reference():
        build.build_oracle()
    kind = "ref" if O.have_reference() else "orc"
    params = make_params(w)
    threads = host_threads()
    mates = 2 if w["paired"] else 1
    n_sample = int(min(w["n"], max(50_000, 150_000 * threads)))
    shards = rank_shards(w, 0, 1, None)
    chunks, keep = workload_chunks(w, shards[:1], pinned=False, threads=min(32, threads), limit_records=n_sample)
    sample, n = cpu_sample(chunks, threads)
    sample.n_records = min(n_sample, chunks[0].n_records)
    n = int(sample.n_records)
    once = O.time_bin_chunk(kind, params, sample, threads, 1)
    reps = int(max(1, min(64, round(2.0 / max(once, 1e-3)))))       # one step = about 2 s of wall time on all cores
    for _ in range(args.warmup):
        O.time_bin_chunk(kind, params, sample, threads, reps)
    t = 0.0
    for _ in range(args.steps):
        t += O.time_bin_chunk(kind, params, sample, threads, reps)
    ms = 1e3 * t / max(args.steps, 1)
    value = mates * n * reps / (ms / 1e3)
    total = args.total_records or w["n"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if "shards" in w else "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config_dict(w, name, args.gpus, total // max(args.gpus, 1) if "shards" in w else total, 0, total),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference" if kind == "ref" else "port",
                             "sample": f"{n * reps} records per step (the first {n} records of the workload x {reps} passes), Categorize+PackToBins on "
                                       f"{threads} threads, one slice per thread like fastore_bin -t{threads}"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def block_dict(blk):
    return {"meta": blk.meta, "dna": blk.dna, "qua": blk.qua, "head": blk.head, "bins": blk.bins, "raw_dna_size": blk.raw_dna_size,
            "raw_head_size": blk.raw_head_size, "n_records": blk.n_records, "read_signature": blk.read_signature, "read_info": blk.read_info}


DUMP_STREAMS = ("meta", "dna", "qua", "head")
DUMP_STREAM_SAMPLE = 2 << 20          # bytes per stream (float32: 8 MB each)
DUMP_BIN_SAMPLE = 1 << 17             # descriptor rows (9 float64 columns: 9 MB)
DUMP_SEED = 20260


def dump_outputs(out_dir, blocks):
    """Writes the blocks of the last timed step as out_dir/<name>.npy, for comparing two builds output for output:

      sizes.npy          float64 [chunk, 8]     n_records, n_bins, meta/dna/qua/head stream sizes, raw_dna_size, raw_head_size
      sha256.npy         float64 [chunk, 5, 8]  SHA-256 of the meta, dna, qua, head streams and the bin descriptors, as 32-bit words
      <stream>.npy       float32 [<= 2 Mi]      a seeded sample of the bytes of that stream, all chunks end to end
      bins.npy           float64 [<= 128 Ki, 9] a seeded sample of descriptor rows: chunk, then the 8 fields of fsb_bin_desc

    The whole output is gigabytes, so the values are sampled (42 MB in all) and the digests cover every byte.  The sample
    positions depend only on the sizes, so two builds that agree on the sizes are sampled at the same positions."""
    import hashlib
    from concurrent.futures import ThreadPoolExecutor
    from fastore_b200 import _native as N

    def view(ptr, nbytes, dtype=np.uint8):
        if not ptr or nbytes == 0:
            return np.zeros(0, dtype=dtype)
        return np.frombuffer((C.c_uint8 * int(nbytes)).from_address(ptr), dtype=dtype)

    streams = [{s: view(getattr(b, s), getattr(b, s + "_size")) for s in DUMP_STREAMS} for b in blocks]
    bins = [view(b.bins, int(b.n_bins) * N.BIN_DESC_DTYPE.itemsize, N.BIN_DESC_DTYPE) for b in blocks]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    sizes = [[b.n_records, b.n_bins, b.meta_size, b.dna_size, b.qua_size, b.head_size, b.raw_dna_size, b.raw_head_size] for b in blocks]
    np.save(out / "sizes.npy", np.array(sizes, dtype=np.float64).reshape(len(blocks), 8))
    parts = [st[s] for st in streams for s in DUMP_STREAMS] + [np.frombuffer(bn.tobytes(), np.uint8) for bn in bins]
    with ThreadPoolExecutor(max_workers=8) as ex:
        digests = list(ex.map(lambda a: np.frombuffer(hashlib.sha256(a).digest(), ">u4"), parts))
    sha = np.array(digests, dtype=np.float64).reshape(5, len(blocks), 8).transpose(1, 0, 2)
    np.save(out / "sha256.npy", np.ascontiguousarray(sha))
    rng = np.random.default_rng(DUMP_SEED)

    def sample(arrays, k):
        """Sorted seeded positions in the arrays laid end to end: (array index, position in it)."""
        ends = np.cumsum([a.shape[0] for a in arrays], dtype=np.int64)
        total = int(ends[-1]) if len(ends) else 0
        pos = np.sort(rng.integers(0, total, min(k, total), dtype=np.int64)) if total else np.zeros(0, np.int64)
        which = np.searchsorted(ends, pos, side="right")
        return which, pos - np.concatenate(([0], ends[:-1]))[which]

    for s in DUMP_STREAMS:
        arrays = [st[s] for st in streams]
        which, pos = sample(arrays, DUMP_STREAM_SAMPLE)
        vals = np.concatenate([arrays[i][pos[which == i]] for i in range(len(arrays))]) if len(pos) else np.zeros(0, np.uint8)
        np.save(out / f"{s}.npy", vals.astype(np.float32))
    which, pos = sample(bins, DUMP_BIN_SAMPLE)
    rows = np.zeros((len(pos), 9), dtype=np.float64)
    rows[:, 0] = which
    for i in range(len(bins)):
        sel = which == i
        for j, f in enumerate(N.BIN_DESC_DTYPE.names):
            rows[sel, 1 + j] = bins[i][f][pos[sel]]
    np.save(out / "bins.npy", rows)


# -------------------------------------------------------------------------------------------------
def run_b200_arm(args, w, name):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # stdout carries exactly one JSON line
        sys.stdout.flush()
        saved = os.dup(1)                                             # NCCL prints its version banner to stdout when the communicator comes up
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from fastore_b200 import _native as N
    from fastore_b200 import build
    from fastore_b200 import sharding
    from fastore_b200.binner import GpuBinner
    build.build_host()
    if not build.CUDA_LIB.exists():
        build.build_cuda()
    lib = N.cuda_lib()
    params = make_params(w)
    mates = 2 if w["paired"] else 1
    total = args.total_records or w["n"]
    shards = rank_shards(w, rank, world, total)
    n_rank = sum(s[2] for s in shards)
    keep_ptrs = []
    t0 = time.time()
    gen_threads = max(1, min(32, host_threads() // max(1, world)))
    chunks, keep = workload_chunks(w, shards, pinned=True, lib=lib, keep=keep_ptrs, threads=gen_threads)
    log(f"[rank {rank}] generated {n_rank} records in {len(chunks)} chunks in {time.time() - t0:.1f}s")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        return sharding.max_over_ranks(x, device="cuda")

    stream = torch.cuda.Stream()
    g = GpuBinner(params, device=local, stream=stream.cuda_stream, profile=True)

    def device_ms(fn):
        """CUDA-event time of what fn enqueues / does on the library's stream, max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(stream):
            e0.record(stream)
            fn()
            e1.record(stream)
        g.sync()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- the three legs one at a time: host->device (with the input check), kernels, device->host ------------------
    g.stage(chunks)                                     # untimed: device buffers get allocated
    g.sync()
    st0 = g.stats()
    h2d_ms = device_ms(lambda: g.stage(chunks))
    st1 = g.stats()
    h2d_leg_bytes = st1["h2d_bytes"] - st0["h2d_bytes"]
    check_ms = g.stage_times(5)[0].get("check", 0.0)   # stage_stats + validate_text kernels of that fsb_stage
    # per-stage times: the batch as ONE pass on one stream (with sub-batches overlapped on two streams the stages of
    # different sub-batches run at the same time and have no duration of their own)
    for _ in range(args.warmup):
        g.run()
    g.sync()
    g.stage_times()                                     # reset the per-stage accumulators
    for _ in range(max(3, min(args.steps, 10))):
        g.run()
    g.sync()
    stage_ms, runs = g.stage_times()
    split = args.run_split
    if split > 1:
        g.set_run_split(split)
        g.stage(chunks)
        for _ in range(args.warmup):
            g.run()
        g.sync()
    launches0 = g.stats()["kernel_launches"]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(args.steps):
            g.run()
        ev1.record(stream)
    g.sync()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = g.stats()["kernel_launches"] - launches0
    g.fetch(copy=False)                                 # untimed: pinned result buffers get allocated
    st0 = g.stats()
    holder = {}
    d2h_ms = device_ms(lambda: holder.__setitem__("b", g.fetch(copy=False)))
    st1 = g.stats()
    d2h_leg_bytes = st1["d2h_bytes"] - st0["d2h_bytes"]
    raw_blocks = holder["b"]
    alg_bytes = st1["algorithmic_bytes"] - st0["algorithmic_bytes"]        # input bytes consumed + output bytes produced, one pass
    out_bytes = sum(int(b.meta_size + b.dna_size + b.qua_size + b.head_size) for b in raw_blocks)
    payload_bytes = sum(int(b.dna_size + b.qua_size + b.head_size) for b in raw_blocks)
    n_bins = sum(int(b.n_bins) for b in raw_blocks)
    ms_per_step = ms_total / args.steps
    n_all = sharding.sum_over_ranks(float(n_rank), device="cuda")           # records of the whole job
    value = mates * n_all / (ms_per_step / 1e3)

    # ---- parity: whole chunks of the resident run against the compiled reference -------------------------------------
    O = oracle()
    kind = "ref" if O.have_reference() else "orc"
    pick = sorted({len(chunks) - 1, len(chunks) // 2} if args.parity_chunks >= 2 else ({len(chunks) - 1} if args.parity_chunks == 1 else set()))
    ok, detail = True, ""
    t0 = time.time()
    from concurrent.futures import ThreadPoolExecutor

    def check(ci):
        got = N.block_to_dict(raw_blocks[ci])
        O.assert_blocks_equal(got, O.bin_chunk(kind, params, chunks[ci]), f"rank {rank} chunk {ci}")
    try:
        with ThreadPoolExecutor(max_workers=max(1, len(pick))) as ex:
            list(ex.map(check, pick))
    except AssertionError as e:
        ok, detail = False, str(e)
    parity_s = time.time() - t0
    all_ok = sharding.sum_over_ranks(0.0 if ok else 1.0, device="cuda") == 0.0
    checked = int(sharding.sum_over_ranks(float(len(pick)), device="cuda"))
    checked_records = int(sharding.sum_over_ranks(float(sum(int(chunks[ci].n_records) for ci in pick)), device="cuda"))
    if not ok:
        log(f"[rank {rank}] PARITY FAILURE: {detail}")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, raw_blocks)
    del raw_blocks, holder

    # ---- end to end through the C ABI with host buffers -----------------------------------------------
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    blocks_c = (N.FsbBlock * len(chunks))()
    g._check(lib.fsb_bin_chunks(g._ctx, g._chunk_array(chunks), len(chunks), blocks_c))   # untimed pass: pinned result buffers get allocated
    st0 = g.stats()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        arr = g._chunk_array(chunks)
        blocks_c = (N.FsbBlock * len(chunks))()
        g._check(lib.fsb_bin_chunks(g._ctx, arr, len(chunks), blocks_c))
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    st1 = g.stats()
    e2e_value = mates * n_all * e2e_steps / e2e_s
    h2d = (st1["h2d_bytes"] - st0["h2d_bytes"]) // e2e_steps
    d2h = (st1["d2h_bytes"] - st0["d2h_bytes"]) // e2e_steps
    # the same call with the chunks handed over as text alone: the library parses them on the device (no record tables over PCIe)
    dp = None
    if w.get("keep_comments", True) and bool(w["params"].get("reads_have_headers", True)):
        text_chunks = []
        for t1, t2, r1, r2 in keep:
            text_chunks.append(N.make_chunk(t1, None, t2))
        blocks_c = (N.FsbBlock * len(chunks))()
        g._check(lib.fsb_bin_chunks(g._ctx, g._chunk_array(text_chunks), len(chunks), blocks_c))     # untimed pass: parse buffers get allocated
        n_parsed = sum(int(b.n_records) for b in blocks_c)
        st2 = g.stats()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            blocks_c = (N.FsbBlock * len(chunks))()
            g._check(lib.fsb_bin_chunks(g._ctx, g._chunk_array(text_chunks), len(chunks), blocks_c))
        torch.cuda.synchronize()
        dp_s = max_over_ranks(time.perf_counter() - t0)
        barrier()
        st3 = g.stats()
        dp = {"value": mates * n_all * e2e_steps / dp_s, "unit": UNIT, "ms_per_step": 1e3 * dp_s / e2e_steps,
              "h2d_bytes_per_step": int((st3["h2d_bytes"] - st2["h2d_bytes"]) // e2e_steps), "records_parsed_equal_tables": bool(n_parsed == n_rank),
              "what": "fsb_bin_chunks with fsb_chunk.records == NULL: FASTQ text in, parsed on the device (parse.cuh), blocks out"}
    clocks = sampler.stop() if rank == 0 else None       # sampled through the timed regions (resident steps and end-to-end steps)

    # ---- roofline -----------------------------------------------------------------------------------------
    peak, peak_src = load_peaks()
    per_stage = {k: v / max(runs, 1) for k, v in stage_ms.items()}
    dom = max(per_stage, key=lambda k: per_stage[k])
    dom_ms = per_stage[dom]
    if not dom_ms > 0:                                 # no per-stage times (should not happen): the line must still come out
        dom, dom_ms = "whole path (per-stage times missing)", ms_per_step
    alg_in = alg_bytes - out_bytes
    # bytes each big kernel moves by itself, algorithmically (DESIGN.md 5): K1 consumes the input and produces the slot
    # payload (the dna / qua / head bits in stored form) + key and card; K4 consumes that payload and produces the streams
    own = {"ingest": alg_in + payload_bytes + 12 * n_rank, "place": payload_bytes + 8 * n_rank + out_bytes}
    traffic, traffic_src = None, None
    try:                                               # dram__bytes_read + write per record of the dominant kernel, from the committed ncu capture
        tj = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        if name in ("c2", "c3") and dom in tj["bytes_per_pair"]:
            traffic = tj["bytes_per_pair"][dom] * n_rank
            traffic_src = tj.get("source", "profiles/traffic.json")
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": dom, "achieved": alg_bytes / (dom_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": alg_bytes / (dom_ms / 1e3) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes,
            "kernel_own_bytes": own.get(dom), "kernel_own_frac": (own[dom] / (dom_ms / 1e3) / 1e9 / peak) if dom in own else None,
            "whole_path_achieved": alg_bytes / (ms_per_step / 1e3) / 1e9,
            "whole_path_frac": alg_bytes / (ms_per_step / 1e3) / 1e9 / peak,
            "stage_ms": per_stage, "stage_ms_note": "stages of an unsplit pass (one stream); ms_per_step is the timed run with run_split sub-batches"}

    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if "shards" in w else "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": config_dict(w, name, world, n_rank, len(chunks), n_all),
                "value_is": "resident: chunks already in HBM, kernels only (no copies, no host parsing); e2e is the headline",
                "records_per_sec": value / mates, "bins_per_step_per_gpu": n_bins, "output_bytes_per_gpu": out_bytes,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                        "h2d_ms": h2d_ms, "h2d_gbs": h2d_leg_bytes / (h2d_ms / 1e3) / 1e9, "kernel_ms": ms_per_step, "d2h_ms": d2h_ms,
                        "d2h_gbs": d2h_leg_bytes / (d2h_ms / 1e3) / 1e9,
                        "device_parse": dp,
                        "legs": "h2d_ms = fsb_stage alone (copies + input check), kernel_ms = fsb_run alone, d2h_ms = fsb_fetch alone, per rank shard, "
                                "max over ranks; ms_per_step = the pipelined fsb_bin_chunks call"},
                "input_check": {"ms": check_ms, "in_timed_region": "e2e yes (inside fsb_bin_chunks); value no (fsb_stage, before the resident steps)",
                                "kernels": "stage_stats_kernel + validate_text_kernel"},
                "parity": {"ok": bool(all_ok) if checked else None, "chunks_checked": checked, "records_checked": checked_records,
                           "against": "oracle/_ref (compiled reference Categorize+PackToBins)" if kind == "ref" else "oracle C port",
                           "what": "streams, descriptors and per-read (signature, position, flags) of whole chunks of the resident run, bit for bit",
                           "seconds": round(parity_s, 1)},
                "run_split": split, "gpu_launches": int(launches), "roofline": roof, "clocks": clocks}
        if world == 1 and not args.no_cpu:
            threads = host_threads()
            sample, n = cpu_sample(chunks, threads)
            once = O.time_bin_chunk(kind, params, sample, threads, 1)            # calibration pass
            reps = int(max(1, min(200, round(12.0 / max(once, 1e-3)))))          # about 12 s of work on all cores
            secs = O.time_bin_chunk(kind, params, sample, threads, reps)
            line["cpu_baseline"] = {"value": mates * n * reps / secs, "unit": UNIT, "cores": threads,
                                    "kind": "reference" if kind == "ref" else "port",
                                    "sample": f"{n} records of chunk 0 x {reps} passes, Categorize+PackToBins, {threads} threads "
                                              f"(one slice per thread like fastore_bin -t{threads}), {secs:.1f} s"}
    g.close()
    for p in keep_ptrs:
        lib.fsb_host_free(p)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)
    if not all_ok:
        log("bench.py: parity check failed -- the numbers above are void")
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto"] + sorted(WORKLOADS),
                    help="auto: configs[1] (c2) on one GPU, configs[2] (c3: 100 M pairs over the ranks) on several")
    ap.add_argument("--total-records", "--total-pairs", "--pairs", dest="total_records", type=int, default=0,
                    help="override the workload's record count (c3: total over all ranks; others: per rank)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--run-split", type=int, default=int(os.environ.get("FSB_BENCH_SPLIT", "2")),
                    help="sub-batches fsb_run overlaps on two streams in the timed resident steps (FSB_OPT_RUN_SPLIT; 1 = one pass on one stream)")
    ap.add_argument("--parity-chunks", type=int, default=1, help="whole chunks per rank compared with the compiled reference (1 or 2)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's chunks) to DIR/*.npy: sizes, digests and a seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    name = args.config
    if name == "auto":
        name = "c3" if max(world, args.gpus) > 1 else "c2"
    w = WORKLOADS[name]
    if args.warmup < 3 and args.impl == "b200":
        log("note: the timing rules ask for >= 3 warm-up steps")
    if args.impl == "reference":
        return run_reference_arm(args, w, name)
    return run_b200_arm(args, w, name)


if __name__ == "__main__":
    sys.exit(main())
