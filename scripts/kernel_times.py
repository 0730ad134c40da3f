"""Per-kernel device times of one resident step of a bench workload, from torch.profiler (GPU box).

    python scripts/kernel_times.py [--config c2] [--run-split 1] [--root DIR]

The step runs unsplit by default, so that every launch of a pass is one sub-batch's kernel over the whole batch.
Prints one JSON line: per kernel, its device time in us for every launch of the profiled step, in launch order.
--root loads the package (and its built library) from another tree, to compare two builds on one GPU.
"""
import argparse
import json
import re
import sys
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--config", default="c2")
ap.add_argument("--run-split", type=int, default=1)
ap.add_argument("--root", default=str(Path(__file__).resolve().parent.parent))
args = ap.parse_args()
sys.path.insert(0, args.root)
sys.dont_write_bytecode = True

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
from fastore_b200 import _native as N  # noqa: E402
from fastore_b200.binner import GpuBinner  # noqa: E402

w = bench.WORKLOADS[args.config]
lib = N.cuda_lib()
keep = []
chunks, _ = bench.workload_chunks(w, bench.rank_shards(w, 0, 1, w["n"]), pinned=True, lib=lib, keep=keep, threads=16)
stream = torch.cuda.Stream()
g = GpuBinner(bench.make_params(w), device=0, stream=stream.cuda_stream, run_split=args.run_split)
g.stage(chunks)
for _ in range(3):
    g.run()
g.sync()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    g.run()
    g.sync()
g.close()

times = {}
for ev in sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start):
    m = re.search(r"(\w+)(<[^(]*>)?\(", ev.name)
    name = m.group(1) if m else ev.name
    times.setdefault(name, []).append(round(ev.time_range.end - ev.time_range.start, 1))
print(json.dumps({"config": args.config, "run_split": args.run_split, "root": Path(args.root).name, "gpu": torch.cuda.get_device_name(0),
                  "kernels_us": times}))
