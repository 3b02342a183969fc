"""Per-kernel device times of eager bench steps under torch.profiler, with the card name and power limit.

    python tools/kernel_table.py ea_128k knorm_128k streaming_128k

KVPRESS_B200_LIB selects the library. Kernels launched with PDL become resident before the kernel in front of them has
finished, so their spans overlap; `after prev` is a kernel's end minus the previous kernel's end, i.e. its time on the
critical path. `GB/s` is given for the compaction kernels: compulsory bytes (read and write every kept K and V row
once) over `after prev`."""
import os
import subprocess
import sys
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torch.autograd import DeviceType  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
from kvpress_b200 import native  # noqa: E402

STEPS = 20
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), "| lib:", native.library_path().name, flush=True)
native.load()
for wl in sys.argv[1:] or ["ea_128k", "knorm_128k"]:
    w = bench.WORKLOADS[wl]
    K, V, extra = bench.make_inputs(w, "cuda:0", 1)
    n_kept = w.get("n_kept") or bench.kept_count(w["S"], w["ratio"])
    for _ in range(5):
        bench.run_native(w, K, V, extra, n_kept)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(STEPS):
            bench.run_native(w, K, V, extra, n_kept)
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start)
    span, crit, count = defaultdict(float), defaultdict(float), defaultdict(int)
    prev_end = None
    for e in evs:
        name = e.name.split("(")[0].split("<")[0].replace("void ", "").replace("kvp::", "")[:40]
        span[name] += e.time_range.elapsed_us()
        end = e.time_range.end
        crit[name] += end - max(prev_end, e.time_range.start) if prev_end is not None else e.time_range.elapsed_us()
        count[name] += 1
        prev_end = end if prev_end is None else max(prev_end, end)
    row_bytes = w["D"] * 2
    rows = w.get("B", 1) * w["Hkv"]
    copy_bytes = 4 * row_bytes * n_kept * rows
    print(f"{wl}: {STEPS} eager steps, us per step")
    print(f"  {'kernel':40s} {'calls':>5s} {'span':>8s} {'after prev':>10s} {'GB/s':>7s}")
    for name in sorted(span, key=lambda n: -crit[n]):
        rate = ""
        if "compact" in name and crit[name] > 0:
            rate = f"{copy_bytes / (crit[name] / STEPS * 1e-6) / 1e9:7.0f}"
        print(f"  {name:40s} {count[name] / STEPS:5.1f} {span[name] / STEPS:8.1f} {crit[name] / STEPS:10.1f} {rate:>7s}".rstrip())
    del K, V, extra
    torch.cuda.empty_cache()
