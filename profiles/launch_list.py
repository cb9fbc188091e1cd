"""Launch list of a bench.py run from torch.profiler (CUDA activities): per kernel its calls and median time, and
for each pair of kernels that follow each other the median gap from the end of the first to the start of the
second (negative: the second was running before the first ended, i.e. an overlapped launch).

    python profiles/launch_list.py OUT.csv -- [bench.py arguments]      e.g. -- --kernel-only --steps 50
"""
import csv
import os
import re
import runpy
import statistics
import sys

import torch
from torch.autograd import DeviceType


def main():
    out, rest = sys.argv[1], sys.argv[sys.argv.index("--") + 1:]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.argv = [os.path.join(root, "bench.py")] + rest
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        try:
            runpy.run_path(sys.argv[0], run_name="__main__")
        except SystemExit as e:
            if e.code not in (None, 0):
                raise
    ks = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA and "memcpy" not in e.name.lower()
                 and "memset" not in e.name.lower()), key=lambda e: e.time_range.start)
    def short(name):   # "void (anonymous namespace)::scan_kernel<...>(...)" -> scan_kernel
        return next((w for w in re.findall(r"([A-Za-z_]\w*)\s*[<(]", name) if w != "void"), name)

    dur, gap = {}, {}
    for a, b in zip(ks, ks[1:]):
        gap.setdefault((short(a.name), short(b.name)), []).append(b.time_range.start - a.time_range.end)
    for e in ks:
        dur.setdefault(short(e.name), []).append(e.time_range.end - e.time_range.start)
    with open(out, "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(["kind", "kernel", "next", "count", "median_us", "min_us", "max_us"])
        for k, v in sorted(dur.items(), key=lambda kv: -sum(kv[1])):
            w.writerow(["kernel", k, "", len(v), f"{statistics.median(v):.2f}", f"{min(v):.2f}", f"{max(v):.2f}"])
        for (a, b), v in sorted(gap.items(), key=lambda kv: -len(kv[1])):
            if len(v) >= 5:
                w.writerow(["gap", a, b, len(v), f"{statistics.median(v):.2f}", f"{min(v):.2f}", f"{max(v):.2f}"])
    print(open(out).read())


if __name__ == "__main__":
    main()
