"""Per-kernel CUDA time of a short bench.py run (--steps 1 --warmup 1, all of its legs), from torch.profiler CUDA activities.  Prints one
line per kernel: total ms and calls, largest first; a kernel's share of one pipeline pass is its total over the pass count.  Usage: python tools/kernel_times.py [extra bench.py args]"""
import os
import runpy
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

if __name__ == "__main__":
    os.chdir(ROOT)
    sys.path.insert(0, ROOT)
    sys.argv = ["bench.py", "--gpus", "1", "--steps", "1", "--warmup", "1", "--no-cpu-baseline"] + sys.argv[1:]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        try:
            runpy.run_path(os.path.join(ROOT, "bench.py"), run_name="__main__")
        except SystemExit as e:
            if e.code not in (None, 0):
                raise
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            rows.append((t / 1e3, ev.count, ev.key))
    rows.sort(reverse=True)
    print("%10s %8s  %s" % ("ms", "calls", "kernel"))
    for ms, n, name in rows:
        print("%10.3f %8d  %s" % (ms, n, name[:140]))
