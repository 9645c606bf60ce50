"""Per-kernel device time of the bench.py workload (PageRank, RMAT scale-24 ef-16, 100 iterations, graph stored transposed)
under torch.profiler with CUDA activities.  Run it in a process of its own: tracing slows the host, so its step time is
not a bench number.

    python scripts/profile_iteration.py [--root TREE] [--scale 24] [--steps 2] [--out DIR]

--root imports cugraph_b200 from another checkout (to profile two builds with one script).  Prints (and, with --out,
writes to DIR/profile_<label>.txt) the device time per kernel name summed over the profiled steps, divided by the
iterations run.
"""
import argparse
import os
import re
import sys
from collections import defaultdict

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--scale", type=int, default=24)
ap.add_argument("--steps", type=int, default=2)
ap.add_argument("--out", default=None)
ap.add_argument("--label", default="current")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402
from cugraph_b200 import pylibcugraph as plc  # noqa: E402
from cugraph_b200.generators import rmat_edgelist  # noqa: E402

ITERS = 100
src, dst = rmat_edgelist(args.scale, 16 << args.scale, seed=0)
h = plc.ResourceHandle()
G = plc.SGGraph(h, plc.GraphProperties(is_symmetric=False, is_multigraph=True), src, dst, store_transposed=True, renumber=True)
del src, dst


def step():
    return plc.pagerank(h, G, None, None, None, None, 0.85, 0.0, ITERS, False, fail_on_nonconvergence=False)


step()  # the first call builds the piece stream and the out-weights
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()

per_kernel = defaultdict(lambda: [0.0, 0])
first, last = None, None
for ev in prof.events():
    if ev.device_type != torch.autograd.DeviceType.CUDA:
        continue
    m = re.search(r"\b(k_\w+)", ev.name)  # the kernel's name without namespace, template arguments and parameters
    name = m.group(1) if m else ev.name
    t0, t1 = ev.time_range.start, ev.time_range.end
    per_kernel[name][0] += t1 - t0
    per_kernel[name][1] += 1
    first = t0 if first is None else min(first, t0)
    last = t1 if last is None else max(last, t1)

iters = ITERS * args.steps
props = torch.cuda.get_device_properties(0)
lines = [f"device: {props.name}; {args.steps} PageRank calls x {ITERS} iterations, RMAT scale-{args.scale} ef-16 "
         f"({args.label})",
         f"span of the traced kernels: {(last - first) / 1e3:.3f} ms ({(last - first) / iters:.2f} us per iteration)",
         f"{'kernel':<48} {'launches/it':>11} {'us/it':>9} {'us/launch':>10}"]
busy = 0.0
for name, (us, n) in sorted(per_kernel.items(), key=lambda kv: -kv[1][0]):
    busy += us
    lines.append(f"{name[:48]:<48} {n / iters:>11.2f} {us / iters:>9.2f} {us / n:>10.2f}")
lines.append(f"{'sum of kernel time':<48} {'':>11} {busy / iters:>9.2f}")
text = "\n".join(lines)
print(text, flush=True)
if args.out:
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, f"profile_{args.label}.txt"), "w") as f:
        f.write(text + "\n")
