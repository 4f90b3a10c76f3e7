"""Per-kernel timeline of PPO updates at bench shapes from torch.profiler (CUDA activities).

usage: python tools/prof_update.py [bf16x3|bf16|fp32] [rows] [updates] [out.json]

Runs the updates the way bench.py's `value` does (resident minibatch, global advantage statistics, L2 flushed between
updates), profiles the last `updates` of them in a run of their own, and prints for the last one every kernel in launch
order: stream, start relative to the update's first kernel, duration and the idle gap before it (the time since the
latest end of any earlier kernel of the update).  The flush kernel between updates delimits them.  With a fourth argument
the per-update rows are also written as JSON.
"""
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from torch.profiler import ProfilerActivity, profile

import bench
from diffusionpolicyoptimization_b200 import _lib as L
from diffusionpolicyoptimization_b200.parallel import advantage_stats

mode = sys.argv[1] if len(sys.argv) > 1 else "bf16x3"
N = int(sys.argv[2]) if len(sys.argv) > 2 else 50000
nup = int(sys.argv[3]) if len(sys.argv) > 3 else 3
out_json = sys.argv[4] if len(sys.argv) > 4 else None

e = bench.make_gpu_engine({"bf16x3": L.PREC_BF16X3, "bf16": L.PREC_BF16, "fp32": L.PREC_FP32}[mode], 0)
b = bench.make_gpu_batches(e, N, 1, seed=10)[0]
st = advantage_stats(b[6].cpu().numpy())
flush = torch.empty(256 << 20, dtype=torch.uint8, device=e.dev)


def step():
    e.ppo_step(*b, lr=1e-4, apply=True, n_global=N, adv_mean=st[0], adv_std=st[1])


for _ in range(5):
    step()
torch.cuda.synchronize()
l0 = e.launch_count()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(nup):
        flush.zero_()
        step()
    torch.cuda.synchronize()
launches = (e.launch_count() - l0) / nup

with tempfile.TemporaryDirectory() as td:
    path = os.path.join(td, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        trace = json.load(f)
kern = sorted((ev for ev in trace["traceEvents"] if ev.get("cat") == "kernel"), key=lambda ev: ev["ts"])
updates, cur = [], None
for ev in kern:
    if "FillFunctor" in ev["name"]:            # flush.zero_() between updates
        cur = []
        updates.append(cur)
        continue
    if cur is not None:
        cur.append(ev)


def short(name):
    name = name.replace("void ", "")
    return name if len(name) <= 60 else name[:57] + "..."


rows_all = []
for u in updates:
    t0 = u[0]["ts"]
    end, rows = t0, []
    for ev in u:
        gap = max(0.0, ev["ts"] - end)
        rows.append({"kernel": short(ev["name"]), "stream": ev["args"].get("stream"), "start_us": ev["ts"] - t0, "dur_us": ev["dur"], "gap_us": gap})
        end = max(end, ev["ts"] + ev["dur"])
    rows_all.append({"rows": rows, "span_us": end - t0, "busy_us": sum(r["dur_us"] for r in rows),
                     "gap_us": sum(r["gap_us"] for r in rows), "kernels": len(rows)})

print(f"{torch.cuda.get_device_name(0)}; mode {mode}, {N} rows; {launches:.1f} library launches per update (launch counter)")
for k, u in enumerate(rows_all):
    print(f"update {k}: {u['kernels']} kernels, first start to last end {u['span_us']:.1f} us, "
          f"kernel time {u['busy_us']:.1f} us, idle gaps {u['gap_us']:.1f} us")
last = rows_all[-1]
print(f"\nlast update in launch order (us):\n{'kernel':<62}{'stream':>7}{'start':>9}{'dur':>8}{'gap':>7}")
for r in last["rows"]:
    print(f"{r['kernel']:<62}{r['stream']:>7}{r['start_us']:>9.1f}{r['dur_us']:>8.1f}{r['gap_us']:>7.1f}")
if out_json:
    with open(out_json, "w") as f:
        json.dump({"device": torch.cuda.get_device_name(0), "mode": mode, "rows": N, "launches_per_update": launches, "updates": rows_all}, f, indent=1)
e.close()
