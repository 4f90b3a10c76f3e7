"""What a wide action chunk costs: the split-precision mode (bf16x3) against the fp32 FFMA path at A = horizon_steps x action_dim in
{24, 56, 128} (walker2d's chunk, a robomimic-transport-sized one, the widest the tensor path covers), H = 512, Hc = 256, T = 20, K = 10:
  * one 50 000-row PPO update (AdamW applied),
  * the log-prob forward pass over the same 50 000 rows,
  * the 18 944-row (148 x 128) sampler.
Median of 7 timed blocks (CUDA events), after warm-up; the card's name and power limit are printed with the numbers.
    python tools/wide_actions_time.py [output.json]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from oracle import dppo_oracle as O  # noqa: E402
from helpers import make_engine  # noqa: E402
from diffusionpolicyoptimization_b200 import _lib as L  # noqa: E402

SHAPES = {24: dict(action_dim=6, horizon_steps=4, obs_dim=17), 56: dict(action_dim=14, horizon_steps=4, obs_dim=59),
          128: dict(action_dim=16, horizon_steps=8, obs_dim=59)}
MODES = {"bf16x3": L.PREC_BF16X3, "fp32": L.PREC_FP32}
N_PPO, B_SAMPLE = 50000, 148 * 128


def timeit(fn, iters, warm=3, blocks=7):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(blocks):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / iters)
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def main():
    if not torch.cuda.is_available():
        sys.exit("wide_actions_time.py: no CUDA device")
    out = {"card": card(), "rows_ppo": N_PPO, "rows_sample": B_SAMPLE, "results": []}
    print(f"card, power limit: {out['card']}", flush=True)
    for A, dims in SHAPES.items():
        o = O.make_oracle("hopper", seed=0, **dims)
        b = O.make_ppo_batch(o, N_PPO, pool=2048, seed=1)
        args = [x.cuda() for x in b]
        for i in (0, 1, 2, 7):
            args[i] = args[i].reshape(N_PPO, -1).contiguous()
        obs = torch.rand(B_SAMPLE, o.d.Do, device="cuda") * 2 - 1
        row = {"A": A, **dims}
        for mode, prec in MODES.items():
            e = make_engine(o, precision=prec)
            slow = mode == "fp32"
            tc0 = e.tc_launch_count()
            ppo = timeit(lambda: e.ppo_step(*args, lr=1e-6, apply=True), iters=2 if slow else 10)
            lp = timeit(lambda: e.logprobs_subsample(args[0], args[1], args[2], args[3]), iters=3 if slow else 10)
            smp = timeit(lambda: e.sample(obs, seed=1, offset=2), iters=2 if slow else 5, warm=2)
            row[mode] = {"ppo_ms": ppo[0], "ppo_min_ms": ppo[1], "logprobs_ms": lp[0], "logprobs_min_ms": lp[1],
                         "sample_ms": smp[0], "sample_min_ms": smp[1], "sample_path": e.last_path(),
                         "tc_launches": e.tc_launch_count() - tc0}
            print(f"A={A:3d} {mode:6s}: PPO update {ppo[0]:8.3f} ms  log-probs {lp[0]:8.3f} ms  sampler {smp[0]:8.3f} ms "
                  f"(path {e.last_path()}, tcgen05 launches {row[mode]['tc_launches']})", flush=True)
            e.close()
        for k in ("ppo", "logprobs", "sample"):
            row[f"speedup_{k}"] = row["fp32"][f"{k}_ms"] / row["bf16x3"][f"{k}_ms"]
        print(f"A={A:3d} fp32 / bf16x3: PPO {row['speedup_ppo']:.1f}x  log-probs {row['speedup_logprobs']:.1f}x  "
              f"sampler {row['speedup_sample']:.1f}x", flush=True)
        out["results"].append(row)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
