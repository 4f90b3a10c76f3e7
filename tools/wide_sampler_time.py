"""What the small-batch rollout sampler costs for wide action chunks: the persistent cluster kernel (path 1) against the
layer-by-layer fp32 sampler (path 2, forced), alternating block by block, at A = horizon_steps x action_dim in {24, 56, 112, 128}
(walker2d's chunk, robomimic-transport-sized ones, the widest the cluster kernel covers), H = 512, T = 20, K = 10:
  * `sample` and `rollout_step` (normalise kernel + sampler with the un-normalising epilogue) for B in {40, 50} env rows
    (the gym configs' n_envs, robomimic's), in the fp32 and bf16x3 modes (below 2048 rows both sample with the same fp32 kernels);
  * `sample` in the fp32 mode for B up to 4096 rows (dppo_sample's row limit for the cluster path), where the layered path's
    SGEMM tiles fill up.
Median and min of 7 timed blocks of 20 calls (CUDA events), after warm-up; the card's name and power limit are printed with them.
    python tools/wide_sampler_time.py [output.json]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import dppo_oracle as O  # noqa: E402
from helpers import make_engine  # noqa: E402
from diffusionpolicyoptimization_b200 import _lib as L  # noqa: E402

SHAPES = {24: dict(action_dim=6, horizon_steps=4, obs_dim=17), 56: dict(action_dim=14, horizon_steps=4, obs_dim=59),
          112: dict(action_dim=14, horizon_steps=8, obs_dim=59), 128: dict(action_dim=16, horizon_steps=8, obs_dim=59)}
MODES = {"fp32": L.PREC_FP32, "bf16x3": L.PREC_BF16X3}
ENVS = (40, 50)
SWEEP = (128, 256, 512, 1024, 2048, 4096)
ITERS, BLOCKS = 20, 7


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def alternate(e, fn, iters):
    """{path: (median, min)} in microseconds per call, the two paths timed in alternating blocks."""
    ts = {1: [], 2: []}
    for path in (1, 2):
        e.force_path(path)
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        if e.last_path() != path:
            sys.exit(f"wide_sampler_time.py: asked for path {path}, ran {e.last_path()}")
    for _ in range(BLOCKS):
        for path in (1, 2):
            e.force_path(path)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            torch.cuda.synchronize()
            ts[path].append(a.elapsed_time(b) / iters * 1e3)
    e.force_path(0)
    return {p: (sorted(v)[len(v) // 2], min(v)) for p, v in ts.items()}


def main():
    if not torch.cuda.is_available():
        sys.exit("wide_sampler_time.py: no CUDA device")
    out = {"card": card(), "iters": ITERS, "blocks": BLOCKS, "results": []}
    print(f"card, power limit: {out['card']}", flush=True)

    def report(A, mode, call, B, r, T):
        (c_med, c_min), (l_med, l_min) = r[1], r[2]
        row = dict(A=A, mode=mode, call=call, B=B, cluster_med_us=c_med, cluster_min_us=c_min, layered_med_us=l_med,
                   layered_min_us=l_min, speedup=l_med / c_med, cluster_us_per_denoising_step=c_med / T)
        out["results"].append(row)
        print(f"A={A:3d} {mode:6s} {call:12s} B={B:4d}: cluster {c_med:8.1f} us (min {c_min:8.1f})  layered {l_med:8.1f} us "
              f"(min {l_min:8.1f})  speed-up {l_med / c_med:5.2f}x  cluster per denoising step {c_med / T:5.2f} us", flush=True)

    for A, dims in SHAPES.items():
        o = O.make_oracle("hopper", seed=0, **dims)
        d, T = o.d, o.d.denoising_steps
        for mode, prec in MODES.items():
            e = make_engine(o, prec)
            Bmax = max(ENVS + (SWEEP if mode == "fp32" else ()))
            rng = np.random.default_rng(0)
            obs_all = torch.from_numpy(rng.uniform(-1, 1, (Bmax, d.obs_dim)).astype(np.float32)).cuda()
            act_all = torch.empty(Bmax, d.A, device="cuda"); ch_all = torch.empty(Bmax, d.ft_denoising_steps + 1, d.A, device="cuda")
            e.set_env_normalization(-np.ones(d.obs_dim, np.float32) * 2, np.ones(d.obs_dim, np.float32) * 3,
                                    -np.ones(d.action_dim, np.float32), np.ones(d.action_dim, np.float32))
            for B in ENVS + (SWEEP if mode == "fp32" else ()):
                obs, act, ch = obs_all[:B], act_all[:B], ch_all[:B]
                r = alternate(e, lambda: e.sample(obs, seed=1, offset=2, actions_out=act, chains_out=ch), ITERS if B <= 1024 else 5)
                report(A, mode, "sample", B, r, T)
                if B in ENVS:
                    raw_obs = torch.from_numpy(rng.uniform(-2, 3, (B, d.obs_dim))).pin_memory()
                    raw_act = torch.zeros(B, d.action_dim).pin_memory()
                    obs_out = torch.empty(B, d.obs_dim, device="cuda")
                    r = alternate(e, lambda: e.rollout_step(raw_obs, obs_out, act, ch, raw_act, 1, seed=1, offset=2), ITERS)
                    report(A, mode, "rollout_step", B, r, T)
            e.close()
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
