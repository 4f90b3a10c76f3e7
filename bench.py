#!/usr/bin/env python
"""bench.py — DPPO hot path on B200 (SURVEY.md §8d, BASELINE.json).

Workload (N=1 default = BASELINE.json configs[1]): walker2d-v2 ft_ppo_diffusion_mlp shapes
(obs 17, act 6, horizon 4, T=20, K=10).  One "step" = one PPO minibatch update of 50 000
(env-step, k) rows PER GPU: log-prob forward of the stored denoising chains under the current
weights, clipped-ratio + value loss, backward, (N>1: one all-reduce of grads+metrics), AdamW.
`value` = PPO log-prob-update samples/s over all ranks (weak scaling).  The other half of the
metric — denoised action chunks/s of the T=20 chain at 40 env copies — is measured in the same
run and reported under "sampling" (it is dependency-latency-bound, not a throughput kernel).

Precision: the headline (`value`, `e2e`, `roofline`) is the fp32-FAITHFUL tensor-core mode `bf16x3` (tcgen05; every operand
as two 16-bit planes (fp16 in the forward pass, bf16 behind it), every product as the sum of exact plane products, fp32 accumulation: it meets north_star's fp32 tolerance,
tests/test_gpu_fullsize_oracle.py), i.e. the reference's own precision.  The faster plain-bf16 tensor mode (looser stated
bounds) and the CUDA-core FFMA mode are measured in the same run and reported under "bf16_mode" / "fp32_ffma_mode".
`--precision bf16|fp32` makes one of those the headline instead.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16x3|bf16|fp32] [--scaling weak|strong]
                  [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

TASK = "walker2d"
N_ROWS = 50_000            # minibatch rows per GPU (cfg train.batch_size, ft_ppo_diffusion_mlp.yaml:69)
N_ENVS = 40                # env copies per rollout step (ft_ppo_diffusion_mlp_run.yaml:26)
METRIC = "ppo_logprob_update_samples_per_sec"
UNIT = "samples/s"
PATHS = {1: "persistent cluster kernel (fp32 FFMA, DSMEM)", 2: "layered fp32", 3: "layered tcgen05", 4: "fused tcgen05 chain (one launch, T steps on chip)"}
WORKLOAD = (f"{TASK}-v2 ft_ppo_diffusion_mlp PPO update: {N_ROWS} (env-step,k) rows per step "
            "(obs 17, act 6, Ta 4, T 20, K 10, actor 512x3 ReLU, critic 256x3 Mish), loss + backward + AdamW")
DTYPES = {"bf16x3": "bf16x3", "bf16": "bf16", "fp32": "fp32"}
PRECISION_NOTE = {
    "bf16x3": "tcgen05, operands as 16-bit planes (two fp16 planes = 22 bits in the actor forward, two bf16 planes elsewhere), exact plane products (3 per multiply-add), fp32 accumulate / masters / loss / AdamW: fp32-faithful (north_star tolerance)",
    "bf16": "tcgen05, bf16 operands, fp32 accumulate / masters / loss / AdamW: looser stated bounds (tests/test_gpu_bf16.py)",
    "fp32": "CUDA-core FFMA everywhere",
}
# kernel classes of the library's live profile (dppo_profile_read_class), per mode
CLASS_NAMES = {
    "bf16x3": ["tsp::pair_gemm_kernel (plane GEMMs on CTA pairs: forward / backward layers, TMA-store epilogue)",
               "tsp::dw_pair_kernel (grouped plane weight-gradient GEMMs on CTA pairs)", "sgemm_kernel", "ts::split_gemm_kernel (narrow output layers)"],
    "bf16": ["fc::chain_kernel<512> (fused tcgen05 actor forward / backward chains, CTA pairs)", "tcp::dw_pair_kernel (tcgen05 grouped split-K weight gradients on CTA pairs)",
             "sgemm_kernel", "fc::chain_kernel<256> (fused tcgen05 Mish critic forward / backward chains)"],
    "fp32": ["-", "-", "sgemm_kernel (fp32 FFMA layers + gradients)", "-"],
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ----------------------------------------------------------------------------- clocks sampler
class Clocks(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- synthetic data
DIMS = dict(obs_dim=17, action_dim=6, horizon_steps=4, cond_steps=1, denoising_steps=20, ft_denoising_steps=10,
            time_dim=16, actor_hidden=512, critic_hidden=256)


class D:
    """Shapes of the workload."""
    def __init__(self):
        self.__dict__.update(DIMS)
        self.A = self.action_dim * self.horizon_steps
        self.Do = self.obs_dim * self.cond_steps
        self.Din = self.A + self.time_dim + self.Do


def make_gpu_engine(precision, device, cond_dim=17, action_dim=6):
    """Engine with Glorot-initialised base policy, fine-tuned copy = base + 5e-3 N(0,1), random critic.
    Uses only the product package (never the oracle)."""
    import diffusionpolicyoptimization_b200 as dp
    from diffusionpolicyoptimization_b200 import _lib as L
    cfg = dp.default_cfg()
    for k in ("obs_dim", "action_dim", "horizon_steps", "cond_steps", "denoising_steps", "ft_denoising_steps", "time_dim",
              "actor_hidden", "critic_hidden"):
        setattr(cfg, k, DIMS[k])
    cfg.precision = precision
    e = dp.Engine(cfg, device)
    actor = dp.DiffusionMLP(action_dim=action_dim, horizon_steps=4, cond_dim=cond_dim, mlp_dims=[512, 512, 512], activation_type="ReLU",
                            residual_style=True, seed=0)
    critic = dp.CriticObs(cond_dim=cond_dim, mlp_dims=[256, 256, 256], residual_style=True, seed=1)
    w = actor.get_flat_weights()
    rng = np.random.default_rng(2)
    e.set_weights(L.NET_ACTOR, w)
    e.set_weights(L.NET_ACTOR_EMA, w)
    e.set_weights(L.NET_ACTOR_FT, w + 5e-3 * rng.standard_normal(w.size).astype(np.float32))
    e.set_weights(L.NET_CRITIC, critic.get_flat_weights())
    return e


def make_gpu_batches(e, n_rows, n_batches, seed):
    """SURVEY.md §8(d): a pool of stored chains produced by the sampler itself (in-kernel Philox),
    old log-probs under the pre-update (base) weights, old values from the critic; minibatch rows
    are random (env-step, k) pairs.  Everything here runs before any timed region."""
    dev, K = e.dev, e.K
    g = torch.Generator(device=dev); g.manual_seed(seed)
    P = 4096
    obs = torch.rand(P, e.Do, device=dev, generator=g) * 2 - 1
    _, chains = e.sample(obs, seed=seed, offset=1)
    oldlogp = e.logprobs(obs, chains, use_base_policy=True).reshape(P, K, e.A)
    values = e.value(obs)
    out = []
    for _ in range(n_batches):
        flat = torch.randint(0, P * K, (n_rows,), device=dev, generator=g)
        b, k = flat // K, flat % K
        out.append([obs[b].contiguous(), chains[b, k].contiguous(), chains[b, k + 1].contiguous(), k.to(torch.int32).contiguous(),
                    torch.randn(n_rows, device=dev, generator=g), (values[b] + 0.1 * torch.randn(n_rows, device=dev, generator=g)).contiguous(),
                    torch.randn(n_rows, device=dev, generator=g), oldlogp[b, k].contiguous()])
    torch.cuda.synchronize()
    return out


def flops_per_sample(d):
    Fa = 2 * (d.Din * d.actor_hidden + 2 * d.actor_hidden ** 2 + d.actor_hidden * d.A)
    Fc = 2 * (d.Do * d.critic_hidden + 2 * d.critic_hidden ** 2 + d.critic_hidden)
    return (3 * Fa - 2 * d.Din * d.actor_hidden) + (3 * Fc - 2 * d.Do * d.critic_hidden), Fa


# ----------------------------------------------------------------------------- reference arm (CPU)
def workload_config(rows_per_gpu, world, scaling):
    """The `config` both arms print (identical strings: the driver compares them)."""
    return {"workload": WORKLOAD, "rows_per_step_per_gpu": rows_per_gpu, "global_rows": rows_per_gpu * world if scaling == "weak" else N_ROWS,
            "parallelism": f"dp{world}"}


def run_reference(args):
    """The reference's CPU implementation of the path = the oracle restatement (TensorFlow is not
    installable here), all host threads, same config/metric, one full 50 000-row minibatch per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import dppo_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    o = O.make_oracle(TASK, seed=0)
    n_cpu = N_ROWS
    batch = O.make_ppo_batch(o, n_cpu, pool=512, seed=1)
    params = [p.clone() for p in o.actor_ft] + [p.clone() for p in o.critic]
    m = [torch.zeros_like(p) for p in params]; v = [torch.zeros_like(p) for p in params]
    last_metrics = [None]

    def step(i):
        oo = O.Oracle(o.d, o.h, o.actor, params[:12], params[12:])
        last_metrics[0], ga, gc = oo.ppo_grads(*batch)
        O.adamw_keras(params, ga + gc, m, v, i + 1, 1e-4, o.h.beta1, o.h.beta2, o.h.adam_eps, o.h.weight_decay)

    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    val = n_cpu * args.steps / dt
    if args.dump_outputs:
        save_outputs(args.dump_outputs, {"ppo_metrics": [float(x) for x in last_metrics[0]],
                                         "actor_ft_weights": O.flatten_params(params[:12]), "critic_weights": O.flatten_params(params[12:])})
    # sampling half of the metric on the CPU, for the "sampling" block
    obs, x_T, noise = O.make_rollout_inputs(o, N_ENVS, seed=3)
    o.sample(obs, x_T, noise)
    t1 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        o.sample(obs, x_T, noise)
    dts = (time.perf_counter() - t1) / reps
    # BASELINE.json configs[0]: the hopper shapes on the CPU
    oh = O.make_oracle("hopper", seed=0)
    obs_h, xT_h, nz_h = O.make_rollout_inputs(oh, N_ENVS, seed=3)
    oh.sample(obs_h, xT_h, nz_h)
    t2 = time.perf_counter()
    for _ in range(reps):
        oh.sample(obs_h, xT_h, nz_h)
    dth = (time.perf_counter() - t2) / reps
    bh = O.make_ppo_batch(oh, n_cpu, pool=512, seed=1)
    oh.ppo_grads(*bh)
    t3 = time.perf_counter()
    for _ in range(3):
        oh.ppo_grads(*bh)
    dtp = (time.perf_counter() - t3) / 3
    cfg = workload_config(N_ROWS, args.gpus, args.scaling)
    cfg["note"] = "oracle = torch-CPU fp32 restatement of the reference TF graph (TF not installable); runs on rank 0 only, one host"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full minibatches of {n_cpu} rows (loss + gradient + AdamW), torch {torch.get_num_threads()} threads"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "sampling": {"chunks_per_sec": N_ENVS / dts, "us_per_rollout_step": dts * 1e6, "n_envs": N_ENVS},
        "hopper": {"sampling_chunks_per_sec": N_ENVS / dth, "sampling_us_per_rollout_step": dth * 1e6, "n_envs": N_ENVS,
                   "ppo_samples_per_sec": n_cpu / dtp, "ppo_ms_per_step": dtp * 1e3, "note": "BASELINE.json configs[0] (loss + gradient, AdamW excluded)"},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm (GPU)
def traffic_from_profiles(kernel_key):
    """dram read+write bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/traffic.json,
    written by tools/ncu_traffic.py from the .ncu-rep of the same bench command)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None, None
    try:
        d = json.load(open(p))
        ent = d.get(kernel_key)
        if ent:
            return float(ent["dram_bytes_per_launch"]), f"profiles/traffic.json [{kernel_key}] <- {ent.get('source', '?')}"
    except Exception:
        pass
    return None, None


def save_outputs(out_dir, arrays):
    """--dump-outputs: what the timed PPO update hands its caller, i.e. the 8 metrics of the last timed step and the weights
    the updates left (fine-tuned actor, critic), as out_dir/<name>.npy in fp32 (about 3 MB).  Weights, batches and seeds
    are fixed, so two builds run with the same arguments can be compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def run_ours(args):
    import hashlib
    import torch.distributed as dist
    from diffusionpolicyoptimization_b200 import _lib as L
    from diffusionpolicyoptimization_b200.parallel import advantage_stats, init_process_group_from_env, shard_range

    rank, world, local = init_process_group_from_env("nccl")
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    PREC = {"bf16x3": L.PREC_BF16X3, "bf16": L.PREC_BF16, "fp32": L.PREC_FP32}
    mode = args.precision
    d = D()
    fps, Fa = flops_per_sample(d)
    pk, pk_src = peaks()
    # rows per GPU: weak scaling keeps 50 000 per rank; strong scaling shards the reference's 50 000-row minibatch
    if args.scaling == "strong":
        lo_r, hi_r = shard_range(N_ROWS, rank, world)
        rows = hi_r - lo_r
        n_global = N_ROWS
    else:
        rows = N_ROWS
        n_global = N_ROWS * world
    e = make_gpu_engine(PREC[mode], local)
    if world > 1:
        e.init_comm()

    # ---- inputs: 2 distinct minibatches per rank, pinned on the host and resident on the device
    devb = make_gpu_batches(e, rows, 2, seed=10 + rank)
    pinned = [[t.cpu().pin_memory() for t in b] for b in devb]

    def global_stats(adv):
        if world > 1:
            sizes = [shard_range(N_ROWS, r, world)[1] - shard_range(N_ROWS, r, world)[0] if args.scaling == "strong" else rows for r in range(world)]
            parts = [torch.empty(n, device=dev, dtype=adv.dtype) for n in sizes]
            dist.all_gather(parts, adv)
            return advantage_stats(torch.cat(parts).cpu().numpy())
        return advantage_stats(adv.cpu().numpy())
    # global advantage statistics (diffusion_ppo.py:74-75 normalises over the whole minibatch)
    stats = [global_stats(devb[i][6]) for i in range(2)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    lr = 1e-4
    metrics_host = torch.empty(8, dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warm):
        for i in range(warm):
            fn(i)
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            flush.zero_()                               # L2 flush between timed steps (outside the event pair)
            evs[i][0].record(); fn(warm + i); evs[i][1].record()
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def step_fn(eng):
        def f(i):
            b = devb[i & 1]; mean, std = stats[i & 1]
            return eng.ppo_step(*b, lr=lr, apply=True, n_global=n_global, adv_mean=mean, adv_std=std)
        return f

    def roofline_of(eng, md, step_ms):
        """Dominant kernel class timed live with CUDA events inside the library (every tensor-class launch is bracketed on its
        launching stream; while the profile is on, kernels that otherwise overlap on two streams run back to back)."""
        eng.profile_enable(True)
        fn = step_fn(eng)
        for i in range(args.steps):
            flush.zero_(); fn(i)
        cls = [eng.profile_read_class(c) for c in range(4)]
        execf = [eng.profile_read_exec(c) for c in range(4)]
        eng.profile_enable(False)
        names = CLASS_NAMES[md]
        dom = max(range(4), key=lambda c: cls[c][0])
        d_ms, d_n, d_fl = cls[dom]
        achieved = d_fl / (d_ms * 1e-3) / 1e12 if d_ms > 0 else 0.0
        all_ms = sum(c[0] for c in cls); all_fl = sum(c[2] for c in cls)
        traffic, tsrc = traffic_from_profiles(names[dom].split(" ")[0])
        roof = {"bound": "tensor", "achieved": achieved, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["bf16_tflops_sustained"], "traffic": traffic, "traffic_source": tsrc,
                "kernel": names[dom],
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({pk_src}); the kernel runs inside a long step",
                "avg_launch_us": d_ms / max(d_n, 1) * 1e3, "launches_timed": d_n,
                "algorithmic_flops_per_launch": d_fl / max(d_n, 1),
                "share_of_step": d_ms / args.steps / step_ms,
                # flops the tensor pipe actually issued for this kernel (padded tiles; 3 or 6 plane products per algorithmic multiply-add)
                "issued_tflops": execf[dom] / (d_ms * 1e-3) / 1e12 if d_ms > 0 else 0.0,
                "issued_frac_of_peak": (execf[dom] / (d_ms * 1e-3) / 1e12 / pk["bf16_tflops_sustained"]) if d_ms > 0 else 0.0,
                "all_tensor_kernels": {"achieved": all_fl / (all_ms * 1e-3) / 1e12 if all_ms > 0 else 0.0,
                                       "share_of_step": all_ms / args.steps / step_ms,
                                       "classes": {names[c].split(" ")[0]: {"ms_per_step": cls[c][0] / args.steps, "launches_per_step": cls[c][1] // args.steps,
                                                                            "tflops": cls[c][2] / (cls[c][0] * 1e-3) / 1e12 if cls[c][0] > 0 else 0.0}
                                                   for c in range(4) if cls[c][1] > 0}}}
        if md == "bf16x3":
            roof["note"] = ("achieved / frac count ALGORITHMIC flops (one multiply-add per weight and row of the unfolded network) against the bf16 tensor peak; "
                            "the plane arithmetic executes 3 tcgen05 products per multiply-add (two 16-bit planes per operand), so the ceiling of this mode is "
                            "1/3 of the pipe; kernels that overlap on two streams in `value` run back to back while they are timed")
        elif md == "bf16":
            roof["note"] = "per-kernel durations are timed with the actor and critic chains serialized; in `value` the critic chain overlaps the actor chain's last wave"
        else:
            ffma = eng.ffma_peak_tflops()
            roof["bound"] = "fp32-fma"; roof["peak"] = ffma; roof["frac"] = achieved / ffma if ffma > 0 else None
            roof["peak_source"] = "measured on this GPU (dppo_debug_ffma_peak: 16 independent fmaf chains per thread, 2048 threads per SM, CUDA events); derived 148 SM x 128 x 2 x 1.965 GHz = 74.5"
            roof["issued_tflops"] = None; roof["issued_frac_of_peak"] = None
            roof["note"] = "CUDA-core FFMA mode: the dominant class is sgemm_kernel (128x128x16 register tiles); frac is against the MEASURED FFMA rate"
        return roof

    clk = Clocks(local); clk.start()
    dev_step = step_fn(e)
    last_metrics = [None]

    def timed_step(i):
        last_metrics[0] = dev_step(i)
    l0 = e.launch_count()
    ms_dev = timed(timed_step, args.steps, args.warmup)
    launches = e.launch_count() - l0
    launches_per_step = launches // (args.steps + args.warmup)
    if args.dump_outputs and rank == 0:
        save_outputs(args.dump_outputs, {"ppo_metrics": last_metrics[0].cpu().numpy(), "actor_ft_weights": e.get_weights(L.NET_ACTOR_FT),
                                         "critic_weights": e.get_weights(L.NET_CRITIC)})

    # ---- e2e (a): host minibatch through dppo_ppo_step_host (H2D of the 18.6 MB minibatch + D2H of the metrics every step)
    def e2e_host_step(i):
        b = pinned[i & 1]; mean, std = stats[i & 1]
        e.ppo_step_host(*[t.numpy() for t in b], metrics_host.numpy(), lr=lr, apply=True, n_global=n_global, adv_mean=mean, adv_std=std)
    ms_e2e_host = timed(e2e_host_step, args.steps, max(3, args.warmup // 2))
    # the same host buffers copied to the device with nothing else running: the host-link floor of that call on this box
    h2d_dst = [torch.empty_like(t, device=dev) for t in pinned[0]]

    def h2d_only(i):
        for hb, db in zip(pinned[i & 1], h2d_dst):
            db.copy_(hb, non_blocking=True)
    ms_h2d = timed(h2d_only, args.steps, 2)
    del h2d_dst
    # ---- e2e (b), the headline `e2e`: the index-driven entry point = the reference's own data flow (train_ppo_diffusion_agent.py
    #      :266-312): the rollout of an iteration (P = 500 steps x 40 envs chains, old log-probs, returns/values/advantages) is uploaded
    #      from pinned host memory once per 20 minibatch updates (update_epochs 5 x 4 minibatches) and stays resident; every step
    #      copies its shuffled flat indices in and the 8 metrics out.  The upload is inside the timed region.
    P_roll, K = 20000, d.ft_denoising_steps
    g2 = torch.Generator(device=dev); g2.manual_seed(99 + rank)
    obs_r = torch.rand(P_roll, d.Do, device=dev, generator=g2) * 2 - 1
    _, chains_r = e.sample(obs_r, seed=5, offset=7)
    olp_r = e.logprobs(obs_r, chains_r, use_base_policy=True).reshape(P_roll, K, d.A)
    val_r = e.value(obs_r)
    roll_host = [t.cpu().pin_memory() for t in (obs_r, chains_r, olp_r, torch.randn(P_roll, device=dev, generator=g2), val_r,
                                                torch.randn(P_roll, device=dev, generator=g2))]
    roll_dev = [torch.empty_like(t, device=dev) for t in roll_host]
    inds_host = [torch.randint(0, P_roll * K, (rows,), dtype=torch.int32).pin_memory() for _ in range(2)]
    UPLOAD_EVERY = 20
    adv_all = roll_host[5].to(dev)
    if world > 1:
        parts = [torch.empty_like(adv_all) for _ in range(world)]
        dist.all_gather(parts, adv_all)
        adv_all = torch.cat(parts)
    idx_mean, idx_std = advantage_stats(adv_all.cpu().numpy())

    def e2e_indexed_step(i):
        if i % UPLOAD_EVERY == 0:
            for hb, db in zip(roll_host, roll_dev):
                db.copy_(hb, non_blocking=True)
        e.ppo_step_indexed(*roll_dev, inds_host[i & 1].numpy(), lr=lr, apply=True, n_global=n_global, adv_mean=idx_mean, adv_std=idx_std,
                           metrics_host=metrics_host.numpy())

    idx_steps = max(args.steps, UPLOAD_EVERY)
    ms_e2e_idx = timed(e2e_indexed_step, idx_steps, UPLOAD_EVERY)     # warm-up and timed region each start with an upload
    roll_bytes = sum(t.numel() * t.element_size() for t in roll_host)
    # the timed regions last only milliseconds: keep the same step running for ~0.3 s so that nvidia-smi (20 ms period)
    # sees the clocks and throttle reasons of this workload under load
    t_load = time.perf_counter(); n_load = 0
    while time.perf_counter() - t_load < 0.3:
        for i in range(20):
            dev_step(i)
        torch.cuda.synchronize(); n_load += 20
    clocks = clk.finish()
    clocks["load_steps_sampled"] = n_load
    step_ms = ms_dev / args.steps
    roof = roofline_of(e, mode, step_ms)

    # ---- multi-rank self-check: (a) the replicas hold bit-identical weights after all those updates; (b) one more update
    #      (loss + gradient only) on the sharded global minibatch equals the same minibatch on ONE rank with the same weights
    selfcheck = None
    if world > 1:
        w_now = np.concatenate([e.get_weights(L.NET_ACTOR_FT), e.get_weights(L.NET_CRITIC)])
        digests = [None] * world
        dist.all_gather_object(digests, hashlib.sha1(w_now.tobytes()).hexdigest())
        b0 = devb[0]; mean0, std0 = stats[0]
        m_n, g_n = e.ppo_step(*b0, lr=0.0, apply=False, n_global=n_global, adv_mean=mean0, adv_std=std0, want_grads=True)
        gathered = []
        for t in b0:
            shp = [list(t.shape)]
            if args.scaling == "strong":
                allshp = [None] * world; dist.all_gather_object(allshp, list(t.shape))
            else:
                allshp = [list(t.shape)] * world
            parts = [torch.empty(sh, device=dev, dtype=t.dtype) for sh in allshp]
            dist.all_gather(parts, t.contiguous())
            gathered.append(torch.cat(parts))
        selfcheck = {"replicas_identical": all(x == digests[0] for x in digests)}
        if rank == 0:
            e1 = make_gpu_engine(PREC[mode], local)
            e1.set_weights(L.NET_ACTOR_FT, e.get_weights(L.NET_ACTOR_FT)); e1.set_weights(L.NET_CRITIC, e.get_weights(L.NET_CRITIC))
            m_1, g_1 = e1.ppo_step(*gathered, lr=0.0, apply=False, n_global=n_global, adv_mean=mean0, adv_std=std0, want_grads=True)
            torch.cuda.synchronize()
            selfcheck["grad_err_vs_single_rank_of_max"] = float((g_n - g_1).abs().max() / g_1.abs().max())
            selfcheck["metrics_abs_err_vs_single_rank"] = float((m_n - m_1).abs().max())
            selfcheck["rows_checked"] = int(gathered[0].shape[0])
            e1.close()
        del gathered
        barrier()

    # ---- sampling half of the metric: 40 env copies, T=20 chain, in-kernel Philox (walker2d = configs[1], hopper = configs[0])
    def sampling_block(eng, dd, label):
        obs40 = torch.rand(N_ENVS, dd.Do, device=dev) * 2 - 1
        obs40_h = obs40.cpu().pin_memory()
        act_h = torch.empty(N_ENVS, dd.A).pin_memory(); ch_h = torch.empty(N_ENVS, dd.ft_denoising_steps + 1, dd.A).pin_memory()
        cnt = [0]

        def samp_dev(i):
            cnt[0] += 1
            eng.sample(obs40, seed=1, offset=cnt[0])

        def samp_e2e(i):
            cnt[0] += 1
            eng.sample_host(obs40_h.numpy(), act_h.numpy(), ch_h.numpy(), seed=1, offset=cnt[0])

        ls0 = eng.launch_count()
        ms_s = timed(samp_dev, 50, 5)
        samp_launches = (eng.launch_count() - ls0) // 55
        samp_path = eng.last_path()
        ms_s_e2e = timed(samp_e2e, 50, 5)
        Fa_l = 2 * (dd.Din * dd.actor_hidden + 2 * dd.actor_hidden ** 2 + dd.actor_hidden * dd.A)
        return {"shapes": label, "chunks_per_sec": world * N_ENVS * 50 / (ms_s * 1e-3), "us_per_rollout_step": ms_s / 50 * 1e3,
                "launches_per_rollout_step": samp_launches, "path": PATHS[samp_path],
                "n_envs_per_gpu": N_ENVS, "e2e_chunks_per_sec": world * N_ENVS * 50 / (ms_s_e2e * 1e-3),
                "e2e_us_per_rollout_step": ms_s_e2e / 50 * 1e3,
                "fp32_fma_frac": (N_ENVS * dd.denoising_steps * Fa_l / (ms_s / 50 * 1e-3)) / 74.5e12}

    sampling = sampling_block(e, d, "walker2d (obs 17, act 6)")
    BL = 148 * 128                                     # one 128-row tile per SM
    obsL = torch.rand(BL, d.Do, device=dev) * 2 - 1
    lcnt = [0]

    def large_fn(eng):
        def f(i):
            lcnt[0] += 1
            eng.sample(obsL, seed=1, offset=lcnt[0], return_chain=True)
        return f

    def large_block(eng, md):
        ms_L = timed(large_fn(eng), 5, 3)
        pth = eng.last_path()
        tf = BL * d.denoising_steps * Fa * 5 / (ms_L * 1e-3) / 1e12
        return {"rows_per_gpu": BL, "dtype": DTYPES[md], "chunks_per_sec": world * BL * 5 / (ms_L * 1e-3), "tflops": tf,
                "frac_of_bf16_sustained": tf / pk["bf16_tflops_sustained"],
                "launches_per_rollout_step": 1 if pth in (1, 4) else None, "path": PATHS[pth]}
    sampling["large_batch"] = large_block(e, mode)

    # ---- BASELINE.json configs[4]: halfcheetah-medium-v2 pre_diffusion_mlp eps-MSE pre-train step, batch 4096 (weak: per GPU; strong: global)
    NBG = 4096
    if args.scaling == "strong":
        lo_p, hi_p = shard_range(NBG, rank, world); NB = hi_p - lo_p; NB_global = NBG; row_off = lo_p
    else:
        NB = NBG; NB_global = NBG * world; row_off = rank * NBG
    x0_p = torch.rand(NB, d.A, device=dev) * 2 - 1
    obs_p = torch.rand(NB, d.Do, device=dev) * 2 - 1
    pcnt = [0]

    def pre_fn(eng):
        def f(i):
            pcnt[0] += 1
            eng.pretrain_step(x0_p, obs_p, lr=1e-3, apply=True, seed=3, offset=pcnt[0], n_global=NB_global, row_offset=row_off)
        return f

    pre_flops = 3 * Fa - 2 * d.Din * d.actor_hidden

    def pre_block(eng, md):
        ms_pre = timed(pre_fn(eng), 20, 5)
        return {"samples_per_sec": NB_global * 20 / (ms_pre * 1e-3), "ms_per_step": ms_pre / 20, "batch_per_gpu": NB, "dtype": DTYPES[md],
                "tflops": pre_flops * NB_global / world * 20 / (ms_pre * 1e-3) / 1e12,
                "note": "latency-bound at this batch (32 row tiles for 148 SMs): 13.7 GFLOP per step"}
    pretrain = pre_block(e, mode)

    # ---- the other precision modes on the same workload, beside the headline
    other = {}
    for md in ("bf16x3", "bf16", "fp32"):
        if md == mode:
            continue
        eo = make_gpu_engine(PREC[md], local)
        if world > 1:
            eo.init_comm()
        nst = args.steps if md != "fp32" else 3
        l1 = eo.launch_count()
        ms_o = timed(step_fn(eo), nst, 3)
        lps = (eo.launch_count() - l1) // (nst + 3)
        blk = {"value": n_global * nst / (ms_o * 1e-3), "unit": UNIT, "ms_per_step": ms_o / nst, "dtype": DTYPES[md], "precision": PRECISION_NOTE[md],
               "gpu_launches_per_step": lps, "step_tflops": fps * rows / (ms_o / nst * 1e-3) / 1e12}
        blk["roofline"] = roofline_of(eo, md, ms_o / nst)
        if md != "fp32":

            def e2e_o(i, eo=eo):
                if i % UPLOAD_EVERY == 0:
                    for hb, db in zip(roll_host, roll_dev):
                        db.copy_(hb, non_blocking=True)
                eo.ppo_step_indexed(*roll_dev, inds_host[i & 1].numpy(), lr=lr, apply=True, n_global=n_global, adv_mean=idx_mean, adv_std=idx_std,
                                    metrics_host=metrics_host.numpy())
            ms_oi = timed(e2e_o, idx_steps, UPLOAD_EVERY)
            blk["e2e"] = {"value": n_global * idx_steps / (ms_oi * 1e-3), "unit": UNIT, "ms_per_step": ms_oi / idx_steps,
                          "api": "Engine.ppo_step_indexed (as the headline e2e)"}
            blk["sampling_large_batch"] = large_block(eo, md)
            blk["pretrain"] = pre_block(eo, md)
        else:
            ffma = blk["roofline"]["peak"]
            blk["fp32_ffma_peak_measured_tflops"] = ffma
            blk["frac_of_fp32_ffma_peak"] = fps * rows / (ms_o / nst * 1e-3) / (ffma * 1e12) if ffma else None

            def e2e_f(i, eo=eo):
                if i % UPLOAD_EVERY == 0:
                    for hb, db in zip(roll_host, roll_dev):
                        db.copy_(hb, non_blocking=True)
                eo.ppo_step_indexed(*roll_dev, inds_host[i & 1].numpy(), lr=lr, apply=True, n_global=n_global, adv_mean=idx_mean, adv_std=idx_std,
                                    metrics_host=metrics_host.numpy())
            ms_fi = timed(e2e_f, 4, 2)
            blk["e2e"] = {"value": n_global * 4 / (ms_fi * 1e-3), "unit": UNIT, "ms_per_step": ms_fi / 4,
                          "api": "Engine.ppo_step_indexed (as the headline e2e; 4 timed steps, rollout resident)"}
        other[md] = blk
        eo.close()

    # ---- BASELINE.json configs[0] / [3]: hopper shapes (obs 11, act 3): 40-env rollout, PPO update, scaled rollout
    hopper = None
    if not args.no_hopper:
        global DIMS
        saved_dims = dict(DIMS)
        DIMS = dict(DIMS, obs_dim=11, action_dim=3)
        try:
            dh = D()
            eh = make_gpu_engine(PREC[mode], local, cond_dim=11, action_dim=3)
            if world > 1:
                eh.init_comm()
            hopper = {"sampling": sampling_block(eh, dh, "hopper (obs 11, act 3)")}
            Fa_h = 2 * (dh.Din * dh.actor_hidden + 2 * dh.actor_hidden ** 2 + dh.actor_hidden * dh.A)
            hb = make_gpu_batches(eh, rows, 1, seed=20 + rank)[0]
            hs = global_stats(hb[6])

            def hop_step(i):
                eh.ppo_step(*hb, lr=lr, apply=True, n_global=n_global, adv_mean=hs[0], adv_std=hs[1])
            ms_h = timed(hop_step, args.steps, 3)
            hopper["ppo"] = {"value": n_global * args.steps / (ms_h * 1e-3), "unit": UNIT, "ms_per_step": ms_h / args.steps, "dtype": DTYPES[mode]}
            scaled = {}
            for tot in (4096, 16384, 65536):
                per = tot // world if args.scaling == "strong" or world > 1 else tot
                if per < 1:
                    continue
                ob = torch.rand(per, dh.Do, device=dev) * 2 - 1
                c2 = [0]

                def sc_fn(i):
                    c2[0] += 1
                    eh.sample(ob, seed=2, offset=c2[0], row_offset=rank * per)
                ms_sc = timed(sc_fn, 5, 3)
                scaled[str(tot)] = {"rows_per_gpu": per, "chunks_per_sec": per * world * 5 / (ms_sc * 1e-3), "ms_per_rollout_step": ms_sc / 5,
                                    "tflops": per * world * dh.denoising_steps * Fa_h * 5 / (ms_sc * 1e-3) / 1e12, "path": PATHS[eh.last_path()]}
            hopper["scaled_rollout_total_envs"] = scaled
            hopper["note"] = "BASELINE.json configs[0] (hopper shapes on the GPU) and configs[3] (4096-65536 env copies sharded over the ranks, in-kernel Philox)"
            eh.close()
        finally:
            DIMS = saved_dims

    # ---- CPU baseline (oracle port) on rank 0, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import dppo_oracle as O      # cpu_baseline leg: the only oracle use in this arm
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        n_cpu = N_ROWS
        o = O.make_oracle(TASK, seed=0)
        batch = O.make_ppo_batch(o, n_cpu, pool=512, seed=1)
        o.ppo_grads(*batch)
        t0 = time.perf_counter(); reps = 0
        while reps < 3 or (time.perf_counter() - t0 < 10 and reps < 20):
            o.ppo_grads(*batch); reps += 1
        dt = (time.perf_counter() - t0) / reps
        cpu = {"value": n_cpu / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{reps} x loss+gradient of one {n_cpu}-row minibatch (AdamW excluded), torch-CPU fp32, {cores} threads"}

    if rank == 0:
        h2d = sum(t.numel() * t.element_size() for t in pinned[0])
        cfg = workload_config(rows, world, args.scaling)
        cfg.update({"precision": PRECISION_NOTE[mode], "l2": "256 MB flush buffer written between timed steps; two alternating minibatches",
                    "flops_per_sample": fps})
        idx_h2d = rows * 4 + roll_bytes * ((idx_steps + UPLOAD_EVERY - 1) // UPLOAD_EVERY) / idx_steps
        line = {
            "metric": METRIC, "value": n_global * args.steps / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": DTYPES[mode], "data": "synthetic",
            "config": cfg,
            "clocks": clocks,
            "e2e": {"value": n_global * idx_steps / (ms_e2e_idx * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e_idx / idx_steps,
                    "steps": idx_steps, "h2d_bytes_per_step": idx_h2d, "d2h_bytes_per_step": 32,
                    "api": "Engine.ppo_step_indexed -> dppo_ppo_step_indexed_host: the reference's data flow (train_ppo_diffusion_agent.py:266-312): the "
                           "rollout buffers are uploaded from pinned host memory every 20 steps (inside the timed region) and stay resident; per step the "
                           "shuffled flat minibatch indices go in and the 8 metrics come out"},
            "e2e_host_minibatch": {"value": n_global * args.steps / (ms_e2e_host * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                                   "ms_per_step": ms_e2e_host / args.steps, "api": "Engine.ppo_step_host -> dppo_ppo_step_host (the whole minibatch from pinned host buffers every step)",
                                   "h2d_alone_ms_per_step": ms_h2d / args.steps, "h2d_alone_gbps": h2d / (ms_h2d / args.steps * 1e-3) / 1e9},
            "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_per_step": launches_per_step,
            "roofline": roof,
            "cpu_baseline": cpu,
            "sampling": sampling,
            "pretrain": pretrain,
            "step_tflops": fps * rows / (ms_dev / args.steps * 1e-3) / 1e12,
            "bf16_mode": other.get("bf16"), "bf16x3_mode": other.get("bf16x3"), "fp32_ffma_mode": other.get("fp32"),
            "hopper": hopper,
            "selfcheck": selfcheck,
        }
        print(json.dumps(line), flush=True)
    e.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("DPPO_BENCH_PRECISION", "bf16x3"), choices=["bf16x3", "bf16", "fp32"])
    ap.add_argument("--scaling", default=os.environ.get("DPPO_BENCH_SCALING", "weak"), choices=["weak", "strong"],
                    help="weak: 50 000 rows per GPU; strong: the reference's 50 000-row minibatch (and 4096-row pre-train batch) sharded over the ranks")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-hopper", action="store_true", help="skip the hopper-shape block (configs[0] / [3])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed update's metrics and the weights it left as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
