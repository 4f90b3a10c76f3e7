"""GPU (-m gpu): the tensor modes away from the default configuration, one switch at a time, against the fp32 oracle.

Every other GPU test builds its engines from the default `Hyper()`: a ReLU actor, a Mish critic, A in {12, 24}, no value clipping,
normalised advantages, reward_horizon = horizon_steps and K = 10 of T = 20.  Code that only a config switch or the input alignment
selects is exercised here, at the benchmarked dimensions (H = 512, Hc = 256, T = 20, time_dim 16):
  act-MR / act-RR / act-MM  actor / critic activations Mish-ReLU, ReLU-ReLU, Mish-Mish: the plane formats of a ReLU critic (fp16 planes,
                            two accumulators) and of a Mish actor (gates and bf16 copies from one epilogue), the per-layer bf16 chain
                            of a Mish actor, the layer-by-layer fp32 sampler
  vclip, noadv, rh2         PPO loss options: value clipping, raw advantages, reward_horizon < horizon_steps
  K1, KT                    K = 1 set at run time (clip coefficient 0), K = T (the chain starts at x_T)
  nodclip, lpclamp          no clip of x0; new log-probs beyond the [-5, 2] clamp
  A9                        A = 9 (A % 4 != 0): the thread-per-row loss and the separate-launch tail, the gathered index-driven update
  unaligned                 prev / nxt / oldlogp 4 bytes off 16-byte alignment: the same fallback, selected by the addresses
  samp                      final action clip with the deterministic, base-policy and minimum-std sampler flags
Each case also checks, on the oracle's side, that its branch is taken by the data (the clipped value arm wins on some rows, some
log-probs are clamped, ...), and that the intended kernels ran (launch counters, sampler path).

Bounds are the modes' own, unchanged: bf16x3 from tests/test_gpu_split.py, bf16 from tests/test_gpu_bf16.py (its general gradient
bound, see GRAD_TOL), fp32 from tests/test_gpu_parity.py.  Largest error over the cases, measured on a B200 (1000 W power limit) in
brackets; the printed lines give each case:
  bf16x3  eps 5e-6 rel [8.6e-7], value 5e-5 rel [4.4e-6], log-probs 1e-3 abs [2.2e-5], PPO / pre-train grads 1e-3 of max [1.2e-4 / 1.2e-6],
          sampled actions 1e-4 rel [1.7e-5]
  bf16    eps / value 2e-2 rel [4.3e-3 / 4.9e-3], log-probs 0.15 abs [6.5e-2], PPO grads 0.15 of max [8.9e-2], pre-train grads 5e-2 [2.5e-3],
          sampled actions mean abs 2e-2 [9.0e-4]
  fp32    eps 2e-5 rel [1.0e-6], value 2e-5 abs [9.5e-7], log-probs 1e-3 abs [5.7e-6], grads 1e-3 of max [3.8e-7 / 2.0e-7], actions 1e-4 rel [8.8e-6]
"""
import dataclasses
import functools
import os

import numpy as np
import pytest
import torch

import diffusionpolicyoptimization_b200 as dp
from diffusionpolicyoptimization_b200 import _lib as L
from oracle import dppo_oracle as O
from helpers import make_cfg, max_abs, rel_err

pytestmark = pytest.mark.gpu

DETERMINISTIC = os.environ.get("DPPO_DETERMINISTIC") == "1"     # bf16: one GEMM launch per product, fixed-order reductions
PREC = {"bf16x3": L.PREC_BF16X3, "bf16": L.PREC_BF16, "fp32": L.PREC_FP32}
TENSOR = ("bf16x3", "bf16")
ALL = ("bf16x3", "bf16", "fp32")

# name -> oracle task, Hyper fields, Dims fields, cfg.reward_horizon, K set with dppo_set_ft_denoising_steps after creation
CASES = {
    "default": dict(task="hopper"),
    "act-MR": dict(task="hopper", hyper=dict(actor_act="Mish", critic_act="ReLU")),
    "act-RR": dict(task="walker2d", hyper=dict(actor_act="ReLU", critic_act="ReLU")),
    "act-MM": dict(task="walker2d", hyper=dict(actor_act="Mish", critic_act="Mish")),
    "vclip": dict(task="hopper", hyper=dict(clip_vloss_coef=0.05)),
    "noadv": dict(task="hopper", hyper=dict(norm_adv=False)),
    "rh2": dict(task="hopper", reward_horizon=2),
    "K1": dict(task="hopper", runtime_k=1),
    "KT": dict(task="hopper", dims=dict(ft_denoising_steps=20)),
    "nodclip": dict(task="hopper", hyper=dict(denoised_clip_value=None)),
    "lpclamp": dict(task="hopper"),                                   # the default config; the batch is changed (ppo_batch)
    "A9": dict(task="hopper", dims=dict(horizon_steps=3)),
    "samp": dict(task="hopper", hyper=dict(final_action_clip_value=0.5)),
}
ACT = ("act-MR", "act-RR", "act-MM")

N_PPO, N_FWD, B_LP, B_SAMPLE, N_PRE = 4099, 3000, 512, 2304, 2304

# the modes' stated bounds
EPS_RTOL = {"bf16x3": 5e-6, "bf16": 2e-2, "fp32": 2e-5}
LOGP_ATOL = {"bf16x3": 1e-3, "bf16": 0.15, "fp32": 1e-3}
# bf16: 0.15 is the mode's general bound (tests/test_gpu_bf16.py states it; that file asserts 8e-2 on its own fixed batches).  A Mish actor
# runs the per-layer bf16 GEMMs, whose bf16 pre-activations feed the Mish gates: act-MM measures 8.9e-2 of max on its batch
GRAD_TOL = {"bf16x3": 1e-3, "bf16": 0.15, "fp32": 1e-3}
METRIC_TOL = {"bf16x3": (2e-3, 2e-6), "bf16": (5e-2, 2e-3), "fp32": (2e-3, 2e-6)}
PRE_GRAD_TOL = {"bf16x3": 1e-3, "bf16": 5e-2, "fp32": 1e-3}


def _value_err(mode, got, want):
    """bf16x3 / bf16: norm-wise relative (5e-5 / 2e-2); fp32: absolute (2e-5)."""
    return (max_abs(got, want), 2e-5) if mode == "fp32" else (rel_err(got, want), 5e-5 if mode == "bf16x3" else 2e-2)


def _pre_loss_tol(mode, want):
    return {"bf16x3": 1e-5 * abs(want), "bf16": 5e-2 * max(1.0, want), "fp32": 1e-4 * max(1.0, want)}[mode]


def _params(spec, mode):
    return pytest.param(spec, mode, id=f"{spec}-{mode}")


def _grid(specs, modes):
    return [_params(s, m) for s in specs for m in modes]


# ---------------------------------------------------------------- oracle side (shared by the modes of a case)
@functools.lru_cache(maxsize=None)
def oracle(name) -> O.Oracle:
    c = CASES[name]
    o = O.make_oracle(c["task"], seed=0, hyper=O.Hyper(**c.get("hyper", {})), **c.get("dims", {}))
    if "runtime_k" in c:
        o = O.Oracle(dataclasses.replace(o.d, ft_denoising_steps=c["runtime_k"]), o.h, o.actor, o.actor_ft, o.critic)
    return o


def reward_horizon(name):
    return CASES[name].get("reward_horizon", oracle(name).d.horizon_steps)


@functools.lru_cache(maxsize=None)
def ppo_batch(name):
    """The update's minibatch and the oracle's metrics and gradients.  lpclamp: the default case with the next-step actions of 5 % of
    the rows moved by +0.5 (about 5 sigma at the 0.1 log-prob std floor), so that their new log-probs fall below the -5 clamp.
    nodclip: the chains come from the default (clipping) sampler.  Twenty unclipped steps of these random weights drive |x| into the
    thousands, and the log-probs' error grows with the inputs' magnitude (bf16x3 measured 1.6e-2 abs there); with O(1) chains |x0|
    still exceeds 1 on many elements."""
    o = oracle(name)
    batch = list(O.make_ppo_batch(oracle("default") if name == "nodclip" else o, N_PPO, pool=512, seed=3))
    rng = np.random.default_rng(11)
    if name == "noadv":
        batch[6] = torch.from_numpy((3.0 + 2.0 * rng.standard_normal(N_PPO)).astype(np.float32))
    if name == "lpclamp":
        nxt = batch[2].clone()
        nxt[torch.from_numpy(rng.choice(N_PPO, N_PPO // 20, replace=False))] += 0.5
        batch[2] = nxt
    metrics, ga, gc = o.ppo_grads(*batch, reward_horizon=reward_horizon(name))
    return tuple(batch), [float(m) for m in metrics], np.concatenate([O.flatten_params(ga), O.flatten_params(gc)])


@functools.lru_cache(maxsize=None)
def rollout(name, B, seed, **flags):
    o = oracle(name)
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=seed)
    okw = dict(flags)
    if "min_sampling_std" in okw:
        okw["min_sampling_denoising_std"] = okw.pop("min_sampling_std")
    return obs, x_T, noise, o.sample(obs, x_T, noise, **okw)


# ---------------------------------------------------------------- engines
@pytest.fixture(scope="module")
def engines():
    made = {}

    def get(name, mode):
        key = ("default" if name in ("lpclamp", "unaligned") else name, mode)
        if key not in made:
            c = CASES[key[0]]
            o = oracle(key[0])
            cfg = make_cfg(o, PREC[mode])
            cfg.reward_horizon = reward_horizon(key[0])
            if "runtime_k" in c:
                cfg.ft_denoising_steps = O.Dims().ft_denoising_steps      # created at K = 10, switched below
            e = dp.Engine(cfg, 0)
            e.set_weights(L.NET_ACTOR, O.flatten_params(o.actor))
            e.set_weights(L.NET_ACTOR_FT, O.flatten_params(o.actor_ft))
            e.set_weights(L.NET_CRITIC, O.flatten_params(o.critic))
            e.set_weights(L.NET_ACTOR_EMA, O.flatten_params(o.actor))
            if "runtime_k" in c:
                e.set_ft_denoising_steps(c["runtime_k"])
                assert e.K == c["runtime_k"]
            made[key] = e
        return made[key]

    yield get
    for e in made.values():
        e.close()


# ---------------------------------------------------------------- which kernels ran
def _counts(e):
    return e.tc_launch_count(), e.fused_launch_count()


def _expect(o, mode, kind):
    """(tcgen05 launches, fused layer-chain launches) of one call.  bf16x3: three plane GEMMs per forward (L0, L1, the folded output
    layer), two backward, one grouped weight-gradient launch.  bf16: the fused chain kernels need a ReLU actor at H = 512 (a Mish
    actor takes the per-layer path: 4 forward, 3 dX and 4 dW GEMMs); the critic at Hc = 256 is fused with either activation."""
    T = o.d.denoising_steps
    if mode == "fp32":
        return (0, 0)
    if mode == "bf16x3":
        return {"fwd": (6, 0), "lp": (3, 0), "ppo": (11, 0), "pre": (6, 0), "sample": (3 * T, 0)}[kind]
    if o.h.actor_act == "ReLU":
        return {"fwd": (2, 2), "lp": (1, 1), "ppo": (5, 4), "pre": (3, 2), "sample": (1, 1)}[kind]
    # per-layer actor; fused critic: forward + backward chain + its grouped dW launch in the update
    return {"fwd": (5, 1), "lp": (4, 0), "ppo": (14, 2), "pre": (11, 0), "sample": (4 * T, 0)}[kind]


def _sample_path(o, mode):
    if mode == "bf16x3":
        return 3                                                     # split layered
    if mode == "bf16":
        return 4 if o.h.actor_act == "ReLU" else 3                  # fused FINAL_SAMPLE chain / per-layer tcgen05
    return 1 if o.h.actor_act == "ReLU" else 2                      # persistent cluster kernel (ReLU only) / layer-by-layer fp32


def _check_counts(o, mode, kind, e, before):
    got = tuple(a - b for a, b in zip(_counts(e), before))
    if DETERMINISTIC and mode == "bf16" and kind in ("ppo", "pre"):
        return
    assert got == _expect(o, mode, kind), (kind, got)


def _flat(x):
    return x.reshape(x.shape[0], -1)


def _ppo_args(batch):
    N = batch[0].shape[0]
    return (_flat(batch[0]), batch[1].reshape(N, -1), batch[2].reshape(N, -1), batch[3], batch[4], batch[5], batch[6],
            batch[7].reshape(N, -1))


def _grad_errs(o, got_g, want_g):
    nA = o.d.n_actor()
    return [float(np.abs(got_g[sl] - want_g[sl]).max() / np.abs(want_g[sl]).max()) for sl in (slice(0, nA), slice(nA, None))]


def _check_ppo_result(name, mode, o, m, g, want_m, want_g, tag=""):
    err_a, err_c = _grad_errs(o, g, want_g)
    m = np.asarray(m)
    print(f"[{name} {mode}{tag}] PPO grads actor {err_a:.2e} critic {err_c:.2e} of max; metrics rel "
          f"{np.abs(m - want_m).max() / max(np.abs(want_m).max(), 1e-30):.2e}")
    assert err_a < GRAD_TOL[mode] and err_c < GRAD_TOL[mode], (err_a, err_c)
    rtol, atol = METRIC_TOL[mode]
    np.testing.assert_allclose(m, want_m, rtol=rtol, atol=atol)


# ---------------------------------------------------------------- forward, value, log-probs
@pytest.mark.parametrize("name,mode", _grid(ACT + ("A9",), ALL))
def test_forward_and_value(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    d = o.d
    rng = np.random.default_rng(N_FWD)
    x = torch.from_numpy(rng.standard_normal((N_FWD, d.horizon_steps, d.action_dim)).astype(np.float32))
    t = torch.from_numpy(rng.integers(0, d.denoising_steps, N_FWD))
    obs = torch.from_numpy(rng.uniform(-1, 1, (N_FWD, 1, d.obs_dim)).astype(np.float32))
    with torch.no_grad():
        want = O.diffusion_mlp(o.actor_ft, x, t, obs, d, o.h.actor_act).reshape(N_FWD, -1)
        wantv = O.critic_obs(o.critic, obs, o.h.critic_act).reshape(-1)
    c0 = _counts(e)
    got = e.actor_forward(L.NET_ACTOR_FT, x.reshape(N_FWD, -1), t, _flat(obs))
    gv = e.value(_flat(obs))
    torch.cuda.synchronize()
    err = rel_err(got, want)
    errv, tolv = _value_err(mode, gv, wantv)
    print(f"[{name} {mode}] eps rel err {err:.2e}, value err {errv:.2e}")
    assert err < EPS_RTOL[mode] and errv < tolv, (err, errv)
    _check_counts(o, mode, "fwd", e, c0)


@pytest.mark.parametrize("name,mode", _grid(ACT + ("A9",), ALL) + _grid(("K1", "KT"), TENSOR))
def test_logprobs_of_whole_chains(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    K = o.d.ft_denoising_steps
    B = max(B_LP, -(-B_SAMPLE // K))                    # K = 1: enough chains for the 2048-row tensor threshold
    obs, _, _, s = rollout(name, B, 3)
    with torch.no_grad():
        want = o.get_logprobs(obs, s.chains).reshape(B * K, -1)
    c0 = _counts(e)
    got = e.logprobs(_flat(obs), s.chains.reshape(B, K + 1, -1))
    torch.cuda.synchronize()
    err = max_abs(got, want)
    print(f"[{name} {mode}] log-prob abs err {err:.2e} ({B} chains, K = {K})")
    assert err < LOGP_ATOL[mode], err
    _check_counts(o, mode, "lp", e, c0)


@pytest.mark.parametrize("name,mode", _grid(ACT, ALL) + _grid(("nodclip",), TENSOR))
def test_logprobs_subsample(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    batch, _, _ = ppo_batch(name)
    N = N_PPO
    with torch.no_grad():
        want, _ = o.get_logprobs_subsample(batch[0], batch[1], batch[2], batch[3])
    if name == "nodclip":
        # the branch is live: without the clip, |x0| exceeds 1 on at least 1 % of the elements
        t = torch.arange(o.d.ft_denoising_steps - 1, -1, -1)[batch[3].long()]
        with torch.no_grad():
            eps = O.diffusion_mlp(o.actor_ft, batch[1], t, batch[0], o.d, o.h.actor_act)
        x0 = o._extract("sqrt_recip_alphas_cumprod", t) * batch[1] - o._extract("sqrt_recipm1_alphas_cumprod", t) * eps
        frac = float((x0.abs() > 1).float().mean())
        print(f"[{name}] |x0| > 1 on {frac:.1%} of the elements")
        assert frac >= 0.01, frac
    c0 = _counts(e)
    got = e.logprobs_subsample(_ppo_args(batch)[0], batch[1].reshape(N, -1), batch[2].reshape(N, -1), batch[3])
    torch.cuda.synchronize()
    err = max_abs(got, want.reshape(N, -1))
    print(f"[{name} {mode}] subsampled log-prob abs err {err:.2e}")
    assert err < LOGP_ATOL[mode], err
    _check_counts(o, mode, "lp", e, c0)


# ---------------------------------------------------------------- the PPO update
@pytest.mark.parametrize("name,mode", _grid(ACT + ("A9",), ALL)
                         + _grid(("vclip", "noadv", "rh2", "K1", "KT", "nodclip", "lpclamp"), TENSOR))
def test_ppo_loss_and_gradients(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    batch, want_m, want_g = ppo_batch(name)
    # every case: the ratio leaves the clip range on some rows (both arms of the policy loss)
    assert want_m[3] > 0.0, want_m
    if name == "vclip":
        with torch.no_grad():
            v = O.critic_obs(o.critic, batch[0], o.h.critic_act).reshape(-1)
        c = o.h.clip_vloss_coef
        vc = batch[5] + torch.clamp(v - batch[5], -c, c)
        frac = float(((vc - batch[4]) ** 2 > (v - batch[4]) ** 2).float().mean())
        print(f"[{name}] the clipped value arm wins on {frac:.1%} of the rows")
        assert 0.05 < frac < 0.95, frac
    if name == "noadv":
        a = batch[6]
        assert abs(float(a.mean())) > 2.0 and float(a.std()) > 1.5
    if name == "rh2":
        m4, _, _ = o.ppo_grads(*batch, reward_horizon=o.d.horizon_steps)
        assert abs(float(m4[0]) - want_m[0]) > 1e-3 * abs(want_m[0]), "reward_horizon = 2 changes nothing on this batch"
    if name == "lpclamp":
        with torch.no_grad():
            lp, _ = o.get_logprobs_subsample(batch[0], batch[1], batch[2], batch[3])
        frac = float(((lp < -5) | (lp > 2)).float().mean())
        print(f"[{name}] {frac:.1%} of the new log-probs lie outside [-5, 2]")
        assert frac >= 0.01, frac
    c0 = _counts(e)
    n0 = e.launch_count()
    m, g = e.ppo_step(*_ppo_args(batch), lr=0.0, apply=False, want_grads=True)
    torch.cuda.synchronize()
    launches = e.launch_count() - n0
    _check_ppo_result(name, mode, o, m.cpu().numpy(), g.cpu().numpy(), want_m, want_g)
    _check_counts(o, mode, "ppo", e, c0)
    if name == "A9" and mode == "bf16x3":
        # A % 4 != 0: the thread-per-row loss and the separate-launch tail, more launches than the default shape's update
        ed = engines("default", mode)
        bd, _, _ = ppo_batch("default")
        ed.ppo_step(*_ppo_args(bd), lr=0.0, apply=False)        # (a fresh engine first builds its folded output layers)
        n1 = ed.launch_count()
        ed.ppo_step(*_ppo_args(bd), lr=0.0, apply=False)
        assert launches > ed.launch_count() - n1, (launches, ed.launch_count() - n1)


@pytest.mark.parametrize("name,mode", _grid(("A9",), ("bf16",)))
def test_bf16_layered_update_into_an_unaligned_critic_slice(name, mode):
    """The flat gradient is [actor_ft | critic]: with A % 4 != 0 the critic's slice starts 4 bytes past a 16-byte boundary.  The
    per-layer bf16 update (force_path 3) accumulates its weight gradients there with the GEMM epilogue's atomics, the fused one with
    the grouped dW kernel's (test_ppo_loss_and_gradients[A9-bf16]): both must fall back from the 16-byte vector reductions."""
    o = oracle(name)
    assert o.d.n_actor() % 4 != 0
    e = dp.Engine(make_cfg(o, PREC[mode]), 0)
    try:
        e.set_weights(L.NET_ACTOR_FT, O.flatten_params(o.actor_ft)); e.set_weights(L.NET_CRITIC, O.flatten_params(o.critic))
        e.force_path(3)
        batch, want_m, want_g = ppo_batch(name)
        n0, f0 = _counts(e)
        m, g = e.ppo_step(*_ppo_args(batch), lr=0.0, apply=False, want_grads=True)
        torch.cuda.synchronize()
        _check_ppo_result(name, mode, o, m.cpu().numpy(), g.cpu().numpy(), want_m, want_g, " layered")
        n1, f1 = _counts(e)
        assert DETERMINISTIC or (n1 - n0, f1 - f0) == (22, 0), (n1 - n0, f1 - f0)     # 8 forward + 6 dX + 8 dW GEMMs
    finally:
        e.close()


@pytest.mark.parametrize("name,mode", _grid(("unaligned",), TENSOR))
def test_ppo_unaligned_rows_take_the_fallback(engines, name, mode):
    """prev / nxt / oldlogp as CUDA views 4 bytes past a 16-byte boundary: the float4 loss kernel is not eligible, the thread-per-row
    loss (and in bf16x3 the separate-launch tail) runs instead.  Only the reduction order differs from the aligned call."""
    o, e = oracle("default"), engines(name, mode)
    batch, want_m, want_g = ppo_batch("default")
    args = [a.cuda() for a in _ppo_args(batch)]
    N, A = N_PPO, o.d.A

    def shifted(x):
        buf = torch.zeros(N * A + 1, device="cuda")
        buf[1:] = x.reshape(-1)
        return buf[1:].view(N, A)

    un = list(args)
    for i in (1, 2, 7):
        un[i] = shifted(args[i])
        assert un[i].data_ptr() % 16 == 4
    e.ppo_step(*args, lr=0.0, apply=False)                        # (a fresh engine first builds its folded output layers)
    n0 = e.launch_count()
    m_al, g_al = e.ppo_step(*args, lr=0.0, apply=False, want_grads=True)
    n1 = e.launch_count()
    c0 = _counts(e)
    m_un, g_un = e.ppo_step(*un, lr=0.0, apply=False, want_grads=True)
    torch.cuda.synchronize()
    n2 = e.launch_count()
    m_al, g_al, m_un, g_un = (x.cpu().numpy() for x in (m_al, g_al, m_un, g_un))
    diff = float(np.abs(g_un - g_al).max() / np.abs(g_al).max())
    print(f"[{name} {mode}] unaligned vs aligned: grads {diff:.2e} of max, metrics rel "
          f"{float(np.abs(m_un - m_al).max() / np.abs(m_al).max()):.2e}")
    assert diff < 1e-5, diff
    # approx_kl = mean(ratio - 1 - logratio) ~ logratio^2 / 2 with logratio = newm - oldm ~ 1e-2: the one-ulp change of a row's log-prob
    # mean (the two loss kernels sum the row in different orders) is amplified by that cancellation (measured 2.9e-5 relative)
    keep = [i for i in range(8) if i != 4]
    np.testing.assert_allclose(m_un[keep], m_al[keep], rtol=1e-5, atol=0)
    np.testing.assert_allclose(m_un[4], m_al[4], rtol=1e-4, atol=0)
    _check_ppo_result(name, mode, o, m_al, g_al, want_m, want_g, " aligned")
    _check_ppo_result(name, mode, o, m_un, g_un, want_m, want_g, " unaligned")
    _check_counts(o, mode, "ppo", e, c0)
    if mode == "bf16x3":
        assert n2 - n1 > n1 - n0, (n2 - n1, n1 - n0)              # the separate-launch tail


@pytest.mark.parametrize("name,mode", _grid(("A9",), ALL))
def test_indexed_update_gathers_unaligned_rows(engines, name, mode):
    """A % 4 != 0: dppo_ppo_step_indexed gathers the minibatch (one kernel) and runs dppo_ppo_step on it; the result is that of
    dppo_ppo_step on the rows gathered on the host (train_ppo_diffusion_agent.py:292-312)."""
    o, e = oracle(name), engines(name, mode)
    d = o.d
    P, K, A, N = 600, d.ft_denoising_steps, d.A, 4096
    obs, _, _, s = rollout(name, P, 77)
    chains = s.chains.reshape(P, K + 1, A)
    g = torch.Generator().manual_seed(5)
    olp = torch.randn(P, K, A, generator=g) * 0.3 - 1.0
    ret, val, adv = torch.randn(P, generator=g), torch.randn(P, generator=g), torch.randn(P, generator=g)
    flat = torch.randint(0, P * K, (N,), generator=g, dtype=torch.int64)
    b, k = flat // K, flat % K
    idx = flat.to(torch.int32).cuda()
    e.ppo_step_indexed(_flat(obs), chains, olp, ret, val, adv, idx, lr=0.0, apply=False)
    n0 = e.launch_count()
    m1, g1 = e.ppo_step_indexed(_flat(obs), chains, olp, ret, val, adv, idx, lr=0.0, apply=False, want_grads=True)
    launches_indexed = e.launch_count() - n0
    n1 = e.launch_count()
    m2, g2 = e.ppo_step(_flat(obs)[b], chains[b, k], chains[b, k + 1], k.to(torch.int32), ret[b], val[b], adv[b], olp[b, k],
                        lr=0.0, apply=False, want_grads=True)
    torch.cuda.synchronize()
    assert launches_indexed == e.launch_count() - n1 + 2          # + the gather kernel + the NaN-on-bad-index kernel
    assert torch.equal(m1, m2)
    if mode == "bf16" and not DETERMINISTIC:                      # dW accumulates with atomics: the order varies run to run
        assert float((g1 - g2).abs().max()) < 2e-3 * float(g2.abs().max())
    else:
        assert torch.equal(g1, g2)


# ---------------------------------------------------------------- pre-training and one applied update
@pytest.mark.parametrize("name,mode", _grid(ACT + ("A9",), ALL))
def test_pretrain_loss_and_gradients(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    d = o.d
    rng = np.random.default_rng(5)
    acts = torch.from_numpy(rng.uniform(-1, 1, (N_PRE, d.horizon_steps, d.action_dim)).astype(np.float32))
    st = torch.from_numpy(rng.uniform(-1, 1, (N_PRE, 1, d.obs_dim)).astype(np.float32))
    tt = torch.from_numpy(rng.integers(0, d.denoising_steps, N_PRE))
    nz = torch.from_numpy(rng.standard_normal((N_PRE, d.horizon_steps, d.action_dim)).astype(np.float32))
    want_l, want_g = o.pretrain_grads(acts, st, tt, nz)
    want_l, wg = float(want_l), O.flatten_params(want_g)
    c0 = _counts(e)
    loss, pg = e.pretrain_step(acts.reshape(N_PRE, -1), _flat(st), lr=0.0, apply=False, t=tt, noise=nz.reshape(N_PRE, -1), want_grads=True)
    torch.cuda.synchronize()
    err_g = float(np.abs(pg.cpu().numpy() - wg).max() / np.abs(wg).max())
    print(f"[{name} {mode}] pre-train loss {float(loss):.6f} vs {want_l:.6f}, grads {err_g:.2e} of max")
    assert abs(float(loss) - want_l) < _pre_loss_tol(mode, want_l) and err_g < PRE_GRAD_TOL[mode], (float(loss), want_l, err_g)
    _check_counts(o, mode, "pre", e, c0)


@pytest.mark.parametrize("name,mode", _grid(ACT, ALL))
def test_applied_update_refreshes_operands(engines, name, mode):
    """After AdamW the operand copies (planes, bf16 copies, folded output layers) must follow the new fp32 weights: the next
    forward agrees with the oracle evaluated at the weights the engine hands back."""
    o, e = oracle(name), engines(name, mode)
    N = 2560
    batch = O.make_ppo_batch(o, N, pool=256, seed=4)
    fb = _ppo_args(batch)
    w_ft0, w_c0 = e.get_weights(L.NET_ACTOR_FT), e.get_weights(L.NET_CRITIC)
    try:
        lp0 = e.logprobs_subsample(*fb[:4]).clone()
        e.ppo_step(*fb, lr=1e-3, apply=True)
        lp1 = e.logprobs_subsample(*fb[:4])
        v1 = e.value(fb[0])
        torch.cuda.synchronize()
        assert float((lp1 - lp0).abs().max()) > 1e-3
        o1 = O.Oracle(o.d, o.h, o.actor, O.unflatten_params(e.get_weights(L.NET_ACTOR_FT), o.d.actor_shapes()),
                      O.unflatten_params(e.get_weights(L.NET_CRITIC), o.d.critic_shapes()))
        with torch.no_grad():
            want_lp, _ = o1.get_logprobs_subsample(batch[0], batch[1], batch[2], batch[3])
            want_v = O.critic_obs(o1.critic, batch[0], o.h.critic_act).reshape(-1)
        err_lp = max_abs(lp1, want_lp.reshape(N, -1))
        err_v, tol_v = _value_err(mode, v1, want_v)
        print(f"[{name} {mode}] after AdamW: log-prob abs err {err_lp:.2e}, value err {err_v:.2e}")
        assert err_lp < LOGP_ATOL[mode] and err_v < tol_v, (err_lp, err_v)
    finally:
        e.set_weights(L.NET_ACTOR_FT, w_ft0); e.set_weights(L.NET_CRITIC, w_c0)     # the engines are shared
        n = e.n_actor + e.n_critic
        e.set_opt_state(L.OPT_FINETUNE, np.zeros(n, np.float32), np.zeros(n, np.float32), 0)


# ---------------------------------------------------------------- sampling
def _check_sample(name, mode, o, e, flags, seed):
    d = o.d
    B = B_SAMPLE
    obs, x_T, noise, want = rollout(name, B, seed, **flags)
    c0 = _counts(e)
    a, ch = e.sample(_flat(obs), x_T=x_T.reshape(B, -1), noise=noise.reshape(d.denoising_steps, B, -1), **flags)
    torch.cuda.synchronize()
    assert e.last_path() == _sample_path(o, mode), e.last_path()
    wa, wc = want.trajectories.reshape(B, -1), want.chains.reshape(B, d.ft_denoising_steps + 1, -1)
    err, err_c = rel_err(a, wa), rel_err(ch, wc)
    mean, mean_c = float((a.cpu() - wa).abs().mean()), float((ch.cpu() - wc).abs().mean())
    print(f"[{name} {mode} {flags}] sampled actions rel {err:.2e} mean abs {mean:.2e}; chains rel {err_c:.2e} mean abs {mean_c:.2e}")
    if mode == "bf16x3":
        assert err < 1e-4 and mean < 1e-6 and mean_c < 1e-6, (err, mean, mean_c)
    elif mode == "bf16":
        assert mean < 2e-2 and err < 0.25 and mean_c < 2e-2, (err, mean, mean_c)
    else:
        assert err < 1e-4 and err_c < 1e-4, (err, err_c)
    _check_counts(o, mode, "sample", e, c0)
    return x_T, ch


@pytest.mark.parametrize("name,mode", _grid(ACT + ("A9",), ALL) + _grid(("KT",), TENSOR))
def test_large_batch_sampler(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    x_T, ch = _check_sample(name, mode, o, e, {}, 6)
    if name == "KT":                                              # K = T: chain[0] is x_T itself (diffusion_vpg.py:286-287)
        assert torch.equal(ch[:, 0].cpu(), x_T.reshape(B_SAMPLE, -1))


@pytest.mark.parametrize("flags", [dict(deterministic=True), dict(use_base_policy=True), dict(min_sampling_std=0.25)],
                         ids=["deterministic", "base", "minstd"])
@pytest.mark.parametrize("name,mode", _grid(("samp",), TENSOR))
def test_large_batch_sampler_flags(engines, name, mode, flags):
    """final_action_clip_value = 0.5 with each sampler flag: the split layered sampler (bf16x3) and the fused one (bf16, whose
    update epilogue is its own)."""
    o, e = oracle(name), engines(name, mode)
    _, _, _, want = rollout(name, B_SAMPLE, 7, **flags)
    assert float((want.trajectories.abs() == 0.5).float().mean()) > 0.01      # the final clip is active
    _check_sample(name, mode, o, e, flags, 7)
