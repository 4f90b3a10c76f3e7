"""GPU (-m gpu): the persistent cluster sampler for actor widths other than 512 (H in {256, 768, 1024}).

sample_cluster_width_kernel<H, AP, R> (csrc/sample_cluster.cuh, AP in {32, 64, 128}) is the rollout sampler of these widths
below the row limits of dppo_sample (path 1); the layer-by-layer fp32 sampler (path 2) and the oracle are the references.  Cases:
  H256-A12    hopper (3 x 4, Do 11)
  H768-A24    walker2d (6 x 4, Do 17), time_dim 32
  H768-A56    14 x 4, Do 59
  H768-A128   16 x 8, Do 59: most of each warp's W1 rows are read from L2 every step
  H1024-A24   walker2d: the W1 slice no longer fits shared memory, part of it is read from L2 every step
  H1024-A128  16 x 8, Do 59: at most 6 rows per cluster pass
  H384-A24    a width the kernel does not cover: stays on the layered path even when path 1 is asked for
  H1024-Mish  a Mish actor: stays on the layered path even when path 1 is asked for
Bounds are the fp32 ones of tests/test_gpu_parity.py: actions and chains within 1e-4 relative (max|a-b| / max|b|).
"""
import functools

import numpy as np
import pytest
import torch

import diffusionpolicyoptimization_b200 as dp
from diffusionpolicyoptimization_b200 import _lib as L
from oracle import dppo_oracle as O
from helpers import make_cfg, make_engine, rel_err

pytestmark = pytest.mark.gpu

ACT_RTOL = 1e-4
WIDE = dict(action_dim=14, horizon_steps=4, obs_dim=59)
WIDEST = dict(action_dim=16, horizon_steps=8, obs_dim=59)
CASES = {
    "H256-A12": ("hopper", dict(actor_hidden=256), "ReLU"),
    "H768-A24": ("walker2d", dict(actor_hidden=768, time_dim=32), "ReLU"),
    "H768-A56": ("hopper", dict(actor_hidden=768, **WIDE), "ReLU"),
    "H768-A128": ("hopper", dict(actor_hidden=768, **WIDEST), "ReLU"),
    "H1024-A24": ("walker2d", dict(actor_hidden=1024), "ReLU"),
    "H1024-A128": ("hopper", dict(actor_hidden=1024, **WIDEST), "ReLU"),
    "H384-A24": ("walker2d", dict(actor_hidden=384), "ReLU"),
    "H1024-Mish": ("walker2d", dict(actor_hidden=1024), "Mish"),
}
NAMES = list(CASES)
LAYERED = ("H384-A24", "H1024-Mish")
CLUSTER = [n for n in NAMES if n not in LAYERED]
# fp32 rows up to which dppo_sample takes the cluster kernel (the measured crossovers, DESIGN.md §5.3)
ROW_LIMITS = {"H256-A12": 2048, "H768-A24": 2048, "H768-A56": 2048, "H768-A128": 1024, "H1024-A24": 1024, "H1024-A128": 1024}


@functools.lru_cache(maxsize=None)
def oracle(name, final_action_clip_value=None, **over):
    task, dims, act = CASES[name]
    hyper = O.Hyper(actor_act=act, final_action_clip_value=final_action_clip_value)
    return O.make_oracle(task, seed=0, hyper=hyper, **dims, **over)


@pytest.fixture(scope="module")
def engines():
    made = {}

    def get(name):
        if name not in made:
            made[name] = make_engine(oracle(name))
        return made[name]

    yield get
    for e in made.values():
        e.close()


def _want_path(name, path):
    return 2 if name in LAYERED else path


def _sample(o, e, B, obs, x_T, noise, **kw):
    return e.sample(obs.reshape(B, -1), x_T=x_T.reshape(B, -1), noise=noise.reshape(o.d.denoising_steps, B, -1), **kw)


def _check(o, want, B, actions, chains):
    assert rel_err(actions, want.trajectories.reshape(B, -1)) < ACT_RTOL
    assert rel_err(chains, want.chains.reshape(B, o.d.ft_denoising_steps + 1, -1)) < ACT_RTOL


def test_case_shapes():
    for name in NAMES:
        d, h = oracle(name).d, oracle(name).h
        H, A = name.split("-")
        assert d.actor_hidden == int(H[1:]), name
        assert A == "Mish" if h.actor_act == "Mish" else d.A == int(A[1:]), name
    assert oracle("H768-A24").d.time_dim == 32


# ---------------------------------------------------------------- oracle match, injected noise
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("B", [1, 5, 40, 50, 67])
@pytest.mark.parametrize("path", [1, 2])     # 1 = persistent cluster sampler, 2 = layer-by-layer fp32
def test_sample_matches_oracle(engines, name, B, path):
    o, e = oracle(name), engines(name)
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=B)
    want = o.sample(obs, x_T, noise)
    e.force_path(path)
    try:
        actions, chains = _sample(o, e, B, obs, x_T, noise)
        torch.cuda.synchronize()
        assert e.last_path() == _want_path(name, path)
    finally:
        e.force_path(0)
    _check(o, want, B, actions, chains)


@pytest.mark.parametrize("name", CLUSTER)
def test_sample_is_one_launch(engines, name):
    o, e = oracle(name), engines(name)
    obs, x_T, noise = O.make_rollout_inputs(o, 40, seed=9)
    _sample(o, e, 40, obs, x_T, noise)        # a first call after new weights also folds the output layers
    n0 = e.launch_count()
    _sample(o, e, 40, obs, x_T, noise)
    torch.cuda.synchronize()
    assert e.last_path() == 1 and e.launch_count() - n0 == 1


# ---------------------------------------------------------------- sampler flags
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("kw", [dict(deterministic=True), dict(use_base_policy=True), dict(min_sampling_std=0.25)])
def test_sample_flags(engines, name, kw):
    o, e = oracle(name), engines(name)
    B = 40
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=21)
    okw = dict(kw)
    if "min_sampling_std" in okw:
        okw["min_sampling_denoising_std"] = okw.pop("min_sampling_std")
    want = o.sample(obs, x_T, noise, **okw)
    for path in (1, 2):
        e.force_path(path)
        try:
            actions, chains = _sample(o, e, B, obs, x_T, noise, **kw)
            torch.cuda.synchronize()
            assert e.last_path() == _want_path(name, path)
        finally:
            e.force_path(0)
        _check(o, want, B, actions, chains)


def _engine_for(o, **cfg_over):
    cfg = make_cfg(o)
    for k, v in cfg_over.items():
        setattr(cfg, k, v)
    e = dp.Engine(cfg, 0)
    e.set_weights(L.NET_ACTOR, O.flatten_params(o.actor))
    e.set_weights(L.NET_ACTOR_FT, O.flatten_params(o.actor_ft))
    e.set_weights(L.NET_CRITIC, O.flatten_params(o.critic))
    return e


@pytest.mark.parametrize("name", ["H256-A12", "H768-A128", "H1024-A24"])
@pytest.mark.parametrize("variant", ["all_steps_finetuned", "runtime_k1", "final_clip"])
def test_sample_chain_variants(name, variant):
    """K = T (x_T is chain[0]), K = 1 set after creation, and a final action clip, on both paths."""
    if variant == "all_steps_finetuned":
        o = oracle(name, ft_denoising_steps=20)
        e = _engine_for(o)
    elif variant == "runtime_k1":
        o = oracle(name, ft_denoising_steps=1)
        e = _engine_for(o, ft_denoising_steps=10)
        e.set_ft_denoising_steps(1)
        assert e.K == 1
    else:
        o = oracle(name, final_action_clip_value=0.5)
        e = _engine_for(o)
    B = 40
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=3)
    want = o.sample(obs, x_T, noise)
    if variant == "all_steps_finetuned":
        np.testing.assert_array_equal(want.chains[:, 0].reshape(B, -1).numpy(), x_T.reshape(B, -1).numpy())
    if variant == "final_clip":
        assert want.trajectories.abs().max() <= 0.5
    for path in (1, 2):
        e.force_path(path)
        actions, chains = _sample(o, e, B, obs, x_T, noise)
        torch.cuda.synchronize()
        assert e.last_path() == path
        assert chains.shape == (B, o.d.ft_denoising_steps + 1, o.d.A)
        _check(o, want, B, actions, chains)
        if variant == "all_steps_finetuned":
            assert torch.equal(chains[:, 0].cpu(), x_T.reshape(B, -1))
    e.close()


# ---------------------------------------------------------------- in-kernel Philox noise
@pytest.mark.parametrize("name", CLUSTER)
def test_philox_cluster_matches_layered_and_shards(engines, name):
    o, e = oracle(name), engines(name)
    B = 40
    obs, _, _ = O.make_rollout_inputs(o, B, seed=5)
    obs = obs.reshape(B, -1)
    got = {}
    for path in (1, 2):
        e.force_path(path)
        try:
            got[path] = e.sample(obs, seed=0x1234567890ABCDEF, offset=77, row_offset=1000)
            torch.cuda.synchronize()
            assert e.last_path() == path
        finally:
            e.force_path(0)
    assert rel_err(got[1][0], got[2][0]) < ACT_RTOL and rel_err(got[1][1], got[2][1]) < ACT_RTOL
    a0, c0 = e.sample(obs, seed=9, offset=4)
    lo = e.sample(obs[:20], seed=9, offset=4, row_offset=0)
    hi = e.sample(obs[20:], seed=9, offset=4, row_offset=20)
    torch.cuda.synchronize()
    assert e.last_path() == 1
    assert torch.equal(torch.cat([lo[0], hi[0]]), a0) and torch.equal(torch.cat([lo[1], hi[1]]), c0)


# ---------------------------------------------------------------- new weights reach the next sample
@pytest.mark.parametrize("name", ["H256-A12", "H768-A56", "H1024-A128"])
def test_set_weights_refreshes_the_resident_slices(name):
    """A new fine-tuned actor reaches the folded output layer, the resident W1 / W_in slices and the W1 rows read from L2."""
    o = oracle(name)
    e = make_engine(o)
    B = 40
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=11)
    _check(o, o.sample(obs, x_T, noise), B, *_sample(o, e, B, obs, x_T, noise))
    rng = np.random.default_rng(5)
    new_ft = [p + 0.05 * torch.from_numpy(rng.standard_normal(tuple(p.shape)).astype(np.float32)) for p in o.actor_ft]
    e.set_weights(L.NET_ACTOR_FT, O.flatten_params(new_ft))
    o2 = O.Oracle(o.d, o.h, o.actor, new_ft, o.critic)
    actions, chains = _sample(o, e, B, obs, x_T, noise)
    torch.cuda.synchronize()
    assert e.last_path() == 1
    _check(o2, o2.sample(obs, x_T, noise), B, actions, chains)
    e.close()


# ---------------------------------------------------------------- precision modes
@pytest.mark.parametrize("name", CLUSTER)
def test_tensor_modes_take_the_same_kernel(engines, name):
    """Below their tensor-core row limits the bf16 and bf16x3 engines sample with the same fp32 kernel on the same weights: the
    results are bit-identical to the fp32 engine's."""
    o, ref = oracle(name), engines(name)
    B = 40
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=17)
    want_inj = [t.clone() for t in _sample(o, ref, B, obs, x_T, noise)]
    want_phx = [t.clone() for t in ref.sample(obs.reshape(B, -1), seed=3, offset=8)]
    for prec in (L.PREC_BF16, L.PREC_BF16X3):
        e = make_engine(o, prec)
        got_inj = _sample(o, e, B, obs, x_T, noise)
        torch.cuda.synchronize()
        assert e.last_path() == 1
        got_phx = e.sample(obs.reshape(B, -1), seed=3, offset=8)
        torch.cuda.synchronize()
        assert e.last_path() == 1
        for g, w in zip(got_inj + got_phx, want_inj + want_phx):
            assert torch.equal(g, w), prec
        e.close()


@pytest.mark.parametrize("name", CLUSTER)
def test_default_path_switches_at_the_row_limit(engines, name):
    """Past each width's measured crossover (DESIGN.md §5.3) the fp32 engine samples on the layered path."""
    o, e = oracle(name), engines(name)
    limit = ROW_LIMITS[name]
    obs = torch.rand(limit + 1, o.d.obs_dim, device="cuda") * 2 - 1
    for B, path in ((limit, 1), (limit + 1, 2)):
        e.sample(obs[:B], seed=1, offset=2)
        torch.cuda.synchronize()
        assert e.last_path() == path, B


# ---------------------------------------------------------------- rollout step with the env epilogue
@pytest.mark.parametrize("name", ["H256-A12", "H768-A24", "H1024-A128"])
def test_rollout_step_is_two_launches(name):
    o = oracle(name)
    e = make_engine(o)
    Do, Da, Ta = o.d.obs_dim, o.d.action_dim, o.d.horizon_steps
    rng = np.random.default_rng(1)
    norm = {"obs_min": -np.ones(Do, np.float32) * 2, "obs_max": np.ones(Do, np.float32) * 3,
            "action_min": -rng.uniform(0.5, 2, Da).astype(np.float32), "action_max": rng.uniform(0.5, 2, Da).astype(np.float32)}
    e.set_env_normalization(**norm)
    B, act_steps = 40, Ta // 2
    raw_obs = torch.from_numpy(rng.uniform(-2, 3, (B, Do))).pin_memory()
    raw_act = torch.zeros(B, act_steps * Da).pin_memory()
    obs_out = torch.zeros(B, Do, device="cuda"); act = torch.zeros(B, o.d.A, device="cuda")
    ch = torch.zeros(B, o.d.ft_denoising_steps + 1, o.d.A, device="cuda")
    e.rollout_step(raw_obs, obs_out, act, ch, raw_act, act_steps, seed=5, offset=9)
    n0 = e.launch_count()
    e.rollout_step(raw_obs, obs_out, act, ch, raw_act, act_steps, seed=5, offset=9)
    torch.cuda.synchronize()
    assert e.launch_count() - n0 == 2 and e.last_path() == 1         # normalise kernel + the persistent sampler
    a = act.cpu().numpy().reshape(B, Ta, Da)[:, :act_steps]
    want_act = ((a + 1) / 2) * (norm["action_max"] - norm["action_min"]) + norm["action_min"]
    np.testing.assert_array_equal(raw_act.numpy().reshape(B, act_steps, Da), want_act.astype(np.float32))
    a2, _ = e.sample(obs_out, seed=5, offset=9)
    assert torch.equal(a2, act)
    e.close()


# ---------------------------------------------------------------- the public shim
def test_ppo_diffusion_1024_wide_actor_samples_on_the_cluster_kernel():
    """PPODiffusion(actor=DiffusionMLP(mlp_dims=[1024] * 3)) samples its rollout on path 1 and matches the oracle."""
    o = oracle("H1024-A24")
    d = o.d
    actor = dp.DiffusionMLP(action_dim=d.action_dim, horizon_steps=d.horizon_steps, cond_dim=d.obs_dim, time_dim=d.time_dim,
                            mlp_dims=[1024] * 3, activation_type="ReLU", residual_style=True)
    critic = dp.CriticObs(cond_dim=d.obs_dim, mlp_dims=[256] * 3, activation_type="Mish", residual_style=True)
    model = dp.PPODiffusion(gamma_denoising=0.99, clip_ploss_coef=0.01, clip_ploss_coef_base=0.01, clip_ploss_coef_rate=3,
                            randn_clip_value=3, min_sampling_denoising_std=0.1, min_logprob_denoising_std=0.1,
                            actor=actor, critic=critic, ft_denoising_steps=d.ft_denoising_steps, horizon_steps=d.horizon_steps,
                            obs_dim=d.obs_dim, action_dim=d.action_dim, denoising_steps=d.denoising_steps, device="cuda:0")
    model.actor.set_flat_weights(O.flatten_params(o.actor))
    model.actor_ft.set_flat_weights(O.flatten_params(o.actor_ft))
    model.critic.set_flat_weights(O.flatten_params(o.critic))
    B = 40
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=1)
    want = o.sample(obs, x_T, noise)
    s = model(cond={"state": obs.cuda()}, deterministic=False, return_chain=True, x_T=x_T, noise=noise)
    torch.cuda.synchronize()
    assert model.engine.last_path() == 1
    assert s.trajectories.shape == (B, d.horizon_steps, d.action_dim)
    assert rel_err(s.trajectories, want.trajectories) < ACT_RTOL and rel_err(s.chains, want.chains) < ACT_RTOL
    s2 = model(cond={"state": obs.numpy()})
    assert model.engine.last_path() == 1 and np.isfinite(s2.chains).all()
