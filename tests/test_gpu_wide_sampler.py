"""GPU (-m gpu): the persistent cluster sampler for action chunks wider than 32 (32 < A = horizon_steps x action_dim <= 128).

sample_cluster_wide_kernel<AP, R> (csrc/sample_cluster.cuh, AP in {64, 128}) is the rollout sampler of these chunks below the
row limits of dppo_sample (path 1); the layer-by-layer fp32 sampler (path 2) and the oracle are the references.  Cases:
  A40   5 x 8, Do 11
  A42   7 x 6, Do 17: A % 4 != 0, the padded columns of the AP = 64 instantiation are masked
  A56   14 x 4, Do 59 (a robomimic-transport-sized chunk)
  A112  14 x 8, Do 59
  A128  16 x 8, Do 59: the widest chunk the kernel covers
  A132  33 x 4, Do 11: wider than 128, stays on the layered path even when path 1 is asked for
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
CASES = {
    "A40": dict(action_dim=5, horizon_steps=8, obs_dim=11),
    "A42": dict(action_dim=7, horizon_steps=6, obs_dim=17),
    "A56": dict(action_dim=14, horizon_steps=4, obs_dim=59),
    "A112": dict(action_dim=14, horizon_steps=8, obs_dim=59),
    "A128": dict(action_dim=16, horizon_steps=8, obs_dim=59),
    "A132": dict(action_dim=33, horizon_steps=4, obs_dim=11),
}
NAMES = list(CASES)
CLUSTER = [n for n in NAMES if n != "A132"]


@functools.lru_cache(maxsize=None)
def oracle(name, **over):
    return O.make_oracle("hopper", seed=0, **CASES[name], **over)


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
    return 2 if name == "A132" else path


def _sample(o, e, B, obs, x_T, noise, **kw):
    return e.sample(obs.reshape(B, -1), x_T=x_T.reshape(B, -1), noise=noise.reshape(o.d.denoising_steps, B, -1), **kw)


def _check(o, want, B, actions, chains):
    assert rel_err(actions, want.trajectories.reshape(B, -1)) < ACT_RTOL
    assert rel_err(chains, want.chains.reshape(B, o.d.ft_denoising_steps + 1, -1)) < ACT_RTOL


def test_case_shapes():
    for name in NAMES:
        A = oracle(name).d.A
        assert A == int(name[1:]) and (32 < A <= 128) == (name in CLUSTER), name
    assert oracle("A42").d.A % 4 != 0


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


@pytest.mark.parametrize("name", ["A42", "A128"])
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
        o = O.make_oracle("hopper", seed=0, hyper=O.Hyper(final_action_clip_value=0.5), **CASES[name])
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
@pytest.mark.parametrize("name", ["A56", "A128"])
def test_set_weights_refreshes_the_folded_output_layer(name):
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


@pytest.mark.parametrize("name,limit", [("A56", 2048), ("A128", 1024)])
def test_default_path_switches_at_the_row_limit(engines, name, limit):
    """Past the measured crossover (DESIGN.md §5.3) the fp32 engine samples wide chunks on the layered path."""
    o, e = oracle(name), engines(name)
    obs = torch.rand(limit + 1, o.d.obs_dim, device="cuda") * 2 - 1
    for B, path in ((limit, 1), (limit + 1, 2)):
        e.sample(obs[:B], seed=1, offset=2)
        torch.cuda.synchronize()
        assert e.last_path() == path, B


# ---------------------------------------------------------------- rollout step with the env epilogue
@pytest.mark.parametrize("name", ["A42", "A112"])
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
