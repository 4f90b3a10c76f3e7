"""GPU (-m gpu): the split-precision (bf16x3) update chain after the weight-gradient launch.

In this mode one launch applies AdamW and rebuilds every table derived from the updated weights (the actor's time tables, the
plane copies of W1 and of the layer-0 rows); `set_weights` rebuilds the same tables with the separate prep kernels.  The time-MLP
backward runs on T + H/32 blocks with a finisher block.  Two configurations at the benchmarked dimensions (H = 512, Hc = 256,
T = 20, time_dim 16):
  bench     walker2d, the default Hyper: ReLU actor, Mish critic, A = 24 (the shapes bench.py times)
  mish-A9   hopper with a Mish actor and horizon 3: A = 9, the thread-per-row loss and the separate-launch tail
Checked:
  * after several applied updates, a fresh engine given the updated actor_ft and critic weights through set_weights gives
    bit-identical log-probs, values and seeded samples (large-batch plane sampler and 40-env cluster sampler): the planes, the time
    tables and the folded output layer built by the update match the ones built from the weights;
  * an update whose minibatch has an out-of-range index leaves the weights, the moments and those outputs untouched;
  * the gradient of the time MLP, of the W_in time rows and of b_in is within the mode's bound (1e-3 of the gradient's max) of
    the fp32 oracle.
"""
import functools

import numpy as np
import pytest
import torch

from diffusionpolicyoptimization_b200 import _lib as L
from oracle import dppo_oracle as O
from helpers import make_engine

pytestmark = pytest.mark.gpu

CASES = {
    "bench": dict(task="walker2d"),
    "mish-A9": dict(task="hopper", hyper=dict(actor_act="Mish"), dims=dict(horizon_steps=3)),
}
N_PPO, B_LP, B_SAMPLE, B_ENV = 4099, 256, 2304, 40
GRAD_TOL = 1e-3


@functools.lru_cache(maxsize=None)
def oracle(name) -> O.Oracle:
    c = CASES[name]
    return O.make_oracle(c["task"], seed=0, hyper=O.Hyper(**c.get("hyper", {})), **c.get("dims", {}))


@functools.lru_cache(maxsize=None)
def ppo_batch(name):
    return tuple(O.make_ppo_batch(oracle(name), N_PPO, pool=512, seed=3))


def _step(e, o, batch, lr, apply=True, want_grads=False):
    N = batch[0].shape[0]
    return e.ppo_step(batch[0].reshape(N, -1), batch[1].reshape(N, -1), batch[2].reshape(N, -1), batch[3], batch[4], batch[5],
                      batch[6], batch[7].reshape(N, -1), lr=lr, apply=apply, want_grads=want_grads)


def _outputs(e, o):
    """log-probs of stored chains, values, and seeded samples of both samplers; everything reads actor_ft / critic"""
    d = o.d
    g = torch.Generator(device="cuda").manual_seed(21)
    obs = torch.rand(B_SAMPLE, d.Do, device="cuda", generator=g) * 2 - 1
    act, chains = e.sample(obs, seed=5, offset=3)
    act_env, _ = e.sample(obs[:B_ENV].contiguous(), seed=6, offset=1)
    lp = e.logprobs(obs[:B_LP].contiguous(), chains[:B_LP].contiguous())
    v = e.value(obs)
    torch.cuda.synchronize()
    return {"sample": act, "sample_env": act_env, "logprobs": lp, "value": v}


def _fresh_with_weights_of(e, o):
    f = make_engine(o, L.PREC_BF16X3)
    f.set_weights(L.NET_ACTOR_FT, e.get_weights(L.NET_ACTOR_FT))
    f.set_weights(L.NET_CRITIC, e.get_weights(L.NET_CRITIC))
    return f


@pytest.mark.parametrize("name", list(CASES))
def test_updated_operands_match_set_weights(name):
    o = oracle(name)
    e = make_engine(o, L.PREC_BF16X3)
    w_start = e.get_weights(L.NET_ACTOR_FT).copy()
    for _ in range(3):
        _step(e, o, ppo_batch(name), lr=1e-3)
    torch.cuda.synchronize()
    assert not np.array_equal(e.get_weights(L.NET_ACTOR_FT), w_start)
    f = _fresh_with_weights_of(e, o)
    got, want = _outputs(e, o), _outputs(f, o)
    for k in want:
        assert torch.equal(got[k], want[k]), k
    e.close(); f.close()


@pytest.mark.parametrize("name", list(CASES))
def test_update_with_a_bad_index_changes_nothing(name):
    o = oracle(name)
    e = make_engine(o, L.PREC_BF16X3)
    _step(e, o, ppo_batch(name), lr=1e-3)                      # moments and tables of an applied step
    torch.cuda.synchronize()
    w0 = e.get_weights(L.NET_ACTOR_FT).copy(); c0 = e.get_weights(L.NET_CRITIC).copy()
    m0, v0, _ = e.get_opt_state(L.OPT_FINETUNE)
    before = _outputs(e, o)
    d = o.d
    P, K, A = 600, d.ft_denoising_steps, d.A
    obs, x_T, noise = O.make_rollout_inputs(o, P, seed=77)
    chains = o.sample(obs, x_T, noise).chains.reshape(P, K + 1, A)
    g = torch.Generator().manual_seed(5)
    olp = torch.randn(P, K, A, generator=g) * 0.3 - 1.0
    ret, val, adv = torch.randn(P, generator=g), torch.randn(P, generator=g), torch.randn(P, generator=g)
    flat = torch.randint(0, P * K, (N_PPO,), generator=g, dtype=torch.int32)
    flat[17] = P * K + 3
    mb = e.ppo_step_indexed(obs.reshape(P, -1), chains, olp, ret, val, adv, flat.cuda(), lr=1e-3, apply=True)
    torch.cuda.synchronize()
    assert torch.isnan(mb).all()
    m1, v1, _ = e.get_opt_state(L.OPT_FINETUNE)
    assert np.array_equal(e.get_weights(L.NET_ACTOR_FT), w0) and np.array_equal(e.get_weights(L.NET_CRITIC), c0)
    assert np.array_equal(m1, m0) and np.array_equal(v1, v0)
    after = _outputs(e, o)
    for k in before:
        assert torch.equal(after[k], before[k]), k
    e.close()


@pytest.mark.parametrize("name", list(CASES))
def test_time_mlp_and_input_bias_gradients(name):
    o = oracle(name)
    d = o.d
    e = make_engine(o, L.PREC_BF16X3)
    batch = ppo_batch(name)
    _, g = _step(e, o, batch, lr=0.0, apply=False, want_grads=True)
    torch.cuda.synchronize()
    _, ga, gc = o.ppo_grads(*batch)
    want = np.concatenate([O.flatten_params(ga), O.flatten_params(gc)])
    got = g.cpu().numpy()
    td, H, A = d.time_dim, d.actor_hidden, d.A
    mlp = 4 * td * td + 3 * td                                 # time MLP: W1, b1, W2, b2
    win = mlp                                                  # W_in rows [x (A) | time (td) | obs]
    bin_ = win + (A + td + d.Do) * H
    sel = np.r_[0:mlp, win + A * H:win + (A + td) * H, bin_:bin_ + H]
    scale = float(np.abs(want).max())
    err = float(np.abs(got[sel] - want[sel]).max()) / scale
    print(f"{name}: time-MLP / W_in time rows / b_in gradient error {err:.2e} of max")
    assert err < GRAD_TOL, err
    assert float(np.abs(want[sel]).max()) > 1e-3 * scale        # the entries carry signal at this scale
    e.close()
