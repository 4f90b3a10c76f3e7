"""GPU (-m gpu): every weight-derived table follows every weight change, and AdamW against the kernels' own gradients.

A handle keeps copies derived from the fp32 master weights: the actor's time tables, the packed FFMA layer-0 weight w0p, the folded
output layer w23 / b23 of the persistent cluster sampler, the bf16 operand copies of the tensor mode and the plane copies and folded
layers of the split-precision mode.  Some are rebuilt by the call that changed the weights, the others lazily by their next reader
(mark_weights_changed marks them stale).  A stale table shows only when a reader ran before the change and runs again after it, so
each mutation test here:
  1. runs every reader once (every lazy table is built and its flag clear),
  2. applies the mutation,
  3. runs every reader again,
  4. forces a full rebuild (set_weights(net, get_weights(net)) for all four nets) and runs every reader a third time,
  5. requires 3 == 4: forward-only readers bit for bit, the PPO gradients (atomics in the tensor modes) within 1e-5 of their largest
     entry, the PPO metrics within 1e-5 relative (measured on a B200 at 1000 W between identical calls: 2.2e-8 in bf16 at hopper
     shapes, 0 elsewhere),
  6. requires every reader of a changed net to differ from 1 and every other reader to equal 1,
  7. (a skipped update) requires weights, moments and every reader to equal 1 while the step counter advances,
  8. compares small-row readers against the float64 oracle at the read-back weights: the 40-row cluster sample at the fp32 bound
     (1e-4 relative) in every mode, since that kernel is FFMA; 1000-row log-probs (1e-3 absolute) and values (2e-5 absolute), FFMA in
     every mode; and the 4096-row forward of each changed net at the mode's bound (eps 2e-5 / 2e-2 / 5e-6 relative for fp32 / bf16 /
     bf16x3, value 2e-5 / 2e-2 / 5e-5), which is what sees a lazy table that the rebuild in 4 does not rebuild either.  Largest
     errors measured on a B200 at 1000 W: sample 1.7e-6, log-probs 6.3e-6, value 7.8e-7 (1000 rows); eps 1.2e-6 / 4.6e-3 / 1.0e-6
     and value 7.8e-7 / 9.9e-3 / 1.3e-5 (4096 rows, fp32 / bf16 / bf16x3).
Geometries: the default hopper one (H 512, Hc 256, ReLU actor, Mish critic, A 12) and walker2d with 8-step chunks (A 48), where bf16
keeps the FFMA path and refreshes through prep_net and bf16x3 runs its wide path.  Each runs in fp32, bf16 and bf16x3.  Every reader
is checked to take the path it is named for (last_path() for the samplers, the tensor-core launch counter for the others).

The AdamW tests set random moments and a step counter of 999 (or 10^6), take one applied step that hands back its gradient, and
recompute w, m and v element by element with oracle.adamw_keras from that gradient (clipped by oracle.clip_by_norm when clipping is
on) and the state read before the step.  Bounds: 4 ulp of the value plus 1e-5 of the element's change, plus 4 ulp of each moment
update's terms and what those move the weight by.  This leaves room for FMA contraction, whose effect on a moment is large where g and
m nearly cancel, and for the clip norm's summation order, and for nothing else.  Measured on a B200 (1000 W): the worst element uses
0.25 of its bound in the fine-tuning slot and 0.44 in the pre-training slot (weight decay 0.1, lr 1e-2); without the moment terms one
pre-training element of 4.9e-4 was off by 15 ulp where the moment update cancelled.
"""
import functools

import numpy as np
import pytest
import torch

import diffusionpolicyoptimization_b200 as dp
from diffusionpolicyoptimization_b200 import _lib as L
from oracle import dppo_oracle as O
from helpers import make_cfg, make_engine, max_abs, rel_err

pytestmark = pytest.mark.gpu

PREC = {"fp32": L.PREC_FP32, "bf16": L.PREC_BF16, "bf16x3": L.PREC_BF16X3}
GEOMS = {"hopper": dict(task="hopper", dims={}), "wide": dict(task="walker2d", dims=dict(horizon_steps=8))}
ACTORS = (L.NET_ACTOR, L.NET_ACTOR_FT, L.NET_ACTOR_EMA)
NET_NAMES = {L.NET_ACTOR: "actor", L.NET_ACTOR_FT: "actor_ft", L.NET_CRITIC: "critic", L.NET_ACTOR_EMA: "actor_ema"}
SMALL, LARGE = 1000, 4096                     # below / above the tensor modes' 2048-row threshold
E_ROLL = 40
LR = 1e-3
GRAD_SPREAD = 1e-5
EPS_RTOL = {"fp32": 2e-5, "bf16": 2e-2, "bf16x3": 5e-6}
VALUE_TOL = {"fp32": 2e-5, "bf16": 2e-2, "bf16x3": 5e-5}       # fp32: absolute, tensor modes: relative


@functools.lru_cache(maxsize=None)
def oracle(geom):
    g = GEOMS[geom]
    return O.make_oracle(g["task"], seed=0, **g["dims"])


def _tensor_shape(geom, mode):
    """The handle's tensor path exists: bf16 covers A <= 32, bf16x3 every A of these geometries."""
    return mode == "bf16x3" or (mode == "bf16" and oracle(geom).d.A <= 32)


def _tensor(geom, mode, rows):
    return rows >= 2048 and _tensor_shape(geom, mode)


def _sample_path(geom, mode, B, force):
    """dppo_sample's choice (sample_impl): 1 cluster, 2 layered fp32, 3 layered tensor, 4 fused bf16 chain."""
    A = oracle(geom).d.A
    tensor = _tensor(geom, mode, B)
    limit = 1024 if mode == "bf16" else (4096 if A <= 32 else 2048)
    if not tensor and force != 2 and (B <= limit or force == 1):
        return 1
    if tensor and mode == "bf16" and force != 3:
        return 4
    return 3 if tensor else 2


# ---------------------------------------------------------------- fixed inputs of the readers and mutations
@functools.lru_cache(maxsize=None)
def inputs(geom):
    o = oracle(geom)
    d = o.d
    K, A, Do, T = d.ft_denoising_steps, d.A, d.Do, d.denoising_steps
    rng = np.random.default_rng(7)
    r = {}
    r["x"] = torch.from_numpy(rng.standard_normal((LARGE, A)).astype(np.float32))
    r["t"] = torch.from_numpy(rng.integers(0, T, LARGE).astype(np.int32))
    r["obs"] = torch.from_numpy(rng.uniform(-1, 1, (LARGE, Do)).astype(np.float32))
    P = 600
    obs, x_T, noise = O.make_rollout_inputs(o, P, seed=77)
    r["pool_obs"] = obs.reshape(P, Do)
    r["pool_chains"] = o.sample(obs, x_T, noise).chains.reshape(P, K + 1, A)
    g = torch.Generator().manual_seed(5)
    r["pool_olp"] = torch.randn(P, K, A, generator=g) * 0.3 - 1.0
    r["pool_ret"], r["pool_val"], r["pool_adv"] = torch.randn(P, generator=g), torch.randn(P, generator=g), torch.randn(P, generator=g)
    r["flat"] = torch.randint(0, P * K, (LARGE,), generator=g, dtype=torch.int64).to(torch.int32)
    for n in (SMALL, LARGE):
        b = O.make_ppo_batch(o, n, pool=256, seed=n)
        r[("ppo", n)] = [b[0].reshape(n, Do), b[1].reshape(n, A), b[2].reshape(n, A), b[3], b[4], b[5], b[6], b[7].reshape(n, A)]
        acts = torch.from_numpy(rng.uniform(-1, 1, (n, A)).astype(np.float32))
        st = torch.from_numpy(rng.uniform(-1, 1, (n, Do)).astype(np.float32))
        tt = torch.from_numpy(rng.integers(0, T, n).astype(np.int32))
        nz = torch.from_numpy(rng.standard_normal((n, A)).astype(np.float32))
        r[("pre", n)] = (acts, st, tt, nz)
    for B in (E_ROLL, LARGE):
        ob, xT, nz = O.make_rollout_inputs(o, B, seed=B + 1)
        r[("roll", B)] = (ob.reshape(B, Do), xT.reshape(B, A), nz.reshape(T, B, A))
    r["raw_obs"] = torch.from_numpy(rng.uniform(-2, 3, (E_ROLL, Do)))
    r["norm"] = dict(obs_min=-np.ones(Do, np.float32) * 2, obs_max=np.ones(Do, np.float32) * 3,
                     action_min=-rng.uniform(0.5, 2, d.action_dim).astype(np.float32),
                     action_max=rng.uniform(0.5, 2, d.action_dim).astype(np.float32))
    return r


@pytest.fixture(scope="module")
def engines():
    made = {}

    def get(geom, mode):
        if (geom, mode) not in made:
            o = oracle(geom)
            e = make_engine(o, PREC[mode])
            ema = O.flatten_params(o.actor) + 0.01 * np.random.default_rng(3).standard_normal(e.n_actor).astype(np.float32)
            e.set_weights(L.NET_ACTOR_EMA, ema)           # the EMA net differs from the actor, so that ema_update changes it
            e.set_env_normalization(**inputs(geom)["norm"])
            made[(geom, mode)] = e
        return made[(geom, mode)]

    yield get
    for e in made.values():
        e.close()


# ---------------------------------------------------------------- readers
class Reader:
    def __init__(self, name, nets, fn, kind="fwd", path=None, tensor=None):
        self.name, self.nets, self.fn, self.kind, self.path, self.tensor = name, frozenset(nets), fn, kind, path, tensor


def readers(geom, mode, e):
    o, r = oracle(geom), inputs(geom)
    d = o.d
    K = d.ft_denoising_steps
    out = []
    for net in ACTORS:
        for n in (SMALL, LARGE):
            out.append(Reader(f"fwd_{NET_NAMES[net]}_{n}", [net],
                              functools.partial(lambda net, n: [e.actor_forward(net, r["x"][:n], r["t"][:n], r["obs"][:n])], net, n),
                              tensor=_tensor(geom, mode, n)))
    for n in (SMALL, LARGE):
        out.append(Reader(f"value_{n}", [L.NET_CRITIC], functools.partial(lambda n: [e.value(r["obs"][:n])], n), tensor=_tensor(geom, mode, n)))
    for base in (0, 1):
        lp_net = L.NET_ACTOR if base else L.NET_ACTOR_FT
        for B in (SMALL // K, (LARGE + K - 1) // K):
            out.append(Reader(f"logprobs_{B * K}_base{base}", [lp_net],
                              functools.partial(lambda B, base: [e.logprobs(r["pool_obs"][:B], r["pool_chains"][:B], use_base_policy=bool(base))], B, base),
                              tensor=_tensor(geom, mode, B * K)))
        for n in (SMALL, LARGE):
            b = r[("ppo", n)]
            out.append(Reader(f"logprobs_sub_{n}_base{base}", [lp_net],
                              functools.partial(lambda b, base: [e.logprobs_subsample(*b[:4], use_base_policy=bool(base))], b, base),
                              tensor=_tensor(geom, mode, n)))
        s_nets = [L.NET_ACTOR] if base else [L.NET_ACTOR, L.NET_ACTOR_FT]
        sample_cases = [(E_ROLL, 1), (E_ROLL, 2), (LARGE, 0)]
        if mode == "bf16" and _tensor_shape(geom, mode):
            sample_cases.append((LARGE, 3))               # the per-layer tensor sampler beside the fused chain
        for B, force in sample_cases:
            def sample(B=B, force=force, base=base):
                ob, xT, nz = r[("roll", B)]
                e.force_path(force)
                try:
                    return list(e.sample(ob, x_T=xT, noise=nz, use_base_policy=bool(base)))
                finally:
                    e.force_path(0)
            out.append(Reader(f"sample_{B}_path{force}_base{base}", s_nets, sample, path=_sample_path(geom, mode, B, force)))

    def rollout():
        obs_out = torch.zeros(E_ROLL, d.Do, device="cuda"); act = torch.zeros(E_ROLL, d.A, device="cuda")
        ch = torch.zeros(E_ROLL, K + 1, d.A, device="cuda")
        raw_act = torch.zeros(E_ROLL, 2 * d.action_dim).pin_memory()
        ob, xT, nz = r[("roll", E_ROLL)]
        if "raw_obs_pinned" not in r:
            r["raw_obs_pinned"] = r["raw_obs"].pin_memory()
        e.rollout_step(r["raw_obs_pinned"], obs_out, act, ch, raw_act, 2, x_T=xT, noise=nz)
        torch.cuda.synchronize()
        return [act, ch, raw_act]
    out.append(Reader("rollout_step", [L.NET_ACTOR, L.NET_ACTOR_FT], rollout, path=1))
    for n in (SMALL, LARGE):
        b = r[("ppo", n)]
        out.append(Reader(f"ppo_grads_{n}", [L.NET_ACTOR_FT, L.NET_CRITIC],
                          functools.partial(lambda b: list(e.ppo_step(*b, lr=0.0, apply=False, want_grads=True)), b),
                          kind="grad", tensor=_tensor(geom, mode, n)))
    return out


def run_readers(e, rds):
    res = {}
    for rd in rds:
        n0 = e.tc_launch_count()
        outs = rd.fn()
        torch.cuda.synchronize()
        if rd.path is not None:
            assert e.last_path() == rd.path, (rd.name, e.last_path(), rd.path)
        if rd.tensor is not None:
            assert (e.tc_launch_count() > n0) == rd.tensor, (rd.name, e.tc_launch_count() - n0)
        res[rd.name] = [t.detach().cpu().numpy().copy() for t in outs]
    return res


def _grad_diff(a, b):
    """(metrics relative difference, gradient difference / largest gradient entry) of a ppo_grads reader."""
    (ma, ga), (mb, gb) = a, b
    dm = float(np.max(np.abs(ma - mb) / np.maximum(np.abs(mb), 1e-6)))
    return dm, float(np.abs(ga - gb).max() / np.abs(gb).max())


def _same(rd, a, b):
    if rd.kind == "grad":
        dm, dg = _grad_diff(a, b)
        return dm <= GRAD_SPREAD and dg <= GRAD_SPREAD
    return all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


def _differs(rd, a, b):
    if rd.kind == "grad":
        return _grad_diff(a, b)[1] > 100 * GRAD_SPREAD
    return not all(np.array_equal(x, y) for x, y in zip(a, b))


def _rebuild_all(e):
    for net in (L.NET_ACTOR, L.NET_ACTOR_FT, L.NET_CRITIC, L.NET_ACTOR_EMA):
        e.set_weights(net, e.get_weights(net))


# ---------------------------------------------------------------- float64 oracle at the read-back weights
def _oracle64(geom, e):
    o = oracle(geom)
    d = o.d
    un = lambda net, shapes: [p.double() for p in O.unflatten_params(e.get_weights(net), shapes)]
    nets = {net: un(net, d.actor_shapes()) for net in ACTORS}
    nets[L.NET_CRITIC] = un(L.NET_CRITIC, d.critic_shapes())
    return O.Oracle(d, o.h, nets[L.NET_ACTOR], nets[L.NET_ACTOR_FT], nets[L.NET_CRITIC]), nets


def check_oracle(geom, mode, e, res, changed, errs):
    o, r = oracle(geom), inputs(geom)
    d = o.d
    K = d.ft_denoising_steps
    o64, nets = _oracle64(geom, e)
    ob, xT, nz = r[("roll", E_ROLL)]
    with torch.no_grad():
        for base in (0, 1):
            want = o64.sample(ob.double().reshape(E_ROLL, 1, -1), xT.double().reshape(E_ROLL, d.horizon_steps, -1),
                              nz.double().reshape(d.denoising_steps, E_ROLL, d.horizon_steps, -1), use_base_policy=bool(base))
            act, ch = res[f"sample_{E_ROLL}_path1_base{base}"]
            err = max(rel_err(act, want.trajectories.reshape(E_ROLL, -1)), rel_err(ch, want.chains.reshape(E_ROLL, K + 1, -1)))
            errs["sample40"] = max(errs.get("sample40", 0.0), err)
            assert err < 1e-4, ("sample40", base, err)
            b = r[("ppo", SMALL)]
            lp, _ = o64.get_logprobs_subsample(b[0].double(), b[1].double().reshape(SMALL, d.horizon_steps, -1),
                                               b[2].double().reshape(SMALL, d.horizon_steps, -1), b[3], use_base_policy=bool(base))
            err = max_abs(res[f"logprobs_sub_{SMALL}_base{base}"][0], lp.reshape(SMALL, -1))
            errs["logp1000"] = max(errs.get("logp1000", 0.0), err)
            assert err < 1e-3, ("logp1000", base, err)
        v = O.critic_obs(nets[L.NET_CRITIC], r["obs"][:SMALL].double(), o.h.critic_act).reshape(-1)
        err = max_abs(res[f"value_{SMALL}"][0], v)
        errs["value1000"] = max(errs.get("value1000", 0.0), err)
        assert err < 2e-5, ("value1000", err)
        for net in changed:
            if net == L.NET_CRITIC:
                v = O.critic_obs(nets[net], r["obs"].double(), o.h.critic_act).reshape(-1)
                got = res[f"value_{LARGE}"][0]
                err = max_abs(got, v) if mode == "fp32" else rel_err(got, v)
                key = f"value{LARGE}"
                tol = VALUE_TOL[mode]
            else:
                want = O.diffusion_mlp(nets[net], r["x"].double().reshape(LARGE, d.horizon_steps, -1), r["t"].long(),
                                       r["obs"].double().reshape(LARGE, 1, -1), d, o.h.actor_act).reshape(LARGE, -1)
                err = rel_err(res[f"fwd_{NET_NAMES[net]}_{LARGE}"][0], want)
                key, tol = f"eps{LARGE}", EPS_RTOL[mode]
            errs[key] = max(errs.get(key, 0.0), err)
            assert err < tol, (key, NET_NAMES[net], err, tol)


# ---------------------------------------------------------------- mutations
def _perturbed(e, net, seed):
    w = e.get_weights(net)
    return w + 1e-3 * np.random.default_rng(seed).standard_normal(w.size).astype(np.float32)


def _ppo(geom, e, n, clip=False):
    e.set_grad_clip_norm(0.05 if clip else None)
    try:
        e.ppo_step(*inputs(geom)[("ppo", n)], lr=LR, apply=True)
        torch.cuda.synchronize()
    finally:
        e.set_grad_clip_norm(None)


def _indexed(geom, e, bad=False):
    r = inputs(geom)
    inds = r["flat"].clone()
    if bad:
        inds[17] = r["pool_chains"].shape[0] * oracle(geom).d.ft_denoising_steps + 3
    m = e.ppo_step_indexed(r["pool_obs"], r["pool_chains"], r["pool_olp"], r["pool_ret"], r["pool_val"], r["pool_adv"], inds.cuda(),
                           lr=LR, apply=True)
    torch.cuda.synchronize()
    assert bool(torch.isnan(m).all()) == bad


def _pretrain(geom, e, n):
    acts, st, tt, nz = inputs(geom)[("pre", n)]
    e.pretrain_step(acts, st, lr=LR, apply=True, t=tt, noise=nz)
    torch.cuda.synchronize()


FT_CRITIC = (L.NET_ACTOR_FT, L.NET_CRITIC)
MUTATIONS = {}
for _net in (L.NET_ACTOR, L.NET_ACTOR_FT, L.NET_CRITIC, L.NET_ACTOR_EMA):
    MUTATIONS[f"set_weights_{NET_NAMES[_net]}_host"] = ((_net,), lambda g, e, net=_net: e.set_weights(net, _perturbed(e, net, 10 + net)))
    MUTATIONS[f"set_weights_{NET_NAMES[_net]}_device"] = (
        (_net,), lambda g, e, net=_net: e.set_weights(net, torch.from_numpy(_perturbed(e, net, 20 + net)).cuda()))
MUTATIONS.update({
    f"ppo_{SMALL}": (FT_CRITIC, lambda g, e: _ppo(g, e, SMALL)),
    f"ppo_{LARGE}": (FT_CRITIC, lambda g, e: _ppo(g, e, LARGE)),
    f"ppo_{SMALL}_clip": (FT_CRITIC, lambda g, e: _ppo(g, e, SMALL, clip=True)),
    f"ppo_{LARGE}_clip": (FT_CRITIC, lambda g, e: _ppo(g, e, LARGE, clip=True)),
    "ppo_indexed": (FT_CRITIC, lambda g, e: _indexed(g, e)),
    f"pretrain_{SMALL}": ((L.NET_ACTOR,), lambda g, e: _pretrain(g, e, SMALL)),
    f"pretrain_{LARGE}": ((L.NET_ACTOR,), lambda g, e: _pretrain(g, e, LARGE)),
    "ema_update": ((L.NET_ACTOR_EMA,), lambda g, e: e.ema_update(0.9)),
    "skipped_update": ((), lambda g, e: _indexed(g, e, bad=True)),
})


def _grid(names):
    return [pytest.param(g, m, n, id=f"{g}-{m}-{n}") for g in GEOMS for m in PREC for n in names]


@pytest.mark.parametrize("geom,mode", [pytest.param(g, m, id=f"{g}-{m}") for g in GEOMS for m in PREC])
def test_readers_are_deterministic(engines, geom, mode):
    """Every forward-only reader gives bit-identical results on an unchanged handle (what the refresh comparison relies on), and the
    PPO gradients agree within their 1e-5 spread."""
    e = engines(geom, mode)
    rds = readers(geom, mode, e)
    a = run_readers(e, rds)
    b = run_readers(e, rds)
    spread = 0.0
    for rd in rds:
        assert _same(rd, a[rd.name], b[rd.name]), rd.name
        if rd.kind == "grad":
            spread = max(spread, _grad_diff(a[rd.name], b[rd.name])[1])
    print(f"{geom}-{mode}: PPO gradient spread between identical calls {spread:.2e} of the largest entry")


@pytest.mark.parametrize("geom,mode,mutation", _grid(list(MUTATIONS)))
def test_tables_follow_weight_changes(engines, geom, mode, mutation):
    e = engines(geom, mode)
    changed, apply = MUTATIONS[mutation]
    rds = readers(geom, mode, e)
    before = run_readers(e, rds)
    w_before = {net: e.get_weights(net) for net in NET_NAMES}
    opt_before = [e.get_opt_state(s) for s in (L.OPT_PRETRAIN, L.OPT_FINETUNE)]
    apply(geom, e)
    after = run_readers(e, rds)
    _rebuild_all(e)
    rebuilt = run_readers(e, rds)
    stale = [rd.name for rd in rds if not _same(rd, after[rd.name], rebuilt[rd.name])]
    assert not stale, f"readers that saw stale tables after {mutation}: {stale}"
    for net in NET_NAMES:
        assert np.array_equal(e.get_weights(net), w_before[net]) != (net in changed), (NET_NAMES[net], "weights")
    for rd in rds:
        if rd.nets & set(changed):
            assert _differs(rd, after[rd.name], before[rd.name]), (rd.name, "did not change")
        else:
            assert _same(rd, after[rd.name], before[rd.name]), (rd.name, "changed")
    if mutation == "skipped_update":
        for slot, (m0, v0, st0) in zip((L.OPT_PRETRAIN, L.OPT_FINETUNE), opt_before):
            m1, v1, st1 = e.get_opt_state(slot)
            assert np.array_equal(m1, m0) and np.array_equal(v1, v0)
            assert st1 == st0 + (slot == L.OPT_FINETUNE)          # the step counter advances even when the update is skipped
    errs = {}
    check_oracle(geom, mode, e, after, changed, errs)
    print(f"{geom}-{mode}-{mutation}: oracle errors " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(errs.items())))


# ---------------------------------------------------------------- AdamW against the kernel's own gradient
def _ulp(x):
    return np.spacing(np.abs(x).astype(np.float32))


def _check_adamw(cfg, w0, m0, v0, g, step, lr, wd, w1, m1, v1, parts):
    """w1 / m1 / v1 (the kernel's) against oracle.adamw_keras from (w0, m0, v0, g) at 1-based `step`; worst error over bound."""
    p, mi, vi = (torch.from_numpy(a.copy()) for a in (w0, m0, v0))
    gt = torch.from_numpy(g)
    O.adamw_keras([p], [gt], [mi], [vi], step, lr, cfg.adam_beta1, cfg.adam_beta2, cfg.adam_eps, wd)
    p, mi, vi = p.numpy(), mi.numpy(), vi.numpy()
    c1, c2 = np.float32(1 - cfg.adam_beta1), np.float32(1 - cfg.adam_beta2)
    # the roundings of each moment update, with or without FMA contraction (large when g and m nearly cancel) ...
    dm = 4 * _ulp(mi) + 4 * _ulp(c1 * (g - m0))
    dv = 4 * _ulp(vi) + 4 * _ulp(c2 * (g * g - v0)) + 4 * c2 * _ulp(g * g)
    # ... and what they move the weight by: step = alpha m / (sqrt(v) + eps)
    alpha = lr * np.sqrt(1 - cfg.adam_beta2 ** step) / (1 - cfg.adam_beta1 ** step)
    den = np.sqrt(vi.astype(np.float64)) + cfg.adam_eps
    bw = 4 * _ulp(np.maximum(np.abs(w0), np.abs(p))) + 1e-5 * np.abs(p - w0) + alpha * dm / den + alpha * np.abs(mi) / den * 0.5 * dv / vi
    bm = dm + 1e-5 * np.abs(c1 * g)
    bv = dv + 1e-5 * c2 * g * g
    worst = 0.0
    for name, sl in parts.items():
        for what, got, want, bound in (("w", w1, p, bw), ("m", m1, mi, bm), ("v", v1, vi, bv)):
            r = np.abs(got[sl] - want[sl]) / np.maximum(bound[sl], 1e-38)
            i = int(np.argmax(r))
            assert r[i] <= 1.0, (name, what, i, float(got[sl][i]), float(want[sl][i]), float(bound[sl][i]))
            worst = max(worst, float(r[i]))
        assert not np.array_equal(w1[sl], w0[sl]), (name, "unchanged")
    return worst


def _clipped(g, d, nA):
    shapes = d.actor_shapes() + d.critic_shapes()
    parts = O.unflatten_params(g, shapes)
    return O.flatten_params(O.clip_by_norm(parts, 0.05))


def _parts(d, nA, n):
    """Index ranges of the flat [actor_ft | critic] vector: the ones ts_update_kernel's last time block writes, and the rest."""
    off = np.cumsum([0] + [int(np.prod(s)) for s in d.actor_shapes()])
    win, bin_ = off[4], off[5]
    t0, t1 = win + d.A * d.actor_hidden, win + (d.A + d.time_dim) * d.actor_hidden
    return {"time_mlp": slice(0, win), "w_in_time_rows": slice(t0, t1), "b_in": slice(bin_, bin_ + d.actor_hidden),
            "w_in_other_rows": slice(win, t0), "rest_of_actor": slice(bin_ + d.actor_hidden, nA), "critic": slice(nA, n)}


def _pretrain_cfg(mode):
    cfg = make_cfg(oracle("hopper"), PREC[mode])
    cfg.pretrain_weight_decay = 0.1                # with lr 1e-2 the decay term is >= 100 ulp of the weight
    return cfg


@pytest.mark.parametrize("mode,rows,clip", [("fp32", SMALL, False), ("fp32", LARGE, False), ("bf16", SMALL, False), ("bf16", LARGE, False),
                                            ("bf16x3", LARGE, False), ("fp32", SMALL, True), ("bf16x3", LARGE, True)])
@pytest.mark.parametrize("step0", [999, 10 ** 6])
def test_adamw_finetune_matches_keras(mode, rows, clip, step0):
    """adamw_kernel (fp32, bf16, the clip path) and ts_update_kernel (bf16x3 without clipping) over two consecutive steps: the second
    also shows that ts_update_kernel's completion counter was reset."""
    o = oracle("hopper")
    d = o.d
    e = make_engine(o, PREC[mode])
    nA, n = e.n_actor, e.n_actor + e.n_critic
    parts = _parts(d, nA, n)
    rng = np.random.default_rng(step0 + rows)
    e.set_opt_state(L.OPT_FINETUNE, 1e-3 * rng.standard_normal(n).astype(np.float32), (1e-6 * rng.uniform(0.5, 2, n)).astype(np.float32), step0)
    e.set_grad_clip_norm(0.05 if clip else None)
    cfg = e.cfg
    worst = 0.0
    for k in range(2):
        w0 = np.concatenate([e.get_weights(L.NET_ACTOR_FT), e.get_weights(L.NET_CRITIC)])
        m0, v0, st0 = e.get_opt_state(L.OPT_FINETUNE)
        _, g = e.ppo_step(*inputs("hopper")[("ppo", rows)], lr=LR, apply=True, want_grads=True)
        g = g.cpu().numpy()
        if clip:
            g = _clipped(g, d, nA)
        w1 = np.concatenate([e.get_weights(L.NET_ACTOR_FT), e.get_weights(L.NET_CRITIC)])
        m1, v1, st1 = e.get_opt_state(L.OPT_FINETUNE)
        assert st1 == st0 + 1 == step0 + k + 1
        worst = max(worst, _check_adamw(cfg, w0, m0, v0, g, st1, LR, cfg.weight_decay, w1, m1, v1, parts))
    e.close()
    print(f"adamw {mode} rows {rows} clip {clip} step {step0 + 1}: worst error / bound {worst:.3f}")


@pytest.mark.parametrize("mode,rows", [("fp32", SMALL), ("bf16", LARGE), ("bf16x3", LARGE)])
@pytest.mark.parametrize("step0", [999, 10 ** 6])
def test_adamw_pretrain_matches_keras(mode, rows, step0):
    """The pre-training slot with a weight decay large enough to be seen (0.1 x lr 1e-2), two consecutive steps."""
    o = oracle("hopper")
    d = o.d
    e = dp.Engine(_pretrain_cfg(mode), 0)
    e.set_weights(L.NET_ACTOR, O.flatten_params(o.actor))
    nA = e.n_actor
    rng = np.random.default_rng(step0 + rows + 1)
    e.set_opt_state(L.OPT_PRETRAIN, 1e-3 * rng.standard_normal(nA).astype(np.float32), (1e-6 * rng.uniform(0.5, 2, nA)).astype(np.float32), step0)
    acts, st, tt, nz = inputs("hopper")[("pre", rows)]
    parts = {k: v for k, v in _parts(d, nA, nA).items() if k != "critic"}
    lr, worst = 1e-2, 0.0
    w_abs = np.abs(e.get_weights(L.NET_ACTOR))
    assert np.median(0.1 * lr * w_abs / np.maximum(_ulp(w_abs), 1e-38)) >= 100
    for k in range(2):
        w0 = e.get_weights(L.NET_ACTOR)
        m0, v0, s0 = e.get_opt_state(L.OPT_PRETRAIN)
        _, g = e.pretrain_step(acts, st, lr=lr, apply=True, t=tt, noise=nz, want_grads=True)
        g = g.cpu().numpy()
        w1 = e.get_weights(L.NET_ACTOR)
        m1, v1, s1 = e.get_opt_state(L.OPT_PRETRAIN)
        assert s1 == s0 + 1 == step0 + k + 1
        worst = max(worst, _check_adamw(e.cfg, w0, m0, v0, g, s1, lr, 0.1, w1, m1, v1, parts))
    e.close()
    print(f"adamw pretrain {mode} rows {rows} step {step0 + 1}: worst error / bound {worst:.3f}")
