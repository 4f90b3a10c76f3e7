"""The three precision modes across the network widths, schedule lengths and time embeddings dppo_create accepts, against the fp32
oracle.  Every other GPU test of the training step runs H = 512, Hc = 256, T = 20, time_dim 16, cond_steps 1.

Cases (ReLU actor, Mish critic, K = 10 unless stated):
  H64-td4     hopper, H = Hc = 64, time_dim 4: one 64-column block, narrower than one plane-GEMM pair tile; smallest time embedding
  H256-To2    hopper, H = Hc = 256, cond_steps 2 (Do = 22): stacked observations
  H384-C192   walker2d, H = 384, Hc = 192: a half-empty last 256-wide pair tile in every actor GEMM and weight-gradient tile
  H768-td32   walker2d, H = 768, time_dim 32: the split-precision update applies AdamW and rebuilds the tables as separate launches
  H768-A56    14 x 4, Do 59, H = 768: the split-precision output-layer gradient assembly does not fit (100.8 KB of shared memory)
  H1024       walker2d, H = 1024: the assembly's k slice (136 rows) exceeds what a block holds
  C512-ReLU   walker2d, Hc = 512 with a ReLU critic: fp16 critic planes / the fused bf16 critic chain at another width
  C1024       walker2d, Hc = 1024: the critic's assembly k slice exceeds what a block holds
  T100        7 x 4, Do 23, T = 100, time_dim 32: KP0 = 192, the per-step column sums of du at exactly 200 KB
  T100-H768   the same at H = 768: per-step column sums of 300 KB
  T255        hopper, T = 255, time_dim 32: KP0 = 320, T x time_dim = 8160, per-step column sums of 510 KB
  T128-td64   hopper, H = Hc = 256, T = 128, time_dim 64: T x time_dim = 8192, the largest time backward (160 KB)
  H100        hopper, H = Hc = 100: not a multiple of 64, every mode stays on FFMA (no tcgen05 launch)
Each case runs in every mode.  A call a mode's tensor path does not cover (fewer than 2048 rows, a shape the mode routes to FFMA for
the whole handle) is held to the fp32 bounds; the launch counters and the sampler path say which kernels ran.  The PPO batches leave
out the rows that lie on a ReLU kink (_off_the_kinks).

Bounds are the modes' own, copied from tests/test_gpu_variants.py:
  bf16x3  eps 5e-6 rel, value 5e-5 rel, log-probs 1e-3 abs, PPO / pre-train grads 1e-3 of max, sampled actions 1e-4 rel
  bf16    eps / value 2e-2 rel, log-probs 0.15 abs, PPO grads 0.15 of max, pre-train grads 5e-2, sampled actions mean abs 2e-2
  fp32    eps 2e-5 rel, value 2e-5 abs, log-probs 1e-3 abs, grads 1e-3 of max, actions 1e-4 rel
"""
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

import diffusionpolicyoptimization_b200 as dp
from diffusionpolicyoptimization_b200 import _lib as L
from oracle import dppo_oracle as O
from helpers import make_engine, max_abs, rel_err

DETERMINISTIC = os.environ.get("DPPO_DETERMINISTIC") == "1"
PREC = {"bf16x3": L.PREC_BF16X3, "bf16": L.PREC_BF16, "fp32": L.PREC_FP32}
MODES = ("bf16x3", "bf16", "fp32")

T100 = dict(action_dim=7, horizon_steps=4, obs_dim=23, denoising_steps=100, time_dim=32)
CASES = {
    "H64-td4": dict(task="hopper", dims=dict(actor_hidden=64, critic_hidden=64, time_dim=4)),
    "H256-To2": dict(task="hopper", dims=dict(actor_hidden=256, critic_hidden=256, cond_steps=2)),
    "H384-C192": dict(task="walker2d", dims=dict(actor_hidden=384, critic_hidden=192)),
    "H768-td32": dict(task="walker2d", dims=dict(actor_hidden=768, time_dim=32)),
    "H768-A56": dict(task="hopper", dims=dict(action_dim=14, horizon_steps=4, obs_dim=59, actor_hidden=768)),
    "H1024": dict(task="walker2d", dims=dict(actor_hidden=1024)),
    "C512-ReLU": dict(task="walker2d", dims=dict(critic_hidden=512), hyper=dict(critic_act="ReLU")),
    "C1024": dict(task="walker2d", dims=dict(critic_hidden=1024)),
    "T100": dict(task="hopper", dims=dict(T100)),
    "T100-H768": dict(task="hopper", dims=dict(T100, actor_hidden=768)),
    "T255": dict(task="hopper", dims=dict(denoising_steps=255, time_dim=32)),
    "T128-td64": dict(task="hopper", dims=dict(actor_hidden=256, critic_hidden=256, denoising_steps=128, time_dim=64)),
    "H100": dict(task="hopper", dims=dict(actor_hidden=100, critic_hidden=100)),
}
NAMES = list(CASES)

# derived sizes (test_case_sizes): KP0 = round_up(A + Do + T + 1, 64), T x time_dim, the per-step column sums T x H x 4 bytes,
# the split-precision assembly's k slice per block ceil((H + A + Do + T) / 8) for actor / critic and its shared memory in bytes
SIZES = {
    "H64-td4": dict(KP0=64, Ttd=80, colsum=5120, kper=(14, 14), dw3_smem=25248),
    "H256-To2": dict(KP0=64, Ttd=320, colsum=20480, kper=(39, 39), dw3_smem=26448),
    "H384-C192": dict(KP0=64, Ttd=320, colsum=30720, kper=(56, 32), dw3_smem=54528),
    "H768-td32": dict(KP0=64, Ttd=640, colsum=61440, kper=(104, 40), dw3_smem=77568),
    "H768-A56": dict(KP0=192, Ttd=320, colsum=61440, kper=(113, 49), dw3_smem=103168),
    "H1024": dict(KP0=64, Ttd=320, colsum=81920, kper=(136, 40), dw3_smem=103168),
    "C512-ReLU": dict(KP0=64, Ttd=320, colsum=40960, kper=(72, 72), dw3_smem=56064),
    "C1024": dict(KP0=64, Ttd=320, colsum=40960, kper=(72, 136), dw3_smem=56064),
    "T100": dict(KP0=192, Ttd=3200, colsum=204800, kper=(83, 51), dw3_smem=66640),
    "T100-H768": dict(KP0=192, Ttd=3200, colsum=307200, kper=(115, 51), dw3_smem=89984),
    "T255": dict(KP0=320, Ttd=8160, colsum=522240, kper=(99, 67), dw3_smem=29328),
    "T128-td64": dict(KP0=192, Ttd=8192, colsum=131072, kper=(51, 51), dw3_smem=27024),
    "H100": dict(KP0=64, Ttd=320, colsum=8000, kper=(18, 18), dw3_smem=25440),
}

N_PPO, N_SMALL, N_FWD, B_LP, B_SAMPLE, B_SMALL, N_PRE = 4099, 1031, 4099, 240, 2304, 40, 2304
TENSOR_MIN_ROWS = 2048                          # TS_MIN_ROWS / TC_MIN_ROWS

EPS_RTOL = {"bf16x3": 5e-6, "bf16": 2e-2, "fp32": 2e-5}
LOGP_ATOL = {"bf16x3": 1e-3, "bf16": 0.15, "fp32": 1e-3}
GRAD_TOL = {"bf16x3": 1e-3, "bf16": 0.15, "fp32": 1e-3}
METRIC_TOL = {"bf16x3": (2e-3, 2e-6), "bf16": (5e-2, 2e-3), "fp32": (2e-3, 2e-6)}
PRE_GRAD_TOL = {"bf16x3": 1e-3, "bf16": 5e-2, "fp32": 1e-3}


def _value_err(mode, got, want):
    return (max_abs(got, want), 2e-5) if mode == "fp32" else (rel_err(got, want), 5e-5 if mode == "bf16x3" else 2e-2)


def _pre_loss_tol(mode, want):
    return {"bf16x3": 1e-5 * abs(want), "bf16": 5e-2 * max(1.0, want), "fp32": 1e-4 * max(1.0, want)}[mode]


def _grid(names=NAMES, modes=MODES):
    return [pytest.param(n, m, id=f"{n}-{m}") for n in names for m in modes]


# ---------------------------------------------------------------- oracle side (shared by the modes of a case)
@functools.lru_cache(maxsize=None)
def oracle(name) -> O.Oracle:
    c = CASES[name]
    return O.make_oracle(c["task"], seed=0, hyper=O.Hyper(**c.get("hyper", {})), **c["dims"])


KINK_CLEARANCE = 3e-5


def _off_the_kinks(o, x, t, obs):
    """Rows whose ReLU pre-activations all lie at least KINK_CLEARANCE x (the unit's mean |pre-activation|) from zero, evaluated in
    float64.  A row closer than that to a kink takes either side of it depending on the last bits of the sum: the mode's rounding, or
    the fp32 oracle's own (on the T100-H768 batch one row's block.l1 pre-activation is 1.5e-7 against a typical 0.13; bf16x3 took the
    other side of that kink, and unit 83's column of dW1 was off by 2.3e-3 of the gradient's max)."""
    d, ok = o.d, torch.ones(x.shape[0], dtype=torch.bool)

    def clear(*pres):
        for pre in pres:
            ok.mul_((pre.abs() >= KINK_CLEARANCE * pre.abs().mean(0)).all(1))

    with torch.no_grad():
        p = [w.double() for w in o.actor_ft]
        temb = O.mish(O.sinusoidal_pos_emb(t, d.time_dim).double() @ p[0] + p[1]) @ p[2] + p[3]
        h0 = torch.cat([x.double().reshape(len(x), -1), temb, obs.double().reshape(len(x), -1)], -1)
        if o.h.actor_act == "ReLU":
            u = h0 @ p[4] + p[5]
            clear(u, torch.relu(u) @ p[6] + p[7])
        if o.h.critic_act == "ReLU":
            c = [w.double() for w in o.critic]
            u = obs.double().reshape(len(x), -1) @ c[0] + c[1]
            clear(u, torch.relu(u) @ c[2] + c[3])
    return ok


@functools.lru_cache(maxsize=None)
def ppo_batch(name, N):
    """N rows of the oracle's own chains, away from the ReLU kinks (_off_the_kinks)."""
    o = oracle(name)
    batch = O.make_ppo_batch(o, N + N // 4, pool=512, seed=3)
    t = torch.arange(o.d.ft_denoising_steps - 1, -1, -1)[batch[3].long()]
    keep = torch.nonzero(_off_the_kinks(o, batch[1], t, batch[0]))[:N, 0]
    assert len(keep) == N, (name, len(keep))
    batch = tuple(x[keep] for x in batch)
    metrics, ga, gc = o.ppo_grads(*batch, reward_horizon=o.d.horizon_steps)
    return batch, [float(m) for m in metrics], np.concatenate([O.flatten_params(ga), O.flatten_params(gc)])


@functools.lru_cache(maxsize=None)
def rollout(name, B, seed):
    o = oracle(name)
    obs, x_T, noise = O.make_rollout_inputs(o, B, seed=seed)
    return obs, x_T, noise, o.sample(obs, x_T, noise)


@functools.lru_cache(maxsize=None)
def pretrain_batch(name, N):
    o = oracle(name)
    d = o.d
    rng = np.random.default_rng(5)
    acts = torch.from_numpy(rng.uniform(-1, 1, (N, d.horizon_steps, d.action_dim)).astype(np.float32))
    st = torch.from_numpy(rng.uniform(-1, 1, (N, d.cond_steps, d.obs_dim)).astype(np.float32))
    tt = torch.from_numpy(rng.integers(0, d.denoising_steps, N))
    nz = torch.from_numpy(rng.standard_normal((N, d.horizon_steps, d.action_dim)).astype(np.float32))
    want_l, want_g = o.pretrain_grads(acts, st, tt, nz)
    return (acts, st, tt, nz), float(want_l), O.flatten_params(want_g)


@pytest.fixture(scope="module")
def engines():
    made = {}

    def get(name, mode):
        if (name, mode) not in made:
            made[(name, mode)] = make_engine(oracle(name), PREC[mode])
        return made[(name, mode)]

    yield get
    for e in made.values():
        e.close()


# ---------------------------------------------------------------- which path each call takes (read from the host code)
def _kper(H, d):
    return -(-(H + d.A + d.Do + d.denoising_steps) // 8)


def _dw3_smem(d):
    """ts_dw3_assemble's dynamic shared memory: per net the larger of the dW3 body ([kper][NO] + [16][32][NC]) and the rank-rows body
    ([8][NO] + H x (N3 + 1)); wide (NO > 32): NC = 16, N3 = 32."""
    def net(H, NO):
        wide = NO > 32
        a = _kper(H, d) * NO + 16 * 32 * (16 if wide else NO)
        b = 8 * NO + H * ((32 if wide else NO) + 1)
        return max(a, b) * 4
    return max(net(d.actor_hidden, d.A), net(d.critic_hidden, 1))


def _tensor_shape(d, mode):
    """The handle's tensor path exists: widths multiples of 64; bf16 covers A <= 32, bf16x3 A <= 128 and the output-layer gradient
    assembly's limits (shared memory <= 100 KB, k slice <= 128 rows per net)."""
    if mode == "fp32" or d.actor_hidden % 64 or d.critic_hidden % 64:
        return False
    if mode == "bf16":
        return d.A <= 32
    return d.A <= 128 and max(_kper(d.actor_hidden, d), _kper(d.critic_hidden, d)) <= 128 and _dw3_smem(d) <= 100 * 1024


def _tensor(o, mode, rows):
    return _tensor_shape(o.d, mode) and rows >= TENSOR_MIN_ROWS


def _kp0(d):
    return -(-(d.A + d.Do + d.denoising_steps + 1) // 64) * 64


def _fused(o, net):
    """bf16: the fused layer-chain kernel covers a ReLU net at 256 / 512 and a Mish net at 256, with KP0 = 64 (fc_net_ok)."""
    d, h = o.d, o.h
    H, act = (d.actor_hidden, h.actor_act) if net == "actor" else (d.critic_hidden, h.critic_act)
    if not _tensor_shape(d, "bf16") or _kp0(d) != 64:
        return False
    return H in (256, 512) if act == "ReLU" else H == 256


def _counts(e):
    return e.tc_launch_count(), e.fused_launch_count()


def _expect(o, mode, kind, rows):
    """(tcgen05 launches, fused layer-chain launches) of one call.  bf16x3: three plane GEMMs per forward (L0, L1, the folded output
    layer), two backward, one grouped weight-gradient launch.  bf16, per net: the fused chain is one launch forward and one backward
    plus a grouped weight-gradient launch (one for both nets when both are fused); the per-layer path 4 forward, 3 dX and 4 dW GEMMs."""
    if not _tensor(o, mode, rows):
        return (0, 0)
    T = o.d.denoising_steps
    if mode == "bf16x3":
        return {"fwd": (6, 0), "lp": (3, 0), "ppo": (11, 0), "pre": (6, 0), "sample": (3 * T, 0)}[kind]
    fa, fc = _fused(o, "actor"), _fused(o, "critic")
    fwd = {True: (1, 1), False: (4, 0)}
    train = {True: (3, 2), False: (11, 0)}
    if kind == "fwd":
        return tuple(a + c for a, c in zip(fwd[fa], fwd[fc]))
    if kind == "lp":
        return fwd[fa]
    if kind == "ppo":
        return (5, 4) if fa and fc else tuple(a + c for a, c in zip(train[fa], train[fc]))
    if kind == "pre":
        return train[fa]
    return (1, 1) if fa else (4 * T, 0)


def _check_counts(o, mode, kind, rows, e, before):
    got = tuple(a - b for a, b in zip(_counts(e), before))
    if DETERMINISTIC and mode == "bf16" and kind in ("ppo", "pre"):
        assert (got[0] == 0) == (_expect(o, mode, kind, rows)[0] == 0), (kind, got)
        return
    assert got == _expect(o, mode, kind, rows), (kind, got, _expect(o, mode, kind, rows))


def _cluster_row_limit(H, A):
    if H == 1024:
        return 1024
    if H != 512:
        return 2048 if A <= 64 else 1024
    return 4096 if A <= 32 else 2048 if A <= 64 else 1024


def _sample_path(o, mode, B):
    """1 persistent cluster kernel, 2 layered fp32, 3 layered tensor, 4 fused bf16 chain (dppo_sample)."""
    d = o.d
    tensor = _tensor(o, mode, B)
    cluster = d.actor_hidden in (256, 512, 768, 1024) and d.A <= 128 and o.h.actor_act == "ReLU"
    limit = 1024 if mode == "bf16" else _cluster_row_limit(d.actor_hidden, d.A)
    if cluster and not tensor and B <= limit:
        return 1
    if tensor and mode == "bf16" and _fused(o, "actor"):
        return 4
    return 3 if tensor else 2


def _bounds(o, mode, rows):
    """The calls a mode's tensor path does not run are held to the fp32 bounds."""
    return mode if _tensor(o, mode, rows) else "fp32"


def _flat(x):
    return x.reshape(x.shape[0], -1)


def _ppo_args(batch):
    N = batch[0].shape[0]
    return (_flat(batch[0]), batch[1].reshape(N, -1), batch[2].reshape(N, -1), batch[3], batch[4], batch[5], batch[6],
            batch[7].reshape(N, -1))


def _grad_errs(o, got_g, want_g):
    nA = o.d.n_actor()
    return [float(np.abs(got_g[sl] - want_g[sl]).max() / np.abs(want_g[sl]).max()) for sl in (slice(0, nA), slice(nA, None))]


# ---------------------------------------------------------------- sizes and limits (no GPU)
def test_case_sizes():
    for name in NAMES:
        d, s = oracle(name).d, SIZES[name]
        assert _kp0(d) == s["KP0"], name
        assert d.denoising_steps * d.time_dim == s["Ttd"], name
        assert d.denoising_steps * d.actor_hidden * 4 == s["colsum"], name
        assert (_kper(d.actor_hidden, d), _kper(d.critic_hidden, d)) == s["kper"], name
        assert _dw3_smem(d) == s["dw3_smem"], name
    assert oracle("T100").d.denoising_steps * oracle("T100").d.actor_hidden * 4 == 200 * 1024
    assert oracle("T128-td64").d.denoising_steps * oracle("T128-td64").d.time_dim * 5 * 4 == 160 * 1024
    # the routing the GPU tests expect
    assert [n for n in NAMES if not _tensor_shape(oracle(n).d, "bf16x3")] == ["H768-A56", "H1024", "C1024", "H100"]
    assert [n for n in NAMES if not _tensor_shape(oracle(n).d, "bf16")] == ["H768-A56", "H100"]


def _accepted(lib, **fields):
    cfg = dp.default_cfg()
    for k, v in fields.items():
        setattr(cfg, k, v)
    n = lib.dppo_num_params(C.byref(cfg), L.NET_ACTOR)
    return n > 0


def test_configuration_limits(lib):
    """dppo_num_params returns 0 for a configuration dppo_create refuses (make_geom), without a device: at every limit the last
    accepted value is accepted and the first refused one is refused."""
    # T x time_dim <= 8192: the time-embedding backward holds 5 T time_dim floats in shared memory (160 KB)
    assert _accepted(lib, denoising_steps=128, time_dim=64)
    assert not _accepted(lib, denoising_steps=129, time_dim=64)
    assert _accepted(lib, denoising_steps=255, time_dim=32)
    assert not _accepted(lib, denoising_steps=255, time_dim=34)
    assert _accepted(lib, denoising_steps=204, time_dim=40) and not _accepted(lib, denoising_steps=205, time_dim=40)
    # the limits that were there before
    assert _accepted(lib, denoising_steps=255, time_dim=16) and not _accepted(lib, denoising_steps=256, time_dim=16)
    assert _accepted(lib, denoising_steps=1, ft_denoising_steps=1) and not _accepted(lib, denoising_steps=0, ft_denoising_steps=0)
    assert _accepted(lib, time_dim=4) and not _accepted(lib, time_dim=2) and not _accepted(lib, time_dim=5)
    assert _accepted(lib, denoising_steps=20, time_dim=64) and not _accepted(lib, time_dim=66)
    for f in ("actor_hidden", "critic_hidden"):
        assert _accepted(lib, **{f: 16}) and not _accepted(lib, **{f: 12})
        assert _accepted(lib, **{f: 1024}) and not _accepted(lib, **{f: 1028})
        assert not _accepted(lib, **{f: 18})


def test_refusal_names_the_limit(lib):
    cfg = dp.default_cfg()
    cfg.denoising_steps, cfg.time_dim = 129, 64
    h = C.c_void_p()
    assert lib.dppo_create(C.byref(cfg), 0, C.byref(h)) != 0
    msg = lib.dppo_last_error()
    assert b"invalid configuration" in msg and b"time_dim" in msg and b"8192" in msg, msg


# ---------------------------------------------------------------- forward, value, log-probs
@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _grid())
def test_forward_and_value(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    d, bm = o.d, _bounds(o, mode, N_FWD)
    rng = np.random.default_rng(N_FWD)
    x = torch.from_numpy(rng.standard_normal((N_FWD, d.horizon_steps, d.action_dim)).astype(np.float32))
    t = torch.from_numpy(rng.integers(0, d.denoising_steps, N_FWD))
    obs = torch.from_numpy(rng.uniform(-1, 1, (N_FWD, d.cond_steps, d.obs_dim)).astype(np.float32))
    with torch.no_grad():
        want = O.diffusion_mlp(o.actor_ft, x, t, obs, d, o.h.actor_act).reshape(N_FWD, -1)
        wantv = O.critic_obs(o.critic, obs, o.h.critic_act).reshape(-1)
    c0 = _counts(e)
    got = e.actor_forward(L.NET_ACTOR_FT, x.reshape(N_FWD, -1), t, _flat(obs))
    gv = e.value(_flat(obs))
    torch.cuda.synchronize()
    err = rel_err(got, want)
    errv, tolv = _value_err(bm, gv, wantv)
    print(f"[{name} {mode}] eps rel err {err:.2e}, value err {errv:.2e}")
    assert err < EPS_RTOL[bm] and errv < tolv, (err, errv)
    _check_counts(o, mode, "fwd", N_FWD, e, c0)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _grid())
def test_logprobs_of_whole_chains(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    K = o.d.ft_denoising_steps
    rows = B_LP * K
    obs, _, _, s = rollout(name, B_LP, 3)
    with torch.no_grad():
        want = o.get_logprobs(obs, s.chains).reshape(rows, -1)
    c0 = _counts(e)
    got = e.logprobs(_flat(obs), s.chains.reshape(B_LP, K + 1, -1))
    torch.cuda.synchronize()
    err = max_abs(got, want)
    print(f"[{name} {mode}] log-prob abs err {err:.2e} ({B_LP} chains, K = {K})")
    assert err < LOGP_ATOL[_bounds(o, mode, rows)], err
    _check_counts(o, mode, "lp", rows, e, c0)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _grid())
def test_logprobs_subsample(engines, name, mode):
    o, e = oracle(name), engines(name, mode)
    batch, _, _ = ppo_batch(name, N_PPO)
    with torch.no_grad():
        want, _ = o.get_logprobs_subsample(batch[0], batch[1], batch[2], batch[3])
    c0 = _counts(e)
    got = e.logprobs_subsample(*_ppo_args(batch)[:4])
    torch.cuda.synchronize()
    err = max_abs(got, want.reshape(N_PPO, -1))
    print(f"[{name} {mode}] subsampled log-prob abs err {err:.2e}")
    assert err < LOGP_ATOL[_bounds(o, mode, N_PPO)], err
    _check_counts(o, mode, "lp", N_PPO, e, c0)


# ---------------------------------------------------------------- the PPO update
@pytest.mark.gpu
@pytest.mark.parametrize("N", [N_PPO, N_SMALL])
@pytest.mark.parametrize("name,mode", _grid())
def test_ppo_loss_and_gradients(engines, name, mode, N):
    """N_PPO rows: the mode's tensor path where the shape has one; N_SMALL rows: the FFMA update in every mode."""
    o, e = oracle(name), engines(name, mode)
    bm = _bounds(o, mode, N)
    batch, want_m, want_g = ppo_batch(name, N)
    c0 = _counts(e)
    m, g = e.ppo_step(*_ppo_args(batch), lr=0.0, apply=False, want_grads=True)
    torch.cuda.synchronize()
    m, g = m.cpu().numpy(), g.cpu().numpy()
    err_a, err_c = _grad_errs(o, g, want_g)
    print(f"[{name} {mode} N={N}] PPO grads actor {err_a:.2e} critic {err_c:.2e} of max; metrics rel "
          f"{np.abs(m - want_m).max() / max(np.abs(want_m).max(), 1e-30):.2e}")
    assert err_a < GRAD_TOL[bm] and err_c < GRAD_TOL[bm], (err_a, err_c)
    rtol, atol = METRIC_TOL[bm]
    np.testing.assert_allclose(m, want_m, rtol=rtol, atol=atol)
    _check_counts(o, mode, "ppo", N, e, c0)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _grid())
def test_indexed_update_matches_the_gathered_minibatch(engines, name, mode):
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
    c0 = _counts(e)
    m1, g1 = e.ppo_step_indexed(_flat(obs), chains, olp, ret, val, adv, idx, lr=0.0, apply=False, want_grads=True)
    if not (DETERMINISTIC and mode == "bf16"):
        assert (_counts(e)[0] - c0[0] == 0) == (not _tensor(o, mode, N))
    m2, g2 = e.ppo_step(_flat(obs)[b], chains[b, k], chains[b, k + 1], k.to(torch.int32), ret[b], val[b], adv[b], olp[b, k],
                        lr=0.0, apply=False, want_grads=True)
    torch.cuda.synchronize()
    assert torch.equal(m1, m2)
    if mode == "bf16" and not DETERMINISTIC and _tensor(o, mode, N):       # dW accumulates with atomics: the order varies
        assert float((g1 - g2).abs().max()) < 2e-3 * float(g2.abs().max())
    else:
        assert torch.equal(g1, g2)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _grid())
def test_applied_update(engines, name, mode):
    """One AdamW step from zero moments: the weights follow the oracle's step within 0.1 lr, and the next log-probs and values agree
    with the oracle evaluated at the weights the engine hands back (the plane copies, time tables and folded output layers were
    rebuilt).  The weights and the optimizer state are restored afterwards: the engines are shared.
    bf16 on its tensor path is held to the second check only: a first step from zero moments moves every weight by about lr sign(g),
    and gradients within the mode's bound (0.15 of max) flip the sign of the small entries (4 - 9 % of the weights)."""
    o, e = oracle(name), engines(name, mode)
    bm = _bounds(o, mode, N_PPO)
    batch, _, _ = ppo_batch(name, N_PPO)
    fb = _ppo_args(batch)
    lr = 1e-3
    n = e.n_actor + e.n_critic
    w_ft0, w_c0 = e.get_weights(L.NET_ACTOR_FT), e.get_weights(L.NET_CRITIC)
    e.set_opt_state(L.OPT_FINETUNE, np.zeros(n, np.float32), np.zeros(n, np.float32), 0)
    try:
        params = [p.clone() for p in o.actor_ft] + [p.clone() for p in o.critic]
        m = [torch.zeros_like(p) for p in params]; v = [torch.zeros_like(p) for p in params]
        _, ga, gc = o.ppo_grads(*batch, reward_horizon=o.d.horizon_steps)
        O.adamw_keras(params, ga + gc, m, v, 1, lr, o.h.beta1, o.h.beta2, o.h.adam_eps, o.h.weight_decay)
        c0 = _counts(e)
        e.ppo_step(*fb, lr=lr, apply=True)
        _check_counts(o, mode, "ppo", N_PPO, e, c0)
        wa, wc = e.get_weights(L.NET_ACTOR_FT), e.get_weights(L.NET_CRITIC)
        frac_bad = float(np.mean(np.abs(np.concatenate([wa, wc]) - O.flatten_params(params)) > 0.1 * lr))
        lp1 = e.logprobs_subsample(*fb[:4])
        v1 = e.value(fb[0])
        torch.cuda.synchronize()
        o1 = O.Oracle(o.d, o.h, o.actor, O.unflatten_params(wa, o.d.actor_shapes()), O.unflatten_params(wc, o.d.critic_shapes()))
        with torch.no_grad():
            want_lp, _ = o1.get_logprobs_subsample(batch[0], batch[1], batch[2], batch[3])
            want_v = O.critic_obs(o1.critic, batch[0], o.h.critic_act).reshape(-1)
        err_lp = max_abs(lp1, want_lp.reshape(N_PPO, -1))
        err_v, tol_v = _value_err(bm, v1, want_v)
        print(f"[{name} {mode}] after AdamW: {frac_bad:.2e} of the weights off the oracle's step by more than 0.1 lr; "
              f"log-prob abs err {err_lp:.2e}, value err {err_v:.2e}")
        if bm != "bf16":
            assert frac_bad < 2e-3, frac_bad
        assert err_lp < LOGP_ATOL[bm] and err_v < tol_v, (err_lp, err_v)
    finally:
        e.set_weights(L.NET_ACTOR_FT, w_ft0); e.set_weights(L.NET_CRITIC, w_c0)
        e.set_opt_state(L.OPT_FINETUNE, np.zeros(n, np.float32), np.zeros(n, np.float32), 0)


# ---------------------------------------------------------------- pre-training, sampling
@pytest.mark.gpu
@pytest.mark.parametrize("N", [N_PRE, N_SMALL])
@pytest.mark.parametrize("name,mode", _grid())
def test_pretrain_loss_and_gradients(engines, name, mode, N):
    o, e = oracle(name), engines(name, mode)
    bm = _bounds(o, mode, N)
    (acts, st, tt, nz), want_l, wg = pretrain_batch(name, N)
    c0 = _counts(e)
    loss, pg = e.pretrain_step(acts.reshape(N, -1), _flat(st), lr=0.0, apply=False, t=tt, noise=nz.reshape(N, -1), want_grads=True)
    torch.cuda.synchronize()
    err_g = float(np.abs(pg.cpu().numpy() - wg).max() / np.abs(wg).max())
    print(f"[{name} {mode} N={N}] pre-train loss {float(loss):.6f} vs {want_l:.6f}, grads {err_g:.2e} of max")
    assert abs(float(loss) - want_l) < _pre_loss_tol(bm, want_l) and err_g < PRE_GRAD_TOL[bm], (float(loss), want_l, err_g)
    _check_counts(o, mode, "pre", N, e, c0)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [B_SAMPLE, B_SMALL])
@pytest.mark.parametrize("name,mode", _grid())
def test_sampler(engines, name, mode, B):
    o, e = oracle(name), engines(name, mode)
    d, bm = o.d, _bounds(o, mode, B)
    obs, x_T, noise, want = rollout(name, B, 6)
    c0 = _counts(e)
    a, ch = e.sample(_flat(obs), x_T=x_T.reshape(B, -1), noise=noise.reshape(d.denoising_steps, B, -1))
    torch.cuda.synchronize()
    assert e.last_path() == _sample_path(o, mode, B), (e.last_path(), _sample_path(o, mode, B))
    wa, wc = want.trajectories.reshape(B, -1), want.chains.reshape(B, d.ft_denoising_steps + 1, -1)
    err, err_c = rel_err(a, wa), rel_err(ch, wc)
    mean, mean_c = float((a.cpu() - wa).abs().mean()), float((ch.cpu() - wc).abs().mean())
    print(f"[{name} {mode} B={B} path {e.last_path()}] sampled actions rel {err:.2e} mean abs {mean:.2e}; "
          f"chains rel {err_c:.2e} mean abs {mean_c:.2e}")
    if bm == "bf16x3":
        assert err < 1e-4 and mean < 1e-6 and mean_c < 1e-6, (err, mean, mean_c)
    elif bm == "bf16":
        assert mean < 2e-2 and err < 0.25 and mean_c < 2e-2, (err, mean, mean_c)
    else:
        assert err < 1e-4 and err_c < 1e-4, (err, err_c)
    _check_counts(o, mode, "sample", B, e, c0)


# ---------------------------------------------------------------- two handles in one process
@pytest.mark.gpu
def test_time_backward_of_a_later_handle_that_needs_more_shared_memory():
    """The time-embedding backward's dynamic shared memory (5 T time_dim floats) is a per-device function attribute: a handle that
    needs more than an earlier handle of the same process set must raise it.  T100 (62.5 KB) first, then T128-td64 (160 KB), each
    through the FFMA update.  (An earlier test file of the same session may already have raised the attribute; run this file alone
    to see the order matter.)"""
    made = []
    try:
        for name in ("T100", "T128-td64"):
            o = oracle(name)
            e = make_engine(o, L.PREC_FP32)
            made.append(e)
            batch, want_m, want_g = ppo_batch(name, N_SMALL)
            m, g = e.ppo_step(*_ppo_args(batch), lr=0.0, apply=False, want_grads=True)
            torch.cuda.synchronize()
            err_a, err_c = _grad_errs(o, g.cpu().numpy(), want_g)
            print(f"[{name} fp32, handle {len(made)}] PPO grads actor {err_a:.2e} critic {err_c:.2e} of max")
            assert err_a < GRAD_TOL["fp32"] and err_c < GRAD_TOL["fp32"], (err_a, err_c)
            np.testing.assert_allclose(m.cpu().numpy(), want_m, rtol=METRIC_TOL["fp32"][0], atol=METRIC_TOL["fp32"][1])
    finally:
        for e in made:
            e.close()
