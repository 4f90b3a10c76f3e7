"""
ORACLE — TEST INFRASTRUCTURE ONLY.  Not part of the product path.

CPU (torch fp32 / numpy) restatement of the reference's DPPO hot path.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg may import this
module; the product (`diffusionpolicyoptimization_b200/`) never does.

PARITY PIN: the reference (jamesmshihua/DiffusionPolicyOptimization) ships no tests, golden
vectors or known-answer files for this path, and its arithmetic lives in TensorFlow / Keras 3 /
tensorflow-probability, none of which is installed (or installable: no network) in the build
image.  The pin is therefore the reference's OWN Python: tests/golden/make_ref_golden.py imports
model/diffusion/*.py and model/common/{mlp,critic}.py unmodified from /root/reference and executes
them over tests/golden/tf_shim/ (a torch-CPU stand-in for the ~60 TF primitives they call); the
resulting fixtures tests/golden/ref_*.npz are checked against this file by tests/test_ref_golden.py
and against the CUDA path by tests/test_gpu_ref_golden.py.  That pins control flow, schedule
arithmetic, indexing, clip order, network switch, chain bookkeeping, loss/metric composition and
gradient variable order to the reference's code.  NOT pinned (TensorFlow itself never ran): the
numerical kernels of the third-party ops, restated here and in the shim from their *published*
semantics:

  * tf.keras.layers.Dense            : y = x @ W[in,out] + b
  * tf.keras.activations.mish        : x * tanh(softplus(x))
  * tfp.distributions.Normal.log_prob: -0.5*((x/s) - (m/s))**2 - (0.5*log(2*pi) + log(s))
  * tf.math.reduce_std               : population std
  * keras.optimizers.AdamW (Keras 3) : decoupled decay  w -= w*wd*lr  applied before the Adam update
                                       m += (g-m)(1-b1); v += (g^2-v)(1-b2);
                                       w -= m * lr*sqrt(1-b2^t)/(1-b1^t) / (sqrt(v)+eps)
    defaults weight_decay=0.004, beta=(0.9,0.999), eps=1e-7; the legacy `decay=` kwarg the
    reference passes (agent/finetune/train_ppo_agent.py:45-49) is ignored by Keras 3.

All file:line citations are relative to the reference repo root.
"""

from __future__ import annotations

import math
from collections import namedtuple
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

Sample = namedtuple("Sample", "trajectories chains")  # model/diffusion/diffusion.py:15


# --------------------------------------------------------------------------------------
# Schedule and DDPM constants
# --------------------------------------------------------------------------------------

def cosine_beta_schedule(timesteps: int, s: float = 0.008) -> np.ndarray:
    """model/diffusion/sampling.py:7-17 — float64 numpy, cast to fp32 at the end."""
    steps = timesteps + 1
    x = np.linspace(0, steps, steps)
    alphas_cumprod = np.cos(((x / steps) + s) / (1 + s) * np.pi * 0.5) ** 2
    alphas_cumprod = alphas_cumprod / alphas_cumprod[0]
    betas = 1 - (alphas_cumprod[1:] / alphas_cumprod[:-1])
    betas_clipped = np.clip(betas, a_min=0, a_max=0.999)
    return betas_clipped.astype(np.float32)


SCHEDULE_ROWS = (
    "betas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
    "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "ddpm_logvar_clipped",
    "ddpm_mu_coef1", "ddpm_mu_coef2",
)


def ddpm_constants(denoising_steps: int) -> dict:
    """model/diffusion/diffusion.py:58-73 — every op after the schedule is fp32."""
    f = np.float32
    betas = cosine_beta_schedule(denoising_steps)
    alphas = (f(1.0) - betas).astype(f)
    # tf.math.cumprod on fp32: sequential running product
    alphas_cumprod = np.empty_like(alphas)
    acc = f(1.0)
    for i in range(len(alphas)):
        acc = f(acc * alphas[i])
        alphas_cumprod[i] = acc
    alphas_cumprod_prev = np.concatenate([np.ones(1, f), alphas_cumprod[:-1]]).astype(f)
    c = {}
    c["betas"] = betas
    c["alphas"] = alphas
    c["alphas_cumprod"] = alphas_cumprod
    c["alphas_cumprod_prev"] = alphas_cumprod_prev
    c["sqrt_alphas_cumprod"] = np.sqrt(alphas_cumprod).astype(f)
    c["sqrt_one_minus_alphas_cumprod"] = np.sqrt((f(1.0) - alphas_cumprod).astype(f)).astype(f)
    c["sqrt_recip_alphas_cumprod"] = np.sqrt((f(1.0) / alphas_cumprod).astype(f)).astype(f)
    c["sqrt_recipm1_alphas_cumprod"] = np.sqrt(((f(1.0) / alphas_cumprod).astype(f) - f(1.0)).astype(f)).astype(f)
    one_m_acp = (f(1.0) - alphas_cumprod).astype(f)
    c["ddpm_var"] = ((betas * (f(1.0) - alphas_cumprod_prev)).astype(f) / one_m_acp).astype(f)
    c["ddpm_logvar_clipped"] = np.log(np.clip(c["ddpm_var"], f(1e-20), None)).astype(f)
    c["ddpm_mu_coef1"] = ((betas * np.sqrt(alphas_cumprod_prev).astype(f)).astype(f) / one_m_acp).astype(f)
    c["ddpm_mu_coef2"] = (((f(1.0) - alphas_cumprod_prev).astype(f) * np.sqrt(alphas).astype(f)).astype(f) / one_m_acp).astype(f)
    return c


def schedule_table(denoising_steps: int) -> np.ndarray:
    """[9, T] fp32 table in SCHEDULE_ROWS order (the layout `dppo_ddpm_schedule` exports)."""
    c = ddpm_constants(denoising_steps)
    return np.stack([c[k] for k in SCHEDULE_ROWS]).astype(np.float32)


# --------------------------------------------------------------------------------------
# Networks
# --------------------------------------------------------------------------------------

def mish(x: torch.Tensor) -> torch.Tensor:
    """tf.keras.activations.mish (model/common/mlp.py:11, mlp_diffusion.py:42)."""
    return x * torch.tanh(torch.nn.functional.softplus(x))


ACT = {"ReLU": torch.relu, "Mish": mish, "Identity": lambda x: x, "Tanh": torch.tanh}


def sinusoidal_pos_emb(t: torch.Tensor, dim: int) -> torch.Tensor:
    """model/diffusion/modules.py:10-15.  t: [N] (any dtype) -> [N, dim]."""
    half_dim = dim // 2
    emb = math.log(10000) / (half_dim - 1)
    emb = torch.exp(torch.arange(half_dim, dtype=torch.float32) * -emb)
    emb = t.to(torch.float32)[:, None] * emb[None, :]
    return torch.cat([torch.sin(emb), torch.cos(emb)], dim=-1)


@dataclass
class Dims:
    obs_dim: int = 11
    action_dim: int = 3
    horizon_steps: int = 4
    cond_steps: int = 1
    denoising_steps: int = 20
    ft_denoising_steps: int = 10
    time_dim: int = 16
    actor_hidden: int = 512
    critic_hidden: int = 256

    @property
    def A(self):
        return self.action_dim * self.horizon_steps

    @property
    def Do(self):
        return self.obs_dim * self.cond_steps

    @property
    def Din(self):
        return self.A + self.time_dim + self.Do

    def actor_shapes(self):
        """Flat variable order = Keras creation order: time Dense32, time Dense16
        (mlp_diffusion.py:40-45), then ResidualMLP input, block.l1, block.l2, output
        (mlp.py:117,170-171,132)."""
        td, H, A = self.time_dim, self.actor_hidden, self.A
        return [(td, 2 * td), (2 * td,), (2 * td, td), (td,),
                (self.Din, H), (H,), (H, H), (H,), (H, H), (H,), (H, A), (A,)]

    def critic_shapes(self):
        """critic.py:27-38 -> ResidualMLP([Do, Hc, Hc, Hc, 1])."""
        Hc = self.critic_hidden
        return [(self.Do, Hc), (Hc,), (Hc, Hc), (Hc,), (Hc, Hc), (Hc,), (Hc, 1), (1,)]

    def n_actor(self):
        return int(sum(int(np.prod(s)) for s in self.actor_shapes()))

    def n_critic(self):
        return int(sum(int(np.prod(s)) for s in self.critic_shapes()))


def init_params(shapes, rng: np.random.Generator, bias_scale: float = 0.05) -> List[torch.Tensor]:
    """Glorot-uniform kernels (Keras Dense default) and small random biases so that the bias
    paths are exercised (Keras would start them at zero; trained checkpoints are non-zero)."""
    out = []
    for s in shapes:
        if len(s) == 2:
            lim = math.sqrt(6.0 / (s[0] + s[1]))
            out.append(torch.from_numpy(rng.uniform(-lim, lim, size=s).astype(np.float32)))
        else:
            out.append(torch.from_numpy((bias_scale * rng.standard_normal(size=s)).astype(np.float32)))
    return out


def flatten_params(params: Sequence[torch.Tensor]) -> np.ndarray:
    return np.concatenate([p.detach().numpy().reshape(-1) for p in params]).astype(np.float32)


def unflatten_params(flat: np.ndarray, shapes) -> List[torch.Tensor]:
    out, off = [], 0
    for s in shapes:
        n = int(np.prod(s))
        out.append(torch.from_numpy(np.asarray(flat[off:off + n], dtype=np.float32).reshape(s).copy()))
        off += n
    assert off == flat.size
    return out


def residual_mlp(p: Sequence[torch.Tensor], x: torch.Tensor, act) -> torch.Tensor:
    """model/common/mlp.py:141-160 with one TwoLayerPreActivationResNetLinear block (:186-206);
    dim_list has 5 entries => num_hidden_layers=2 => exactly one block (:112-127)."""
    w_in, b_in, w1, b1, w2, b2, w_out, b_out = p
    x = x @ w_in + b_in
    x_input = x
    h = act(x)
    h = h @ w1 + b1
    h = act(h)
    h = h @ w2 + b2
    x = h + x_input
    return x @ w_out + b_out


def time_embedding(p: Sequence[torch.Tensor], t: torch.Tensor, time_dim: int) -> torch.Tensor:
    """mlp_diffusion.py:40-45: SinusoidalPosEmb -> Dense(2*td, mish) -> Dense(td)."""
    tw1, tb1, tw2, tb2 = p
    e = sinusoidal_pos_emb(t, time_dim).to(tw1.dtype)       # float64 parameters evaluate the whole net in float64
    return mish(e @ tw1 + tb1) @ tw2 + tb2


def diffusion_mlp(params: Sequence[torch.Tensor], x, t, obs, dims: Dims, act="ReLU") -> torch.Tensor:
    """DiffusionMLP.call, model/diffusion/mlp_diffusion.py:65-90.
    x [N,Ta,Da], t [N], obs [N,To,Do] -> eps [N,Ta,Da]; concat order [x, time_emb, state] (:86)."""
    B = x.shape[0]
    xf = x.reshape(B, -1)
    state = obs.reshape(B, -1)
    temb = time_embedding(params[:4], t.reshape(B), dims.time_dim)
    h = torch.cat([xf, temb, state], dim=-1)
    out = residual_mlp(params[4:], h, ACT[act])
    return out.reshape(B, dims.horizon_steps, dims.action_dim)


def critic_obs(params: Sequence[torch.Tensor], obs, act="Mish") -> torch.Tensor:
    """CriticObs.call, model/common/critic.py:40-54 -> [N,1]."""
    B = obs.shape[0]
    return residual_mlp(params, obs.reshape(B, -1), ACT[act])


# --------------------------------------------------------------------------------------
# Diffusion policy
# --------------------------------------------------------------------------------------

@dataclass
class Hyper:
    """cfg.model.* / cfg.train.* values of cfg/gym/finetune/hopper-v2/ft_ppo_diffusion_mlp.yaml."""
    denoised_clip_value: Optional[float] = 1.0          # diffusion.py:28
    randn_clip_value: float = 3.0                       # yaml:83
    final_action_clip_value: Optional[float] = None     # diffusion.py:30
    min_sampling_denoising_std: float = 0.1             # yaml:84
    min_logprob_denoising_std: float = 0.1              # yaml:85
    gamma_denoising: float = 0.99                       # yaml:79
    clip_ploss_coef: float = 0.01                       # yaml:80
    clip_ploss_coef_base: float = 0.01                  # yaml:81
    clip_ploss_coef_rate: float = 3.0                   # yaml:82
    clip_vloss_coef: Optional[float] = None
    norm_adv: bool = True
    vf_coef: float = 0.5                                # yaml:71
    actor_act: str = "ReLU"                             # yaml:94
    critic_act: str = "Mish"                            # yaml:103
    # Keras-3 AdamW defaults (see module docstring)
    lr: float = 1e-4
    beta1: float = 0.9
    beta2: float = 0.999
    adam_eps: float = 1e-7
    weight_decay: float = 0.004


class Oracle:
    """VPGDiffusion / PPODiffusion restated on explicit parameter lists."""

    def __init__(self, dims: Dims, hyper: Hyper, actor, actor_ft, critic):
        self.d, self.h = dims, hyper
        self.actor, self.actor_ft, self.critic = actor, actor_ft, critic
        c = ddpm_constants(dims.denoising_steps)
        self.c = {k: torch.from_numpy(v) for k, v in c.items()}

    # sampling.py:20-24
    def _extract(self, name, t, ndim=3):
        return self.c[name][t.long()].reshape([t.shape[0]] + [1] * (ndim - 1))

    def p_mean_var(self, x, t, obs, use_base_policy=False, actor_ft=None):
        """VPGDiffusion.p_mean_var DDPM branch, model/diffusion/diffusion_vpg.py:151-245.
        The base-net evaluation at :161 is dead compute whenever the ft net overwrites it
        (:165-180, decision by the FIRST row only) and is skipped here."""
        d, h = self.d, self.h
        actor_ft = self.actor_ft if actor_ft is None else actor_ft
        if bool(t[0] < d.ft_denoising_steps) and not use_base_policy:
            noise = diffusion_mlp(actor_ft, x, t, obs, d, h.actor_act)
        else:
            noise = diffusion_mlp(self.actor, x, t, obs, d, h.actor_act)
        x_recon = self._extract("sqrt_recip_alphas_cumprod", t) * x \
            - self._extract("sqrt_recipm1_alphas_cumprod", t) * noise            # :198-201
        if h.denoised_clip_value is not None:
            x_recon = torch.clamp(x_recon, -h.denoised_clip_value, h.denoised_clip_value)  # :206
        mu = self._extract("ddpm_mu_coef1", t) * x_recon + self._extract("ddpm_mu_coef2", t) * x  # :239-242
        logvar = self._extract("ddpm_logvar_clipped", t)                          # :243
        etas = torch.ones_like(mu)                                                # :244
        return mu, logvar, etas

    @torch.no_grad()
    def sample(self, obs, x_T, noise, deterministic=False, use_base_policy=False,
               min_sampling_denoising_std=None):
        """VPGDiffusion.call, diffusion_vpg.py:249-339, with the Gaussian draws injected:
        x_T [B,Ta,Da] replaces :280, noise[i] (i-th loop iteration, t = T-1-i) replaces :319."""
        d, h = self.d, self.h
        B = obs.shape[0]
        min_std = h.min_sampling_denoising_std if min_sampling_denoising_std is None else min_sampling_denoising_std
        x = x_T.clone()
        t_all = list(reversed(range(d.denoising_steps)))
        chain = []
        if d.ft_denoising_steps == d.denoising_steps:                              # :286-287
            chain.append(x)
        for i, t in enumerate(t_all):
            t_b = torch.full((B,), t, dtype=torch.int64)
            mean, logvar, _ = self.p_mean_var(x, t_b, obs, use_base_policy=use_base_policy)
            std = torch.exp(0.5 * logvar)                                          # :301
            if deterministic and t == 0:
                std = torch.zeros_like(std)                                        # :310-311
            elif deterministic:
                std = torch.clamp(std, 1e-3, 1e6)                                  # :312-313
            else:
                std = torch.clamp(std, min_std, 1e6)                               # :315
            eps = torch.clamp(noise[i], -h.randn_clip_value, h.randn_clip_value)   # :319
            x = mean + std * eps                                                   # :320
            if h.final_action_clip_value is not None and i == len(t_all) - 1:      # :323-327
                x = torch.clamp(x, -h.final_action_clip_value, h.final_action_clip_value)
            if t <= d.ft_denoising_steps:                                          # :330-331
                chain.append(x)
        return Sample(x, torch.stack(chain, dim=1))                                # :338-339

    @staticmethod
    def normal_log_prob(x, loc, scale):
        """tfp.distributions.Normal._log_prob."""
        log_unnormalized = -0.5 * ((x / scale) - (loc / scale)) ** 2
        log_normalization = 0.5 * math.log(2.0 * math.pi) + torch.log(scale)
        return log_unnormalized - log_normalization

    def get_logprobs(self, obs, chains, use_base_policy=False, actor_ft=None):
        """VPGDiffusion.get_logprobs, diffusion_vpg.py:343-425 -> [B*K, Ta, Da]."""
        d, h = self.d, self.h
        K = d.ft_denoising_steps
        B = chains.shape[0]
        obs_rep = obs.unsqueeze(1).repeat(1, K, *([1] * (obs.ndim - 1))).reshape(-1, *obs.shape[1:])  # :374-379
        t_single = torch.arange(K - 1, -1, -1)
        t_all = t_single.unsqueeze(0).repeat(B, 1).reshape(-1)                      # :385-390
        prev = chains[:, :-1].reshape(-1, d.horizon_steps, d.action_dim)           # :402-407
        nxt = chains[:, 1:].reshape(-1, d.horizon_steps, d.action_dim)
        mean, logvar, _ = self.p_mean_var(prev, t_all, obs_rep, use_base_policy=use_base_policy,
                                          actor_ft=actor_ft)                      # :410
        std = torch.clamp(torch.exp(0.5 * logvar), h.min_logprob_denoising_std, 1e6)  # :417-418
        return self.normal_log_prob(nxt, mean, std)                                # :419-422

    def get_logprobs_subsample(self, obs, chains_prev, chains_next, denoising_inds,
                               use_base_policy=False, actor_ft=None):
        """VPGDiffusion.get_logprobs_subsample, diffusion_vpg.py:427-481 -> (logp, eta)."""
        d, h = self.d, self.h
        t_single = torch.arange(d.ft_denoising_steps - 1, -1, -1)
        t_all = t_single[denoising_inds.long()]                                    # :456-458
        mean, logvar, eta = self.p_mean_var(chains_prev, t_all, obs, use_base_policy=use_base_policy,
                                            actor_ft=actor_ft)                    # :466
        std = torch.clamp(torch.exp(0.5 * logvar), h.min_logprob_denoising_std, 1e6)
        return self.normal_log_prob(chains_next, mean, std), eta

    def ppo_loss(self, obs, chains_prev, chains_next, denoising_inds, returns, oldvalues,
                 advantages, oldlogprobs, reward_horizon=4, actor_ft=None, critic=None):
        """PPODiffusion.c_loss, model/diffusion/diffusion_ppo.py:32-132 (use_bc_loss False)."""
        d, h = self.d, self.h
        K = d.ft_denoising_steps
        critic = self.critic if critic is None else critic
        newlogprobs, eta = self.get_logprobs_subsample(obs, chains_prev, chains_next, denoising_inds,
                                                       actor_ft=actor_ft)
        entropy_loss = -eta.mean()                                                 # :49
        newlogprobs = torch.clamp(newlogprobs, -5, 2)                              # :50
        oldlogprobs = torch.clamp(oldlogprobs, -5, 2)                              # :51
        newlogprobs = newlogprobs[:, :reward_horizon, :]                           # :54
        oldlogprobs = oldlogprobs[:, :reward_horizon, :]
        newlogprobs = newlogprobs.mean(dim=(-1, -2)).reshape(-1)                   # :58
        oldlogprobs = oldlogprobs.mean(dim=(-1, -2)).reshape(-1)
        bc_loss = torch.zeros(())
        if h.norm_adv:                                                             # :74-75
            advantages = (advantages - advantages.mean()) / (advantages.std(unbiased=False) + 1e-8)
        dinds = denoising_inds.to(torch.float32)
        discount = torch.pow(torch.tensor(h.gamma_denoising, dtype=torch.float32), K - dinds - 1)  # :83-85
        advantages = advantages * discount
        logratio = newlogprobs - oldlogprobs
        ratio = torch.exp(logratio)                                                # :89-90
        t = dinds / (K - 1) if K > 1 else dinds
        if K > 1:                                                                  # :94-99
            clip = h.clip_ploss_coef_base + (h.clip_ploss_coef - h.clip_ploss_coef_base) * (
                torch.exp(h.clip_ploss_coef_rate * t) - 1) / (math.exp(h.clip_ploss_coef_rate) - 1)
        else:
            clip = t
        pg_loss1 = -advantages * ratio
        pg_loss2 = -advantages * torch.minimum(torch.maximum(ratio, 1 - clip), 1 + clip)
        pg_loss = torch.maximum(pg_loss1, pg_loss2).mean()                         # :104-106
        newvalues = critic_obs(critic, obs, h.critic_act).squeeze(-1)              # :109
        if h.clip_vloss_coef is not None:                                          # :110-116
            v_un = (newvalues - returns) ** 2
            v_cl = oldvalues + torch.clamp(newvalues - oldvalues, -h.clip_vloss_coef, h.clip_vloss_coef)
            v_loss = 0.5 * torch.maximum(v_un, (v_cl - returns) ** 2).mean()
        else:
            v_loss = 0.5 * ((newvalues - returns) ** 2).mean()                     # :118
        approx_kl = ((ratio - 1) - logratio).mean()                                # :121
        clipfrac = ((ratio - 1.0).abs() > clip).to(torch.float32).mean()           # :122
        return (pg_loss, entropy_loss, v_loss, clipfrac, approx_kl, ratio.mean(), bc_loss, eta.mean())

    def ppo_grads(self, *batch, reward_horizon=4):
        """Caller side, agent/finetune/train_ppo_diffusion_agent.py:340-346:
        loss = pg_loss + vf_coef*v_loss; gradients wrt actor_ft + critic variables."""
        ft = [p.clone().requires_grad_(True) for p in self.actor_ft]
        cr = [p.clone().requires_grad_(True) for p in self.critic]
        out = self.ppo_loss(*batch, reward_horizon=reward_horizon, actor_ft=ft, critic=cr)
        loss = out[0] + out[2] * self.h.vf_coef
        grads = torch.autograd.grad(loss, ft + cr)
        return [o.detach() for o in out], [g.detach() for g in grads[:len(ft)]], [g.detach() for g in grads[len(ft):]]

    # ---- pre-training (DiffusionModel) ----
    def q_sample(self, x_start, t, noise):
        """model/diffusion/diffusion.py:196-202."""
        return self._extract("sqrt_alphas_cumprod", t) * x_start \
            + self._extract("sqrt_one_minus_alphas_cumprod", t) * noise

    def p_losses(self, x_start, obs, t, noise, network=None):
        """model/diffusion/diffusion.py:186-194 with the draw at :187 injected."""
        network = self.actor if network is None else network
        x_noisy = self.q_sample(x_start, t, noise)
        x_recon = diffusion_mlp(network, x_noisy, t, obs, self.d, self.h.actor_act)
        return ((x_recon - noise) ** 2).mean()

    def pretrain_grads(self, x_start, obs, t, noise):
        net = [p.clone().requires_grad_(True) for p in self.actor]
        loss = self.p_losses(x_start, obs, t, noise, network=net)
        grads = torch.autograd.grad(loss, net)
        return loss.detach(), [g.detach() for g in grads]


def adamw_keras(params, grads, m, v, step, lr, beta1=0.9, beta2=0.999, eps=1e-7, weight_decay=0.004):
    """Keras-3 AdamW.apply_gradients (see module docstring).  `step` is the 1-based iteration.
    Operates in place on lists of fp32 tensors; returns nothing."""
    f = torch.float32
    lr_t = torch.tensor(lr, dtype=f)
    b1p = torch.tensor(beta1, dtype=f) ** step
    b2p = torch.tensor(beta2, dtype=f) ** step
    alpha = lr_t * torch.sqrt(1 - b2p) / (1 - b1p)
    for p, g, mi, vi in zip(params, grads, m, v):
        if weight_decay:
            p.sub_(p * (weight_decay * lr))
        mi.add_((g - mi) * (1 - beta1))
        vi.add_((g * g - vi) * (1 - beta2))
        p.sub_(mi * alpha / (torch.sqrt(vi) + eps))


def clip_by_norm(grads, clip_norm=1.0):
    """[tf.clip_by_norm(g, clip_norm) for g in gradients], agent/finetune/train_ppo_diffusion_agent.py:352
    (published TF semantics: t * clip_norm / max(sqrt(sum(t*t)), clip_norm), the sqrt guarded for an all-zero t)."""
    out = []
    for g in grads:
        l2sum = (g * g).sum()
        l2norm = torch.sqrt(torch.where(l2sum > 0, l2sum, torch.ones_like(l2sum)))
        out.append(g * clip_norm / torch.maximum(l2norm, torch.tensor(clip_norm, dtype=g.dtype)))
    return out


def gae(rewards: np.ndarray, terminated: np.ndarray, values: np.ndarray, next_values: np.ndarray,
        reward_scale_const: float = 1.0, gamma: float = 0.999, gae_lambda: float = 0.95):
    """agent/finetune/train_ppo_diffusion_agent.py:242-263 — NumPy float64 backward scan over the rollout.
    rewards / terminated / values: [n_steps, n_envs]; next_values: [n_envs] (critic of the last observation).
    Returns (advantages, returns) as float64 [n_steps, n_envs] (the reference casts them to fp32 at :277-279)."""
    rewards = np.asarray(rewards, np.float64); values = np.asarray(values, np.float64)
    n_steps = rewards.shape[0]
    advantages = np.zeros_like(rewards)
    lastgaelam = 0
    for t in reversed(range(n_steps)):
        # :252 the bootstrap value is the critic's fp32 output, and `self.gamma * nextvalues` (Python float x fp32 array) is an fp32
        # product in NumPy; the other steps read the float64 holder `values_trajs` (pinned by tests/golden/ref_gae.npz)
        gnext = (np.float32(gamma) * np.asarray(next_values, np.float32).reshape(1, -1)) if t == n_steps - 1 else gamma * values[t + 1]
        nonterminal = 1.0 - np.asarray(terminated[t], np.float64)
        delta = rewards[t] * reward_scale_const + gnext * nonterminal - values[t]
        lastgaelam = delta + gamma * gae_lambda * nonterminal * lastgaelam
        advantages[t] = lastgaelam
    return advantages, advantages + values


def ema_update(ema_params, params, decay=0.995):
    """agent/pretrain/train_agent.py:53-58: ema <- decay*ema + (1-decay)*w."""
    for e, p in zip(ema_params, params):
        e.mul_(decay).add_(p * (1 - decay))


# --------------------------------------------------------------------------------------
# Synthetic problem instances (SURVEY.md §8(d) recipe)
# --------------------------------------------------------------------------------------

TASKS = {
    "hopper": dict(obs_dim=11, action_dim=3),
    "walker2d": dict(obs_dim=17, action_dim=6),
    "halfcheetah": dict(obs_dim=17, action_dim=6),
}


def make_oracle(task="hopper", seed=0, hyper: Optional[Hyper] = None, ft_perturb: float = 5e-3, **dim_over) -> Oracle:
    dims = Dims(**{**TASKS[task], **dim_over})
    rng = np.random.default_rng(seed)
    actor = init_params(dims.actor_shapes(), rng)
    # ft = base + small perturbation so that the two nets differ
    actor_ft = [p + ft_perturb * torch.from_numpy(rng.standard_normal(size=tuple(p.shape)).astype(np.float32))
                for p in actor]
    critic = init_params(dims.critic_shapes(), rng)
    return Oracle(dims, hyper or Hyper(), actor, actor_ft, critic)


def make_rollout_inputs(o: Oracle, B: int, seed=1):
    d = o.d
    rng = np.random.default_rng(seed)
    obs = torch.from_numpy(rng.uniform(-1, 1, size=(B, d.cond_steps, d.obs_dim)).astype(np.float32))
    x_T = torch.from_numpy(rng.standard_normal(size=(B, d.horizon_steps, d.action_dim)).astype(np.float32))
    noise = torch.from_numpy(rng.standard_normal(
        size=(d.denoising_steps, B, d.horizon_steps, d.action_dim)).astype(np.float32))
    return obs, x_T, noise


def make_ppo_batch(o: Oracle, N: int, pool: int = 256, seed=2):
    """N (env-step, k) rows drawn from `pool` chains produced by the oracle sampler itself."""
    d = o.d
    K = d.ft_denoising_steps
    rng = np.random.default_rng(seed)
    obs, x_T, noise = make_rollout_inputs(o, pool, seed=seed + 100)
    chains = o.sample(obs, x_T, noise).chains                     # [pool, K+1, Ta, Da]
    with torch.no_grad():
        oldlogp_all = o.get_logprobs(obs, chains, actor_ft=o.actor).reshape(pool, K, d.horizon_steps, d.action_dim)
        values_all = critic_obs(o.critic, obs, o.h.critic_act).reshape(-1)
    flat = torch.from_numpy(rng.integers(0, pool * K, size=N))
    b_inds, k_inds = flat // K, flat % K
    batch = (
        obs[b_inds],                                              # [N,To,Do]
        chains[b_inds, k_inds],                                   # prev  [N,Ta,Da]
        chains[b_inds, k_inds + 1],                               # next
        k_inds.to(torch.int32),                                   # denoising_inds
        torch.from_numpy(rng.standard_normal(N).astype(np.float32)),   # returns
        values_all[b_inds] + 0.1 * torch.from_numpy(rng.standard_normal(N).astype(np.float32)),  # oldvalues
        torch.from_numpy(rng.standard_normal(N).astype(np.float32)),   # advantages
        oldlogp_all[b_inds, k_inds],                              # oldlogprobs [N,Ta,Da]
    )
    return batch
