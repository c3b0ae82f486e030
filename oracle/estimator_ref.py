"""CPU oracle: functional fp32/fp64 restatement of the StableTTS CFM/DiT path.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Every function cites
the reference site it follows (paths relative to the reference checkout).  The
restatement is weight-dict driven (``state`` maps the reference's
``estimator.*``-relative parameter names to tensors) and deliberately uses the
same torch library calls as the reference (``F.conv1d``, dense-float-mask
``F.scaled_dot_product_attention``) so that, timed on host cores, it is a fair
stand-in for the reference's own CPU path.

Pinned by: ``tests/test_oracle.py`` (against ``tests/golden/*.npz``, outputs of ``models.estimator.Decoder`` and its
RoPE module).
Solver stepping (``odeint_fixed``) restates torchdiffeq's fixed-grid tableaux
from the published algorithm: parity unpinned for solver behaviour.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional

import torch
import torch.nn.functional as F

State = Dict[str, torch.Tensor]


# --------------------------------------------------------------------------- #
# time embedding  (models/estimator.py:35-62, :117)
# --------------------------------------------------------------------------- #
def sinusoidal_pos_emb(t: torch.Tensor, dim: int, scale: float = 1000.0) -> torch.Tensor:
    """models/estimator.py:41-49 — note the (half_dim - 1) denominator."""
    if t.ndim < 1:
        t = t.unsqueeze(0)
    half = dim // 2
    step = math.log(10000) / (half - 1)
    freqs = torch.exp(torch.arange(half, device=t.device).float() * -step)
    if t.dtype == torch.float64:
        freqs = freqs.double()
    e = scale * t.unsqueeze(1) * freqs.unsqueeze(0)
    return torch.cat((e.sin(), e.cos()), dim=-1)


def time_embedding(state: State, t: torch.Tensor, hidden: int) -> torch.Tensor:
    """models/estimator.py:55-62 applied to :41-49 — Linear, SiLU, Linear."""
    e = sinusoidal_pos_emb(t, hidden).to(state["time_mlp.layer.0.weight"].dtype)
    h = F.linear(e, state["time_mlp.layer.0.weight"], state["time_mlp.layer.0.bias"])
    h = F.silu(h)
    return F.linear(h, state["time_mlp.layer.2.weight"], state["time_mlp.layer.2.bias"])


# --------------------------------------------------------------------------- #
# RoPE  (models/diffusion_transformer.py:123-198)
# --------------------------------------------------------------------------- #
def rope_partial(x: torch.Tensor, d_rot: int, base: float = 10000.0) -> torch.Tensor:
    """x: (B, nh, T, dh).  Rotates the first ``d_rot`` dims, pairs (j, j+d_rot/2),
    theta_i = base^(-2i/d_rot); position = frame index from 0
    (models/diffusion_transformer.py:157-178,190-198)."""
    T = x.shape[2]
    theta = 1.0 / (base ** (torch.arange(0, d_rot, 2, device=x.device).float() / d_rot))
    pos = torch.arange(T, device=x.device).float()
    ang = torch.einsum("n,d->nd", pos, theta)
    ang = torch.cat([ang, ang], dim=1)                      # (T, d_rot)
    cos, sin = ang.cos().to(x.dtype), ang.sin().to(x.dtype)
    xr, xp = x[..., :d_rot], x[..., d_rot:]
    half = d_rot // 2
    rot = torch.cat([-xr[..., half:], xr[..., :half]], dim=-1)
    xr = xr * cos[None, None] + rot * sin[None, None]
    return torch.cat((xr, xp), dim=-1)


# --------------------------------------------------------------------------- #
# DiT block  (models/diffusion_transformer.py:82-121)
# --------------------------------------------------------------------------- #
def _attention(state: State, pfx: str, x: torch.Tensor, attn_mask: torch.Tensor, n_heads: int) -> torch.Tensor:
    """models/diffusion_transformer.py:58-79."""
    q = F.conv1d(x, state[pfx + "conv_q.weight"], state[pfx + "conv_q.bias"])
    k = F.conv1d(x, state[pfx + "conv_k.weight"], state[pfx + "conv_k.bias"])
    v = F.conv1d(x, state[pfx + "conv_v.weight"], state[pfx + "conv_v.bias"])
    b, d, t = q.shape
    dh = d // n_heads
    q = q.view(b, n_heads, dh, t).transpose(2, 3)
    k = k.view(b, n_heads, dh, t).transpose(2, 3)
    v = v.view(b, n_heads, dh, t).transpose(2, 3)
    d_rot = int(dh * 0.5)                                   # :48-49
    q = rope_partial(q, d_rot)
    k = rope_partial(k, d_rot)
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=attn_mask, dropout_p=0.0)   # :77
    o = o.transpose(2, 3).contiguous().view(b, d, t)
    return F.conv1d(o, state[pfx + "conv_o.weight"], state[pfx + "conv_o.bias"])


def _ffn(state: State, pfx: str, x: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """models/diffusion_transformer.py:25-30 (eval: dropout is a no-op)."""
    w1, b1 = state[pfx + "conv_1.weight"], state[pfx + "conv_1.bias"]
    w2, b2 = state[pfx + "conv_2.weight"], state[pfx + "conv_2.bias"]
    h = F.conv1d(x * mask, w1, b1, padding=w1.shape[-1] // 2)
    h = F.silu(h)
    h = F.conv1d(h * mask, w2, b2, padding=w2.shape[-1] // 2)
    return h * mask


def _layer_norm_c(x: torch.Tensor) -> torch.Tensor:
    """LayerNorm over the channel axis of (B, C, T), no affine, eps 1e-5
    (models/diffusion_transformer.py:88,90,111-112)."""
    return F.layer_norm(x.transpose(1, 2), (x.shape[1],), eps=1e-5).transpose(1, 2)


def dit_block(state: State, pfx: str, x: torch.Tensor, c: torch.Tensor, mask: torch.Tensor, n_heads: int) -> torch.Tensor:
    """models/diffusion_transformer.py:98-121."""
    x = x * mask
    am = mask.unsqueeze(1) * mask.unsqueeze(-1)                               # (B,1,T,T) :107
    am = torch.zeros_like(am).masked_fill(am == 0, -torch.finfo(x.dtype).max)  # :108
    mod = F.linear(F.silu(c), state[pfx + "adaLN_modulation.2.weight"], state[pfx + "adaLN_modulation.2.bias"])
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = mod.unsqueeze(2).chunk(6, dim=1)
    u = _layer_norm_c(x) * (1 + scale_msa) + shift_msa
    x = x + gate_msa * _attention(state, pfx + "attn.", u, am, n_heads) * mask
    u = _layer_norm_c(x) * (1 + scale_mlp) + shift_mlp
    x = x + gate_mlp * _ffn(state, pfx + "mlp.", u, mask)
    return x


# --------------------------------------------------------------------------- #
# Estimator  (models/estimator.py:103-137)
# --------------------------------------------------------------------------- #
def cond_proj(state: State, mu: torch.Tensor) -> torch.Tensor:
    """models/estimator.py:83-89,118 — three k=3 convs, SiLU between, UNMASKED."""
    h = mu
    for i, last in ((0, False), (2, False), (4, True)):
        w, b = state[f"cond_proj.{i}.weight"], state[f"cond_proj.{i}.bias"]
        h = F.conv1d(h, w, b, padding=w.shape[-1] // 2)
        if not last:
            h = F.silu(h)
    return h


def estimator_forward(state: State, t: torch.Tensor, x: torch.Tensor, mask: torch.Tensor,
                      mu: torch.Tensor, c: torch.Tensor, n_heads: int = 4) -> torch.Tensor:
    """models/estimator.py:103-137.  t: 0-dim or (B,); x, mu: (B,M,T); mask (B,1,T); c (B,gin)."""
    hidden = state["in_proj.weight"].shape[0]
    n_layers = 1 + max(int(k.split(".")[1]) for k in state if k.startswith("blocks."))
    n_lsc = n_layers // 2
    temb = time_embedding(state, t, hidden)                                   # :117
    h = cond_proj(state, mu)                                                  # :118
    h = torch.cat((x, h), dim=1)                                              # :120
    h = F.conv1d(h, state["in_proj.weight"], state["in_proj.bias"])          # :121
    skips = []
    for i in range(n_layers):
        if i < n_lsc:
            skips.append(h)                                                   # :128-129
        else:
            h = torch.cat((h, skips.pop()), dim=1)                            # :131
            w, b = state[f"lsc_layers.{i - n_lsc}.weight"], state[f"lsc_layers.{i - n_lsc}.bias"]
            h = F.conv1d(h, w, b, padding=w.shape[-1] // 2)                   # :132
        pfx = f"blocks.{i}."
        film = F.conv1d(temb.unsqueeze(2), state[pfx + "time_fusion.film.weight"], state[pfx + "time_fusion.film.bias"])
        gamma, beta = torch.chunk(film, 2, dim=1)                             # :30-33
        h = (gamma * h + beta) * mask                                         # :16
        h = dit_block(state, pfx + "block.", h, c, mask, n_heads)             # :17
    out = F.conv1d(h * mask, state["final_proj.weight"], state["final_proj.bias"])   # :136
    return out * mask                                                         # :137


def cfg_estimator(state: State, t, x, mask, mu, c, fake_speaker, fake_content, cfg_strength: float,
                  n_heads: int = 4) -> torch.Tensor:
    """models/flow_matching.py:58-67 — two sequential estimator calls + lerp."""
    fs = fake_speaker.repeat(x.size(0), 1)
    fc = fake_content.repeat(x.size(0), 1, x.size(-1))
    cond = estimator_forward(state, t, x, mask, mu, c, n_heads)
    uncond = estimator_forward(state, t, x, mask, fc, fs, n_heads)
    return uncond + cfg_strength * (cond - uncond)


# --------------------------------------------------------------------------- #
# Fixed-grid ODE driver — restated from torchdiffeq's published fixed-grid
# solvers (call site models/flow_matching.py:54).  PARITY UNPINNED: the package
# is absent; tableaux below are the textbook ones torchdiffeq documents.
# --------------------------------------------------------------------------- #
# Dormand–Prince 5(4) tableau, used WITHOUT error control for "dopri5_fixed".
_DP_C = (0.0, 1 / 5, 3 / 10, 4 / 5, 8 / 9, 1.0)
_DP_A = (
    (),
    (1 / 5,),
    (3 / 40, 9 / 40),
    (44 / 45, -56 / 15, 32 / 9),
    (19372 / 6561, -25360 / 2187, 64448 / 6561, -212 / 729),
    (9017 / 3168, -355 / 33, 46732 / 5247, 49 / 176, -5103 / 18656),
)
_DP_B = (35 / 384, 0.0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84)


def odeint_fixed(f: Callable, y0: torch.Tensor, t_span: torch.Tensor, method: str = "euler") -> torch.Tensor:
    """Returns the final state y(t_span[-1]).  f(t, y) with t a 0-dim tensor."""
    y = y0
    for i in range(len(t_span) - 1):
        t0, t1 = t_span[i], t_span[i + 1]
        dt = t1 - t0
        if method == "euler":
            y = y + dt * f(t0, y)
        elif method == "midpoint":
            half = 0.5 * dt
            y_mid = y + half * f(t0, y)
            y = y + dt * f(t0 + half, y_mid)
        elif method == "rk4":      # torchdiffeq's "rk4" is the 3/8-rule variant
            k1 = f(t0, y)
            k2 = f(t0 + dt / 3, y + dt * k1 / 3)
            k3 = f(t0 + dt * 2 / 3, y + dt * (k2 - k1 / 3))
            k4 = f(t1, y + dt * (k1 - k2 + k3))
            y = y + (k1 + 3 * (k2 + k3) + k4) * dt * 0.125
        elif method == "dopri5_fixed":
            ks = []
            for s in range(6):
                ys = y
                for j, a in enumerate(_DP_A[s]):
                    ys = ys + (dt * a) * ks[j]
                ks.append(f(t0 + _DP_C[s] * dt, ys))
            inc = 0
            for b, k in zip(_DP_B, ks):
                if b != 0.0:
                    inc = inc + b * k
            y = y + dt * inc
        else:
            raise ValueError(f"unknown fixed-grid method {method!r}")
    return y


def cfm_forward(state: State, mu: torch.Tensor, mask: torch.Tensor, n_timesteps: int, z: torch.Tensor,
                c: torch.Tensor, method: str = "euler", cfg: Optional[dict] = None, n_heads: int = 4) -> torch.Tensor:
    """models/flow_matching.py:24-55 with the noise ``z`` (= randn_like(mu)*temperature,
    UNMASKED, :45) passed in so both sides consume the same draw."""
    t_span = torch.linspace(0, 1, n_timesteps + 1, device=mu.device).to(mu.dtype)   # :46
    if cfg is None:
        f = lambda t, y: estimator_forward(state, t, y, mask, mu, c, n_heads)
    else:
        f = lambda t, y: cfg_estimator(state, t, y, mask, mu, c, cfg["fake_speaker"], cfg["fake_content"],
                                       cfg["cfg_strength"], n_heads)
    with torch.inference_mode():
        return odeint_fixed(f, z, t_span, method)


def cfm_loss(state: State, x1: torch.Tensor, mask: torch.Tensor, mu: torch.Tensor, c: torch.Tensor, u01: torch.Tensor,
             z: torch.Tensor, sigma_min: float = 1e-4, n_heads: int = 4):
    """models/flow_matching.py:69-100 (eval mode, no autograd) with the two random draws passed in:
    ``u01`` = the ``torch.rand([b,1,1])`` draw (:92), ``z`` = ``randn_like(x1)`` (:96).  Returns (loss, y)."""
    t = 1 - torch.cos(u01 * 0.5 * torch.pi)                                     # :93
    y = (1 - (1 - sigma_min) * t) * z + t * x1                                  # :98
    u = x1 - (1 - sigma_min) * z                                                # :99
    with torch.inference_mode():
        v = estimator_forward(state, t.squeeze(), y, mask, mu, c, n_heads)
    loss = F.mse_loss(v, u, reduction="sum") / (torch.sum(mask) * u.size(1))    # :101
    return loss, y
