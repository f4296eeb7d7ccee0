"""Functional fp32 restatement of the MicroDiT training hot path -- the travelling CPU oracle.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Plain torch on CPU, no nn.Module: every function
takes the flat reference state_dict (`P`: key -> tensor, the 478-entry scheme of SURVEY.md section 8b)
and derives the architecture from the tensor shapes.  Each function cites the reference code it follows
(paths relative to the reference root).  All random draws are explicit inputs so that a seeded run of
the unmodified reference can be replayed draw for draw (SURVEY.md section 3.2: sigma-normal -> eps ->
mask noise).

Pinned against the reference by tests/test_oracle_pinned.py through the committed fixtures tests/golden/*.pt,
generated from the reference by oracle/make_golden.py.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


@dataclass(frozen=True)
class PortConfig:
    patch_size: int = 2
    head_dim: int = 64
    num_experts: int = 8
    expert_capacity: float = 2.0
    norm_eps: float = 1e-6
    sigma_data: float = 0.9  # model.py:79
    p_mean: float = -0.6
    p_std: float = 1.2
    freq_dim: int = 512  # utils.py:256


# ---------------------------------------------------------------------------------------------- pieces

def _lin(P, name: str, x: Tensor) -> Tensor:
    return F.linear(x, P[name + ".weight"], P.get(name + ".bias"))


def _ln(x: Tensor, w, eps: float) -> Tensor:
    """create_norm: weight-only LayerNorm or non-affine LayerNorm (utils.py:71-78)."""
    return F.layer_norm(x, (x.shape[-1],), w, None, eps)


def _gelu_tanh(x: Tensor) -> Tensor:
    return F.gelu(x, approximate="tanh")


def _mlp(P, pre: str, x: Tensor, eps: float) -> Tensor:
    """timm-style Mlp with the norm between activation and fc2 (utils.py:63-68)."""
    h = _gelu_tanh(_lin(P, pre + ".fc1", x))
    if pre + ".norm.weight" in P:
        h = _ln(h, P[pre + ".norm.weight"], eps)
    return _lin(P, pre + ".fc2", h)


def _heads(x: Tensor, hd: int) -> Tensor:  # (B,N,H*hd) -> (B,H,N,hd)
    b, n, c = x.shape
    return x.view(b, n, c // hd, hd).transpose(1, 2)


def self_attention(P, pre: str, x: Tensor, cfg: PortConfig) -> Tensor:
    """utils.py:178-196: qkv -> LN(q), LN(k) over the full hidden width -> SDPA -> proj."""
    q, k, v = _lin(P, pre + ".qkv", x).chunk(3, dim=-1)
    q = _ln(q, None, cfg.norm_eps)
    k = _ln(k, None, cfg.norm_eps)
    o = F.scaled_dot_product_attention(_heads(q, cfg.head_dim), _heads(k, cfg.head_dim), _heads(v, cfg.head_dim))
    o = o.transpose(1, 2).reshape(x.shape[0], x.shape[1], -1)
    return _lin(P, pre + ".proj", o)


def cross_attention(P, pre: str, x: Tensor, y: Tensor, cfg: PortConfig) -> Tensor:
    """utils.py:116-136: q from x, k/v from the caption tokens, same QK-LayerNorm."""
    q = _lin(P, pre + ".q_linear", x)
    k, v = _lin(P, pre + ".kv_linear", y).chunk(2, dim=-1)
    q = _ln(q, None, cfg.norm_eps)
    k = _ln(k, None, cfg.norm_eps)
    o = F.scaled_dot_product_attention(_heads(q, cfg.head_dim), _heads(k, cfg.head_dim), _heads(v, cfg.head_dim))
    o = o.transpose(1, 2).reshape(x.shape[0], x.shape[1], -1)
    return _lin(P, pre + ".proj", o)


def swiglu(P, pre: str, x: Tensor) -> Tensor:
    """dit.py:88-89."""
    return _lin(P, pre + ".w3", F.silu(_lin(P, pre + ".w1", x)) * _lin(P, pre + ".w2", x))


def ecmoe_route(probs: Tensor, k: int):
    """Expert-choice routing (dit.py:131-133): every expert takes its top-k tokens of each sample.
    probs (n,t,e) -> gate values g (n,e,k), token ids m (n,e,k)."""
    return torch.topk(probs.permute(0, 2, 1), k, dim=-1)


def ecmoe(P, pre: str, x: Tensor, cfg: PortConfig) -> Tensor:
    """dit.py:126-143, with the one-hot dispatch/combine einsums written as gather / index_add
    (algorithmically identical: p is a 0/1 selection matrix)."""
    n, t, d = x.shape
    e = cfg.num_experts
    k = int(cfg.expert_capacity * t / e)
    probs = F.softmax(F.linear(x, P[pre + ".gate.weight"]), dim=-1)
    g, m = ecmoe_route(probs, k)  # (n,e,k)
    xin = torch.gather(x.unsqueeze(1).expand(n, e, t, d), 2, m.unsqueeze(-1).expand(n, e, k, d))
    h = torch.einsum("nekd,edf->nekf", xin, P[pre + ".w1"])
    h = F.gelu(h)
    h = torch.einsum("nekf,efd->nekd", h, P[pre + ".w2"])
    out = torch.zeros_like(x)
    out.scatter_add_(1, m.reshape(n, e * k, 1).expand(n, e * k, d), (g.unsqueeze(-1) * h).reshape(n, e * k, d))
    return out


def dit_block(P, pre: str, x: Tensor, y: Tensor, c: Tensor, cfg: PortConfig) -> Tensor:
    """DiTBlock.forward (dit.py:232-239)."""
    mod = F.linear(_gelu_tanh(c), P[pre + ".adaLN_modulation.1.weight"], P[pre + ".adaLN_modulation.1.bias"])
    sh_a, sc_a, g_a, sh_m, sc_m, g_m = mod.unsqueeze(1).chunk(6, dim=-1)
    eps = cfg.norm_eps
    h = _ln(x, P[pre + ".norm1.weight"], eps) * (1 + sc_a) + sh_a
    x = x + g_a * self_attention(P, pre + ".attn", h, cfg)
    x = x + cross_attention(P, pre + ".cross_attn", _ln(x, P[pre + ".norm2.weight"], eps), y, cfg)
    h = _ln(x, P[pre + ".norm3.weight"], eps) * (1 + sc_m) + sh_m
    if pre + ".mlp.gate.weight" in P:
        f = ecmoe(P, pre + ".mlp", h, cfg)
    else:
        f = swiglu(P, pre + ".mlp", h)
    return x + g_m * f


def timestep_embedding(t: Tensor, dim: int) -> Tensor:
    """utils.py:265-281 ([cos | sin], max_period 10000)."""
    half = dim // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    a = t[:, None].float() * freqs[None]
    return torch.cat([torch.cos(a), torch.sin(a)], dim=-1)


def sincos_pos_embed(dim: int, grid: int, pos_interp_scale: float, base_size: int) -> Tensor:
    """get_2d_sincos_pos_embed (utils.py:330-379): float32 grid, float64 omega, w-axis first,
    [sin | cos] halves per axis."""
    import numpy as np
    ax = np.arange(grid, dtype=np.float32) / (grid / base_size) / pos_interp_scale
    gw, gh = np.meshgrid(ax, ax)  # gw varies along columns (w), gh along rows (h)
    omega = 1.0 / 10000 ** (np.arange(dim // 4, dtype=np.float64) / (dim / 4.0))

    def one(pos):
        o = np.einsum("m,d->md", pos.reshape(-1), omega)
        return np.concatenate([np.sin(o), np.cos(o)], axis=1)

    return torch.from_numpy(np.concatenate([one(gw), one(gh)], axis=1)).float()


def random_mask(noise: Tensor, mask_ratio: float):
    """get_mask (utils.py:382-403) with the uniform noise passed in."""
    b, t = noise.shape
    keep = int(t * (1 - mask_ratio))
    shuffle = torch.argsort(noise, dim=1)
    restore = torch.argsort(shuffle, dim=1)
    mask = torch.ones(b, t, device=noise.device)
    mask[:, :keep] = 0
    mask = torch.gather(mask, 1, restore)
    return shuffle[:, :keep], restore, mask


def _depth(P, stem: str) -> int:
    n = 0
    while f"{stem}.{n}.norm1.weight" in P:
        n += 1
    return n


def conditioning_stem(P, cfg: PortConfig, t: Tensor, y: Tensor):
    """dit.py:480-485: returns (caption tokens (N,L,D), conditioning vector c (N,D))."""
    n = y.shape[0]
    temb = timestep_embedding(t.expand(n), cfg.freq_dim)
    temb = _lin(P, "t_embedder.mlp.2", _gelu_tanh(_lin(P, "t_embedder.mlp.0", temb)))
    yt = _mlp(P, "y_embedder.y_proj", y, cfg.norm_eps).squeeze(1)  # (N,L,D)
    eps = cfg.norm_eps
    hd_cfg = cfg
    yt = yt + self_attention(P, "y_emb_preprocess.attn", _ln(yt, P["y_emb_preprocess.norm1.weight"], eps), hd_cfg)
    yt = yt + swiglu(P, "y_emb_preprocess.mlp", _ln(yt, P["y_emb_preprocess.norm2.weight"], eps))
    pooled = _mlp(P, "pooled_y_emb_process", yt.mean(dim=1), eps)
    return yt, temb + pooled


def dit_forward(P, cfg: PortConfig, x: Tensor, t: Tensor, y: Tensor, mask_ratio: float = 0.0,
                mask_noise: Tensor | None = None):
    """DiT.forward_without_cfg (dit.py:455-519).  x (N,C,H,W), t (N,) or (1,), y (N,1,L,Dc).
    Returns dict(sample (N,C,H,W), mask (N,T) or None, ids_keep, ids_restore, tokens (N,T',p*p*C))."""
    p = cfg.patch_size
    n = x.shape[0]
    w = P["x_embedder.proj.weight"]
    tok = F.conv2d(x, w, P["x_embedder.proj.bias"], stride=p).flatten(2).transpose(1, 2) + P["pos_embed"]
    yt, c = conditioning_stem(P, cfg, t, y)
    mixer_depth = _depth(P, "patch_mixer")
    if mixer_depth:
        eps = cfg.norm_eps
        if "patch_mixer_map_xin.1.weight" in P:
            tok = _lin(P, "patch_mixer_map_xin.1", _ln(tok, P["patch_mixer_map_xin.0.weight"], eps))
            ym = _lin(P, "patch_mixer_map_y.1", _ln(yt, P["patch_mixer_map_y.0.weight"], eps))
        else:
            ym = yt
        for i in range(mixer_depth):
            tok = dit_block(P, f"patch_mixer.{i}", tok, ym, c, cfg)
    mask = ids_keep = ids_restore = None
    if mask_ratio > 0:
        ids_keep, ids_restore, mask = random_mask(mask_noise, mask_ratio)
        tok = torch.gather(tok, 1, ids_keep.unsqueeze(-1).expand(-1, -1, tok.shape[-1]))
    if mixer_depth and "patch_mixer_map_xout.1.weight" in P:
        tok = _lin(P, "patch_mixer_map_xout.1", _ln(tok, P["patch_mixer_map_xout.0.weight"], cfg.norm_eps))
    for i in range(_depth(P, "blocks")):
        tok = dit_block(P, f"blocks.{i}", tok, yt, c, cfg)
    mod = F.linear(_gelu_tanh(c), P["final_layer.adaLN_modulation.1.weight"], P["final_layer.adaLN_modulation.1.bias"])
    sh, sc = mod.unsqueeze(1).chunk(2, dim=-1)
    out_tok = _lin(P, "final_layer.linear", _ln(tok, P["final_layer.norm_final.weight"], cfg.norm_eps) * (1 + sc) + sh)
    full = out_tok
    if mask_ratio > 0:
        t_all = ids_restore.shape[1]
        pad = P["mask_token"].expand(n, t_all - out_tok.shape[1], -1)
        full = torch.gather(torch.cat([out_tok, pad], 1), 1, ids_restore.unsqueeze(-1).expand(-1, -1, out_tok.shape[-1]))
    g = int(round(full.shape[1] ** 0.5))
    cch = full.shape[-1] // (p * p)
    sample = full.reshape(n, g, g, p, p, cch).permute(0, 5, 1, 3, 2, 4).reshape(n, cch, g * p, g * p)
    return {"sample": sample, "mask": mask, "ids_keep": ids_keep, "ids_restore": ids_restore, "tokens": out_tok}


def edm_precondition(cfg: PortConfig, sigma: Tensor):
    """model.py:153-164 (sigma shaped (N,1,1,1))."""
    sd = cfg.sigma_data
    c_skip = sd ** 2 / (sigma ** 2 + sd ** 2)
    c_out = sigma * sd / (sigma ** 2 + sd ** 2).sqrt()
    c_in = 1 / (sd ** 2 + sigma ** 2).sqrt()
    c_noise = sigma.log() / 4
    return c_skip, c_out, c_in, c_noise


def denoise(P, cfg: PortConfig, x_noisy: Tensor, sigma: Tensor, y: Tensor, mask_ratio=0.0, mask_noise=None):
    """model_forward_wrapper (model.py:144-179)."""
    sigma = sigma.to(x_noisy.dtype).reshape(-1, 1, 1, 1)
    c_skip, c_out, c_in, c_noise = edm_precondition(cfg, sigma)
    out = dit_forward(P, cfg, c_in * x_noisy, c_noise.flatten(), y, mask_ratio, mask_noise)
    out["F"] = out["sample"]
    out["sample"] = c_skip * x_noisy + c_out * out["sample"]
    return out


def edm_loss(P, cfg: PortConfig, x: Tensor, y: Tensor, rnd_normal: Tensor, eps_noise: Tensor,
             mask_ratio: float = 0.0, mask_noise: Tensor | None = None):
    """edm_loss (model.py:181-210) with the three random draws passed in.
    Returns (loss scalar, dict with D_x, mask, per-sample losses)."""
    sd = cfg.sigma_data
    sigma = (rnd_normal.reshape(-1, 1, 1, 1) * cfg.p_std + cfg.p_mean).exp()
    weight = (sigma ** 2 + sd ** 2) / (sigma * sd) ** 2
    out = denoise(P, cfg, x + eps_noise * sigma, sigma, y, mask_ratio, mask_noise)
    loss = weight * (out["sample"] - x) ** 2
    if mask_ratio > 0:
        loss = F.avg_pool2d(loss.mean(dim=1), cfg.patch_size).flatten(1)
        unmask = 1 - out["mask"]
        per_sample = (loss * unmask).sum(dim=1) / unmask.sum(dim=1)
    else:
        per_sample = loss.flatten(1).mean(dim=1)
    out["per_sample"] = per_sample
    out["sigma"] = sigma.flatten()
    # model.py:210 takes loss.mean() over all elements when unmasked == mean of per-sample means
    return per_sample.mean(), out


def latent_diffusion_forward(P, cfg: PortConfig, batch: dict, rnd_normal, eps_noise, mask_ratio=0.0, mask_noise=None):
    """LatentDiffusion.forward (model.py:104-142) for precomputed latents: caption drop + fp32 casts."""
    latents = batch["image_latents"]
    cond = batch["caption_latents"]
    if "drop_caption_mask" in batch:
        cond = (cond * batch["drop_caption_mask"].view([-1] + [1] * (cond.dim() - 1))).to(cond.dtype)
    return edm_loss(P, cfg, latents.float(), cond.float(), rnd_normal, eps_noise, mask_ratio, mask_noise)


def edm_sampler(P, cfg: PortConfig, x: Tensor, y: Tensor, steps: int, guidance: float = 1.0, sigma_min: float = 0.002,
                sigma_max: float = 80.0, rho: float = 7.0) -> Tensor:
    """edm_sampler_loop (model.py:232-297) with the defaults of edm_config (model.py:74-88: S_churn 0, S_noise 1, so
    gamma = 0 and the churn noise term vanishes -- `randn_like` is still drawn by the reference but multiplied by 0);
    guidance > 1 goes through DiT.forward_with_cfg (dit.py:521-550).  fp64 state, fp32 denoiser."""
    P = {k: v.detach() for k, v in P.items()}
    i = torch.arange(steps, dtype=torch.float64)
    t_steps = (sigma_max ** (1 / rho) + i / (steps - 1) * (sigma_min ** (1 / rho) - sigma_max ** (1 / rho))) ** rho
    t_steps = torch.cat([t_steps, torch.zeros(1, dtype=torch.float64)])

    def den(xf: Tensor, sigma: Tensor) -> Tensor:
        sg = sigma.to(torch.float32).reshape(1).expand(xf.shape[0])
        if guidance > 1.0:
            c_skip, c_out, c_in, c_noise = edm_precondition(cfg, sg.view(-1, 1, 1, 1))
            xin = (c_in * xf)
            out = dit_forward(P, cfg, torch.cat([xin, xin], 0), torch.cat([c_noise.flatten()] * 2),
                              torch.cat([y, torch.zeros_like(y)], 0))["sample"]
            cond, unc = torch.split(out, xf.shape[0], dim=0)
            return c_skip * xf + c_out * (unc + guidance * (cond - unc))
        return denoise(P, cfg, xf, sg.view(-1, 1, 1, 1), y)["sample"]

    with torch.no_grad():
        x_next = x.to(torch.float64) * t_steps[0]
        for k in range(steps):
            t_hat, t_next = t_steps[k], t_steps[k + 1]
            x_hat = x_next
            d_cur = (x_hat - den(x_hat.float(), t_hat).double()) / t_hat
            x_next = x_hat + (t_next - t_hat) * d_cur
            if k < steps - 1:
                d_prime = (x_next - den(x_next.float(), t_next).double()) / t_next
                x_next = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * d_prime)
    return x_next.float()
