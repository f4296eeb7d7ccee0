"""Generate the fixtures under tests/golden/ from the UNMODIFIED reference (needs its source tree, see oracle.ref_import).

    python -m oracle.make_golden             # parity_<cfg>.pt
    python -m oracle.make_golden sampler     # sampler_<cfg>.pt
    python -m oracle.make_golden reference   # reference_grads_<cfg>.pt, reference_get_mask.pt, reference_configs/

For every config in oracle.configs.PARITY_CONFIGS: synthetic non-degenerate weights (oracle.weights, seed 7),
synthetic batch (seed 11), the reference's three random draws replayed from torch.manual_seed(123)
(SURVEY.md section 3.2).  Stored (fp32, fp32-reference arithmetic):
  loss, per-sample D_x ('sample' of model_forward_wrapper), mask, and per-parameter gradient fingerprints
  (L2 norm + dot with a fixed seeded probe) plus a few complete gradient tensors.
Also the reference's own amp-bf16 deviation from its fp32 result (loss / gradient), which is the yardstick
the bf16 kernel path is held to (DESIGN.md "Numerics").
The weights and inputs are NOT stored: they are pure functions of the seeds (oracle.weights).
"""
from __future__ import annotations

import os
import sys
import zlib

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import configs, ref_import, weights  # noqa: E402

WEIGHT_SEED, BATCH_SEED, DRAW_SEED = 7, 11, 123
FULL_GRADS = ("final_layer.linear.weight", "x_embedder.proj.weight", "patch_mixer.1.mlp.gate.weight",
              "blocks.0.norm1.weight", "y_embedder.y_proj.norm.weight", "t_embedder.mlp.0.bias")


def fingerprint(name, g):
    pr = weights.synth_tensor("probe:" + name, g.shape, 99)
    return float(g.norm()), float((g * pr).sum())


def reference_case(ref_dit, c):
    """The reference DiT of config `c` with the seeded weights, its LatentDiffusion (train mode) and the seeded batch."""
    ct = c["ctor"]
    net = ref_dit.DiT(**ct)
    sd = weights.synth_state_dict(net.state_dict(), seed=WEIGHT_SEED)
    net.load_state_dict(sd)
    ld = ref_import.build_reference_latent_diffusion(net, c["p_mean"], c["p_std"], c["mask_ratio"], ct["input_size"])
    ld.train()
    batch = weights.synth_batch(c["batch"], ct["in_channels"], ct["input_size"], seed=BATCH_SEED)
    return net, sd, ld, batch


def main():
    ref_dit, ref_model, _ = ref_import.load_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    for name, c in configs.PARITY_CONFIGS.items():
        ct = c["ctor"]
        net, sd, ld, batch = reference_case(ref_dit, c)
        res = {}
        for mode in ("fp32", "bf16"):
            net.zero_grad()
            torch.manual_seed(DRAW_SEED)
            with torch.autocast("cpu", dtype=torch.bfloat16, enabled=mode == "bf16"):
                loss, _, _ = ld({k: v.clone() for k, v in batch.items()})
            loss.backward()
            res[mode] = (float(loss), {k: p.grad.detach().clone() for k, p in net.named_parameters()})
        l32, g32 = res["fp32"]
        l16, g16 = res["bf16"]
        dev = sorted(float((g16[k] - g32[k]).norm() / (g32[k].norm() + 1e-12)) for k in g32)
        # denoiser output D_x on the same draws (fp32)
        g = ct["input_size"] // ct["patch_size"]
        rnd, eps, noise = weights.replay_draws(DRAW_SEED, (c["batch"], ct["in_channels"], ct["input_size"], ct["input_size"]),
                                               g * g, c["mask_ratio"])
        torch.manual_seed(DRAW_SEED)
        r2 = torch.randn([c["batch"], 1, 1, 1])
        assert torch.equal(r2, rnd), "generator replay does not match the global RNG stream"
        sigma = (rnd * c["p_std"] + c["p_mean"]).exp()
        x = batch["image_latents"].float()
        y = (batch["caption_latents"] * batch["drop_caption_mask"].view(-1, 1, 1, 1)).to(torch.float16).float()
        with torch.no_grad():
            torch.manual_seed(DRAW_SEED + 1)
            net.eval()
            den = ld.model_forward_wrapper(x + eps * sigma, sigma, y, net, mask_ratio=0.0)["sample"]
            net.train()
        fixture = {
            "config": name, "seeds": (WEIGHT_SEED, BATCH_SEED, DRAW_SEED),
            "loss": l32, "ref_amp_bf16_loss_rel": abs(l16 - l32) / l32,
            "ref_amp_bf16_grad_rel_median": dev[len(dev) // 2], "ref_amp_bf16_grad_rel_max": dev[-1],
            "denoised_unmasked": den.clone(),
            "grad_fingerprint": {k: fingerprint(k, v) for k, v in g32.items()},
            "grad_full": {k: g32[k].clone() for k in FULL_GRADS if k in g32},
            "pos_embed_sum": float(sd["pos_embed"].double().sum()), "pos_embed_probe": sd["pos_embed"][0, ::7, ::13].clone(),
            "torch_version": torch.__version__,
        }
        path = os.path.join(out_dir, f"parity_{name}.pt")
        torch.save(fixture, path)
        print(f"{name}: loss {l32:.6f}  ref amp-bf16 loss rel {fixture['ref_amp_bf16_loss_rel']:.2e} "
              f"grad rel median {fixture['ref_amp_bf16_grad_rel_median']:.2e} -> {path} "
              f"({os.path.getsize(path) / 1024:.0f} KiB)")


SAMPLER_SEED, SAMPLER_STEPS = 31, 3


def sampler_inputs(name):
    """Start noise and captions of the sampler fixture: pure functions of the seed."""
    c = configs.PARITY_CONFIGS[name]
    ct = c["ctor"]
    g = torch.Generator().manual_seed(SAMPLER_SEED)
    x = torch.randn(2, ct["in_channels"], ct["input_size"], ct["input_size"], generator=g)
    y = torch.randn(2, 1, 77, ct.get("caption_channels", 1024), generator=g).half().float()
    return x, y


def main_sampler(names=("P", "S")):
    """tests/golden/sampler_<cfg>.pt: edm_sampler_loop (model.py:232-297) of the unmodified reference, fp32, 3 Heun
    steps, with and without classifier-free guidance."""
    ref_dit, ref_model, _ = ref_import.load_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    for name in names:
        c = configs.PARITY_CONFIGS[name]
        ct = c["ctor"]
        net = ref_dit.DiT(**ct)
        net.load_state_dict(weights.synth_state_dict(net.state_dict(), seed=WEIGHT_SEED))
        ld = ref_import.build_reference_latent_diffusion(net, c["p_mean"], c["p_std"], c["mask_ratio"], ct["input_size"])
        ld.eval()
        x, y = sampler_inputs(name)
        fx = {"steps": SAMPLER_STEPS}
        for cfg in (1.0, 3.0):
            fx[f"out_cfg{cfg}"] = ld.edm_sampler_loop(x.clone(), y.clone(), steps=SAMPLER_STEPS, cfg=cfg).float()
        torch.save(fx, os.path.join(out_dir, f"sampler_{name}.pt"))
        print(name, {k: (tuple(v.shape), float(v.abs().mean())) for k, v in fx.items() if torch.is_tensor(v)})


GRAD_SAMPLE, GRAD_SAMPLE_SEED = 128, 41


def grad_sample_index(key, numel):
    """Flat indices of the gradient entries of parameter `key` kept in reference_grads_<cfg>.pt: all of them up to
    GRAD_SAMPLE, else a fixed sample drawn from a generator seeded by the key."""
    if numel <= GRAD_SAMPLE:
        return torch.arange(numel)
    g = torch.Generator().manual_seed((GRAD_SAMPLE_SEED * 1000003 + zlib.crc32(key.encode())) % (2 ** 31 - 1))
    return torch.randperm(numel, generator=g)[:GRAD_SAMPLE]


def main_reference_grads():
    """tests/golden/reference_grads_<cfg>.pt: the reference's fp32 loss and, for every parameter in `names` order, its
    gradient at the entries grad_sample_index() picks, concatenated -- the same case as main()."""
    ref_dit, _, _ = ref_import.load_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    for name, c in configs.PARITY_CONFIGS.items():
        net, _, ld, batch = reference_case(ref_dit, c)
        torch.manual_seed(DRAW_SEED)
        loss, _, _ = ld({k: v.clone() for k, v in batch.items()})
        loss.backward()
        names = [k for k, _ in net.named_parameters()]
        sample = torch.cat([p.grad.detach().reshape(-1)[grad_sample_index(k, p.numel())] for k, p in net.named_parameters()])
        path = os.path.join(out_dir, f"reference_grads_{name}.pt")
        torch.save({"config": name, "loss": loss.item(), "names": names, "grad_sample": sample,
                    "torch_version": torch.__version__}, path)
        print(f"{name}: loss {loss.item():.7f}, {len(names)} gradients -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


def main_reference_mask():
    """tests/golden/reference_get_mask.pt: get_mask (utils.py:383-399) of the reference after torch.manual_seed(5)."""
    _, _, ref_utils = ref_import.load_reference()
    torch.manual_seed(5)
    m = ref_utils.get_mask(3, 64, 0.75, torch.device("cpu"))
    torch.save({k: m[k].clone() for k in ("ids_keep", "ids_restore", "mask")},
               os.path.join(ROOT, "tests", "golden", "reference_get_mask.pt"))


def main_reference_configs():
    """tests/golden/reference_configs/: the reference's training YAML files, byte for byte."""
    import shutil
    src = os.path.join(ref_import.REFERENCE_ROOT, "configs")
    dst = os.path.join(ROOT, "tests", "golden", "reference_configs")
    os.makedirs(dst, exist_ok=True)
    for f in sorted(os.listdir(src)):
        if f.endswith(".yaml"):
            shutil.copyfile(os.path.join(src, f), os.path.join(dst, f))
            print(f"{f} -> {dst}")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "sampler":
        main_sampler()
    elif len(sys.argv) > 1 and sys.argv[1] == "reference":
        main_reference_grads()
        main_reference_mask()
        main_reference_configs()
    else:
        main()
