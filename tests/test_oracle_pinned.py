"""The CPU oracle (oracle.port) is pinned to committed golden fixtures generated from the unmodified reference
(oracle/make_golden.py): loss, D_x, gradient fingerprints and sampled gradients of every parameter, the sampler and
the token mask.  fp32 vs fp32, so the tolerance is reassociation-level: 1e-5 relative."""
import os

import pytest
import torch

from oracle import configs, port, weights
from tests import parity_common as pc

CASES = list(configs.PARITY_CONFIGS)


def _template(name):
    from micro_diffusion_b200.arch import DiTConfig
    cfg = DiTConfig(**configs.PARITY_CONFIGS[name]["ctor"])
    sd = {k: torch.zeros(s) for k, s in cfg.buffer_specs() + cfg.param_specs()}
    ct = configs.PARITY_CONFIGS[name]["ctor"]
    g = ct["input_size"] // ct["patch_size"]
    sd["pos_embed"] = port.sincos_pos_embed(ct["dim"], g, ct.get("pos_interp_scale", 1.0), g).unsqueeze(0)
    return sd


@pytest.mark.parametrize("name", CASES)
def test_port_matches_golden(name):
    fx = torch.load(os.path.join(pc.GOLDEN, f"parity_{name}.pt"), weights_only=False)
    loss, grads, den, sd = pc.oracle_run(name, _template(name))
    assert abs(loss - fx["loss"]) / fx["loss"] < 1e-5
    assert pc.rel_l2(den, fx["denoised_unmasked"]) < 1e-5
    assert abs(float(sd["pos_embed"].double().sum()) - fx["pos_embed_sum"]) < 1e-3
    assert torch.allclose(sd["pos_embed"][0, ::7, ::13], fx["pos_embed_probe"], atol=1e-6)
    for k, (norm, dot) in fx["grad_fingerprint"].items():
        g = grads[k]
        assert abs(float(g.norm()) - norm) <= 1e-4 * norm + 1e-7, k
        pr = weights.synth_tensor("probe:" + k, g.shape, 99)
        assert abs(float((g * pr).sum()) - dot) <= 2e-4 * norm * float(pr.norm()) + 1e-7, k
    for k, g in fx["grad_full"].items():
        assert pc.rel_l2(grads[k], g) < 1e-4, k


@pytest.mark.parametrize("name", CASES)
def test_port_matches_reference_grads(name):
    """Loss and the gradient of every parameter against the reference's own fp32 run of the same case (fixture from
    `oracle.make_golden reference`: the loss and a fixed seeded sample of each gradient)."""
    from oracle.make_golden import GRAD_SAMPLE, grad_sample_index
    fx = torch.load(os.path.join(pc.GOLDEN, f"reference_grads_{name}.pt"), weights_only=False)
    oloss, ograds, _, _ = pc.oracle_run(name, _template(name))
    assert abs(oloss - fx["loss"]) / fx["loss"] < 1e-6
    names = fx["names"]
    assert set(names) == set(ograds)
    ref = fx["grad_sample"].split([min(ograds[k].numel(), GRAD_SAMPLE) for k in names])
    for k, r in zip(names, ref):
        assert pc.rel_l2(ograds[k].reshape(-1)[grad_sample_index(k, ograds[k].numel())], r) < 1e-4, k


def test_mask_and_routing_match_reference():
    """port.random_mask against get_mask (utils.py:383-399) of the reference, both after torch.manual_seed(5)."""
    m = torch.load(os.path.join(pc.GOLDEN, "reference_get_mask.pt"))
    torch.manual_seed(5)
    noise = torch.rand(3, 64)
    keep, restore, mask = port.random_mask(noise, 0.75)
    assert torch.equal(keep, m["ids_keep"]) and torch.equal(restore, m["ids_restore"]) and torch.equal(mask, m["mask"])


@pytest.mark.parametrize("name", ["P", "S"])
def test_port_sampler_matches_golden(name):
    """edm_sampler_loop of the unmodified reference (fixture from oracle.make_golden sampler) vs the restatement."""
    from oracle.make_golden import SAMPLER_STEPS, sampler_inputs
    fx = torch.load(os.path.join(pc.GOLDEN, f"sampler_{name}.pt"), weights_only=False)
    c = configs.PARITY_CONFIGS[name]
    sd = weights.synth_state_dict(_template(name), seed=pc.WEIGHT_SEED)
    x, y = sampler_inputs(name)
    cfg = pc.port_config(c, c["ctor"])
    for g in (1.0, 3.0):
        out = port.edm_sampler(sd, cfg, x, y, SAMPLER_STEPS, guidance=g)
        assert pc.rel_l2(out, fx[f"out_cfg{g}"]) < 1e-5, g
