"""Row f-2: the reference's YAML configs drive the Composer-free trainer (config parsing is host logic: CPU)."""
import os

import pytest
import torch
import yaml

from tests import parity_common as pc

# the reference's configs/*.yaml, stored unchanged (oracle/make_golden.py reference)
REF_CONFIGS = os.path.join(pc.GOLDEN, "reference_configs")

MINI = """
exp_name: mini_run
seed: 18
algorithms:
  low_precision_layernorm:
    precision: amp_bf16
  gradient_clipping:
    clipping_type: norm
    clip_norm: 0.25
model:
  _target_: micro_diffusion.models.model.create_latent_diffusion
  dit_arch: MicroDiT_Tiny_2
  precomputed_latents: true
  in_channels: 4
  latent_res: 32
  train_mask_ratio: 0.75
dataset:
  image_size: 256
  train_batch_size: 8
  cap_drop_prob: 0.1
  train:
    _target_: micro_diffusion.datasets.latents_loader.build_streaming_latents_dataloader
    datadir:
      - DATADIR
    drop_last: true
    shuffle: true
optimizer:
  _target_: torch.optim.AdamW
  lr: 2.4e-4
  weight_decay: 0.1
  eps: 1.0e-8
  betas:
    - 0.9
    - 0.999
scheduler:
  _target_: composer.optim.CosineAnnealingWithWarmupScheduler
  t_warmup: 2ba
  alpha_f: 0.33
logger:
  progress:
    _target_: composer.loggers.TensorboardLogger
callbacks:
  nan_catcher:
    _target_: micro_diffusion.models.callbacks.NaNCatcher
trainer:
  _target_: composer.Trainer
  max_duration: 3ba
  save_interval: 2ba
  device_train_microbatch_size: 4
  run_name: ${exp_name}
  seed: ${seed}
  save_folder: SAVEDIR/${exp_name}/
  fsdp_config:
    sharding_strategy: "SHARD_GRAD_OP"
misc:
  compile: true
"""


def test_interpolation_overrides_and_trainer_kwargs(tmp_path):
    from micro_diffusion_b200 import train
    p = tmp_path / "mini.yaml"
    p.write_text(MINI.replace("DATADIR", "/data").replace("SAVEDIR", "/out"))
    cfg = train.load_config(str(p), ["trainer.device_train_microbatch_size=2", "optimizer.lr=1.0e-3",
                                     "dataset.train.datadir=[/a,/b]"])
    assert cfg["trainer"]["run_name"] == "mini_run" and cfg["trainer"]["seed"] == 18  # type-preserving ${seed}
    assert cfg["trainer"]["save_folder"] == "/out/mini_run/"
    assert cfg["dataset"]["train"]["datadir"] == ["/a", "/b"]
    kw = train.trainer_kwargs(cfg)
    assert kw["lr"] == 1e-3 and kw["device_train_microbatch_size"] == 2 and kw["clip_norm"] == 0.25
    assert kw["t_warmup"] == "2ba" and kw["alpha_f"] == 0.33 and kw["max_duration"] == "3ba"
    assert kw["betas"] == (0.9, 0.999) and kw["weight_decay"] == 0.1 and kw["eps"] == 1e-8
    notes = " ".join(train.ignored_sections(cfg))
    assert "logger" in notes and "fsdp_config" in notes and "compile" in notes and "low_precision" in notes
    assert "nan_catcher" not in notes
    with pytest.raises(ValueError):
        train.trainer_kwargs({"optimizer": {"_target_": "torch.optim.SGD"}})
    with pytest.raises(ValueError):
        train.apply_overrides({}, ["novalue"])


@pytest.mark.parametrize("name", ["res_256_pretrain", "res_256_finetune", "res_512_pretrain", "res_512_finetune"])
def test_every_reference_yaml_maps_onto_the_trainer(name):
    from micro_diffusion_b200 import train
    from micro_diffusion_b200.trainer import parse_batches
    cfg = train.load_config(os.path.join(REF_CONFIGS, name + ".yaml"))
    kw = train.trainer_kwargs(cfg)
    assert parse_batches(kw["max_duration"]) > 0 and parse_batches(kw["t_warmup"]) >= 0
    assert kw["clip_norm"] == cfg["algorithms"]["gradient_clipping"]["clip_norm"]
    assert kw["lr"] == float(cfg["optimizer"]["lr"]) and kw["device_train_microbatch_size"] > 0
    m = cfg["model"]
    assert m["_target_"] == "micro_diffusion.models.model.create_latent_diffusion" and m["precomputed_latents"]
    assert cfg["dataset"]["image_size"] == 8 * m["latent_res"]
    if "512" in name and "pretrain" in name:  # res_512_pretrain.yaml:117-123
        assert kw["load_weights_only"] and not kw["load_strict_model_weights"]
        assert "state/model/dit.pos_embed" in kw["load_ignore_keys"]
    # the `_target_` of dataset.train is the function name this repo re-exports
    import micro_diffusion_b200.data as data
    assert cfg["dataset"]["train"]["_target_"].endswith(".build_streaming_latents_dataloader")
    assert hasattr(data, "build_streaming_latents_dataloader")


def test_build_and_fit_from_yaml_on_cpu_kernels(tmp_path):
    """End to end on the CPU kernel contracts: YAML -> dataset shards -> device loader -> Trainer.fit -> checkpoint."""
    import numpy as np
    from micro_diffusion_b200 import train
    from micro_diffusion_b200.data import write_mds
    from oracle.emu_ops import EmuOps
    rng = np.random.default_rng(0)
    samples = [{"caption": "c", "caption_latents": rng.standard_normal(77 * 1024).astype(np.float16).tobytes(),
                "latents_256": rng.standard_normal(4 * 32 * 32).astype(np.float16).tobytes()} for _ in range(16)]
    write_mds(str(tmp_path / "data"), samples, {"caption": "str", "caption_latents": "bytes", "latents_256": "bytes"})
    p = tmp_path / "mini.yaml"
    p.write_text(MINI.replace("DATADIR", str(tmp_path / "data")).replace("SAVEDIR", str(tmp_path / "out")))
    cfg = train.load_config(str(p))
    model = pc.build_product("P", ops_factory=lambda d: EmuOps(d, exact=True))  # injected: Tiny_2 on CPU kernels is slow
    _, loader, tr = train.build(cfg, torch.device("cpu"), model=model)
    assert len(loader) == 2 and tr.microbatch == 4 and tr.t_max == 3
    logs = []
    tr.log, tr.log_every = logs.append, 1
    tr.fit()
    assert tr.batch == 3 and len(logs) == 3
    assert os.path.exists(os.path.join(str(tmp_path / "out"), "mini_run", "ba2.pt"))
