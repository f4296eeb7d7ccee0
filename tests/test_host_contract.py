"""Host-side contract tests (no GPU): state_dict scheme, C-ABI surface, loud failure without CUDA, flat storage."""
import ctypes
import json
import os
import re

import pytest
import torch

from tests import parity_common as pc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_keys_match_reference_zoo():
    """Names, shapes and ORDER of the 478-entry state_dict (golden list dumped from the reference's own modules)."""
    from micro_diffusion_b200.arch import DiTConfig, micro_dit_tiny_2_kwargs, micro_dit_xl_2_kwargs
    gold = json.load(open(os.path.join(pc.GOLDEN, "state_dict_keys.json")))
    cases = {"MicroDiT_Tiny_2_32_4": micro_dit_tiny_2_kwargs(input_size=32, in_channels=4),
             "MicroDiT_Tiny_2_64_16": micro_dit_tiny_2_kwargs(input_size=64, in_channels=16, pos_interp_scale=2.0),
             "MicroDiT_XL_2_32_4": micro_dit_xl_2_kwargs(input_size=32, in_channels=4)}
    for name, kw in cases.items():
        cfg = DiTConfig(**kw)
        mine = [[k, list(s)] for k, s in cfg.buffer_specs() + cfg.param_specs()]
        assert mine == gold[name], name
    assert len(gold["MicroDiT_XL_2_32_4"]) == 478


def test_module_state_dict_and_flat_views():
    from micro_diffusion_b200.models.dit import MicroDiT_Tiny_2
    from oracle.emu_ops import EmuOps
    gold = json.load(open(os.path.join(pc.GOLDEN, "state_dict_keys.json")))["MicroDiT_Tiny_2_32_4"]
    net = MicroDiT_Tiny_2(ops_factory=lambda d: EmuOps(d))
    sd = net.state_dict()
    assert [[k, list(v.shape)] for k, v in sd.items()] == gold
    # default init reproduces the reference's degeneracy: zero-initialised adaLN / output layers
    assert float(sd["final_layer.linear.weight"].abs().max()) == 0.0
    assert float(sd["blocks.3.adaLN_modulation.1.weight"].abs().max()) == 0.0
    assert abs(float(sd["blocks.0.norm1.weight"].mean()) - 1.0) < 1e-6
    st = net.store
    for n, p in net.named_parameters():
        assert p.data_ptr() == st.p[n].data_ptr() and p.dtype == torch.float32
    # load_state_dict writes through the views into the flat buffer
    new = {k: torch.full_like(v, 0.5) for k, v in sd.items()}
    net.load_state_dict(new)
    assert float(st.flat[st.layout.slots["blocks.0.attn.qkv.weight"][0]]) == 0.5
    # the stacked GEMM groups are contiguous
    assert st.W("ada").shape == (st.layout.ada_rows, 512)
    assert st.W("blocks.0.mlp.w12").shape[0] == 2 * net.cfg.blocks[0].ffn_dim


def test_c_abi_exports_every_declared_symbol():
    from micro_diffusion_b200 import _lib
    from micro_diffusion_b200.ops import _PROTOS, EXPORTED_SYMBOLS
    header = open(os.path.join(ROOT, "include", "microdit_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = re.findall(r"MD_API\s+(?:const\s+char\*|int)\s+(md_\w+)\s*\(([^;]*?)\)\s*;", header, flags=re.S)
    assert len(declared) >= 39
    lib = _lib.load()
    for name, args in declared:
        assert hasattr(lib, name), f"{name} declared in include/microdit_b200.h but not exported"
        assert name in EXPORTED_SYMBOLS
        if name in _PROTOS:
            nargs = len([a for a in args.split(",") if a.strip()])
            assert nargs == len(_PROTOS[name]), f"ctypes prototype of {name} is out of date"
    assert lib.md_abi_version() == 4
    # struct layout of md_gemm_args must match the header field order
    fields = re.search(r"typedef struct md_gemm_args \{(.*?)\} md_gemm_args;", header, flags=re.S).group(1)
    names = re.findall(r"(\w+)\s*(?:,|;)", re.sub(r"\b(const|void|int64_t|int32_t|float)\b|\*", " ", fields))
    assert names == [f[0] for f in _lib.GemmArgs._fields_]


def test_argument_validation_without_gpu():
    """Validation happens before any launch, so it can be exercised on a CPU-only box."""
    from micro_diffusion_b200 import _lib
    lib = _lib.load()
    lib.md_last_error.restype = ctypes.c_char_p
    lib.md_ln_fwd.restype = ctypes.c_int
    rc = lib.md_ln_fwd(None, 0, None, None, None, None, None, None, None, ctypes.c_int64(0), ctypes.c_int64(1), None,
                       None, None, ctypes.c_int64(4), ctypes.c_int64(100), ctypes.c_float(1e-6), 0, None)
    assert rc == -3 and b"D=100" in lib.md_last_error()
    args = _lib.GemmArgs()
    assert lib.md_gemm_bf16(ctypes.byref(args), None) == -1


def test_product_path_fails_loudly_without_cuda():
    from micro_diffusion_b200._lib import MicroditLibraryError
    from micro_diffusion_b200.models.dit import DiT
    from micro_diffusion_b200.ops import CudaOps
    from oracle import configs
    with pytest.raises(MicroditLibraryError):
        CudaOps("cpu")
    # the model lives on the CPU, so its first forward asks for CudaOps("cpu") whether or not a GPU is present
    net = DiT(**configs.PARITY_CONFIGS["P"]["ctor"])  # default ops factory = CUDA
    with pytest.raises(MicroditLibraryError), torch.no_grad():
        net(torch.zeros(1, 4, 32, 32), torch.zeros(1), torch.zeros(1, 1, 77, 1024).half())
    with pytest.raises(RuntimeError):  # training-mode autograd through DiT.forward is refused, not silently wrong
        net(torch.zeros(1, 4, 32, 32), torch.zeros(1), torch.zeros(1, 1, 77, 1024).half())


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "micro_diffusion_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"


def test_drop_in_namespace_and_factory():
    import micro_diffusion.models.model as m
    import micro_diffusion.models.utils as u
    from micro_diffusion_b200.models.model import PrecomputedLatentStubs
    from oracle.emu_ops import EmuOps
    assert u.text_encoder_embedding_format("openclip:hf-hub:apple/DFN5B-CLIP-ViT-H-14-378") == (77, 1024)
    with pytest.raises(ValueError):
        u.text_encoder_embedding_format("nope")
    vae, te, tok = PrecomputedLatentStubs.make()
    ld = m.create_latent_diffusion(dit_arch="MicroDiT_Tiny_2", latent_res=32, in_channels=4, train_mask_ratio=0.75,
                                   vae=vae, text_encoder=te, tokenizer=tok)
    assert ld.dit.in_channels == 4 and ld.dit.patch_size == 2 and ld.train_mask_ratio == 0.75
    assert ld.edm_config.sigma_data == 0.9 and ld.edm_config.P_mean == -0.6 and ld.latent_res == 32
    assert ld.dit._fsdp_wrap is True and callable(ld.randn_like)
    assert len(list(ld.dit.named_parameters())) == 288
    with pytest.raises(AttributeError):
        m.create_latent_diffusion(dit_arch="NoSuchArch", vae=vae, text_encoder=te, tokenizer=tok)
    assert "loss" in ld.get_metrics()


def test_pos_embed_matches_golden_probe():
    from micro_diffusion_b200.models.utils import get_2d_sincos_pos_embed
    fx = torch.load(os.path.join(pc.GOLDEN, "parity_S.pt"), weights_only=False)
    pe = torch.from_numpy(get_2d_sincos_pos_embed(256, 8, pos_interp_scale=2.0, base_size=8)).float()
    assert torch.allclose(pe[::7, ::13], fx["pos_embed_probe"], atol=1e-6)


def test_gemm_args_struct_layout_matches_the_header(tmp_path):
    """The ctypes mirror of md_gemm_args (micro_diffusion_b200/_lib.py) must have the field order, offsets and size
    the C header declares: compile a probe against include/microdit_b200.h with gcc and compare."""
    import ctypes
    import shutil
    import subprocess
    from micro_diffusion_b200._lib import GemmArgs
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = [f[0] for f in GemmArgs._fields_]
    src = tmp_path / "probe.c"
    body = "\n".join(f'  printf("{n} %zu\\n", offsetof(md_gemm_args, {n}));' for n in names)
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "microdit_b200.h"\nint main(void) {\n' + body +
                   '\n  printf("sizeof %zu\\n", sizeof(md_gemm_args));\n  return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.run([gcc, "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for n in names:
        assert int(out[n]) == getattr(GemmArgs, n).offset, n
    assert int(out["sizeof"]) == ctypes.sizeof(GemmArgs)


def test_cast_table_covers_every_operand_copy():
    """ParamStore._cast_table (one md_cast_transpose_multi launch per exchange range) must produce exactly the copies the
    per-matrix entry point produces, including the 32-row interleave of the fused-SwiGLU stacks and the expert banks."""
    import torch
    from oracle.emu_ops import EmuOps
    from tests import parity_common as pc
    ld = pc.build_product("S", device="cpu", ops_factory=lambda d: EmuOps(d, exact=False))
    st = ld.dit.store
    ops = ld.dit.engine.ops
    st.flat.copy_(torch.randn(st.flat.shape, generator=torch.Generator().manual_seed(3)))
    assert st.interleave, "the S configuration has SwiGLU stacks with f % 32 == 0"
    st.refresh_copies(ops, None, force=True)
    wb, wbt = st.wb.clone(), st.wbt.clone()
    ref_b, ref_t = torch.zeros_like(wb), torch.zeros_like(wbt)
    covered = 0
    for g in st.layout.groups.values():
        src = st.flat[g.offset: g.offset + g.numel].view(g.batch, g.rows, g.cols)
        b = ref_b[g.offset: g.offset + g.numel].view(g.batch, g.rows, g.cols)
        t = ref_t[g.offset: g.offset + g.numel].view(g.batch, g.cols, g.rows) if g.need_t else None
        ops.cast_transpose(src, b, t, interleave_half=st.interleave.get(g.name, 0))
        covered += g.numel
        assert torch.equal(wb[g.offset: g.offset + g.numel], ref_b[g.offset: g.offset + g.numel]), g.name
        if g.need_t:
            assert torch.equal(wbt[g.offset: g.offset + g.numel], ref_t[g.offset: g.offset + g.numel]), g.name
    for part in ("front", "back"):
        desc, tiles = st._cast_table(part)
        d = desc.tolist()
        assert all(d[i][5] < d[i + 1][5] for i in range(len(d) - 1)) and tiles == d[-1][5] + d[-1][6] * ((d[-1][1] + 63) // 64)
    assert covered > 0
