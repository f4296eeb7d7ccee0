#!/usr/bin/env python
"""bench.py -- training throughput of the MicroDiT hot path on B200 (contract: see README / task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c3|c4|c5|tiny]
                    [--dump-outputs DIR]

One "step" = one optimisation step at global batch 2048 (BASELINE.json metric): every rank runs its
2048/N images as microbatches through LatentDiffusion.forward + backward (the CUDA path through the C ABI),
then the data-parallel gradient mean (NCCL), then global-norm clip + AdamW.  Synthetic data of the reference's
batch contract (fp16 latents / fp16 77x1024 captions / caption-drop mask), random non-degenerate weights.

`value`  : img/s with the step's inputs already resident in HBM (device-timed, max over ranks).
`e2e`    : the same through the public API from PINNED HOST buffers, H2D copies and the loss read-back inside
           the timed region.
`--dump-outputs DIR` : after the timed steps, what the last of them handed its caller, as DIR/<name>.npy (float32):
           `loss` (the step's mean loss), `params` (updated fp32 parameters) and `adamw_m` (AdamW's first moment, the
           running mean of the clipped gradient), the latter two at DUMP_SAMPLE fixed seeded positions of the flat
           buffers.  Weights, batch and the EDM / mask draws are seeded, and the run uses the library's deterministic
           mode (DESIGN.md section 5.4; `config.deterministic` in the line): the fast path's cross-block float atomics
           make the gradients differ in the last bits from run to run, and AdamW and the following steps amplify that
           far beyond rounding.  With fixed-order sums the outputs are a function of the arguments alone, so two runs
           agree bit for bit and two builds can be compared output for output.
`--impl reference` : the reference algorithm on the host CPU cores (oracle.port -- the reference itself is pure
           Python/torch and /root/reference does not exist on the GPU box), bounded sample per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GLOBAL_BATCH = 2048
# algorithmic training GFLOP per image (3 x forward; SURVEY.md section 8d / BASELINE.md section 3)


def read_gemm_traffic():
    """roofline.traffic: DRAM bytes of one launch of the dominant kernel from a committed ncu capture, or null."""
    path = os.path.join(ROOT, "profiles", "ncu_gemm_traffic.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return {"traffic": d["dram_bytes"], "traffic_launch": d.get("launch"), "traffic_source": d.get("source")}
    except Exception:
        return {"traffic": None, "traffic_launch": None, "traffic_source": "no committed capture"}


def stock_torch_leg(args):
    """SURVEY.md section 8d's honest GPU comparator: the reference algorithm (oracle.port) run by stock PyTorch on this
    B200 under autocast(bf16) -- eager, and through torch.compile (train.py:115) -- forward + backward, no optimizer,
    in a subprocess with a time limit (tools/stock_torch_gpu.py).  Reported beside the line, never part of `value`."""
    out = {}
    for mode, extra, limit in (("eager", [], 240), ("compile", ["--compile"], 420)):
        cmd = [sys.executable, os.path.join(ROOT, "tools", "stock_torch_gpu.py"), "--workload", args.workload,
               "--batch", "128", "--iters", "3", "--warmup", "2", *extra]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=limit)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            out[mode] = json.loads(line[-1]) if line else {"error": (r.stderr or "no output")[-200:]}
        except subprocess.TimeoutExpired:
            out[mode] = {"error": f"timed out after {limit} s"}
        except Exception as e:
            out[mode] = {"error": f"{type(e).__name__}: {e}"[:200]}
    return out

WORKLOADS = {
    "c2": dict(arch="MicroDiT_XL_2", res=32, ch=4, mask=0.75, pos=1.0, p_mean=-0.6, p_std=1.2, micro=512, gf=282.30,
               name="MicroDiT_XL_2 res_256_pretrain mask=0.75 (32x32x4 latents)"),
    "c3": dict(arch="MicroDiT_XL_2", res=32, ch=4, mask=0.0, pos=1.0, p_mean=-0.6, p_std=1.2, micro=256, gf=714.41,
               name="MicroDiT_XL_2 res_256_finetune mask=0 (32x32x4 latents)"),
    "c4": dict(arch="MicroDiT_XL_2", res=64, ch=4, mask=0.75, pos=2.0, p_mean=0.0, p_std=0.6, micro=128, gf=1069.36,
               name="MicroDiT_XL_2 res_512_pretrain mask=0.75 (64x64x4 latents)"),
    "c5": dict(arch="MicroDiT_XL_2", res=64, ch=16, mask=0.0, pos=2.0, p_mean=0.0, p_std=0.6, micro=64, gf=3003.38,
               name="MicroDiT_XL_2 res_512 mask=0 (64x64x16 latents)"),
    "tiny": dict(arch="MicroDiT_Tiny_2", res=32, ch=4, mask=0.75, pos=1.0, p_mean=-0.6, p_std=1.2, micro=256, gf=None,
                 name="MicroDiT_Tiny_2 res_256 mask=0.75"),
}


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(bf16_burst=d.get("bf16_tflops"), bf16_sustained=d.get("bf16_tflops_sustained"), hbm=d.get("hbm_gbs"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._halt = gpu_index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.gpu)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = int(float(self.rows[0][2])) if self.rows and self.rows[0][2].replace(".", "").isdigit() else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def synth_host_batch(B, wl, seed, pinned):
    g = torch.Generator().manual_seed(seed)
    lat = (0.8 * torch.randn(B, wl["ch"], wl["res"], wl["res"], generator=g)).half()
    cap = torch.randn(B, 1, 77, 1024, generator=g).half()
    drop = (torch.rand(B, generator=g) >= 0.1).double()
    b = {"image_latents": lat, "caption_latents": cap, "drop_caption_mask": drop}
    if pinned:
        b = {k: v.pin_memory() for k, v in b.items()}
    return b


DUMP_SAMPLE = 1 << 22  # entries kept of each flat buffer by --dump-outputs: 16 MiB of float32 each


def timed_outputs(ld, opt, loss):
    """The arrays of --dump-outputs (see the module docstring), on the host."""
    flat = ld.dit.store.flat
    idx = None
    if flat.numel() > DUMP_SAMPLE:
        g = torch.Generator().manual_seed(1234)
        idx = torch.randint(flat.numel(), (DUMP_SAMPLE,), generator=g).sort().values.to(flat.device)
    pick = lambda t: (t if idx is None else t[idx]).float().cpu().numpy()  # noqa: E731
    return {"loss": loss.float().reshape(1).cpu().numpy(), "params": pick(flat), "adamw_m": pick(opt.m)}


def randomize_weights(dit, seed):
    """De-degenerate the zero-initialised tensors (dit.py:615-627) so every block carries signal."""
    g = torch.Generator(device=dit.store.device).manual_seed(seed)
    with torch.no_grad():
        for n, p in dit.named_parameters():
            if p.dim() >= 2 and float(p.abs().max()) == 0.0:
                p.normal_(0.0, 0.02, generator=g)
    dit.mark_weights_dirty()


def build_model(wl, device):
    from micro_diffusion_b200.models import dit as zoo
    from micro_diffusion_b200.models.model import LatentDiffusion, PrecomputedLatentStubs
    net = getattr(zoo, wl["arch"])(input_size=wl["res"], caption_channels=1024, pos_interp_scale=wl["pos"],
                                   in_channels=wl["ch"]).to(device)
    vae, te, tok = PrecomputedLatentStubs.make()
    ld = LatentDiffusion(net, vae, te, tok, p_mean=wl["p_mean"], p_std=wl["p_std"], train_mask_ratio=wl["mask"],
                         latent_res=wl["res"])
    ld.train()
    randomize_weights(net, 18)
    return ld


# ------------------------------------------------------------------------------------------ CPU legs
def host_threads():
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 32))  # torch's CPU GEMMs stop scaling (and regress) beyond ~32 threads at these sizes


def cpu_reference_img_per_s(wl, batch, iters, threads, state_dict=None, budget_s=60.0, warmup=0):
    """The reference algorithm (oracle.port, fp32) forward+backward on the host cores.
    Runs `warmup` untimed passes, then up to `iters` timed passes, stopping early once `budget_s` is spent (None: all).
    Returns (img/s, timed passes done)."""
    from oracle import port, weights
    torch.set_num_threads(threads)
    if state_dict is None:
        from micro_diffusion_b200.arch import DiTConfig, micro_dit_tiny_2_kwargs, micro_dit_xl_2_kwargs
        kw = (micro_dit_xl_2_kwargs if wl["arch"] == "MicroDiT_XL_2" else micro_dit_tiny_2_kwargs)(
            input_size=wl["res"], in_channels=wl["ch"], pos_interp_scale=wl["pos"])
        cfg = DiTConfig(**kw)
        state_dict = {}
        for k, s in cfg.buffer_specs() + cfg.param_specs():
            if k == "pos_embed":
                state_dict[k] = port.sincos_pos_embed(cfg.dim, cfg.grid, cfg.pos_interp_scale, cfg.grid).unsqueeze(0)
            elif k == "mask_token":
                state_dict[k] = torch.zeros(s)
            elif len(s) == 1:
                state_dict[k] = torch.ones(s) if not k.endswith("bias") else torch.zeros(s)
            else:  # cheap non-degenerate fill (a 1.2 B-element randn costs a minute of host time)
                n = 1
                for d in s:
                    n *= d
                state_dict[k] = (((torch.arange(n, dtype=torch.float32) * 0.6180339887) % 1.0) - 0.5).mul_(0.07).view(s)
    hd = 64 if wl["arch"] == "MicroDiT_XL_2" else 32
    pcfg = port.PortConfig(patch_size=2, head_dim=hd, num_experts=8, expert_capacity=2.0, p_mean=wl["p_mean"], p_std=wl["p_std"])
    P = {k: v.detach().float().cpu().requires_grad_(k not in ("pos_embed", "mask_token")) for k, v in state_dict.items()}
    T = (wl["res"] // 2) ** 2
    times = []
    t_start = time.perf_counter()
    for it in range(warmup + iters):
        b = weights.synth_batch(batch, wl["ch"], wl["res"], seed=100 + it)
        rnd, eps, noise = weights.replay_draws(200 + it, (batch, wl["ch"], wl["res"], wl["res"]), T, wl["mask"])
        for v in P.values():
            v.grad = None
        t0 = time.perf_counter()
        loss, _ = port.latent_diffusion_forward(P, pcfg, b, rnd, eps, wl["mask"], noise)
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if budget_s is not None and time.perf_counter() - t_start > budget_s and times:
            break
    return batch * len(times) / sum(times), len(times)


def run_reference_arm(args, wl):
    """`--impl reference`: the reference algorithm on the host cores (oracle.port; /root/reference and its Python
    dependencies do not exist on the GPU box).  Each "step" is a bounded sample: forward+backward of `sample` images."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    sample = 8 if wl["res"] == 32 else 2
    t0 = time.perf_counter()
    ips, done = cpu_reference_img_per_s(wl, sample, args.steps, threads, budget_s=None, warmup=1 if args.warmup > 0 else 0)
    wall = time.perf_counter() - t0
    line = {
        "impl": "reference", "metric": "training images/sec (global batch 2048)", "value": ips, "unit": "img/s",
        "n_gpus": args.gpus, "steps": done, "warmup": 1 if args.warmup > 0 else 0, "ms_per_step": 1000.0 * sample / ips,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "global_batch": GLOBAL_BATCH,
                   "sample": f"{sample} images per step (forward+backward)"},
        "cpu_baseline": {"value": ips, "unit": "img/s", "cores": threads, "kind": "port",
                         "sample": f"{sample}-image forward+backward x {done}, fp32, oracle.port, {threads} threads"},
        "e2e": {"value": ips, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": wall,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--microbatch", type=int, default=0)
    ap.add_argument("--global-batch", type=int, default=GLOBAL_BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-out", default="")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the brief c3/c4/c5 legs of the N=1 run")
    ap.add_argument("--no-stock-torch", action="store_true", help="skip the stock-PyTorch-on-B200 comparator leg")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the last timed step's loss, parameters and AdamW first moment as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the B200 path")
    wl = dict(WORKLOADS[args.workload])
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    import torch.distributed as dist
    from micro_diffusion_b200.train_step import FlatAdamW, GradReducer, train_step

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the MicroDiT hot path has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"
    W, K = max(3, args.warmup), args.steps
    per_rank = args.global_batch // world
    micro = min(args.microbatch or wl["micro"], per_rank)

    def measure(wl, micro, K, W, with_e2e=True, with_probe=True, with_outputs=False):
        """Build the model of workload `wl`, run W warm-up + K timed steps (inputs resident), optionally the end-to-end
        pass from pinned host memory and the per-launch roofline probe; returns a dict of raw numbers and frees the model.
        `with_outputs`: also the host copies of what the last timed step returned (timed_outputs)."""
        torch.manual_seed(18)  # weight init and the EDM / mask draws of every step
        ld = build_model(wl, device)
        opt = FlatAdamW(ld.dit, lr=2.4e-4, weight_decay=0.1, clip_norm=0.25)
        reducer = GradReducer(ld.dit.store, ops=ld.dit.engine.ops) if world > 1 else None
        ops = ld.dit.engine.ops
        deterministic = with_outputs or os.environ.get("MD_DETERMINISTIC", "0") == "1"
        if with_outputs:
            ops.set_deterministic(True)

        host = synth_host_batch(per_rank, wl, seed=18 + rank, pinned=True)
        h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())
        resident = {k: v.to(device, non_blocking=True) for k, v in host.items()}
        torch.cuda.synchronize()

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def max_over_ranks(ms):
            if world == 1:
                return ms
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t)

        def step_resident():
            # the caption-drop mask is applied in place (reference semantics), so hand the step a fresh device copy
            b = {"image_latents": resident["image_latents"], "caption_latents": resident["caption_latents"].clone(),
                 "drop_caption_mask": resident["drop_caption_mask"]}
            return train_step(ld, b, opt, reducer, micro)

        def step_e2e():
            b = {k: v.to(device, non_blocking=True) for k, v in host.items()}
            loss = train_step(ld, b, opt, reducer, micro)
            return loss.item()  # device -> host read of the step's result

        for _ in range(W):
            step_resident()
        barrier()
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        l0 = ops.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.profiler.start()  # cudaProfilerStart: `ncu --profile-from-start off` lists exactly the timed steps
        e0.record()
        for _ in range(K):
            loss_t = step_resident()
        e1.record()
        torch.cuda.profiler.stop()
        barrier()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        launches = (ops.launches - l0)
        clocks = sampler.stop() if sampler else None
        ms_step = ms_total / K
        value = args.global_batch / (ms_step / 1e3)

        r = dict(value=value, ms_step=ms_step, launches=launches, clocks=clocks, loss=float(loss_t), micro=micro,
                 h2d_bytes=h2d_bytes, step_tflops=(value / world) * wl["gf"] / 1e3 if wl["gf"] else None,
                 deterministic=deterministic)
        if with_outputs:
            opt.gather_state()  # sharded optimizer: complete the moments (a collective: every rank calls it)
            r["outputs"] = timed_outputs(ld, opt, loss_t) if rank == 0 else None
        # ---- end to end from pinned host memory
        if with_e2e:
            step_e2e()
            barrier()
            e0.record()
            for _ in range(K):
                r["last_loss"] = step_e2e()
            e1.record()
            barrier()
            r["ms_e2e"] = max_over_ranks(e0.elapsed_time(e1)) / K
            r["e2e_value"] = args.global_batch / (r["ms_e2e"] / 1e3)
        # ---- roofline probe: one extra step with CUDA events around every launch (same stream, same work)
        if with_probe:
            ops.profile = []
            f0 = ops.gemm_flops
            step_resident()
            torch.cuda.synchronize()
            prof = ops.profile_summary()
            ops.profile = None
            probe_flops = ops.gemm_flops - f0
            tot_ms = sum(v[1] for v in prof.values())
            gemm = {k: v for k, v in prof.items() if k.startswith("md_gemm_bf16")}
            gemm_ms = sum(v[1] for v in gemm.values())
            attn_ms = sum(v[1] for k, v in prof.items() if k.startswith("md_attn"))
            # launches whose epilogue only stores (epi 0-3) vs the fused tails (GELU / GELU' / SwiGLU: epi 4-7), which do the
            # work of a former element-wise pass inside the GEMM and are epilogue- rather than tensor-bound
            plain = {k: v for k, v in gemm.items() if " epi=" in k and int(k.split(" epi=")[1].split(" ")[0]) < 4}
            plain_ms, plain_fl = sum(v[1] for v in plain.values()), sum(v[2] for v in plain.values())
            r.update(prof=prof, tot_ms=tot_ms, gemm_ms=gemm_ms, gemm_n=sum(v[0] for v in gemm.values()), attn_ms=attn_ms,
                     gemm_tflops=probe_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None,
                     plain_tflops=plain_fl / (plain_ms * 1e-3) / 1e12 if plain_ms > 0 else None,
                     fused_share=(gemm_ms - plain_ms) / gemm_ms if gemm_ms > 0 else None)
        r["grad_exchange"] = None
        if reducer is not None:
            r["grad_exchange"] = (
                (f"NCCL reduce-scatter (mean) of the flat fp32 gradient -> clip + AdamW on 1/{world} per rank -> all-gather of "
                 f"the fp32 parameters (backbone range under the next step's patch-mixer forward)") if reducer.shard else
                "NCCL all-reduce (mean) of the flat fp32 gradient, replicated clip + AdamW") + \
                f"; overlap with backward={reducer.overlap}, {reducer.reserve} SMs left to NCCL while it overlaps"
        r["peak_hbm_gb"] = torch.cuda.max_memory_allocated(device) / 2 ** 30
        if deterministic and os.environ.get("MD_DETERMINISTIC", "0") != "1":
            ops.set_deterministic(False)  # process-wide switch: the other workloads' legs run the fast path
        r["state_dict"] = ({k: v.detach().cpu() for k, v in ld.dit.state_dict().items()}
                           if (rank == 0 and with_probe and not args.no_cpu_baseline and world == 1) else None)
        del ld, opt, ops, resident, host, reducer, step_resident, step_e2e
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(device)
        return r

    peaks = read_peaks()
    m = measure(wl, micro, K, W, with_outputs=bool(args.dump_outputs))
    value, ms_step, launches, clocks = m["value"], m["ms_step"], m["launches"], m["clocks"]
    prof, tot_ms, gemm_ms, gemm_n, gemm_tflops, step_tflops = (m["prof"], m["tot_ms"], m["gemm_ms"], m["gemm_n"],
                                                               m["gemm_tflops"], m["step_tflops"])
    e2e_value, ms_e2e, last_loss, h2d_bytes = m["e2e_value"], m["ms_e2e"], m["last_loss"], m["h2d_bytes"]

    # ---- the other BASELINE.json configurations, briefly (N=1 default run only): 1 warm-up + 2 timed steps each
    others = None
    if world == 1 and args.workload == "c2" and not args.no_other_configs:
        others = {}
        for key in ("c3", "c4", "c5"):
            try:
                o = measure(WORKLOADS[key], min(WORKLOADS[key]["micro"], per_rank), 2, 1, with_e2e=False, with_probe=False)
                others[key] = {"workload": WORKLOADS[key]["name"], "value": o["value"], "unit": "img/s",
                               "ms_per_step": o["ms_step"], "steps": 2, "warmup": 1, "microbatch": o["micro"],
                               "step_algorithmic_tflops_per_gpu": o["step_tflops"],
                               "step_frac": o["step_tflops"] / peaks["bf16_sustained"] if o["step_tflops"] else None,
                               "peak_hbm_gb": o["peak_hbm_gb"], "loss": o["loss"]}
            except Exception as e:  # an auxiliary leg must never take the headline line down
                others[key] = {"workload": WORKLOADS[key]["name"], "error": f"{type(e).__name__}: {e}"[:200]}

    if rank == 0:
        if args.profile_out:
            os.makedirs(os.path.dirname(args.profile_out) or ".", exist_ok=True)
            with open(args.profile_out, "w") as f:
                f.write(f"# per-op CUDA-event times of one {args.workload} step (per rank {per_rank} imgs, microbatch {micro})\n")
                f.write("op,launches,total_ms,share,algorithmic_tflops\n")
                agg = {}
                for k, (n, ms, fl) in prof.items():
                    kk = k.split(" ")[0]
                    a = agg.get(kk, (0, 0.0, 0))
                    agg[kk] = (a[0] + n, a[1] + ms, a[2] + fl)
                for k, (n, ms, fl) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                    tf = f"{fl / (ms * 1e-3) / 1e12:.1f}" if fl else ""
                    f.write(f"{k},{n},{ms:.3f},{ms / tot_ms:.4f},{tf}\n")
                f.write("# GEMM / attention launches by shape\n")
                for k, (n, ms, fl) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
                    if " " not in k:
                        continue
                    tf = f"{fl / (ms * 1e-3) / 1e12:.1f}" if fl else ""
                    f.write(f"{k},{n},{ms:.3f},{ms / tot_ms:.4f},{tf}\n")
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in m["outputs"].items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        cpu_base = None
        if not args.no_cpu_baseline and world == 1:
            threads = host_threads()
            sample = 8 if wl["res"] == 32 else 2
            t0 = time.perf_counter()
            sd = m["state_dict"]
            ips, done = cpu_reference_img_per_s(wl, sample, 3, threads, sd, budget_s=25.0, warmup=1)
            cpu_base = {"value": ips, "unit": "img/s", "cores": threads, "kind": "port",
                        "sample": f"{done} x {sample}-image forward+backward after one warm-up pass, fp32 oracle.port on "
                                  f"{threads} threads, same weights as the GPU arm ({time.perf_counter() - t0:.0f} s wall)"}
        line = {
            "metric": "training images/sec (global batch 2048)", "value": value, "unit": "img/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["name"], "global_batch": args.global_batch, "per_gpu_batch": per_rank,
                       "microbatch": micro, "parallelism": f"dp{world}", "deterministic": m["deterministic"],
                       "optimizer": "clip0.25+AdamW (fused, in step)",
                       "l2": "per-step working set (activations > 40 GB per microbatch) far exceeds the 126 MB L2",
                       "grad_exchange": m["grad_exchange"]},
            "e2e": {"value": e2e_value, "unit": "img/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "loss": last_loss},
            "gpu_launches": launches,
            "peak_hbm_gb": m["peak_hbm_gb"],
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (md_gemm_bf16)",
                         "achieved": gemm_tflops, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                         "frac": (gemm_tflops / peaks["bf16_sustained"]) if gemm_tflops else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel, read from the
                         # committed summary of an `ncu --set full` capture (profiles/ncu_gemm_traffic.json, written by
                         # tools/summarize_ncu_raw.py); null when no capture of the current kernel is committed
                         **read_gemm_traffic(),
                         "achieved_store_only_launches": m.get("plain_tflops"),
                         "frac_store_only_launches": (m["plain_tflops"] / peaks["bf16_sustained"]) if m.get("plain_tflops") else None,
                         "fused_tail_share_of_kernel_time": m.get("fused_share"),
                         "peak_source": peaks["source"] + " sustained", "launches_per_step": gemm_n,
                         "share_of_step_kernel_time": gemm_ms / tot_ms if tot_ms else None,
                         "step_algorithmic_tflops_per_gpu": step_tflops,
                         "step_frac": (step_tflops / peaks["bf16_sustained"]) if step_tflops else None},
            "cpu_baseline": cpu_base,
            "loss": m["loss"],
            "attention_share_of_step_kernel_time": m["attn_ms"] / tot_ms if tot_ms else None,
            "other_configs": others,
            "stock_torch_gpu": stock_torch_leg(args) if (world == 1 and not args.no_stock_torch) else None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
