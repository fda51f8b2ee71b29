#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on BASELINE.json's configs.

Main workload (configs[1]): SD-XL base 1.0 UNet2DConditionModel, batch 8 per GPU, 1024x1024 (latent 128x128), DDIM
(50-step schedule), bf16, synthetic inputs and random-init weights of the SDXL architecture. One bench "step" = one
denoising timestep = one UNet forward over the batch + the fused DDIM update. Metric = denoiser-forward latents/s
(images pushed through one denoiser forward per second, whole job); finished latents/s = that / 50.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

K timed steps in every GPU section (SDXL, SD3, STDiT2, Qwen2-VL prefill). --dump-outputs writes what the last timed SDXL
step returned; inputs and weights are seeded, so runs with the same arguments see identical inputs.

N > 1 is launched by `python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...`: one rank per GPU,
images sharded, weights replicated, no per-step communication, one NCCL all_gather of the finished latents.

The same JSON line carries, as extra keys (all timed with CUDA events, max over ranks):
  job            K steps + the all_gather of the finished latents + the D2H copy of the gathered result on rank 0
                 (the path's only collective INSIDE a timed region)
  sdxl_strong    strong scaling of configs[1]: the global batch stays 8, each rank takes 8 / N images
  sd3_b32        configs[2]: SD3-medium MMDiT, global batch 32 (32 / N images per rank), 1024^2, FlowMatchEuler-28 step,
                 plus its own job-level number with the all_gather
  stdit2_b4      configs[4]: STDiT2-XL, 16 x 512^2, global batch 4 over min(N, 4) GPUs
  qwen2vl_prefill  configs[3] (N = 1): Qwen2-VL-7B prefill tokens/s
  cpu_baseline / parity (N = 1): the CPU restatement of the reference on ONE full 1024^2 image, and the GPU output on
                 the same weights / inputs compared with it (cosine, max-rel; tolerance cosine >= 0.999, max-rel <= 0.04)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "denoiser_forward_latents_per_sec_sdxl_1024"
UNIT = "latents/s"
SDXL = dict(down_block_types=("DownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D"),
            up_block_types=("CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "UpBlock2D"), block_out_channels=(320, 640, 1280),
            cross_attention_dim=2048, transformer_layers_per_block=(1, 2, 10), attention_head_dim=(5, 10, 20),
            use_linear_projection=True, addition_embed_type="text_time", addition_time_embed_dim=256,
            projection_class_embeddings_input_dim=2816)
SD3_MEDIUM = dict(sample_size=128, patch_size=2, in_channels=16, num_layers=24, attention_head_dim=64,
                  num_attention_heads=24, joint_attention_dim=4096, caption_projection_dim=1536,
                  pooled_projection_dim=2048, out_channels=16, pos_embed_max_size=192)
DDIM = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
            set_alpha_to_one=False, steps_offset=1)
SDXL_TFLOP_PER_SAMPLE = 6.761  # 2*MAC over conv/linear/QK^T/PV, SURVEY.md §8d (oracle.unet.unet_flops reproduces it)
SD3_TFLOP_PER_SAMPLE = 8.437
STDIT2_TFLOP_PER_SAMPLE = 24.39
PARITY_TOL = {"cosine_min": 0.999, "max_rel_err": 0.04}
REF_STEPS, REF_WARMUP = 3, 1  # reference / cpu_baseline legs: fixed sample count, independent of --steps
DUMP_BYTES = 64_000_000  # --dump-outputs: upper bound of all files together


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def igemm_traffic_per_launch():
    """DRAM bytes (read + write) per igemm launch, averaged over the launches of one SDXL forward. NOT measured in this
    run: it comes from a committed `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` pass of the same forward
    (tools/gpu_ncu.sh); returns (value, source file) or (None, None)."""
    for name in ("r02_igemm_dram_traffic.json", "r01_igemm_dram_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)["dram_bytes_per_launch"], f"profiles/{name} (ncu pass, not measured in this run)"
        except Exception:  # noqa: BLE001
            continue
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------
# CPU restatement of the reference (oracle, kind = "port"): one full-size image, fixed sample count
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_forward(steps=REF_STEPS, warmup=REF_WARMUP, keep=False):
    """Times the CPU restatement of the reference's UNet forward (oracle/unet.py; PaddlePaddle itself is not
    installable here) on a bounded sample of the workload: ONE image (B = 1) of the SDXL 1024^2 forward, `warmup`
    untimed + `steps` timed passes. The thread count is chosen once by a short probe at latent 64x64 (all logical cores
    vs half of them: oversubscribed SMT threads are often slower for oneDNN); the SAME policy runs in the cpu_baseline
    leg and in --impl reference. Returns a dict; with keep=True also the weights, inputs and the fp32 output (for the
    parity leg)."""
    import torch

    from oracle import unet as O
    ncpu = os.cpu_count() or 1
    cfg = O.UNET_CONFIGS["sdxl"]
    P = O.init_params(O.unet_param_shapes(cfg), seed=1)  # fan-in scaled, bf16-representable values
    g = torch.Generator().manual_seed(7)
    bf = torch.bfloat16
    x = torch.randn(1, 4, 128, 128, generator=g).to(bf).float()
    ctx = torch.randn(1, 77, 2048, generator=g).to(bf).float()
    added = {"text_embeds": torch.randn(1, 1280, generator=g).to(bf).float(),
             "time_ids": torch.tensor([[1024., 1024., 0, 0, 1024., 1024.]])}
    best, threads = None, ncpu
    for nt in sorted({ncpu, max(1, ncpu // 2)}, reverse=True):
        torch.set_num_threads(nt)
        t0 = time.perf_counter()
        with torch.no_grad():
            O.unet_forward(cfg, P, x[:, :, :64, :64], 981, ctx, added)
        dtp = time.perf_counter() - t0
        if best is None or dtp < best:
            best, threads = dtp, nt
    torch.set_num_threads(threads)
    with torch.no_grad():
        for _ in range(warmup):
            ref = O.unet_forward(cfg, P, x, 981, ctx, added)
        t0 = time.perf_counter()
        for _ in range(steps):
            ref = O.unet_forward(cfg, P, x, 981, ctx, added)
        dt = (time.perf_counter() - t0) / steps
    out = {"value": 1.0 / dt, "seconds_per_sample": dt, "cores": threads, "kind": "port",
           "sample": (f"1 image (B=1) SDXL UNet forward at 1024x1024 (latent 128x128), fp32, torch-CPU restatement of the "
                      f"reference (oracle/unet.py), {warmup} warm-up + {steps} timed passes, {threads} threads")}
    if keep:
        out["_keep"] = (cfg, P, x, ctx, added, ref)
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores. The reference is pure
    Python on PaddlePaddle, which cannot be installed offline, so this runs the oracle port (cpu_baseline.kind='port')
    on the same config as the b200 arm's cpu_baseline leg: one full 1024^2 image, fixed sample count."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_forward()
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": REF_STEPS, "warmup": REF_WARMUP, "ms_per_step": r["seconds_per_sample"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "SDXL-base UNet2DConditionModel forward, 1024x1024, DDIM timestep (configs[1])",
                       "sample": r["sample"], "requested_steps": args.steps, "requested_warmup": args.warmup},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# helpers shared by the GPU sections
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    """Process-group context of one rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            from paddlemix_b200 import distributed as bdist
            bdist.init_comm(self.local)  # the path's collective goes through the C ABI (b200mix_allgather_latents)
        self.dist = dist

    def sync_all(self):
        import torch
        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
            torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, *vals):
        import torch
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def timed(self, fn, steps, warmup):
        """W untimed calls, then exactly K calls between barrier + synchronize on both sides, CUDA events; ms total
        (max over ranks)."""
        import torch
        for i in range(warmup):
            fn(i)
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        self.sync_all()
        return self.max_over_ranks(e0.elapsed_time(e1))[0]


def dump_outputs(c, outputs, out_dir):
    """Writes each device tensor of `outputs` as out_dir/<name>.npy in float32 (rank 0; with N ranks the global batch in
    rank order). An array over its share of DUMP_BYTES is replaced by a fixed seeded sample of its flattened elements,
    so two builds run with the same arguments can be compared element for element."""
    import numpy as np
    import torch
    cap = (DUMP_BYTES // len(outputs) - 4096) // 4  # float32 elements per file, .npy header included
    for name, t in outputs.items():
        t = t.float().contiguous()
        if c.world > 1:
            full = torch.empty((c.world * t.shape[0],) + tuple(t.shape[1:]), device=t.device, dtype=t.dtype)
            c.dist.all_gather_into_tensor(full, t)
            t = full
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0))
            t = t.flatten()[idx.to(t.device)]
        if c.rank == 0:
            os.makedirs(out_dir, exist_ok=True)
            np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def sdxl_setup(c, B, height):
    """Model, graph, scheduler and pinned host inputs of the SDXL workload for B images on this rank."""
    import torch

    from paddlemix_b200.ppdiffusers.pipelines import GraphedUNet
    from paddlemix_b200.ppdiffusers.schedulers import DDIMScheduler
    H, L = height // 8, 77
    g = torch.Generator().manual_seed(2 + c.rank)
    s = {"B": B, "H": H}
    s["lat_h"] = torch.randn(B, 4, H, H, generator=g).pin_memory()
    s["ctx_h"] = torch.randn(B, L, 2048, generator=g).to(torch.bfloat16).pin_memory()
    s["te_h"] = torch.randn(B, 1280, generator=g).to(torch.bfloat16).pin_memory()
    s["ids_h"] = torch.tensor([[float(height), float(height), 0, 0, float(height), float(height)]] * B).pin_memory()
    s["out_h"] = torch.empty(B, 4, H, H).pin_memory()
    sched = DDIMScheduler(**DDIM)
    sched.set_timesteps(50)
    s["sched"], s["timesteps"] = sched, [int(t) for t in sched.timesteps]
    return s


def sdxl_section(c, unet, B, height, steps, warmup, with_e2e=True, sample_clocks=False, keep_outputs=False):
    """Device-resident steps, end-to-end steps (host buffers), job-level (steps + all_gather + D2H) for B images/rank.
    keep_outputs: res["outputs"] holds what the last timed step returned (noise prediction, next latents)."""
    import torch

    from paddlemix_b200 import ops
    from paddlemix_b200.ppdiffusers.pipelines import GraphedUNet, all_gather_latents
    dev = c.dev
    s = sdxl_setup(c, B, height)
    H, sched, timesteps = s["H"], s["sched"], s["timesteps"]
    den = GraphedUNet(unet, (B, 4, H, H), (B, 77, 2048), {"text_embeds": (B, 1280), "time_ids": (B, 6)})
    state = {"lat": s["lat_h"].to(dev), "nxt": torch.empty(B, 4, H, H, device=dev)}
    den(state["lat"], 981.0, s["ctx_h"].to(dev), {"text_embeds": s["te_h"].to(dev), "time_ids": s["ids_h"].to(dev)})

    def step_resident(i):
        t = timesteps[i % len(timesteps)]
        eps = den(state["lat"], float(t))
        sched.step(eps, t, state["lat"], out=state["nxt"])
        state["lat"], state["nxt"] = state["nxt"], state["lat"]

    sampler = ClockSampler(c.local) if (sample_clocks and c.rank == 0) else None
    for i in range(warmup):
        step_resident(i)
    c.sync_all()
    if sampler:
        sampler.start()
    n0 = ops.launches()
    ms = c.timed(step_resident, steps, 0)
    launches = ops.launches() - n0
    if sampler:
        sampler.stop_flag = True
    res = {"ms": ms, "launches": launches, "clocks": sampler.summary() if sampler else None, "den": den, "state": s}
    if keep_outputs:  # copied now: the job leg below steps the same state further
        res["outputs"] = {"noise_pred": den.out.float(), "latents": state["lat"].clone()}

    # job level: K steps + the path's only collective (all_gather of the finished latents) + D2H of the gathered result
    gathered_h = torch.empty(B * c.world, 4, H, H).pin_memory() if c.rank == 0 else None

    def job(_):
        for i in range(steps):
            step_resident(i)
        fin = all_gather_latents(state["lat"])
        if c.rank == 0:
            gathered_h.copy_(fin, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    job(0)  # warm-up (NCCL communicator set-up, pinned buffers)
    t0 = time.perf_counter()
    ms_job = c.timed(job, 1, 0)
    wall_job = (time.perf_counter() - t0) * 1e3
    c.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fin = all_gather_latents(state["lat"])
    if c.rank == 0:
        gathered_h.copy_(fin, non_blocking=True)
    e1.record()
    c.sync_all()
    ms_coll = c.max_over_ranks(e0.elapsed_time(e1))[0]
    res["job"] = {"steps": steps, "ms_total": round(ms_job, 3), "wall_ms_total": round(c.max_over_ranks(wall_job)[0], 3),
                  "ms_allgather_plus_d2h": round(ms_coll, 3), "value": round(B * c.world * steps / (ms_job * 1e-3), 3),
                  "unit": UNIT, "gathered_bytes": B * c.world * 4 * H * H * 4,
                  "what": "K timesteps + all_gather of the finished latents (NCCL) + D2H of the gathered tensor on rank 0"}

    if with_e2e:
        def step_e2e(i):
            t = timesteps[i % len(timesteps)]
            x = s["lat_h"].to(dev, non_blocking=True)
            eps = den(x, float(t), s["ctx_h"].to(dev, non_blocking=True),
                      {"text_embeds": s["te_h"].to(dev, non_blocking=True), "time_ids": s["ids_h"].to(dev, non_blocking=True)})
            out = sched.step(eps, t, x)
            s["out_h"].copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()  # the caller reads the result every step

        for i in range(min(warmup, 3)):
            step_e2e(i)
        c.sync_all()
        t0 = time.perf_counter()
        ms_e2e = c.timed(step_e2e, steps, 0)
        wall = c.max_over_ranks((time.perf_counter() - t0) * 1e3)[0]
        res["e2e"] = {"ms": ms_e2e, "wall_ms": wall,
                      "h2d": s["lat_h"].numel() * 4 + s["ctx_h"].numel() * 2 + s["te_h"].numel() * 2 + s["ids_h"].numel() * 4,
                      "d2h": s["out_h"].numel() * 4}
    return res


def roofline_section(c, unet, B, height):
    """Per-launch CUDA events in one eager forward: achieved rate of every kernel family, igemm as the dominant kernel."""
    import torch

    from paddlemix_b200 import ops
    dev = c.dev
    H = height // 8
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(B, 4, H, H, generator=g).to(dev)
    x_nhwc = ops.nchw_to_nhwc(lat)
    added = {"text_embeds": torch.randn(B, 1280, generator=g).to(torch.bfloat16).to(dev),
             "time_ids": torch.tensor([[float(height), float(height), 0, 0, float(height), float(height)]] * B).to(dev)}
    tt = torch.full((B,), 981.0, device=dev)
    ctx_d = torch.randn(B, 77, 2048, generator=g).to(torch.bfloat16).to(dev)
    unet.forward_nhwc(x_nhwc, tt, ctx_d, added)  # eager warm-up
    torch.cuda.synchronize(dev)
    ops.profile_begin()
    unet.forward_nhwc(x_nhwc, tt, ctx_d, added)
    prof = ops.profile_end()
    # The shipped path folds the transformer blocks' LayerNorms into the GEMM epilogues either side (DESIGN.md §3): the
    # igemm family then carries ~4 ms of normalisation work and its TFLOP/s drop although the step gets faster. For
    # comparison with the numbers of earlier rounds the same forward is profiled once more with explicit LayerNorm kernels.
    from paddlemix_b200.ppdiffusers import unet_2d_condition as U
    unfused = None
    if U._Transformer2D.FOLD_LAYERNORM:
        try:
            U._Transformer2D.FOLD_LAYERNORM = False
            unet.forward_nhwc(x_nhwc, tt, ctx_d, added)
            torch.cuda.synchronize(dev)
            ops.profile_begin()
            unet.forward_nhwc(x_nhwc, tt, ctx_d, added)
            p2 = ops.profile_end()
        finally:
            U._Transformer2D.FOLD_LAYERNORM = True
        if p2.get("igemm"):
            pk = measured_peaks()[0]
            a2 = p2["igemm"]["work"] / (p2["igemm"]["ms"] * 1e-3) / 1e12
            unfused = {"what": "same forward with explicit LayerNorm kernels (B200MIX_FOLD_LN=0), eager per-launch events",
                       "igemm_ms": round(p2["igemm"]["ms"], 3), "igemm_achieved": round(a2, 1), "igemm_frac": round(a2 / pk, 4),
                       "layernorm_ms": round(p2.get("layernorm", {}).get("ms", 0.0), 3),
                       "sum_of_families_ms": round(sum(v["ms"] for v in p2.values()), 3)}
    peak_tf, peak_gbs, how = measured_peaks()
    ig = prof.get("igemm")
    if not ig:
        return None
    ach = ig["work"] / (ig["ms"] * 1e-3) / 1e12
    total_ms = sum(v["ms"] for v in prof.values())
    traffic, tsrc = igemm_traffic_per_launch()
    fam = {}
    for k, v in prof.items():
        flop = v["unit"] == "flop"
        a = v["work"] / (v["ms"] * 1e-3) / (1e12 if flop else 1e9)
        fam[k] = {"ms": round(v["ms"], 3), "achieved": round(a, 1), "unit": "TFLOP/s" if flop else "GB/s",
                  "frac": round(a / (peak_tf if flop else peak_gbs), 4), "launches": v["calls"]}
    return {"kernel": "igemm_kernel (tcgen05 implicit GEMM: linear + conv3x3)", "bound": "tensor",
            "achieved": round(ach, 1), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(ach / peak_tf, 4),
            "traffic": traffic, "traffic_source": tsrc, "peak_source": how, "launches_per_step": ig["calls"],
            "avg_launch_ms": round(ig["ms"] / ig["calls"], 4), "share_of_step": round(ig["ms"] / total_ms, 3),
            "algorithmic_tflop_per_step": round(ig["work"] / 1e12, 2), "hbm_peak_gbs": peak_gbs,
            "sum_of_families_ms": round(total_ms, 3), "layernorm": "folded into the igemm epilogues (no LayerNorm launches)"
            if "layernorm" not in prof else "explicit kernels", "unfused_layernorm": unfused, "by_kernel": fam}


def sd3_section(c, steps, warmup, global_batch=32):
    """configs[2]: SD3-medium MMDiT, global batch 32 sharded over the ranks, 1024^2, FlowMatchEuler (28-step schedule);
    one step = one MMDiT forward over the rank's images + the fused Euler update; job = steps + all_gather + D2H."""
    import torch

    from paddlemix_b200 import ops
    from paddlemix_b200.ppdiffusers.pipelines import all_gather_latents, shard_batch
    from paddlemix_b200.ppdiffusers.schedulers import FlowMatchEulerDiscreteScheduler
    from paddlemix_b200.ppdiffusers.transformer_sd3 import SD3Transformer2DModel
    dev = c.dev
    lo, hi = shard_batch(global_batch, c.rank, c.world)
    B = hi - lo
    model = SD3Transformer2DModel(**SD3_MEDIUM).init_synthetic_weights(seed=3, device=c.local)
    g = torch.Generator().manual_seed(20 + c.rank)
    lat = torch.randn(B, 16, 128, 128, generator=g).to(dev)
    nxt = torch.empty_like(lat)
    ctx = torch.randn(B, 154, 4096, generator=g).to(torch.bfloat16).to(dev)
    pooled = torch.randn(B, 2048, generator=g).to(torch.bfloat16).to(dev)
    sched = FlowMatchEulerDiscreteScheduler(shift=3.0)
    sched.set_timesteps(28)
    ts = list(sched.timesteps)
    tvec = torch.empty(B, device=dev, dtype=torch.float32)
    st = {"lat": lat, "nxt": nxt}

    def step(i):
        if i % len(ts) == 0:
            sched.set_timesteps(28)  # the scheduler counts its steps: restart the 28-step schedule when the bench wraps
        t = ts[i % len(ts)]
        tvec.fill_(float(t))
        v = model(hidden_states=st["lat"], timestep=tvec, encoder_hidden_states=ctx, pooled_projections=pooled,
                  return_dict=False)[0]
        sched.step(v, t, st["lat"], out=st["nxt"])
        st["lat"], st["nxt"] = st["nxt"], st["lat"]

    n0 = ops.launches()
    ms = c.timed(step, steps, warmup)
    launches = (ops.launches() - n0) // (steps + warmup)
    gathered_h = torch.empty(global_batch, 16, 128, 128).pin_memory() if c.rank == 0 else None

    def job(_):
        for i in range(steps):
            step(i)
        fin = all_gather_latents(st["lat"])
        if c.rank == 0:
            gathered_h.copy_(fin, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    job(0)
    ms_job = c.timed(job, 1, 0)
    del model
    torch.cuda.empty_cache()
    per_step = ms / steps
    return {"metric": "denoiser_forward_latents_per_sec_sd3_medium_1024", "value": round(global_batch / (per_step * 1e-3), 2),
            "unit": UNIT, "ms_per_step": round(per_step, 3), "scaling": "strong", "n_gpus": c.world,
            "model_tflops_per_sec": round(SD3_TFLOP_PER_SAMPLE * global_batch / (per_step * 1e-3), 1),
            "gpu_launches_per_step": launches,
            "job": {"steps": steps, "ms_total": round(ms_job, 3), "value": round(global_batch * steps / (ms_job * 1e-3), 2),
                    "unit": UNIT, "what": "K steps + all_gather of the finished latents + D2H on rank 0"},
            "config": {"workload": "SD3-medium MMDiT (24 layers, 4096 image + 154 text tokens) forward + fused FlowMatchEuler "
                                   "update per timestep (configs[2])", "global_batch": global_batch, "batch_per_gpu": B,
                       "resolution": "1024x1024", "scheduler": "FlowMatchEulerDiscrete 28 steps, shift 3.0", "cfg": "off",
                       "parallelism": f"dp{c.world} (images sharded, weights replicated, one all_gather of finished latents)",
                       "weights": "random init, SD3-medium architecture (2.0 B params)", "dtype": "bf16", "cuda_graph": False}}


def stdit2_section(c, steps, warmup, global_batch=4):
    """configs[4]: Open-Sora STDiT2-XL, 16 frames x 512^2 (latent 64x64 -> 16 x 1024 tokens), 120 text tokens, global
    batch 4 sharded over min(N, 4) ranks (ranks beyond the 4th hold one extra sample each: weak beyond N = 4)."""
    import torch

    from paddlemix_b200.opensora import STDiT2
    dev = c.dev
    B = max(1, global_batch // c.world)
    total = B * c.world
    m = STDiT2(dict(qk_norm=True)).init_synthetic_weights(seed=5, device=c.local)
    g = torch.Generator().manual_seed(30 + c.rank)
    x = torch.randn(B, 4, 16, 64, 64, generator=g).to(dev)
    y = torch.randn(B, 1, 120, 4096, generator=g).to(torch.bfloat16).to(dev)
    kw = dict(num_frames=torch.full((B,), 16.0), height=torch.full((B,), 512.0), width=torch.full((B,), 512.0),
              ar=torch.full((B,), 1.0), fps=torch.full((B,), 24.0))
    t = torch.full((B,), 500.0, device=dev)
    ms = c.timed(lambda i: m(x, t, y, **kw), steps, warmup)
    del m
    torch.cuda.empty_cache()
    per = ms / steps
    return {"metric": "denoiser_forward_samples_per_sec_stdit2_xl_16x512", "value": round(total / (per * 1e-3), 3),
            "unit": "video-latents/s", "ms_per_step": round(per, 3), "n_gpus": c.world,
            "model_tflops_per_sec": round(STDIT2_TFLOP_PER_SAMPLE * total / (per * 1e-3), 1),
            "config": {"workload": "Open-Sora STDiT2-XL forward, 16 frames x 512x512 (16 x 1024 tokens), 120 text tokens "
                                   "(configs[4])", "global_batch": total, "batch_per_gpu": B, "dtype": "bf16"}}


def bench_qwen2vl_prefill(dev, steps=20, warmup=5):
    """Second half of BASELINE.json's metric: Qwen2-VL-7B prefill tokens/s (configs[3]: 4 x (one 448x448 image +
    512 text tokens) = 4 x 768 tokens, bf16, 1 x B200, ViT + 28 decoder layers + lm_head over all positions)."""
    import torch

    from paddlemix_b200 import ops
    from paddlemix_b200.qwen2_vl import Qwen2VLForConditionalGeneration
    model = Qwen2VLForConditionalGeneration({}).init_synthetic_weights(seed=4, device=dev.index)
    c = model.config
    g = torch.Generator().manual_seed(4)
    B, n_img_tok, n_txt = 4, 256, 510
    grid = [[1, 32, 32]] * B
    pv_h = torch.randn(B * 1024, 1176, generator=g).to(torch.bfloat16).pin_memory()
    rows = [[c.vision_start_token_id] + [c.image_token_id] * n_img_tok + [c.vision_end_token_id] +
            torch.randint(0, 151643, (n_txt,), generator=g).tolist() for _ in range(B)]
    ids_h = torch.tensor(rows).pin_memory()
    S = ids_h.shape[1]
    # device-resident variant: index math done once on the host, inputs already in HBM
    pos, _ = model.get_rope_index(ids_h, torch.tensor(grid))
    cos, sin = model._mrope_tables(pos)
    ids_d = ids_h.to(dev).reshape(-1)
    idx_d = (ids_h.reshape(-1) == c.image_token_id).nonzero().reshape(-1).to(dev)
    pv_d = pv_h.to(dev)
    for _ in range(warmup):  # also brings the clocks back up after an idle phase
        logits = model.prefill_device(ids_d, B, S, cos, sin, pv_d, grid, idx_d)
    torch.cuda.synchronize(dev)
    n0 = ops.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        logits = model.prefill_device(ids_d, B, S, cos, sin, pv_d, grid, idx_d)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    launches = (ops.launches() - n0) // steps
    # end to end through the public forward(): host token ids + pixel values in, logits of the LAST position out (what
    # generation consumes, modeling_qwen2_vl.py generate path; the forward itself produces all positions on the device)
    out_h = torch.empty(B, c.vocab_size).pin_memory()
    gt = torch.tensor(grid)
    for _ in range(3):
        model(input_ids=ids_h, pixel_values=pv_h, image_grid_thw=gt)
    torch.cuda.synchronize(dev)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    f0.record()
    for _ in range(steps):
        out = model(input_ids=ids_h, pixel_values=pv_h, image_grid_thw=gt)
        out_h.copy_(out.logits[:, -1], non_blocking=True)
        torch.cuda.current_stream().synchronize()
    f1.record()
    torch.cuda.synchronize(dev)
    wall_e2e = (time.perf_counter() - t0) * 1e3 / steps
    ms_e2e = max(f0.elapsed_time(f1) / steps, wall_e2e)
    tflop = 12.58 * B  # oracle.qwen2vl.qwen2vl_flops for this input (SURVEY.md §8d quotes 12.46 per 768-token sample)
    del model, logits
    torch.cuda.empty_cache()
    return {"metric": "qwen2vl_7b_prefill_tokens_per_sec", "value": round(B * S / (ms * 1e-3), 1), "unit": "tokens/s",
            "ms_per_prefill": round(ms, 3), "model_tflops_per_sec": round(tflop / (ms * 1e-3), 1), "steps": steps,
            "warmup": warmup,
            "config": {"workload": "Qwen2-VL-7B prefill, 4 x (448x448 image -> 1024 patches -> 256 merged tokens + 512 "
                                   "text tokens) = 3072 tokens, ViT + LLM + lm_head (all positions, fp32 logits) (configs[3])",
                       "weights": "random init, Qwen2-VL-7B architecture (8.3 B params)", "dtype": "bf16"},
            "gpu_launches": launches,
            "e2e": {"value": round(B * S / (ms_e2e * 1e-3), 1), "unit": "tokens/s", "ms_per_prefill": round(ms_e2e, 3),
                    "wall_ms_per_prefill": round(wall_e2e, 3),
                    "h2d_bytes_per_step": pv_h.numel() * 2 + ids_h.numel() * 8, "d2h_bytes_per_step": out_h.numel() * 4,
                    "d2h": "last-position logits [B, vocab] fp32"}}


def parity_section(c, keep):
    """C2 parity in the bench run: the GPU model on the cpu_baseline leg's weights / inputs vs its fp32 output."""
    import torch

    from paddlemix_b200.ppdiffusers.unet_2d_condition import UNet2DConditionModel
    cfg, P, x, ctx, added, ref = keep
    keys = ("in_channels", "out_channels", "flip_sin_to_cos", "freq_shift", "down_block_types", "up_block_types",
            "block_out_channels", "layers_per_block", "norm_num_groups", "norm_eps", "cross_attention_dim",
            "transformer_layers_per_block", "attention_head_dim", "use_linear_projection", "addition_embed_type",
            "addition_time_embed_dim", "projection_class_embeddings_input_dim", "resnet_out_scale_factor")
    model = UNet2DConditionModel(**{k: cfg[k] for k in keys}).load_state_dict(P, device=c.local)
    out = model(x.to(c.dev), 981, ctx.to(c.dev), added_cond_kwargs={k: v.to(c.dev) for k, v in added.items()}).sample
    o = out.float().cpu()
    cos = torch.nn.functional.cosine_similarity(o.flatten().double(), ref.flatten().double(), dim=0).item()
    err = (o - ref).abs().max().item() / ref.abs().max().item()
    del model
    torch.cuda.empty_cache()
    return {"config": "configs[1] shape: SDXL-base UNet, latent 128x128, B=1, t=981 (GPU bf16 kernels vs CPU fp32 oracle, "
                      "same weights and inputs)", "cosine": round(cos, 6), "max_rel_err": round(err, 5),
            "tolerance": PARITY_TOL, "pass": bool(cos >= PARITY_TOL["cosine_min"] and err <= PARITY_TOL["max_rel_err"]),
            "more": "tests/test_baseline_parity_gpu.py covers configs[1..4] shapes; profiles/ holds the recorded values"}


def run_b200(args):
    import torch

    c = Ctx()
    from paddlemix_b200.ppdiffusers.unet_2d_condition import UNet2DConditionModel
    world, rank = c.world, c.rank
    B, height = args.batch, args.height
    unet = UNet2DConditionModel(**SDXL).init_synthetic_weights(seed=1, device=c.local)

    main = sdxl_section(c, unet, B, height, args.steps, args.warmup, with_e2e=True, sample_clocks=True,
                        keep_outputs=args.dump_outputs is not None)
    if args.dump_outputs is not None:
        dump_outputs(c, main.pop("outputs"), args.dump_outputs)
    ms, ms_e2e = main["ms"], main["e2e"]["ms"]
    roof = roofline_section(c, unet, B, height) if rank == 0 else None

    extras = {}
    if not args.no_extras:
        # strong scaling of configs[1]: global batch 8 stays fixed, 8 / N images per rank
        if world > 1 and 8 % world == 0:
            del main["den"]
            torch.cuda.empty_cache()
            bs = 8 // world
            st = sdxl_section(c, unet, bs, height, args.steps, args.warmup, with_e2e=False)
            extras["sdxl_strong"] = {"metric": METRIC, "scaling": "strong", "global_batch": 8, "batch_per_gpu": bs,
                                     "value": round(8 * args.steps / (st["ms"] * 1e-3), 3), "unit": UNIT,
                                     "ms_per_step": round(st["ms"] / args.steps, 3), "n_gpus": world, "job": st["job"]}
            del st
        elif world == 1:
            extras["sdxl_strong"] = {"metric": METRIC, "scaling": "strong", "global_batch": 8, "batch_per_gpu": 8,
                                     "value": round(B * args.steps / (ms * 1e-3), 3), "unit": UNIT,
                                     "ms_per_step": round(ms / args.steps, 3), "n_gpus": 1,
                                     "note": "N = 1: identical to the main (weak) workload"}
    job = main["job"]
    clocks = main["clocks"]
    launches = main["launches"]
    h2d, d2h, wall_e2e = main["e2e"]["h2d"], main["e2e"]["d2h"], main["e2e"]["wall_ms"]
    del main, unet
    torch.cuda.empty_cache()

    if not args.no_extras:
        try:
            extras["sd3_b32"] = sd3_section(c, steps=args.steps, warmup=args.warmup)
        except Exception as ex:  # noqa: BLE001
            extras["sd3_b32"] = {"error": repr(ex)[:300]}
        try:
            extras["stdit2_b4"] = stdit2_section(c, steps=args.steps, warmup=args.warmup)
        except Exception as ex:  # noqa: BLE001
            extras["stdit2_b4"] = {"error": repr(ex)[:300]}

    if rank != 0:
        if world > 1:
            c.dist.destroy_process_group()
        return

    qwen = None
    if world == 1 and not args.no_qwen:
        try:
            qwen = bench_qwen2vl_prefill(c.dev, steps=args.steps)
        except Exception as ex:  # noqa: BLE001
            qwen = {"metric": "qwen2vl_7b_prefill_tokens_per_sec", "value": None, "error": repr(ex)[:300]}

    cpu = parity = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_reference_forward(keep=True)
            keep = r.pop("_keep")
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
                   "seconds_per_sample": round(r["seconds_per_sample"], 2)}
            try:
                parity = parity_section(c, keep)
            except Exception as ex:  # noqa: BLE001
                parity = {"error": repr(ex)[:300]}
        except Exception as ex:  # the baseline is a report, never a reason to lose the GPU number
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port", "sample": f"failed: {ex}"}

    value = B * world * args.steps / (ms * 1e-3)
    ms_e2e_eff = max(ms_e2e, wall_e2e)  # device events and the host clock around the same loop: report the larger
    e2e = B * world * args.steps / (ms_e2e_eff * 1e-3)
    step_tflop = SDXL_TFLOP_PER_SAMPLE * B if height == 1024 else None
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "SDXL-base UNet2DConditionModel forward + fused DDIM update per timestep (configs[1])",
                   "batch_per_gpu": B, "global_batch": B * world, "resolution": f"{height}x{height}",
                   "latent": f"{height // 8}x{height // 8}", "scheduler": "DDIM 50 steps (scaled_linear, steps_offset 1)",
                   "cfg": "off (UNet rows = batch)",
                   "parallelism": f"dp{world} (images sharded, weights replicated, one all_gather of finished latents)",
                   "weights": "random init, SDXL-base architecture (2.57 B params)", "cuda_graph": True,
                   "l2": "no explicit flush: 5.1 GB of weights + >10 GB of activations stream per step (>> 126 MB L2)"},
        "finished_latents_per_sec_50_steps": round(value / 50.0, 4),
        "model_tflops_per_sec": None if step_tflop is None else round(step_tflop * world / (ms / args.steps * 1e-3), 1),
        "clocks": clocks,
        "e2e": {"value": round(e2e, 3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": round(ms_e2e_eff / args.steps, 3), "device_ms_per_step": round(ms_e2e / args.steps, 3),
                "wall_ms_per_step": round(wall_e2e / args.steps, 3)},
        "gpu_launches": launches,
        "roofline": roof,
        "job": job,
        "cpu_baseline": cpu,
        "parity": parity,
        "qwen2vl_prefill": qwen,
    }
    line.update(extras)
    print(json.dumps(line), flush=True)
    if world > 1:
        c.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-qwen", action="store_true", help="skip the Qwen2-VL-7B prefill section")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling / SD3 / STDiT2 sections")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed SDXL steps, write what the last one returned (noise_pred, latents) as "
                         "float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
