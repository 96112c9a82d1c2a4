#!/usr/bin/env python
"""Benchmark of the Ctrl-Adapter denoising hot path on B200 (contract: see the task brief / DESIGN.md section 6).

  python bench.py --gpus N --steps K --warmup W            ours: CUDA path (this repo's kernels)
  python bench.py --impl reference --gpus N ...            reference arm: the oracle restatement of the reference's
                                                           PyTorch path on the host CPU cores (diffusers is not
                                                           installable here, so the reference itself cannot run)
  python bench.py ... --dump-outputs DIR                   also writes the final latents of the last timed step to
                                                           DIR/latents.npy, for comparing the outputs of two builds

Workloads (--workload):
  sdxl   (default, the headline) BASELINE.json configs[1]: SDXL + depth ControlNet + Ctrl-Adapter, 1024x1024, batch 8
  i2vgen BASELINE.json configs[2]: I2VGen-XL + depth adapter, 16 frames 512x512, batch 4
  svd    BASELINE.json configs[3]: SVD + adapter, 14 frames 576x1024, batch 2 per GPU (use_size_512=False)
  multi  BASELINE.json configs[4]: I2VGen-XL + 3 ControlNets (depth, canny, softedge) + MoE router, 16 frames 512x512,
         batch 8 over 8 GPUs = 1 clip per GPU
Synthetic latents / embeddings of the named shapes, random weights of the real architectures, bf16.
One "step" = one iteration of the pipeline loop for the whole per-GPU batch:
[pool] -> ControlNet(s) -> [router merge] -> Ctrl-Adapter -> UNet(+injection) -> CFG -> scheduler update.
Step-invariant work (prompt K/V projections, the ControlNet's conditioning-image embedding, router weights) is done once
in prepare(), outside the timed steps, exactly as a pipeline call would do it once per generation.

Every line carries, next to `value` (CUDA-graph replay, inputs resident in HBM): `e2e` (the step as the pipeline classes run it
-- CUDA-graph replay by default, `--no-graph`: eager module forward()s through the C ABI -- with pinned host latents copied
in and out every step and the host waiting for each result), `roofline` (dominant kernel family, CUDA events),
`eager_gpu_baseline` + `vs_eager` (the oracle restatement of the reference loop as eager bf16-autocast PyTorch on the same
GPU: BASELINE.md's "reference single-GPU eager PyTorch" denominator) and `cpu_baseline` (the same oracle on the host cores).

Multi-GPU (--gpus N under torchrun): batch-axis sharding, every rank runs its own batch with no per-step
communication (weak scaling) and one NCCL all-gather of the final latents after the last step.
"""
from __future__ import annotations

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
sys.dont_write_bytecode = True  # the benchmark leaves the tree as the build left it (it may be read-only)

import torch  # noqa: E402

BF16 = torch.bfloat16
# algorithmic TFLOP per frame-sample (SURVEY.md section 8d / BASELINE.md section 2)
TF = {"cn64": 0.2833, "cn72x128": 0.7735, "ad_sdxl": 2.2565, "ad_video64": 0.6564, "ad_video72x128": 1.679,
      "unet_sdxl": 6.761, "unet_i2vgen": 1.308, "unet_svd72x128": 3.192}
WORKLOADS = {
    "sdxl": dict(metric="denoising steps/sec (SDXL 1024x1024 + depth ControlNet + Ctrl-Adapter, batch 8)",
                 base="BASELINE.json configs[1]", batch=8, frames=1, tflop=TF["cn64"] + TF["ad_sdxl"] + TF["unet_sdxl"]),
    "i2vgen": dict(metric="denoising steps/sec (I2VGen-XL 16f 512x512 + depth ControlNet + Ctrl-Adapter, batch 4)",
                   base="BASELINE.json configs[2]", batch=4, frames=16,
                   tflop=TF["cn64"] + TF["ad_video64"] + TF["unet_i2vgen"]),
    "svd": dict(metric="denoising steps/sec (SVD 14f 576x1024 + depth ControlNet + Ctrl-Adapter, batch 2 per GPU)",
                base="BASELINE.json configs[3]", batch=2, frames=14,
                tflop=TF["cn72x128"] + TF["ad_video72x128"] + TF["unet_svd72x128"]),
    "multi": dict(metric="denoising steps/sec (I2VGen-XL 16f 512x512 + depth/canny/softedge ControlNets + MoE router + "
                         "Ctrl-Adapter, batch 8 over 8 GPUs)",
                  base="BASELINE.json configs[4]", batch=1, frames=16,
                  tflop=3 * TF["cn64"] + TF["ad_video64"] + TF["unet_i2vgen"]),
}
VIDEO_ADAPTER_KW = dict(num_blocks=1, cross_attention_dim=1024, add_spatial_resnet=True, add_temporal_resnet=True,
                        add_spatial_transformer=True, add_temporal_transformer=True, add_adapter_location_A=True,
                        add_adapter_location_B=True, add_adapter_location_C=True, add_adapter_location_D=True,
                        add_adapter_location_M=True)
SDXL_ADAPTER_KW = dict(num_blocks=1, num_frames=1, cross_attention_dim=2048, add_spatial_resnet=True,
                       add_spatial_transformer=True, add_adapter_location_A=True, add_adapter_location_B=True,
                       add_adapter_location_C=True)
ROUTER_KW = dict(num_experts=7, backbone_model_name="i2vgenxl", router_type="simple_weights", num_routers=12,
                 add_mid_block_router=True)
ROUTER_MASK = [1, 1, 0, 1, 0, 0, 0]  # inference.py:343-345: control types depth, canny, softedge


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--batch", type=int, default=0, help="images / clips per GPU (0 = the BASELINE config's)")
    p.add_argument("--res", type=int, default=1024, help="sdxl only")
    p.add_argument("--workload", default="sdxl", choices=list(WORKLOADS))
    p.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    p.add_argument("--skip-cpu-baseline", action="store_true")
    p.add_argument("--skip-e2e", action="store_true")
    p.add_argument("--skip-eager-baseline", action="store_true",
                   help="do not time the oracle (restated reference) as eager bf16-autocast PyTorch on this GPU")
    p.add_argument("--skip-profile", action="store_true", help="skip the per-kernel CUDA-event profile (roofline block)")
    p.add_argument("--cpu-budget-s", type=float, default=45.0, help="wall-clock budget of the cpu_baseline leg")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the latents of the last timed step to DIR/latents.npy (float32) so that two builds can be "
                        "compared output for output; the inputs and weights are seeded, so equal arguments give equal inputs. "
                        "The outputs themselves vary slightly from run to run (the GroupNorm statistics are summed with "
                        "atomics), and the variation grows with the number of steps: compare with a tolerance")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return a


# ----------------------------------------------------------------------------------------------------
# synthetic inputs of the named shapes (identical for our loop, the eager-GPU oracle and the CPU oracle)
# ----------------------------------------------------------------------------------------------------
def synthetic_inputs(workload, batch, res, device, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g).to(device)  # noqa: E731
    u = lambda *s: torch.rand(*s, generator=g).to(device)   # noqa: E731
    if workload == "sdxl":
        lat = res // 8
        return dict(latents=r(batch, 4, lat, lat), prompt_embeds=r(2 * batch, 77, 2048),
                    add_text_embeds=r(2 * batch, 1280),
                    add_time_ids=torch.tensor([[res, res, 0, 0, res, res]] * (2 * batch), dtype=torch.float32).to(device),
                    controlnet_prompt_embeds=r(2 * batch, 77, 768), control_images=u(2 * batch, 3, 512, 512))
    if workload in ("i2vgen", "multi"):
        f = WORKLOADS[workload]["frames"]
        n = 2 * batch * f
        d = dict(latents=r(batch, 4, f, 64, 64), prompt_embeds=r(2 * batch, 77, 1024),
                 image_latents=r(2 * batch, 4, f, 64, 64), image_embeddings=r(2 * batch, 1, 1024),
                 fps=torch.full((2 * batch,), 16.0, device=device), controlnet_prompt_embeds=r(n, 77, 768))
        d["control_images"] = [u(n, 3, 512, 512) for _ in range(3)] if workload == "multi" else u(n, 3, 512, 512)
        return d
    f, lh, lw = WORKLOADS["svd"]["frames"], 72, 128  # 576 x 1024 video -> 72 x 128 latents (needs use_size_512=False)
    n = 2 * batch * f
    il = r(batch, f, 4, lh, lw)
    return dict(latents=r(batch, f, 4, lh, lw), image_latents=torch.cat([torch.zeros_like(il), il]),
                image_embeddings=torch.cat([torch.zeros(batch, 1, 1024, device=device), r(batch, 1, 1024)]),
                added_time_ids=torch.tensor([[13.0, 127.0, 0.02]] * (2 * batch)).to(device),
                controlnet_prompt_embeds=r(n, 77, 768), control_images=u(n, 3, 8 * lh, 8 * lw))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each tensor as <out_dir>/<name>.npy in float32.  If they exceed DUMP_LIMIT_BYTES in all, each is replaced by
    the same share of its flattened elements, at positions drawn from a fixed seed (so two runs sample alike)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(4 * t.numel() for t in arrays.values())
    keep = min(1.0, DUMP_LIMIT_BYTES / total) if total else 1.0
    for name, t in arrays.items():
        flat = t.detach().float().reshape(-1).cpu()
        if keep < 1.0:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:int(flat.numel() * keep)]
            flat = flat[idx.sort().values]
        else:
            flat = flat.reshape(t.shape)
        np.save(os.path.join(out_dir, f"{name}.npy"), flat.numpy())


def _randomise_controlnet_heads(cn):
    """zero-initialised ControlNet heads would make every residual exactly 0: give them random values"""
    for m in list(cn.controlnet_down_blocks) + [cn.controlnet_mid_block, cn.controlnet_cond_embedding.conv_out]:
        torch.nn.init.normal_(m.weight, std=0.02)


def build_ours(workload, batch, res, dev, seed):
    """Our modules + loop for one workload; returns (loop, inputs)."""
    from ctrl_adapter_b200.adapter import ControlNetAdapter, ControlNetRouter
    from ctrl_adapter_b200.controlnet import ControlNetModel, MultiControlNetModel
    n_nets = 3 if workload == "multi" else 1
    nets = []
    for _ in range(n_nets):
        with torch.device(dev):
            cn = ControlNetModel(cross_attention_dim=768)
        _randomise_controlnet_heads(cn)
        nets.append(cn.to(BF16).eval())
    inp = synthetic_inputs(workload, batch, res, dev, seed)
    if workload == "sdxl":
        from ctrl_adapter_b200.pipeline_sdxl import SDXLControlNetAdapterLoop
        from ctrl_adapter_b200.unet_sdxl import UNet2DConditionModel
        with torch.device(dev):
            ad, un = ControlNetAdapter("sdxl", **SDXL_ADAPTER_KW), UNet2DConditionModel()
        loop = SDXLControlNetAdapterLoop(nets[0], ad.to(BF16).eval(), un.to(BF16).eval(), num_inference_steps=50,
                                         guidance_scale=5.0, controlnet_conditioning_scale=1.0)
    elif workload == "svd":
        from ctrl_adapter_b200.pipeline_svd import SVDControlNetAdapterLoop
        from ctrl_adapter_b200.unet_svd import UNetSpatioTemporalConditionModel
        f = WORKLOADS["svd"]["frames"]
        with torch.device(dev):
            ad = ControlNetAdapter("svd", num_frames=f, **VIDEO_ADAPTER_KW)
            un = UNetSpatioTemporalConditionModel(num_attention_heads=(5, 10, 20, 20), num_frames=f)
        loop = SVDControlNetAdapterLoop(nets[0], ad.to(BF16).eval(), un.to(BF16).eval(), num_inference_steps=25,
                                        min_guidance_scale=1.0, max_guidance_scale=3.0, use_size_512=False,
                                        skip_conv_in=True)
    else:
        from ctrl_adapter_b200.pipeline_i2vgen import I2VGenXLControlNetAdapterLoop
        from ctrl_adapter_b200.unet_i2vgen import I2VGenXLUNet
        f = WORKLOADS[workload]["frames"]
        with torch.device(dev):
            ad, un = ControlNetAdapter("i2vgenxl", num_frames=f, **VIDEO_ADAPTER_KW), I2VGenXLUNet()
        router, masks, cnm = None, None, nets[0]
        if workload == "multi":
            with torch.device(dev):
                router = ControlNetRouter(**ROUTER_KW)
            for m in list(router.down_blocks_router) + [router.mid_block_router]:
                torch.nn.init.normal_(m.wg.weight, std=1.0)
            masks, cnm = ROUTER_MASK, MultiControlNetModel(nets)
        loop = I2VGenXLControlNetAdapterLoop(cnm, ad.to(BF16).eval(), un.to(BF16).eval(), router,
                                             num_inference_steps=50, guidance_scale=9.0, inference_expert_masks=masks)
    loop.prepare(**inp)
    return loop, inp


def build_oracle_stepper(workload, inp, device, dtype, batch):
    """The restated reference loop on the oracle modules (fresh random weights of the same architectures).
    Returns step(i, latents) -> latents and the initial latents."""
    from oracle.adapter import ControlNetAdapter as OA, ControlNetRouter as OR
    from oracle.controlnet import ControlNetModel as OC, MultiControlNetModel as OM
    with torch.device(device):
        nets = [OC(cross_attention_dim=768) for _ in range(3 if workload == "multi" else 1)]
    for cn in nets:
        _randomise_controlnet_heads(cn)
    # .to(device): legacy torch.Tensor([...]) parameters of the restated modules ignore the device context
    cast = lambda m: m.to(device=device, dtype=dtype).eval()  # noqa: E731
    ei = {k: ([t.to(dtype) for t in v] if isinstance(v, list) else (v.to(dtype) if v.is_floating_point() else v))
          for k, v in inp.items()}
    if workload == "sdxl":
        from oracle.pipeline_sdxl import EulerDiscreteScheduler, sdxl_step
        from oracle.unet_sdxl import UNet2DConditionModel as OU
        with torch.device(device):
            ad, un = OA("sdxl", **SDXL_ADAPTER_KW), OU()
        cn, ad, un = cast(nets[0]), cast(ad), cast(un)
        sch = EulerDiscreteScheduler()
        sch.set_timesteps(50, device=device)
        lat0 = ei["latents"] * sch.init_noise_sigma

        def step(i, lat):
            return sdxl_step(cn, ad, un, sch, i, lat, ei["prompt_embeds"], ei["add_text_embeds"], ei["add_time_ids"],
                             ei["controlnet_prompt_embeds"], ei["control_images"])
        return step, lat0
    if workload == "svd":
        from oracle.pipeline_svd import EulerDiscreteSchedulerSVD, svd_step
        from oracle.unet_svd import UNetSpatioTemporalConditionModel as OU
        f = WORKLOADS["svd"]["frames"]
        with torch.device(device):
            ad = OA("svd", num_frames=f, **VIDEO_ADAPTER_KW)
            un = OU(num_attention_heads=(5, 10, 20, 20), num_frames=f)
        cn, ad, un = cast(nets[0]), cast(ad), cast(un)
        sch = EulerDiscreteSchedulerSVD()
        sch.set_timesteps(25, device=device)
        lat0 = (ei["latents"] * sch.init_noise_sigma).to(dtype)

        def step(i, lat):
            return svd_step(cn, ad, un, sch, i, lat, ei["image_latents"], ei["image_embeddings"], ei["added_time_ids"],
                            ei["controlnet_prompt_embeds"], ei["control_images"], use_size_512=False, skip_conv_in=True,
                            skip_time_emb=False).to(dtype)
        return step, lat0
    from oracle.pipeline_i2vgen import DDIMScheduler, i2vgen_step
    from oracle.unet_i2vgen import I2VGenXLUNet as OU
    f = WORKLOADS[workload]["frames"]
    with torch.device(device):
        ad, un = OA("i2vgenxl", num_frames=f, **VIDEO_ADAPTER_KW), OU()
    ad, un = cast(ad), cast(un)
    router, masks = None, None
    if workload == "multi":
        with torch.device(device):
            router = OR(**ROUTER_KW)
        router, masks, cn = cast(router), ROUTER_MASK, OM([cast(c) for c in nets])
    else:
        cn = cast(nets[0])
    sch = DDIMScheduler()
    sch.set_timesteps(50, device=device)

    def step(i, lat):
        return i2vgen_step(cn, ad, un, sch, i, lat, ei["prompt_embeds"], ei["image_latents"], ei["image_embeddings"],
                           ei["fps"], ei["controlnet_prompt_embeds"], ei["control_images"], router=router, masks=masks)
    return step, ei["latents"]


# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------
# CPU legs: the oracle (restated reference PyTorch path) on the host cores
# ----------------------------------------------------------------------------------------------------
def _cpu_threads():
    """Threads for the CPU legs: one per PHYSICAL core this process may run on, whatever OMP_NUM_THREADS says (torchrun
    sets it to 1).  BASELINE.md section 3 says os.cpu_count(), but on the pool's 2-way SMT hosts 128 logical threads
    make the oracle 34x SLOWER than 64 (218 s vs 6.4 s for the same 512x512 frame-sample, round-2 run 6 vs round 1:
    OpenMP spin-waits fighting over the shared cores), so the reference's CPU path would be misrepresented."""
    try:
        allowed = os.sched_getaffinity(0)
        cores, phys, cid, cpu = set(), None, None, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id"):
                cid = int(line.split(":")[1])
                if cpu in allowed:
                    cores.add((phys, cid))
        if cores:
            return len(cores)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return ""


def _oracle_frame_sample(cn, ad, un, inp, lat, t, res):
    """One SDXL frame-sample through ControlNet (at res/2, SURVEY.md section 8a) -> adapter -> UNet, restated reference
    modules (the quick CPU sample of the default run)."""
    F = torch.nn.functional
    down, mid = cn(F.adaptive_avg_pool2d(lat, (res // 16, res // 16)), t,
                   encoder_hidden_states=inp["controlnet_prompt_embeds"][:1],
                   controlnet_cond=F.adaptive_avg_pool2d(inp["control_images"][:1], (res // 2, res // 2)),
                   conditioning_scale=1.0, return_dict=False)
    da, _ = ad(down, num_frames=1, timestep=t, encoder_hidden_states=inp["prompt_embeds"][:1])
    un(lat, t, encoder_hidden_states=inp["prompt_embeds"][:1],
       added_cond_kwargs={"text_embeds": inp["add_text_embeds"][:1], "time_ids": inp["add_time_ids"][:1]},
       down_block_additional_residuals=da, mid_block_additional_residual=0)


def _sdxl_oracle_modules(device):
    from oracle.adapter import ControlNetAdapter
    from oracle.controlnet import ControlNetModel
    from oracle.unet_sdxl import UNet2DConditionModel
    with torch.device(device):
        return (ControlNetModel(cross_attention_dim=768).eval(), ControlNetAdapter("sdxl", **SDXL_ADAPTER_KW).eval(),
                UNet2DConditionModel().eval())


def _oracle_flops_per_frame_sample(res):
    """Exact matmul / conv / attention FLOPs of one SDXL frame-sample at `res`, counted on meta tensors (no compute)."""
    from torch.utils.flop_counter import FlopCounterMode
    cn, ad, un = _sdxl_oracle_modules("meta")
    inp = {k: (v.to("meta") if torch.is_tensor(v) else v) for k, v in synthetic_inputs("sdxl", 1, res, "cpu", 1234).items()}
    with FlopCounterMode(display=False) as fc, torch.no_grad():
        _oracle_frame_sample(cn, ad, un, inp, inp["latents"][:1], torch.tensor(500.0), res)
    return float(fc.get_total_flops())


def cpu_quick_sdxl_rate(res, budget_s, sample_res=512):
    """The cpu_baseline leg of the DEFAULT run (must stay well inside a minute; a full-resolution pass of the reference
    path costs ~190 s on the pool's hosts): ONE SDXL frame-sample at `sample_res` (ControlNet -> adapter -> UNet, fp32
    eager, one thread per physical core), >= 3 timed passes after one warm-up, scaled to the 16-frame-sample `res` step by the
    exact FLOP ratio (torch FlopCounterMode on meta tensors).  `--impl reference` times the un-scaled full-resolution
    sample instead; both state their extrapolation factor."""
    cores = _cpu_threads()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    t0 = time.time()
    cn, ad, un = _sdxl_oracle_modules("cpu")
    build_s = time.time() - t0
    f_pass = _oracle_flops_per_frame_sample(sample_res)
    f_step = 2 * WORKLOADS["sdxl"]["batch"] * _oracle_flops_per_frame_sample(res)
    from oracle.pipeline_sdxl import EulerDiscreteScheduler
    sch = EulerDiscreteScheduler()
    sch.set_timesteps(50)
    inp = synthetic_inputs("sdxl", 1, sample_res, "cpu", 1234)
    lat = (inp["latents"] * sch.init_noise_sigma)[:1]
    times, t_start = [], time.time()
    for i in range(1 + 8):
        t1 = time.time()
        with torch.no_grad():
            _oracle_frame_sample(cn, ad, un, inp, sch.scale_model_input(lat, i % 50), sch.timesteps[i % 50], sample_res)
        dt = time.time() - t1
        spent = time.time() - t_start
        if i >= 1 or spent > budget_s:
            times.append(dt)
        if len(times) >= 3 and spent + dt > budget_s:
            break
        if spent > budget_s and times:
            break
    med, mn = statistics.median(times), min(times)
    factor = f_step / f_pass
    rate = 1.0 / (med * factor)
    info = {"value": rate, "unit": "steps/s", "cores": cores, "kind": "port",
            "sample": f"one frame-sample (ControlNet -> adapter -> UNet) at {sample_res}x{sample_res} = {f_pass / 1e12:.3f} TFLOP, "
                      f"fp32 eager, {cores} threads, {len(times)} timed passes after 1 warm-up: median {med:.2f} s, min {mn:.2f} s; "
                      f"scaled to the 16-frame-sample {res}x{res} step ({f_step / 1e12:.1f} TFLOP) by the exact FLOP ratio "
                      f"x{factor:.1f} (a full-resolution pass is timed by `--impl reference`); oracle restatement of the "
                      f"reference path (the reference itself needs diffusers, not installable here); cpu: {_cpu_model()}",
            "s_per_sample_median": med, "s_per_sample_min": mn, "value_from_min": 1.0 / (mn * factor),
            "extrapolation_factor": factor, "timed_passes": len(times), "cpu_tflops": f_pass / med / 1e12,
            "model_build_s": build_s, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"), "logical_cpus": os.cpu_count()}
    return rate, info


def cpu_reference_step_rate(workload, res, steps, warmup, budget_s):
    """Oracle on the host CPU: fp32 eager, one thread per physical core (_cpu_threads) whatever OMP_NUM_THREADS says.  A full step of any workload costs many CPU-minutes, so a timed pass is a BOUNDED sample of the
    same workload at its real resolution and frame count: one denoising iteration of ONE batch element (sdxl: one image
    = 2 CFG frame-samples at `res`; video: one clip = 2 x F frame-samples).  Batch elements are independent on this path
    (no op mixes samples), so the step time is the sample time x the per-GPU batch -- the only extrapolation, stated in
    `sample`.  At least 3 timed passes unless the budget runs out; min and median are both reported, `value` uses the
    median."""
    cores = _cpu_threads()
    torch.set_num_threads(cores)
    w = WORKLOADS[workload]
    batch = w["batch"]
    torch.manual_seed(0)
    t0 = time.time()
    inp = synthetic_inputs(workload, 1, res, "cpu", 1234)
    step, lat = build_oracle_stepper(workload, inp, "cpu", torch.float32, 1)
    build_s = time.time() - t0
    times, done = [], 0
    t_start = time.time()
    want = max(3, steps)
    for i in range(warmup + want):
        t1 = time.time()
        with torch.no_grad():
            lat = step(i % 25, lat)
        dt = time.time() - t1
        done += 1
        spent = time.time() - t_start
        if i >= warmup or spent > budget_s:
            times.append(dt)  # a warm-up pass is promoted to a timed one when the budget is already spent
        # stop when the next pass would overrun the budget (but always keep one timed pass)
        if times and spent + dt > budget_s and (len(times) >= 3 or spent > budget_s):
            break
    med, mn = statistics.median(times), min(times)
    rate = 1.0 / (med * batch)
    n_fs = 2 * w["frames"]
    info = {"value": rate, "unit": "steps/s", "cores": cores, "kind": "port",
            "sample": f"one denoising iteration of ONE batch element ({n_fs} CFG frame-samples at the workload's real "
                      f"resolution / frame count: {n_fs * w['tflop']:.1f} TFLOP), fp32 eager, {cores} threads, {len(times)} timed "
                      f"pass(es) of {done} executed: median {med:.2f} s, min {mn:.2f} s; step time = sample x {batch} "
                      f"(the per-GPU batch; batch elements are independent); oracle restatement of the reference path (the "
                      f"reference itself needs diffusers, not installable here); cpu: {_cpu_model()}",
            "s_per_sample_median": med, "s_per_sample_min": mn, "value_from_min": 1.0 / (mn * batch),
            "extrapolation_factor": batch, "timed_passes": len(times), "cpu_tflops": n_fs * w["tflop"] / med,
            "model_build_s": build_s, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"), "logical_cpus": os.cpu_count()}
    return rate, info


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[a.workload]
    rate, info = cpu_reference_step_rate(a.workload, a.res, a.steps, a.warmup, budget_s=150.0)
    line = {"impl": "reference", "metric": w["metric"], "value": rate, "unit": "steps/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1000.0 / rate if rate > 0 else None,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a.workload, w["batch"], a.res), "baseline_config": w["base"],
                       "sample": info["sample"], "extrapolation_factor": info["extrapolation_factor"]},
            "cpu_baseline": info,
            "e2e": {"value": rate, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_name(workload, batch, res):
    w = WORKLOADS[workload]
    n = 2 * batch * w["frames"]
    return {"sdxl": f"SDXL+depth ControlNet+Ctrl-Adapter {res}x{res}, batch {batch} per GPU",
            "i2vgen": f"I2VGen-XL+depth ControlNet+Ctrl-Adapter 16 frames 512x512, batch {batch} per GPU",
            "svd": f"SVD+depth ControlNet+Ctrl-Adapter 14 frames 576x1024, batch {batch} per GPU",
            "multi": f"I2VGen-XL + 3 ControlNets (depth, canny, softedge) + MoE router + Ctrl-Adapter 16 frames 512x512, "
                     f"batch {batch} per GPU"}[workload] + f" (CFG: {n} frame-samples), one pipeline-loop iteration per step"


# ----------------------------------------------------------------------------------------------------
_RESULT_FD = None


def _quiet_stdout():
    """The contract is ONE JSON line on stdout: route everything libraries print there (e.g. NCCL's version banner)
    to stderr and keep the real stdout for emit()."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    a = parse()
    _quiet_stdout()
    if a.impl == "reference":
        run_reference_arm(a)
        return
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours) needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from ctrl_adapter_b200 import _lib, ops
    _lib.check(_lib.load().ca_device_ok(), "ca_device_ok")

    w = WORKLOADS[a.workload]
    batch = a.batch or w["batch"]
    torch.manual_seed(1234 + rank)
    loop, inp = build_ours(a.workload, batch, a.res, dev, 1234 + rank)
    n_samples = 2 * batch * w["frames"]

    use_graph = not a.no_graph
    nsteps = loop.num_inference_steps  # the schedule wraps around when more steps are timed than it has
    l0 = ops.PROFILER.launches
    loop.step(0)  # packs weights, sets kernel attributes
    launches_per_step = ops.PROFILER.launches - l0
    torch.cuda.synchronize()
    if use_graph:
        loop.capture(warmup=1)
    stepfn = loop.step_graph if use_graph else loop.step
    for i in range(a.warmup):
        stepfn(i % nsteps)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(a.steps):
        stepfn((a.warmup + i) % nsteps)
    if dist:  # the single collective of the job: gather every rank's final latents (C1 in SURVEY.md)
        from ctrl_adapter_b200.distributed import gather_latents
        gathered = gather_latents(loop.latents, loop.latents.shape[0] * world)  # noqa: F841
    ev1.record()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    if dist:
        tt = torch.tensor([ms_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt)
    ms_step = ms_total / a.steps
    value = world * a.steps / (ms_total / 1000.0)
    finite = bool(torch.isfinite(loop.latents).all())
    if a.dump_outputs and rank == 0:  # before the e2e and profile legs below step the loop again
        dump_outputs(a.dump_outputs, {"latents": gathered if dist else loop.latents})

    # ---- e2e: public module API, host buffers, H2D/D2H of the step's inputs/outputs inside the timed region ----
    e2e = None
    if not a.skip_e2e:
        host_lat = torch.empty(loop.latents.shape, dtype=torch.float32).pin_memory()
        host_lat.copy_(loop.latents.cpu())
        host_in = torch.empty(loop.model_in.shape, dtype=BF16).pin_memory()
        host_in.copy_(loop.model_in.cpu())
        ke = max(3, min(a.steps, 10))
        for _ in range(2):
            stepfn(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(ke):
            loop.latents.copy_(host_lat, non_blocking=True)       # H2D: this step's latents
            loop.model_in.copy_(host_in, non_blocking=True)       # H2D: scaled model input
            stepfn(i % nsteps)                                    # the pipeline classes' step (graph replay unless --no-graph)
            host_lat.copy_(loop.latents, non_blocking=True)       # D2H: the step's result
            host_in.copy_(loop.model_in, non_blocking=True)
            torch.cuda.current_stream().synchronize()             # the host consumes the result every step
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms_e = e0.elapsed_time(e1)
        if dist:
            tt = torch.tensor([ms_e], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms_e = float(tt)
        nbytes = host_lat.numel() * 4 + host_in.numel() * 2
        e2e = {"value": world * ke / (ms_e / 1000.0), "unit": "steps/s", "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": nbytes, "steps": ke, "ms_per_step": ms_e / ke, "wall_ms_per_step": 1000 * wall / ke,
               "path": ("CUDA-graph replay of the step (the pipeline classes' default)" if use_graph else
                        "eager module forward() calls through the C ABI") +
                       ", pinned host latents copied in/out every step, host waits for every result"}

    # ---- per-kernel-family CUDA-event profile of one eager step -> roofline of the dominant kernel ----
    roofline, families = None, None
    peaks, peak_src = measured_peaks()
    if not a.skip_profile and rank == 0:
        ops.PROFILER.start()
        loop.step(0)
        ops.PROFILER.stop()
        fam = ops.PROFILER.summary()
        tot = sum(v["ms"] for v in fam.values())
        families = {k: {"launches": v["launches"], "ms": round(v["ms"], 3), "share": round(v["ms"] / tot, 4),
                        "tflops": round(v["flops"] / (v["ms"] * 1e9), 2) if v["ms"] > 0 and v["flops"] else None,
                        "gbs": round(v["bytes"] / (v["ms"] * 1e6), 1) if v["ms"] > 0 and v["bytes"] else None}
                    for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
        top = max(fam.items(), key=lambda kv: kv[1]["ms"])
        # DRAM bytes per launch of the dominant kernel: ncu dram__bytes_{read,write}.sum over every launch of one step
        # (profiles/r?_traffic_<workload>.json, made by scripts/launch_share.py from the committed launch list)
        traffic = None
        for rnd in ("r2", "r1"):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", f"{rnd}_traffic_{a.workload}.json")))
                kn = {"gemm": "gemm_conv_kernel", "attention": "attention_kernel"}.get(top[0])
                if kn in tj:
                    traffic = round(tj[kn]["dram_bytes_per_launch"], 0)
                    break
            except Exception:
                continue
        if top[0] in ("gemm", "attention"):
            ach = top[1]["flops"] / (top[1]["ms"] * 1e9)
            peak = peaks["bf16_tflops_sustained"]
            roofline = {"kernel": {"gemm": "gemm_conv_kernel (tcgen05 multi-tap GEMM / implicit conv)",
                                   "attention": "attention_kernel (tcgen05 flash attention)"}[top[0]],
                        "bound": "tensor", "achieved": round(ach, 2), "peak": peak, "unit": "TFLOP/s",
                        "frac": round(ach / peak, 4), "traffic": traffic,
                        "how": f"sum of algorithmic FLOPs of the {top[1]['launches']} launches of one step / sum of their "
                               f"CUDA-event durations ({top[1]['ms']:.1f} ms = {100 * top[1]['ms'] / tot:.0f}% of the step); "
                               f"peak = bf16_tflops_sustained, {peak_src}"}
        else:
            ach = top[1]["bytes"] / (top[1]["ms"] * 1e6)
            roofline = {"kernel": top[0], "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"],
                        "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": None,
                        "how": f"algorithmic bytes / CUDA-event time of one step; peak {peak_src}"}

    # ---- "reference single-GPU eager PyTorch" (BASELINE.md section 3, the north-star denominator): oracle modules, bf16
    # params, torch.autocast, default SDPA backend, no compile, same synthetic tensors and batch; >= 10 steps after 3 ----
    eager_gpu = None
    del loop
    torch.cuda.empty_cache()
    if not a.skip_eager_baseline and rank == 0 and world == 1:  # N > 1 lines: see the N = 1 line of the same workload
        try:
            estep, lat = build_oracle_stepper(a.workload, inp, dev, BF16, batch)

            def run(i, lat):
                with torch.no_grad(), torch.autocast("cuda", dtype=BF16):
                    return estep(i, lat)
            for i in range(3):
                lat = run(i, lat)
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ne = 10
            q0.record()
            for i in range(ne):
                lat = run(3 + i, lat)
            q1.record()
            torch.cuda.synchronize()
            ems = q0.elapsed_time(q1) / ne
            eager_gpu = {"value": 1000.0 / ems, "unit": "steps/s", "ms_per_step": ems, "steps": ne, "warmup": 3,
                         "what": "oracle restatement of the reference loop, eager PyTorch bf16 autocast on this GPU "
                                 "(cuDNN / cuBLAS / SDPA), same batch and shapes, random weights of the same architectures"}
            del estep, lat
            torch.cuda.empty_cache()
        except Exception as e:
            eager_gpu = {"value": None, "error": repr(e)[:300]}

    cpu_baseline = None
    if rank == 0 and world == 1 and not a.skip_cpu_baseline:
        try:
            if a.workload == "sdxl":
                _, cpu_baseline = cpu_quick_sdxl_rate(a.res, budget_s=a.cpu_budget_s)
            else:  # video workloads (not the default run): the full-resolution one-clip sample
                _, cpu_baseline = cpu_reference_step_rate(a.workload, a.res, 3, 1, budget_s=a.cpu_budget_s)
        except Exception as e:  # the CPU leg must never hide the GPU numbers
            cpu_baseline = {"value": None, "error": repr(e)[:300]}

    if rank == 0:
        step_tflop = n_samples * w["tflop"]
        line = {
            "metric": w["metric"],
            "value": value, "unit": "steps/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": workload_name(a.workload, batch, a.res), "baseline_config": w["base"],
                       "parallelism": f"batch-sharded dp{world}", "cuda_graph": use_graph,
                       "l2": "per-step working set (multi-GB bf16 weights + multi-GB activations) exceeds the 126 MB L2; "
                             "no explicit flush",
                       "algorithmic_tflop_per_step": round(step_tflop, 1),
                       "step_tflops_achieved": round(step_tflop / (ms_step / 1000.0), 1),
                       "step_frac_of_sustained_peak": round(step_tflop / (ms_step / 1000.0) / peaks["bf16_tflops_sustained"], 4)},
            "finite_outputs": finite, "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * a.steps,
            "launches_per_step": launches_per_step, "roofline": roofline, "kernel_families": families,
            "cpu_baseline": cpu_baseline, "eager_gpu_baseline": eager_gpu,
            "vs_eager": (value / world / eager_gpu["value"]) if eager_gpu and eager_gpu.get("value") else None,
        }
        emit(line)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
